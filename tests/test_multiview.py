"""Multiview without a GPU: argument validation of gsr_set_views / gsr_render_views, and the XR camera helpers (stereo_pair,
the off-axis frustum) against hand-computed matrices."""
import ctypes as C

import numpy as np

from godotgaussiansplatting_b200 import _lib
from godotgaussiansplatting_b200 import camera as cam


def test_set_views_rejects_bad_arguments_without_a_device():
    L = _lib.lib()
    for k in (0, 1, 2, 4, 5, -1):
        assert L.gsr_set_views(None, k) == _lib.GSR_ERR_INVALID
    vp = np.zeros(64, dtype=np.float32)
    ub = bytes(64)
    assert L.gsr_render_views(None, vp.ctypes.data_as(C.POINTER(C.c_float)), ub, 0.0, None) == _lib.GSR_ERR_INVALID
    assert L.gsr_render_views_async(None, vp.ctypes.data_as(C.POINTER(C.c_float)), ub, 0.0, None, 0) == _lib.GSR_ERR_INVALID
    assert L.gsr_render_views_async(None, vp.ctypes.data_as(C.POINTER(C.c_float)), ub, 0.0, None, 0x77) == _lib.GSR_ERR_INVALID
    assert _lib.GSR_MAX_VIEWS == 4


def test_frustum_matches_hand_computed_matrix():
    # window [-0.3, 0.1] x [-0.2, 0.2] at near 0.5, far 100
    m = cam.frustum(-0.3, 0.1, -0.2, 0.2, 0.5, 100.0).reshape(4, 4)   # m[column][row]
    want = np.zeros((4, 4), dtype=np.float64)
    want[0][0] = 2 * 0.5 / 0.4
    want[1][1] = 2 * 0.5 / 0.4
    want[2][0] = (0.1 - 0.3) / 0.4
    want[2][1] = 0.0
    want[2][2] = -(100.5) / 99.5
    want[2][3] = -1.0
    want[3][2] = -(2 * 100 * 0.5) / 99.5
    np.testing.assert_allclose(m, want, rtol=1e-6, atol=1e-7)
    assert m.dtype == np.float32


def test_symmetric_frustum_equals_the_perspective():
    near, far, fov, aspect = 0.05, 4000.0, 75.0, 16 / 9
    top = near * np.tan(np.radians(fov / 2))
    np.testing.assert_allclose(cam.frustum(-top * aspect, top * aspect, -top, top, near, far), cam.perspective(fov, aspect, near, far),
                               rtol=2e-6, atol=1e-9)


def test_stereo_pair_offsets_the_eyes_along_the_right_axis():
    head = cam.orbit_camera(37, aspect=16 / 9)
    left, right = cam.stereo_pair(head, ipd=0.063)
    r = head.basis[0].astype(np.float64)
    np.testing.assert_allclose(left.global_position, head.global_position - 0.0315 * r, atol=1e-6)
    np.testing.assert_allclose(right.global_position, head.global_position + 0.0315 * r, atol=1e-6)
    np.testing.assert_allclose(np.linalg.norm(right.global_position.astype(np.float64) - left.global_position), 0.063, rtol=1e-5)
    for e in (left, right):
        np.testing.assert_array_equal(e.basis, head.basis)
        np.testing.assert_array_equal(e.get_camera_projection(), head.get_camera_projection())
    # the eyes' push constants differ from the head's only in the translation column of the view matrix
    vh = cam.pack_camera_push_constants(head.get_camera_transform(), head.get_camera_projection())
    vl = cam.pack_camera_push_constants(left.get_camera_transform(), left.get_camera_projection())
    np.testing.assert_array_equal(vh[:12], vl[:12])
    np.testing.assert_array_equal(vh[16:], vl[16:])
    # an eye sees the head's view-space origin shifted by +-ipd/2 along x (mirrored x of the reference's packing: -x row)
    assert abs(abs(float(vl[12] - vh[12])) - 0.0315) < 1e-5


# ---------------------------------------------------------------------------------------------------------------------
# The multiview kernels under the CPU emulator (tests/kernel_emu/multiview_emu.cpp, built with the g++ flags of
# tests/kernel_emu/build.py): logic only -- the memory model and timing need the GPU (tests/test_gpu_multiview.py).
# ---------------------------------------------------------------------------------------------------------------------
import os  # noqa: E402
import subprocess  # noqa: E402

import pytest  # noqa: E402

from oracle import oracle as orc  # noqa: E402
from tests import test_kernel_emu as kemu  # noqa: E402
from tests.scenes import uniforms_bytes  # noqa: E402

_HERE = os.path.dirname(os.path.abspath(__file__))
_MV_SRC = os.path.join(_HERE, "kernel_emu", "multiview_emu.cpp")
_MV_OUT = os.path.join(_HERE, "kernel_emu", "libmultiview_emu.so")
_MV = None


def mv_lib():
    global _MV
    if _MV is None:
        csrc = os.path.join(os.path.dirname(_HERE), "godotgaussiansplatting_b200", "csrc")
        deps = [_MV_SRC, os.path.join(_HERE, "kernel_emu", "cuda_shim.h")] + [os.path.join(csrc, f) for f in
                                                                                ("compositor.cu", "ranges.cu", "projection.cu", "common.cuh")]
        if not os.path.exists(_MV_OUT) or os.path.getmtime(_MV_OUT) < max(os.path.getmtime(d) for d in deps):
            b = kemu._emu_build
            subprocess.run([b.CXX, "-std=gnu++17", "-O1", "-march=x86-64-v3", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-w",
                            "-I", b.CUDA_INC, _MV_SRC, "-o", _MV_OUT], check=True)
        L = C.CDLL(_MV_OUT)
        L.emu_projection_views.restype = C.c_longlong
        L.emu_projection_views.argtypes = [C.c_void_p, C.c_ulonglong, C.c_uint, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_uint, C.c_int, C.POINTER(C.c_uint), C.POINTER(C.c_int)]
        L.emu_tile_ranges_views.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_int]
        L.emu_composite_views.argtypes = [C.c_int, C.c_void_p, C.c_ulonglong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float,
                                          C.c_uint32, C.c_void_p]
        _MV = L
    return _MV


def emu_views(soa, stride, n, vps, ubs, cap, sh_bulk_min=0):
    K = len(vps)
    vp = np.ascontiguousarray(np.concatenate(vps), dtype=np.float32)
    recs = np.zeros((K, n), dtype=orc.RECORD_DTYPE)
    keys = np.zeros(cap, dtype=np.uint32)
    vals = np.zeros(cap, dtype=np.uint32)
    vis, last = C.c_uint(0), C.c_int(0)
    m = mv_lib().emu_projection_views(soa.ctypes.data, stride, n, K, vp.ctypes.data, b"".join(ubs), recs.ctypes.data, keys.ctypes.data, vals.ctypes.data,
                                      cap, sh_bulk_min, C.byref(vis), C.byref(last))
    assert 0 <= m <= cap
    return recs, keys[:m], vals[:m], int(vis.value), int(last.value)


def emu_ranges_views(keys, T, K, quirks, grid=5):
    keys = np.ascontiguousarray(keys, dtype=np.uint32)
    bounds = np.zeros((K, T, 2), dtype=np.uint32)
    assert mv_lib().emu_tile_ranges_views(keys.ctypes.data, keys.size, bounds.ctypes.data, T, K, int(quirks), grid) == 0
    return bounds


def views_cameras(K, w, h):
    """K different cameras, view 1 with an asymmetric (off-axis) frustum."""
    vps, ubs = [], []
    for v in range(K):
        c = cam.orbit_camera((0, 23, 61, 140)[v], aspect=w / h)
        if v == 1:
            top = 0.05 * np.tan(np.radians(37.5))
            right = top * w / h
            proj = cam.frustum(-0.8 * right, 1.2 * right, -top, top, 0.05, 4000.0)
        else:
            proj = c.get_camera_projection()
        vps.append(cam.pack_camera_push_constants(c.get_camera_transform(), proj))
        ubs.append(uniforms_bytes(c.global_position, 1.0, w, h, 10.0))
    return vps, ubs


def concatenated_reference(per_view, T):
    """The sorted pairs of a K-view frame: the single-view sorted pairs, view v with tile ids + v*T, view after view."""
    keys = np.concatenate([k + np.uint32((v * T) << 16) for v, (k, _) in enumerate(per_view)]) if per_view else np.zeros(0, np.uint32)
    vals = np.concatenate([vv for _, vv in per_view]) if per_view else np.zeros(0, np.uint32)
    return keys.astype(np.uint32), vals.astype(np.uint32)


def assert_lists_equal(bounds_v, ref_bounds, start, msg):
    got, want = bounds_v.astype(np.int64), ref_bounds.astype(np.int64)
    cg, cw = np.maximum(0, got[:, 1] - got[:, 0]), np.maximum(0, want[:, 1] - want[:, 0])
    np.testing.assert_array_equal(cg, cw, err_msg=msg)
    busy = cw > 0
    np.testing.assert_array_equal(got[busy, 0] - start, want[busy, 0], err_msg=msg)


@pytest.mark.parametrize("K,w,h", [(2, 96, 64), (3, 96, 64), (2, 333, 257), (3, 333, 257)])
def test_emulated_multiview_projection_ranges_and_compositor(K, w, h):
    n = 3000
    T = ((w + 15) // 16) * ((h + 15) // 16)
    splat60 = kemu.make_scene(n, 21 + K, w, h, scale_boost=0.5)[0]
    vps, ubs = views_cameras(K, w, h)
    soa, stride = kemu.emu_upload(splat60)
    recs, ukeys, uvals, vis, last = emu_views(soa, stride, n, vps, ubs, cap=200 * n)
    single = [kemu.emu_project(soa, stride, n, vp, ub, w, h, cap=200 * n) for vp, ub in zip(vps, ubs)]
    assert ukeys.size == sum(s["m"] for s in single) and vis == sum(s["visible"] for s in single)
    lasts = [v * T + s["last_tile"] for v, s in enumerate(single) if s["last_tile"] >= 0]
    assert last == (max(lasts) if lasts else -1)
    # records per view; the pairs of view v, in emission order, are the single-view emission with tile ids + v*T
    tile_view = (ukeys >> 16) // T
    for v, s in enumerate(single):
        vis_ids = np.unique(s["values"])
        for f in orc.RECORD_DTYPE.names:
            np.testing.assert_array_equal(kemu.bits(recs[v][f][vis_ids]), kemu.bits(s["records"][f][vis_ids]), err_msg=f"view {v} field {f}")
        sel = tile_view == v
        np.testing.assert_array_equal(ukeys[sel] - np.uint32((v * T) << 16), s["keys"])
        np.testing.assert_array_equal(uvals[sel], s["values"])
    # one stable sort of the concatenation, then the multiview ranges kernel in both quirk modes
    skeys, svals = orc.sort_pairs(ukeys, uvals)
    ref = [orc.sort_pairs(s["keys"], s["values"]) for s in single]
    want_k, want_v = concatenated_reference(ref, T)
    np.testing.assert_array_equal(skeys, want_k)
    np.testing.assert_array_equal(svals, want_v)
    for quirks in (True, False):
        bounds = emu_ranges_views(skeys, T, K, quirks)
        start = 0
        for v, (k, _) in enumerate(ref):
            assert_lists_equal(bounds[v], orc.boundaries(k, T, quirks=quirks), start, f"view {v} quirks={quirks}")
            start += k.size
    # the compositor over K*T tiles: layer v = orc.render of view v
    bounds = emu_ranges_views(skeys, T, K, True)
    out = np.zeros((K, h, w, 4), dtype=np.float32)
    pick = np.zeros(4, dtype=np.float32)
    vals_pad = np.concatenate([svals, np.zeros(512, dtype=np.uint32)])
    assert mv_lib().emu_composite_views(0, recs.ctypes.data, n, vals_pad.ctypes.data, bounds.ctypes.data, out.ctypes.data, w, h, K, 0.0, 0xFFFFFFFF,
                                        pick.ctypes.data) == 0
    for v, (k, vv) in enumerate(ref):
        want, _, _ = orc.render(single[v]["records"], vv, orc.boundaries(k, T, quirks=True), w, h)
        np.testing.assert_array_equal(kemu.bits(out[v]), kemu.bits(want), err_msg=f"layer {v}")


def _keys(tiles, depth=7):
    return (np.asarray(tiles, dtype=np.uint32) << 16) | np.uint32(depth)


@pytest.mark.parametrize("quirks", [True, False])
def test_emulated_multiview_ranges_edge_views(quirks):
    """Per-view Q10: a view whose last occupied tile is its T-1, a view with 0 pairs, a view with exactly 1 pair, a view whose pairs
    all sit in its first tile -- each view's lists equal orc.boundaries of that view alone."""
    T = 12
    views = [
        [0, 0, 0, 0],                 # view 0: every pair in its first tile
        [],                           # view 1: no pairs
        [5],                          # view 2: exactly one pair
        [1, 1, 4, 9, 11, 11],         # view 3: last occupied tile is T-1
    ]
    for order in ([0, 1, 2, 3], [3, 2, 1, 0], [2, 0, 3, 1], [1, 3, 0, 2]):
        per = [views[i] for i in order]
        keys = np.concatenate([_keys(np.asarray(t, dtype=np.int64) + v * T) for v, t in enumerate(per)]).astype(np.uint32)
        bounds = emu_ranges_views(keys, T, len(per), quirks, grid=3)
        start = 0
        for v, t in enumerate(per):
            assert_lists_equal(bounds[v], orc.boundaries(_keys(t), T, quirks=quirks), start, f"order {order} view {v}")
            start += len(t)
