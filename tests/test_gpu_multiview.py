"""Multiview frames (gsr_set_views / gsr_render_views): layer v of a K-view frame against the CPU oracle's frame of camera v and
against gsr_render of camera v in a single-view context, bit for bit; the concatenated sort keys, tile ranges and record tables;
flags, capacity, read-back formats, pick and the state / argument errors of the multiview calls."""
import ctypes as C

import numpy as np
import pytest

from godotgaussiansplatting_b200 import _lib
from godotgaussiansplatting_b200 import camera as cam
from godotgaussiansplatting_b200.ply_file import swizzle_splats
from godotgaussiansplatting_b200.synthetic import synthetic_ply_chunks, synthetic_ply_table
from oracle import oracle as orc
from tests.gsr_direct import REC_DTYPE, Ctx
from tests.scenes import uniforms_bytes

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def eye_frustum(aspect, offset, near=0.05, far=4000.0, fov=75.0):
    """An asymmetric per-eye frustum (XR style): the fov-75 window shifted sideways by `offset` of its half-width."""
    top = near * np.tan(np.radians(fov / 2.0))
    right = top * aspect
    return cam.frustum(-right + offset * right, right + offset * right, -top, top, near, far)


def view_set(K, w, h, frames=(0, 37, 90, 181), offaxis=(1,), time=10.0, model_scale=1.0):
    """K cameras (orbit frames); the views listed in `offaxis` use an asymmetric frustum.  Returns ([vp32], [uniforms])."""
    vps, ubs = [], []
    for v in range(K):
        c = cam.orbit_camera(frames[v % len(frames)] + 7 * (v // len(frames)), aspect=w / h)
        proj = eye_frustum(w / h, 0.15 if v % 2 else -0.15) if v in offaxis else c.get_camera_projection()
        vps.append(cam.pack_camera_push_constants(c.get_camera_transform(), proj))
        ubs.append(uniforms_bytes(c.global_position, model_scale, w, h, time))
    return vps, ubs


def scene(n, seed, scale_boost=0.0, creation_time=0.0):
    table = synthetic_ply_table(n, seed)
    if scale_boost:
        table[:, 55:58] += scale_boost
    return swizzle_splats(table, creation_time)


def render_views(c, vps, ubs, heatmap=0.0):
    K = len(vps)
    vp = np.ascontiguousarray(np.concatenate(vps), dtype=np.float32)
    out = np.empty((K, c.hgt, c.w, 4), dtype=np.float32)
    _lib.check(c.L.gsr_render_views(c.h, vp.ctypes.data_as(C.POINTER(C.c_float)), b"".join(ubs), float(heatmap), C.c_void_p(out.ctypes.data)),
               "gsr_render_views")
    return out


def set_views(c, k):
    _lib.check(c.L.gsr_set_views(c.h, k), "gsr_set_views")


def check_views(splat60, vps, ubs, w, h, flags=0, heatmap=0.0, oracle=True, factor=10):
    """Render the K views in one multiview context; compare with K single-view frames of libgsr and (oracle=True) of the oracle."""
    n, K = splat60.shape[0], len(vps)
    T = ((w + 15) // 16) * ((h + 15) // 16)
    quirks = not (flags & _lib.GSR_FLAG_FIXED_RANGES)
    with Ctx(n, w, h, flags=flags, factor=factor) as c:
        c.upload(splat60)
        singles, sstats = [], []
        for vp, ub in zip(vps, ubs):
            singles.append(c.render(vp, ub, heatmap=heatmap))
            sstats.append(c.stats())
        set_views(c, K)
        layers = render_views(c, vps, ubs, heatmap)
        st = c.stats()
        m = int(min(st.duplicates, st.capacity))
        keys = c.copy(_lib.GSR_BUF_KEYS, m, np.uint32)
        vals = c.copy(_lib.GSR_BUF_VALUES, m, np.uint32)
        bounds = c.copy(_lib.GSR_BUF_BOUNDS, K * T * 2, np.uint32).reshape(K, T, 2)
        recs = c.copy(_lib.GSR_BUF_RECORDS, K * n, REC_DTYPE).reshape(K, n)
        fb = c.copy(_lib.GSR_BUF_FRAMEBUFFER, K * h * w * 4, np.float32).reshape(K, h, w, 4)
    assert not st.overflow
    assert st.duplicates == sum(s.duplicates for s in sstats)
    assert st.visible == sum(s.visible for s in sstats)
    lasts = [v * T + s.last_tile for v, s in enumerate(sstats) if s.last_tile >= 0]
    assert st.last_tile == (max(lasts) if lasts else -1)
    np.testing.assert_array_equal(bits(fb), bits(layers))
    refs = []
    if oracle:
        for vp, ub in zip(vps, ubs):
            refs.append(orc.frame(splat60, vp, orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8)), heatmap=heatmap, quirks=quirks,
                                  cap=1000 * n))
    start = 0
    for v in range(K):
        np.testing.assert_array_equal(bits(layers[v]), bits(singles[v]), err_msg=f"layer {v} vs single-view gsr_render")
        if not refs:
            continue
        ref = refs[v]
        assert ref.duplicates == sstats[v].duplicates
        np.testing.assert_array_equal(bits(layers[v]), bits(ref.rgba), err_msg=f"layer {v} vs oracle")
        # concatenation rule: view v's sorted pairs are the single-view pairs with tile ids + v*T, after those of views < v
        mv = ref.duplicates
        np.testing.assert_array_equal(keys[start:start + mv], ref.keys + np.uint32((v * T) << 16))
        np.testing.assert_array_equal(vals[start:start + mv], ref.values)
        # per-tile lists: same count max(0, end - start) and, where non-empty, the same list
        got = bounds[v].astype(np.int64)
        want = ref.bounds.astype(np.int64)
        cnt_got, cnt_want = np.maximum(0, got[:, 1] - got[:, 0]), np.maximum(0, want[:, 1] - want[:, 0])
        np.testing.assert_array_equal(cnt_got, cnt_want, err_msg=f"tile list lengths of view {v}")
        busy = cnt_want > 0
        np.testing.assert_array_equal(got[busy, 0] - start, want[busy, 0])
        vis = np.unique(ref.values)
        for f in ("image_pos", "pos_xy", "conic", "pos_z", "color"):
            np.testing.assert_array_equal(bits(recs[v][f][vis]), bits(ref.records[f][vis]), err_msg=f"view {v} record field {f}")
        start += mv
    return layers, refs, st


@pytest.mark.parametrize("K", [2, 3, 4])
@pytest.mark.parametrize("n,seed,w,h", [(2000, 1, 320, 240), (20000, 2, 640, 480), (60000, 3, 1920, 1080), (5000, 4, 333, 257)])
def test_layers_equal_single_view_frames_and_the_oracle(K, n, seed, w, h):
    vps, ubs = view_set(K, w, h)
    layers, refs, st = check_views(scene(n, seed), vps, ubs, w, h)
    assert all(r.duplicates > 0 for r in refs)


def test_stereo_at_full_c3_size():
    """6 M splats, 1920x1080 per eye, an orbit frame, ipd 0.063, both eyes off-axis."""
    n, w, h = 6_000_000, 1920, 1080
    splat60 = np.empty((n, 60), dtype=np.float32)
    for lo, blk in synthetic_ply_chunks(n, 2):
        splat60[lo:lo + blk.shape[0]] = swizzle_splats(blk, 0.0)
    head = cam.orbit_camera(37, aspect=w / h)
    eyes = cam.stereo_pair(head, 0.063)
    vps = [cam.pack_camera_push_constants(e.get_camera_transform(), eye_frustum(w / h, off)) for e, off in zip(eyes, (0.1, -0.1))]
    ubs = [uniforms_bytes(e.global_position, 1.0, w, h, 10.0) for e in eyes]
    layers, refs, st = check_views(splat60, vps, ubs, w, h)
    assert st.duplicates == sum(r.duplicates for r in refs) and st.visible == sum(r.visible for r in refs)


@pytest.mark.parametrize("case", ["fixed_ranges", "uncontracted", "heatmap_scale", "load_in"])
def test_flags_and_uniforms(case):
    w, h = 640, 480
    kw, flags, heat, sc = {}, 0, 0.0, dict()
    if case == "fixed_ranges":
        flags = _lib.GSR_FLAG_FIXED_RANGES
    elif case == "uncontracted":
        flags = _lib.GSR_FLAG_UNCONTRACTED_BLEND
    elif case == "heatmap_scale":
        heat, kw = 1.0, dict(model_scale=1.7)
    else:
        kw, sc = dict(time=0.6), dict(creation_time=0.0)
    vps, ubs = view_set(2, w, h, **kw)
    if flags & _lib.GSR_FLAG_UNCONTRACTED_BLEND:
        orc.set_blend_contraction(False)
    try:
        check_views(scene(20000, 7, **sc), vps, ubs, w, h, flags=flags, heatmap=heat)
    finally:
        orc.set_blend_contraction(True)


def test_all_culled_view_beside_a_full_one():
    w, h = 640, 480
    vps, ubs = view_set(2, w, h, offaxis=())
    c = cam.default_camera(aspect=w / h)
    c.look_at_from_position((0.0, 0.0, -50.0), (0.0, 0.0, -100.0))   # looks away from the cloud
    vps[0] = cam.pack_camera_push_constants(c.get_camera_transform(), c.get_camera_projection())
    ubs[0] = uniforms_bytes(c.global_position, 1.0, w, h, 10.0)
    layers, refs, st = check_views(scene(20000, 8), vps, ubs, w, h)
    assert refs[0].duplicates == 0 and refs[1].duplicates > 0


def test_views_that_differ_in_the_last_tile_rule():
    """Q10: views whose last occupied tile is their tile T-1 (big splats cover the frame), then views where it is not: an empty
    view beside views of exactly one pair."""
    w, h = 320, 240
    splat60 = scene(3000, 9, scale_boost=2.5)
    vps, ubs = view_set(3, w, h, offaxis=())
    refs = [orc.frame(splat60, vp, orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8)), cap=1000 * 3000) for vp, ub in zip(vps, ubs)]
    T = 20 * 15
    assert any(r.last_tile == T - 1 for r in refs)
    check_views(splat60, vps, ubs, w, h)
    # one splat: no pair in view 0 (culled), exactly one pair in views 1 and 2 (so the last occupied tile is not T-1)
    one = scene(2000, 10)[:1].copy()
    c = cam.default_camera(aspect=w / h)
    vp_center = cam.pack_camera_push_constants(c.get_camera_transform(), c.get_camera_projection())
    ub_center = uniforms_bytes(c.global_position, 1.0, w, h, 10.0)
    away = cam.default_camera(aspect=w / h)
    away.look_at_from_position((0.0, 0.0, -50.0), (0.0, 0.0, -100.0))
    vp_away = cam.pack_camera_push_constants(away.get_camera_transform(), away.get_camera_projection())
    ub_away = uniforms_bytes(away.global_position, 1.0, w, h, 10.0)
    _, refs1, _ = check_views(one, [vp_away, vp_center, vp_center], [ub_away, ub_center, ub_center], w, h)
    assert [r.duplicates for r in refs1] == [0, 1, 1] and refs1[1].last_tile != T - 1


def test_capacity_factor_one_and_static_capacity():
    w, h = 640, 480
    splat60 = scene(3000, 9, scale_boost=2.5)
    vps, ubs = view_set(2, w, h, offaxis=())
    check_views(splat60, vps, ubs, w, h, factor=1)   # grows: the synchronous call never returns a truncated frame
    with Ctx(3000, w, h, flags=_lib.GSR_FLAG_STATIC_CAPACITY, factor=1) as c:
        c.upload(splat60)
        set_views(c, 2)
        render_views(c, vps, ubs)
        st = c.stats()
    assert st.overflow and st.duplicates > st.capacity


@pytest.mark.parametrize("fmt", [0, 1, 2, 3, 0x100, 0x101, 0x102, 0x103])
def test_async_readback_formats_and_present_device(fmt):
    import torch
    n, w, h, K = 20000, 333, 257, 2
    splat60 = scene(n, 11)
    vps, ubs = view_set(K, w, h)
    refs = [orc.frame(splat60, vp, orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8)), cap=1000 * n) for vp, ub in zip(vps, ubs)]
    per = int(c_output_bytes(fmt, w, h))
    host = torch.zeros(K * per, dtype=torch.uint8).pin_memory()
    with Ctx(n, w, h) as c:
        c.upload(splat60)
        set_views(c, K)
        vp = np.ascontiguousarray(np.concatenate(vps), dtype=np.float32)
        _lib.check(c.L.gsr_render_views_async(c.h, vp.ctypes.data_as(C.POINTER(C.c_float)), b"".join(ubs), 0.0, C.c_void_p(host.data_ptr()), fmt), "async")
        c.sync()
        dev = torch.zeros(K * per, dtype=torch.uint8, device="cuda")
        _lib.check(c.L.gsr_present_device(c.h, C.c_void_p(dev.data_ptr()), fmt), "present")
        c.sync()
        got_dev = dev.cpu().numpy()
    got = host.numpy()
    for v in range(K):
        want = orc.present(refs[v].rgba, fmt).view(np.uint8).reshape(-1)
        np.testing.assert_array_equal(got[v * per:(v + 1) * per], want, err_msg=f"read-back layer {v}")
        np.testing.assert_array_equal(got_dev[v * per:(v + 1) * per], want, err_msg=f"present_device layer {v}")


def c_output_bytes(fmt, w, h):
    return _lib.lib().gsr_output_bytes(fmt, w, h)


def test_pipelined_frames_equal_synchronous_frames():
    import torch
    n, w, h, K = 20000, 640, 480, 2
    splat60 = scene(n, 12)
    sets = [view_set(K, w, h, frames=(f, f + 11)) for f in (0, 20, 40, 60, 80, 100)]
    with Ctx(n, w, h) as c:
        c.upload(splat60)
        set_views(c, K)
        want = [render_views(c, vps, ubs) for vps, ubs in sets]
        hosts = [torch.zeros((K, h, w, 4), dtype=torch.float32).pin_memory() for _ in sets]
        for (vps, ubs), out in zip(sets, hosts):
            vp = np.ascontiguousarray(np.concatenate(vps), dtype=np.float32)
            _lib.check(c.L.gsr_render_views_async(c.h, vp.ctypes.data_as(C.POINTER(C.c_float)), b"".join(ubs), 0.0, C.c_void_p(out.data_ptr()), 0), "async")
        _lib.check(c.L.gsr_stream_join(c.h), "join")
        c.sync()
    for a, b in zip(hosts, want):
        np.testing.assert_array_equal(bits(a.numpy()), bits(b))


def test_pick_takes_concatenated_tile_ids():
    n, w, h, K = 20000, 640, 480, 3
    T = 40 * 30
    splat60 = scene(n, 13)
    vps, ubs = view_set(K, w, h)
    refs = [orc.frame(splat60, vp, orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8)), cap=1000 * n) for vp, ub in zip(vps, ubs)]
    with Ctx(n, w, h) as c:
        c.upload(splat60)
        set_views(c, K)
        render_views(c, vps, ubs)
        for v, ref in enumerate(refs):
            counts = ref.bounds[:, 1].astype(np.int64) - ref.bounds[:, 0]
            busy = int(np.argmax(counts))
            got = c.pick(v * T + busy)
            _, _, want = orc.render(ref.records, ref.values, ref.bounds, w, h, target_tile=busy, pick=np.zeros(4, np.float32))
            np.testing.assert_array_equal(bits(got), bits(want))


def test_state_and_validation_errors():
    n, w, h = 2000, 320, 240
    splat60 = scene(n, 14)
    vps, ubs = view_set(2, w, h)
    L = _lib.lib()
    with Ctx(n, w, h) as c:
        c.upload(splat60)
        # contexts that multiview cannot join
        c.set_band(0, 5)
        assert L.gsr_set_views(c.h, 2) == _lib.GSR_ERR_STATE
        c.set_band(0, 15)
        c.set_row_interleave(0, 2)
        assert L.gsr_set_views(c.h, 2) == _lib.GSR_ERR_STATE
        c.set_row_interleave(0, 1)
        _lib.check(L.gsr_debug_pipeline(c.h, 1), "overlap on")
        assert L.gsr_set_views(c.h, 2) == _lib.GSR_ERR_STATE
        _lib.check(L.gsr_debug_pipeline(c.h, -1), "overlap default")
        assert L.gsr_set_views(c.h, 0) == _lib.GSR_ERR_INVALID and L.gsr_set_views(c.h, 5) == _lib.GSR_ERR_INVALID
        set_views(c, 2)
        # single-view entries and multi-GPU set-ups refuse while K > 1
        vp0 = np.ascontiguousarray(vps[0], dtype=np.float32)
        assert L.gsr_render(c.h, vp0.ctypes.data_as(C.POINTER(C.c_float)), ubs[0], 0.0, None) == _lib.GSR_ERR_STATE
        assert L.gsr_render_async(c.h, vp0.ctypes.data_as(C.POINTER(C.c_float)), ubs[0], 0.0, None) == _lib.GSR_ERR_STATE
        assert L.gsr_set_band(c.h, 0, 5) == _lib.GSR_ERR_STATE
        assert L.gsr_set_row_interleave(c.h, 0, 2) == _lib.GSR_ERR_STATE
        assert L.gsr_debug_pipeline(c.h, 1) == _lib.GSR_ERR_STATE
        blob = (C.c_ubyte * _lib.GSR_GROUP_BLOB_BYTES)()
        assert L.gsr_group_export(c.h, blob) == _lib.GSR_ERR_STATE
        handles = (C.c_ubyte * 128)()
        assert L.gsr_peer_export_framebuffers(c.h, handles) == _lib.GSR_ERR_STATE
        # uniform blocks must agree on dims, time and scale
        vp = np.ascontiguousarray(np.concatenate(vps), dtype=np.float32)
        for bad in (uniforms_bytes([0, 0, 0], 1.0, w, h, 11.0), uniforms_bytes([0, 0, 0], 1.5, w, h, 10.0), uniforms_bytes([0, 0, 0], 1.0, w + 1, h, 10.0)):
            assert L.gsr_render_views(c.h, vp.ctypes.data_as(C.POINTER(C.c_float)), ubs[0] + bad, 0.0, None) == _lib.GSR_ERR_INVALID
        # K*T > 65536: refused by gsr_set_views and gsr_resize, the context unchanged
        c.resize(1920, 1080)
        assert L.gsr_set_views(c.h, 4) == _lib.GSR_OK                    # 4 x 8160 tiles fit
        assert L.gsr_resize(c.h, 3840, 2160) == _lib.GSR_ERR_INVALID      # 4 x 32400 do not
        assert c.stats().width == 1920
        set_views(c, 1)
        c.resize(3840, 2160)
        assert L.gsr_set_views(c.h, 3) == _lib.GSR_ERR_INVALID
        assert L.gsr_set_views(c.h, 2) == _lib.GSR_OK
        # back to one view: single-view frames equal the oracle
        set_views(c, 1)
        c.resize(w, h)
        img = c.render(vps[0], ubs[0])
    ref = orc.frame(splat60, vps[0], orc.uniforms_from_bytes(np.frombuffer(ubs[0], dtype=np.uint8)))
    np.testing.assert_array_equal(bits(img), bits(ref.rgba))
