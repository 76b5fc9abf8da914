"""GPU parity tests proper: the CUDA path (through the C-ABI) against the CPU oracle on the same inputs.

Bar (BASELINE.json north_star): sort keys and tile ranges bit-exact; per-pixel RGBA within 1e-4 abs.
Because both sides implement the same "gsr deterministic math" contract the tests additionally check that
RGBA and the 48-byte records are bit-identical, which removes the tile-stop-rule flakiness (SURVEY 7).
"""
import numpy as np
import pytest

from godotgaussiansplatting_b200 import _lib
from oracle import oracle as orc
from tests.gsr_direct import Ctx
from tests.scenes import make_scene

pytestmark = pytest.mark.gpu

RGBA_TOL = 1e-4  # north_star tolerance (abs)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def run_both(n, seed, w, h, frame=None, flags=0, heatmap=0.0, band=None, time=10.0, model_scale=1.0, scale_boost=0.0, factor=10):
    splat60, vp, ub = make_scene(n, seed, w, h, frame=frame, time=time, model_scale=model_scale, scale_boost=scale_boost)
    quirks = not (flags & _lib.GSR_FLAG_FIXED_RANGES)
    # default contexts grow their duplicate capacity (the synchronous render never returns a truncated frame): the oracle gets room
    # for every instance; GSR_FLAG_STATIC_CAPACITY keeps the reference's fixed factor * N and its truncation
    cap = factor * n if (flags & _lib.GSR_FLAG_STATIC_CAPACITY) else max(factor, 1000) * n
    ref = orc.frame(splat60, vp, orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8)), heatmap=heatmap, quirks=quirks,
                    band=band, cap=cap)
    with Ctx(n, w, h, flags=flags, factor=factor) as c:
        c.upload(splat60)
        if band is not None:
            c.set_band(*band)
        c.keep_unsorted()
        rgba = c.render(vp, ub, heatmap=heatmap)
        t = c.taps()
        t["rgba"] = rgba
        t["ukeys"] = c.copy(_lib.GSR_BUF_KEYS_UNSORTED, t["m"], np.uint32)
        t["uvals"] = c.copy(_lib.GSR_BUF_VALUES_UNSORTED, t["m"], np.uint32)
    return ref, t


def assert_frame_equal(ref, t, band=None, h=None):
    st = t["stats"]
    assert st.duplicates == ref.duplicates, (st.duplicates, ref.duplicates)
    assert st.visible == ref.visible
    assert st.last_tile == ref.last_tile
    assert bool(st.overflow) == ref.overflow
    if ref.overflow:
        return
    # emission order (Q13 fixed to splat-id order) and the projection outputs
    np.testing.assert_array_equal(t["ukeys"], orc_unsorted(ref)[0])
    np.testing.assert_array_equal(t["uvals"], orc_unsorted(ref)[1])
    vis = np.unique(ref.values)
    for f in ("image_pos", "pos_xy", "conic", "pos_z", "color"):
        np.testing.assert_array_equal(bits(t["records"][f][vis]), bits(ref.records[f][vis]), err_msg=f"record field {f}")
    # sort keys + values bit-exact, tile ranges bit-exact
    np.testing.assert_array_equal(t["keys"], ref.keys)
    np.testing.assert_array_equal(t["values"], ref.values)
    np.testing.assert_array_equal(t["bounds"], ref.bounds)
    # pixels: tolerance from the north star, and (stronger) bit-exact
    a, b = t["rgba"], ref.rgba
    if band is not None:
        y0, y1 = band[0] * 16, min(band[1] * 16, a.shape[0])
        a, b = a[y0:y1], b[y0:y1]
    assert a.size == 0 or np.abs(a - b).max() <= RGBA_TOL
    np.testing.assert_array_equal(bits(a), bits(b))


_UNSORTED = {}


def orc_unsorted(ref):
    """Oracle emission order = stable order before sorting; recover it from the projection call."""
    return ref._unsorted


@pytest.fixture(autouse=True)
def _patch_unsorted(monkeypatch):
    # orc.frame sorts in place; keep the unsorted pairs by projecting once more (cheap at test sizes)
    real = orc.frame

    def wrapped(splat60, vp, u, **kw):
        fr = real(splat60, vp, u, **kw)
        pr = orc.project(splat60, vp, u, band=kw.get("band"), cap=kw.get("cap"))
        fr._unsorted = (pr.keys, pr.values)
        return fr

    monkeypatch.setattr(orc, "frame", wrapped)


@pytest.mark.parametrize("n,seed,w,h", [(2000, 1, 320, 240), (20000, 2, 640, 480), (60000, 3, 1920, 1080), (5000, 4, 333, 257)])
def test_frame_parity_default_camera(n, seed, w, h):
    ref, t = run_both(n, seed, w, h)
    assert ref.duplicates > 0
    assert_frame_equal(ref, t)


@pytest.mark.parametrize("frame", [0, 37, 90, 181, 270])
def test_frame_parity_orbit(frame):
    ref, t = run_both(30000, 5, 640, 360, frame=frame)
    assert_frame_equal(ref, t)


def test_fixed_ranges_flag():
    ref, t = run_both(20000, 6, 640, 480, flags=_lib.GSR_FLAG_FIXED_RANGES)
    assert_frame_equal(ref, t)


def test_heatmap_and_model_scale():
    ref, t = run_both(20000, 7, 640, 480, heatmap=1.0, model_scale=1.7)
    assert_frame_equal(ref, t)


def test_load_in_animation():
    # splats 0.5 s old: time factors < 1 shift image_pos and double the scale (Q14)
    ref, t = run_both(20000, 8, 640, 480, time=0.5)
    assert_frame_equal(ref, t)
    ref2, t2 = run_both(20000, 8, 640, 480, time=0.2)  # opacity factor is exactly 0 => pow(0, .2) = 0
    assert_frame_equal(ref2, t2)


def test_big_splats_many_tiles_per_splat():
    ref, t = run_both(3000, 9, 640, 480, scale_boost=2.5)
    assert ref.duplicates / max(ref.visible, 1) > 20
    assert_frame_equal(ref, t)


def test_overflow_is_reported():
    """GSR_FLAG_STATIC_CAPACITY = the reference's fixed factor*N capacity (rasterizer.gd:79): overflow is reported, not repaired."""
    ref, t = run_both(3000, 9, 640, 480, scale_boost=2.5, factor=2, flags=_lib.GSR_FLAG_STATIC_CAPACITY)
    assert ref.overflow
    assert_frame_equal(ref, t)


def test_capacity_grows_instead_of_truncating():
    """Scope row f4 (rasterizer.gd:79 'FIXME: This should not be a static value!'): by default the duplicate capacity grows.  The
    scene that overflows a 2 x N capacity must come out exactly like the oracle run with room for every instance -- through the
    synchronous call at once, through the asynchronous one from the frame after the (flagged) overflow."""
    n, w, h = 3000, 640, 480
    splat60, vp, ub = make_scene(n, 9, w, h, scale_boost=2.5)
    ref = orc.frame(splat60, vp, orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8)), cap=400 * n)
    assert not ref.overflow and ref.duplicates > 2 * n
    with Ctx(n, w, h, factor=2) as c:          # synchronous: never a truncated frame
        c.upload(splat60)
        img = c.render(vp, ub)
        t = c.taps()
        assert not t["stats"].overflow and t["stats"].capacity >= ref.duplicates > 2 * n
        np.testing.assert_array_equal(t["keys"], ref.keys)
        np.testing.assert_array_equal(t["values"], ref.values)
        np.testing.assert_array_equal(t["bounds"], ref.bounds)
        np.testing.assert_array_equal(bits(img), bits(ref.rgba))
    with Ctx(n, w, h, factor=2) as c:          # asynchronous: the overflowing frame is flagged, the next one has room
        c.upload(splat60)
        c.render_async(vp, ub)
        c.sync()
        assert c.stats().overflow == 1 and c.stats().duplicates == ref.duplicates
        c.render_async(vp, ub)
        c.sync()
        t = c.taps()
        assert not t["stats"].overflow
        np.testing.assert_array_equal(t["keys"], ref.keys)
        img = c.copy(_lib.GSR_BUF_FRAMEBUFFER, w * h * 4, np.float32).reshape(h, w, 4)
        np.testing.assert_array_equal(bits(img), bits(ref.rgba))


def test_not_yet_loaded_splats_are_dispatched_like_the_reference():
    """The reference dispatches the projection over point_cloud.size every frame (rasterizer.gd:83,134), i.e. also over the
    zero-initialised structs of splats the loader thread has not delivered yet; libgsr does the same (max_splats, zeroed SoA)."""
    n, loaded, w, h = 20000, 12345, 640, 480
    splat60, vp, ub = make_scene(n, 12, w, h)
    partial = splat60.copy()
    partial[loaded:] = 0.0
    ref = orc.frame(partial, vp, orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8)))
    with Ctx(n, w, h) as c:
        c.upload(splat60[:loaded])
        img = c.render(vp, ub)
        t = c.taps()
    assert t["stats"].duplicates == ref.duplicates
    np.testing.assert_array_equal(t["keys"], ref.keys)
    np.testing.assert_array_equal(t["values"], ref.values)
    np.testing.assert_array_equal(t["bounds"], ref.bounds)
    np.testing.assert_array_equal(bits(img), bits(ref.rgba))


@pytest.mark.parametrize("band", [(0, 7), (7, 20), (20, 30), (29, 30), (12, 12)])
def test_tile_row_band_matches_oracle_band(band):
    ref, t = run_both(20000, 10, 640, 480, band=band)
    assert_frame_equal(ref, t, band=band)


def test_bands_concatenate_to_full_frame():
    """SURVEY 8e: per-band sorted keys concatenated in band order == single-GPU sorted keys; pixels too."""
    n, w, h = 20000, 640, 480
    splat60, vp, ub = make_scene(n, 11, w, h)
    with Ctx(n, w, h) as c:
        c.upload(splat60)
        full = c.render(vp, ub)
        tf = c.taps()
        keys, vals, img = [], [], np.zeros_like(full)
        for band in [(0, 8), (8, 16), (16, 24), (24, 30)]:
            c.set_band(*band)
            part = c.render(vp, ub)
            tb = c.taps()
            keys.append(tb["keys"]); vals.append(tb["values"])
            img[band[0] * 16:band[1] * 16] = part[band[0] * 16:band[1] * 16]
    np.testing.assert_array_equal(np.concatenate(keys), tf["keys"])
    np.testing.assert_array_equal(np.concatenate(vals), tf["values"])
    np.testing.assert_array_equal(bits(img), bits(full))


def test_empty_scene_and_all_culled():
    n, w, h = 1000, 320, 240
    splat60, vp, ub = make_scene(n, 12, w, h)
    splat60[:, 2] = -5.0  # behind the camera: everything culled
    with Ctx(n, w, h) as c:
        c.upload(splat60)
        img = c.render(vp, ub)
        st = c.stats()
    assert st.duplicates == 0 and st.visible == 0 and st.last_tile == -1
    assert np.all(img[..., :3] == 0) and np.all(img[..., 3] == 1)


def test_rerender_is_deterministic_and_resize_works():
    n = 20000
    splat60, vp, ub = make_scene(n, 13, 640, 480)
    with Ctx(n, 640, 480) as c:
        c.upload(splat60)
        a = c.render(vp, ub)
        b = c.render(vp, ub)
        np.testing.assert_array_equal(bits(a), bits(b))
        splat60b, vp2, ub2 = make_scene(n, 13, 800, 450)
        c.resize(800, 450)
        img = c.render(vp2, ub2)
    ref = orc.frame(splat60, vp2, orc.uniforms_from_bytes(np.frombuffer(ub2, dtype=np.uint8)))
    np.testing.assert_array_equal(bits(img), bits(ref.rgba))


def test_chunked_upload_equals_single_upload():
    n = 10000
    splat60, vp, ub = make_scene(n, 14, 320, 240)
    with Ctx(n, 320, 240) as c:
        c.upload(splat60)
        a = c.render(vp, ub)
    with Ctx(n, 320, 240) as c:
        for lo in range(0, n, 1234):
            c.upload(splat60[lo:lo + 1234], first=lo)
        b = c.render(vp, ub)
    np.testing.assert_array_equal(bits(a), bits(b))


def test_pick_matches_oracle():
    n, w, h = 20000, 640, 480
    splat60, vp, ub = make_scene(n, 15, w, h)
    ref = orc.frame(splat60, vp, orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8)))
    counts = ref.bounds[:, 1].astype(np.int64) - ref.bounds[:, 0]
    busy = int(np.argmax(counts))
    empty = int(np.argmin(counts))
    with Ctx(n, w, h) as c:
        c.upload(splat60)
        c.render(vp, ub, readback=False)
        got_empty = c.pick(empty)
        got = c.pick(busy)
    _, _, want = orc.render(ref.records, ref.values, ref.bounds, w, h, target_tile=busy, pick=np.zeros(4, np.float32))
    np.testing.assert_array_equal(bits(got), bits(want))
    if counts[empty] <= 0:
        assert got_empty[3] == 0  # nothing written: rasterizer.gd:171 returns Vector3.INF


def test_pipelined_readback_matches_sync_render():
    """gsr_render_async + copy stream: every host frame equals the synchronous render of the same camera."""
    import ctypes as C
    n, w, h = 20000, 640, 480
    frames = [make_scene(n, 16, w, h, frame=f) for f in (0, 20, 40, 60, 80)]
    with Ctx(n, w, h) as c:
        c.upload(frames[0][0])
        want = [c.render(vp, ub) for _, vp, ub in frames]
        hosts = [np.zeros((h, w, 4), dtype=np.float32) for _ in frames]
        for (_, vp, ub), out in zip(frames, hosts):
            vp = np.ascontiguousarray(vp, dtype=np.float32)
            _lib.check(c.L.gsr_render_async(c.h, vp.ctypes.data_as(C.POINTER(C.c_float)), ub, 0.0, C.c_void_p(out.ctypes.data)), "async")
        _lib.check(c.L.gsr_stream_join(c.h), "join")
        _lib.check(c.L.gsr_sync(c.h), "sync")
    for a, b in zip(hosts, want):
        np.testing.assert_array_equal(bits(a), bits(b))


def test_overlapped_frames_equal_serial_frames():
    """Front / back overlap (gsr_debug_pipeline): frame f+1's projection runs beside frame f's compositor on a second stream, consecutive
    frames alternate between two sort inputs and two record tables.  Back-to-back frames through pinned host memory, an upload in
    the middle of the sequence (it must not overtake a projection in flight), a pick after the last frame: bit-identical to the
    serial pipeline, and the first and last frame equal the oracle's."""
    import ctypes as C
    import torch
    n, w, h = 150000, 1280, 720
    cams = [make_scene(n, 23, w, h, frame=f) for f in range(0, 96, 6)]
    splat60 = cams[0][0]
    late = make_scene(n, 24, w, h, frame=0)[0][: n // 3]   # replaces the first third of the splats half-way through
    results = {}
    for overlap in (0, 1):
        with Ctx(n, w, h) as c:
            _lib.check(c.L.gsr_debug_pipeline(c.h, overlap), "pipeline")
            c.upload(splat60)
            hosts = [torch.zeros((h, w, 4), dtype=torch.float32).pin_memory() for _ in cams]
            for i, (_, vp, ub) in enumerate(cams):
                if i == len(cams) // 2:
                    c.upload(late)
                c.render_async(vp, ub, host_ptr=hosts[i].data_ptr())
            _lib.check(c.L.gsr_stream_join(c.h), "join")
            c.sync()
            picked = c.pick(c.stats().last_tile // 2)
            results[overlap] = ([t.numpy().copy() for t in hosts], picked, c.taps())
    for a, b in zip(results[0][0], results[1][0]):
        np.testing.assert_array_equal(bits(a), bits(b))
    np.testing.assert_array_equal(bits(results[0][1]), bits(results[1][1]))
    np.testing.assert_array_equal(results[0][2]["keys"], results[1][2]["keys"])
    np.testing.assert_array_equal(results[0][2]["values"], results[1][2]["values"])
    for idx, scene in ((0, splat60), (len(cams) - 1, np.concatenate([late, splat60[n // 3:]]))):
        _, vp, ub = cams[idx]
        ref = orc.frame(scene, vp, orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8)), cap=1000 * n)
        np.testing.assert_array_equal(bits(results[1][0][idx]), bits(ref.rgba))


def test_golden_demo_subset_on_gpu():
    """Real data: 8216 splats of the reference's demo.ply (tests/golden/demo_subset.npz: oracle outputs + the reference shaders' own outputs)."""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "demo_subset.npz"))
    w, h = int(g["width"]), int(g["height"])
    with Ctx(g["splat60"].shape[0], w, h) as c:
        c.upload(g["splat60"])
        img = c.render(g["vp"], g["uniforms"].tobytes())
        t = c.taps()
    assert t["stats"].duplicates == int(g["duplicates"]) and t["stats"].visible == int(g["visible"])
    np.testing.assert_array_equal(t["keys"], g["keys"])
    np.testing.assert_array_equal(t["values"], g["values"])
    np.testing.assert_array_equal(t["bounds"], g["bounds"])
    assert np.abs(img - g["rgba"]).max() <= RGBA_TOL
    np.testing.assert_array_equal(bits(img), bits(g["rgba"]))
    # ref_*: the same frame minted by the reference's own shaders executed on the CPU (tests/golden/make_golden.py)
    np.testing.assert_array_equal(t["keys"], g["ref_keys"])
    np.testing.assert_array_equal(t["values"], g["ref_values"])
    np.testing.assert_array_equal(t["bounds"], g["ref_bounds"])
    assert np.abs(img - g["ref_rgba"]).max() <= RGBA_TOL


def test_mirror_class_end_to_end():
    """The GDScript-mirror class drives the same path: _init -> rasterize -> get_splat_position -> cleanup_gpu."""
    from godotgaussiansplatting_b200 import camera as cam
    from godotgaussiansplatting_b200.ply_file import swizzle_splats
    from godotgaussiansplatting_b200.rasterizer import GaussianSplattingRasterizer, RenderTexture
    from godotgaussiansplatting_b200.synthetic import synthetic_ply
    ply = synthetic_ply(5000, 17)
    w, h = 400, 300
    camera = cam.default_camera(aspect=w / h)
    tex = RenderTexture()
    r = GaussianSplattingRasterizer(ply, (w, h), tex, camera, clock=lambda: 100.0)
    loaded = []
    r.loaded_callbacks.append(lambda: loaded.append(True))
    r.update_camera_matrices()
    r.rasterize(time=100.0)                       # lazily calls init_gpu (rasterizer.gd:123)
    assert loaded == [True] and r.is_loaded and r.num_splats_loaded[0] == 5000 and tex.device_ptr != 0
    img = tex.read()
    st = r.stats()
    splat60 = swizzle_splats(ply.table, 0.0)      # chunks were stamped with creation time 0 (clock - t0)
    ref = orc.frame(splat60, r.camera_push_constants, orc.uniforms_from_bytes(np.frombuffer(r.uniforms_bytes(100.0), dtype=np.uint8)))
    assert st.duplicates == ref.duplicates
    np.testing.assert_array_equal(bits(img), bits(ref.rgba))
    pos = r.get_splat_position((200, 150))
    assert pos.shape == (3,)
    r.texture_size = (200, 150)                   # resize path (rasterizer.gd:26-48)
    r.camera.aspect = 200 / 150
    r.update_camera_matrices()
    r.rasterize(time=100.0)
    assert tex.read().shape == (150, 200, 4)
    r.cleanup_gpu()
    assert tex.device_ptr == 0


@pytest.mark.parametrize("w,h", [(640, 480), (333, 257)])
def test_rgb_readback_equals_rgba_frame(w, h):
    import ctypes as C
    n = 8000
    splat60, vp, ub = make_scene(n, 18, w, h)
    with Ctx(n, w, h) as c:
        c.upload(splat60)
        want = c.render(vp, ub)
        hosts = [np.zeros((h, w, 3), dtype=np.float32) for _ in range(3)]
        vpc = np.ascontiguousarray(vp, dtype=np.float32)
        for out in hosts:
            _lib.check(c.L.gsr_render_async_rgb(c.h, vpc.ctypes.data_as(C.POINTER(C.c_float)), ub, 0.0, C.c_void_p(out.ctypes.data)), "async rgb")
        _lib.check(c.L.gsr_sync(c.h), "sync")
    assert np.all(want[..., 3] == 1.0)
    for out in hosts:
        np.testing.assert_array_equal(bits(out), bits(np.ascontiguousarray(want[..., :3])))


@pytest.mark.parametrize("flags", [0, _lib.GSR_FLAG_FAST_REJECT])
@pytest.mark.parametrize("G,n,seed,boost", [(2, 20000, 19, 0.0), (3, 20000, 20, 0.0), (5, 6000, 21, 1.5), (8, 30000, 22, 0.5)])
def test_row_interleave_fast_mode_reassembles_the_full_frame(G, n, seed, boost, flags):
    """Cyclic tile-row ownership + conservative early reject + all-reduced last tile + fix-up (emulated on one GPU):
    per-rank sorted pairs are exactly the full frame's pairs of the owned rows, and the assembled frame equals the
    oracle's frame bit for bit (including the blanked last occupied tile of the reference's Q10 quirk)."""
    w, h = 640, 360
    gx = (w + 15) // 16
    splat60, vp, ub = make_scene(n, seed, w, h, frame=30, scale_boost=boost)
    factor = 60 if boost > 1.0 else 10
    ref = orc.frame(splat60, vp, orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8)), cap=factor * n)
    assert not ref.overflow
    rows = (ref.keys >> 16) // gx
    with Ctx(n, w, h, factor=factor, flags=flags) as c:
        c.upload(splat60)
        words = []
        for rem in range(G):
            c.set_row_interleave(rem, G)
            c.render(vp, ub, readback=False)
            t = c.taps()
            sel = rows % G == rem
            np.testing.assert_array_equal(t["keys"], ref.keys[sel])
            np.testing.assert_array_equal(t["values"], ref.values[sel])
            assert t["stats"].duplicates == int(sel.sum())
            words.append(c.sync_word())
            assert words[-1] == (int(ref.keys[sel][-1] >> 16) + 1 if sel.any() else 0)
        assert max(words) == ref.last_tile + 1
        for rem in range(G):  # emulate all-reduce(MAX) + fix-up on every "rank"
            c.set_row_interleave(rem, G)
            c.sync_word(max(words))
            c.band_fixup()
        img = c.copy(_lib.GSR_BUF_FRAMEBUFFER, w * h * 4, np.float32).reshape(h, w, 4)
    np.testing.assert_array_equal(bits(img), bits(ref.rgba))


def test_device_ply_ingest_matches_host_ingest():
    """Scope row f1: gsr_upload_ply_raw (exp/sigmoid/quat->cov/SH interleave on the GPU) feeds the projection the same
    splats as the host mirror + oracle restatement of util/ply_file.gd:44-69: identical keys, ranges and pixels."""
    from godotgaussiansplatting_b200 import camera as cam
    from godotgaussiansplatting_b200.ply_file import swizzle_splats
    from godotgaussiansplatting_b200.synthetic import synthetic_ply_table
    from tests.scenes import uniforms_bytes
    n, w, h = 50000, 640, 480
    table = synthetic_ply_table(n, 23)
    table[:5, 54] = [np.inf, -np.inf, 40.0, -40.0, 0.0]           # opacity-logit extremes (demo.ply has +inf)
    table[5, 58:62] = (1.0, 0.0, 0.0, 0.0)                          # identity rotation: exact zeros in the covariance
    table = np.concatenate([table, np.zeros((n, 3), np.float32)], axis=1)  # 65 properties: extra columns are ignored
    c0 = cam.default_camera(aspect=w / h)
    vp = cam.pack_camera_push_constants(c0.get_camera_transform(), c0.get_camera_projection())
    ub = uniforms_bytes(c0.global_position, 1.0, w, h, 10.0)
    splat60 = swizzle_splats(table, 2.5)
    np.testing.assert_array_equal(splat60.view(np.uint32), orc.preprocess_ply(table, 2.5).view(np.uint32))
    with Ctx(n, w, h) as c:
        c.upload(splat60)
        a = c.render(vp, ub)
        ta = c.taps()
    with Ctx(n, w, h) as c:
        for lo in range(0, n, 17000):
            c.upload_ply_raw(table[lo:lo + 17000], first=lo, creation_time=2.5)
        b = c.render(vp, ub)
        tb = c.taps()
    np.testing.assert_array_equal(ta["keys"], tb["keys"])
    np.testing.assert_array_equal(ta["values"], tb["values"])
    np.testing.assert_array_equal(ta["bounds"], tb["bounds"])
    np.testing.assert_array_equal(bits(a), bits(b))


@pytest.mark.parametrize("fmt", [_lib.GSR_OUT_RGBA32F, _lib.GSR_OUT_RGB32F, _lib.GSR_OUT_RGBA16F, _lib.GSR_OUT_RGBA8,
                                 _lib.GSR_OUT_RGBA32F | _lib.GSR_OUT_SRGB_TO_LINEAR, _lib.GSR_OUT_RGBA16F | _lib.GSR_OUT_SRGB_TO_LINEAR,
                                 _lib.GSR_OUT_RGBA8 | _lib.GSR_OUT_SRGB_TO_LINEAR])
def test_presentation_formats_match_the_oracle_frame_through_the_same_conversion(fmt):
    """Scope row f3: the fused copy-out conversions (csrc/present.cu; main.gdshader:7-11 for the sRGB -> linear variants) applied to
    the frame equal oracle.present() of the oracle's frame byte for byte -- through the pipelined host read-back and through the
    device-to-device hand-off (gsr_present_device, the path an imported Vulkan image takes)."""
    import ctypes as C
    import torch
    n, w, h = 40000, 645, 363     # ragged: neither a tile multiple nor a multiple of 4 pixels
    splat60, vp, ub = make_scene(n, 21, w, h, scale_boost=0.7)
    ref = orc.frame(splat60, vp, orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8)), heatmap=1.0)
    want = orc.present(ref.rgba, fmt)
    nbytes = _lib.lib().gsr_output_bytes(fmt, w, h)
    assert nbytes == want.nbytes
    with Ctx(n, w, h) as c:
        c.upload(splat60)
        host = torch.zeros(nbytes, dtype=torch.uint8).pin_memory()
        c.render_async_fmt(vp, ub, host.data_ptr(), fmt, heatmap=1.0)
        c.sync()
        np.testing.assert_array_equal(host.numpy(), want.view(np.uint8).reshape(-1))
        dev = torch.zeros(nbytes + 64, dtype=torch.uint8, device="cuda")
        _lib.check(_lib.lib().gsr_present_device(c.h, C.c_void_p(dev.data_ptr()), fmt), "gsr_present_device")
        c.sync()
        np.testing.assert_array_equal(dev[:nbytes].cpu().numpy(), want.view(np.uint8).reshape(-1))
        assert not dev[nbytes:].any()


def test_uncontracted_blend_flag_is_bit_identical_to_the_reference_shader_text():
    """GSR_FLAG_UNCONTRACTED_BLEND (VERDICT r01 weak #3): with no fma contraction anywhere in gsplat_render.glsl:84-90 the GPU frame is
    bit-identical to the oracle's uncontracted evaluation -- the evaluation the reference's own shader text gives when it is executed
    on the CPU (its frame's digest is stored in tests/golden/refshaders.json)."""
    n, w, h = 30000, 640, 360
    splat60, vp, ub = make_scene(n, 23, w, h, scale_boost=0.8)
    u = orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8))
    orc.set_blend_contraction(False)
    try:
        ref = orc.frame(splat60, vp, u)
    finally:
        orc.set_blend_contraction(True)
    spec = orc.frame(splat60, vp, u)
    with Ctx(n, w, h, flags=_lib.GSR_FLAG_UNCONTRACTED_BLEND) as c:
        c.upload(splat60)
        img = c.render(vp, ub)
        t = c.taps()
    np.testing.assert_array_equal(t["keys"], ref.keys)
    np.testing.assert_array_equal(bits(img), bits(ref.rgba))
    assert float(np.abs(img - spec.rgba).max()) <= 1e-4 and not np.array_equal(bits(img), bits(spec.rgba))   # a different member of the legal set
    from tests.refgolden import digest, golden
    assert digest(img) == golden("uncontracted_blend")["rgba"], "frame differs from the reference shaders' frame"
