"""CPU tests of the oracle itself (no GPU): deterministic-math pins, the literal shader-emulation of the radix sort,
the float64 numpy transliteration, host mirrors (ingest, camera packing) and the SURVEY Appendix-B statistics."""
import os

import numpy as np
import pytest

from godotgaussiansplatting_b200 import camera as cam
from godotgaussiansplatting_b200.ply_file import swizzle_splats
from godotgaussiansplatting_b200.synthetic import radix_keys, synthetic_ply_table
from oracle import oracle as orc
from oracle import refmath_numpy as ref64
from tests.refgolden import digest, golden
from tests.scenes import demo_subset_scene, make_scene

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


# ---------------------------------------------------------------- deterministic math (gsr spec) vs libm
def test_det_exp_accuracy_and_edges():
    x = np.concatenate([np.linspace(-100, 5, 20001), -np.logspace(-8, 2, 500)]).astype(np.float32)
    got = orc.det_exp(x).astype(np.float64)
    want = np.exp(x.astype(np.float64))
    ok = want > 1e-37
    rel = np.abs(got[ok] - want[ok]) / want[ok]
    # Vulkan's bound for exp is 3 + 2|x| ULP; the single-rounded x*log2e argument costs ~|x| ULP/1.44
    assert np.all(rel <= (3 + 2 * np.abs(x[ok])) * 2.0 ** -23)
    assert orc.det_exp([0.0])[0] == 1.0
    assert orc.det_exp([-200.0])[0] == 0.0          # 2^-127 scale underflows to exactly 0
    assert orc.det_exp([-1e30])[0] == 0.0
    assert np.isinf(orc.det_exp([100.0])[0])         # 2^128 -> +inf


def test_det_pow_fifth_root():
    x = np.concatenate([np.logspace(-38, 0, 4000), [1.0, 0.5, 1e-45, 2.0 ** -126]]).astype(np.float32)
    got = orc.det_pow(x, 0.2).astype(np.float64)
    want = np.power(x.astype(np.float64), np.float64(np.float32(0.2)))
    rel = np.abs(got - want) / want
    # Vulkan: pow inherits exp2(y*log2(x)) = (3 + 2|y log2 x|) ULP on top of log2's 3 ULP
    assert np.all(rel <= (6 + 2 * np.abs(0.2 * np.log2(x.astype(np.float64)))) * 2.0 ** -23)
    assert np.max(rel[x >= 1e-3]) < 4e-7      # realistic opacities: a few ULP
    assert orc.det_pow([0.0], 0.2)[0] == 0.0
    assert orc.det_pow([1.0], 0.2)[0] == 1.0


def test_det_log2_exact_powers():
    for e in (-149, -130, -126, -1, 0, 1, 10, 100):
        assert orc.det_log2([np.float32(2.0) ** e])[0] == float(e)


# ---------------------------------------------------------------- radix sort: literal shader emulation == stable sort
@pytest.mark.parametrize("n", [1, 2, 100, 4095, 4096, 4097, 9000, 20000])
def test_shader_emulation_is_a_stable_sort(n):
    keys = radix_keys(n, n, "tile_depth")
    vals = np.arange(n, dtype=np.uint32)[::-1].copy()
    k, v = orc.sort_pairs_shader_emulation(keys, vals, cap=max(n, 1) + 123)
    order = np.argsort(keys, kind="stable")
    np.testing.assert_array_equal(k, keys[order])
    np.testing.assert_array_equal(v, vals[order])
    k2, v2 = orc.sort_pairs(keys, vals)
    np.testing.assert_array_equal(k2, k)
    np.testing.assert_array_equal(v2, v)


def test_oracle_sort_threaded_large():
    n = 300000
    keys = radix_keys(n, 3, "uniform32")
    vals = np.arange(n, dtype=np.uint32)
    k, v = orc.sort_pairs(keys, vals)
    order = np.argsort(keys, kind="stable")
    np.testing.assert_array_equal(k, keys[order])
    np.testing.assert_array_equal(v, vals[order])


# ---------------------------------------------------------------- boundaries quirks (Q10)
def test_boundaries_quirks():
    T = 8
    keys = (np.array([1, 1, 1, 3, 3, 5], dtype=np.uint32) << 16) | 7
    b = orc.boundaries(keys, T, quirks=True)
    assert b[1].tolist() == [0, 3] and b[3].tolist() == [3, 5]
    assert b[5].tolist() == [5, 0]                 # last occupied tile != T-1: end never written => renders nothing
    b = orc.boundaries(keys, T, quirks=False)
    assert b[5].tolist() == [5, 6]
    keys = (np.array([1, 7, 7, 7], dtype=np.uint32) << 16)
    b = orc.boundaries(keys, T, quirks=True)
    assert b[7].tolist() == [1, 3]                 # tile T-1: end = M-1, final splat dropped
    b = orc.boundaries(np.array([7 << 16], dtype=np.uint32), T, quirks=True)
    assert b[7].tolist() == [0, 0]                 # M == 1: thread 0 returns early, nothing written
    # sharded: band-local last tile that is not the frame's last gets its end
    keys = (np.array([1, 1, 2], dtype=np.uint32) << 16)
    assert orc.boundaries(keys, T, quirks=True, global_last_tile=5)[2].tolist() == [2, 3]
    assert orc.boundaries(keys, T, quirks=True, global_last_tile=2)[2].tolist() == [2, 0]


# ---------------------------------------------------------------- host mirrors
def test_ingest_numpy_mirror_matches_oracle_bitwise():
    table = synthetic_ply_table(5000, 42)
    table[:7, 54] = [np.inf, -np.inf, 88.0, -88.0, -104.0, 0.0, -0.0]   # opacity-logit extremes (demo.ply has +inf)
    a = swizzle_splats(table, 1.25)
    b = orc.preprocess_ply(table, 1.25)
    np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32))
    assert a[0, 10] == 1.0 and a[1, 10] == 0.0


def test_camera_pack_mirror_matches_oracle_bitwise():
    for f in (0, 33, 200):
        c = cam.orbit_camera(f)
        a = cam.pack_camera_push_constants(c.get_camera_transform(), c.get_camera_projection())
        b = orc.pack_camera(c.get_camera_transform(), c.get_camera_projection())
        np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32))
    c = cam.default_camera(aspect=640 / 480)
    vp = cam.pack_camera_push_constants(c.get_camera_transform(), c.get_camera_projection())
    # SURVEY 8c: the default camera gives view = diag(1,1,-1) in the packed convention (up to sin(pi) ~ 8.7e-8)
    np.testing.assert_allclose(vp[:16].reshape(4, 4), np.diag([1, 1, -1, 1]), atol=1e-6)
    assert vp[16 + 11] == -1.0 and vp[16 + 15] == 0.0


def test_orbit_camera_looks_at_centroid():
    s = np.zeros((1, 60), dtype=np.float32)
    s[0, 0:3] = (0.0, 0.0, 2.5)
    s[0, 4], s[0, 7], s[0, 9], s[0, 10] = 1e-4, 1e-4, 1e-4, 0.9
    for f in (0, 90, 181, 300):
        c = cam.orbit_camera(f, aspect=16 / 9)
        vp = cam.pack_camera_push_constants(c.get_camera_transform(), c.get_camera_projection())
        p = c.global_position
        pr = orc.project(s, vp, orc.make_uniforms([-p[0], -p[1], p[2]], 1.0, 1920, 1080, 10.0))
        assert pr.visible == 1
        np.testing.assert_allclose(pr.records["image_pos"][0], [959.5, 539.5], atol=0.05)


# ---------------------------------------------------------------- float64 transliteration vs the float32 oracle
def test_float64_transliteration_agrees_with_oracle():
    n, w, h = 4000, 320, 240
    splat60, vp, ub = make_scene(n, 21, w, h, scale_boost=0.7)
    u = orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8))
    fr = orc.frame(splat60, vp, u)
    pr = ref64.project(splat60, vp, list(u.camera_pos), u.model_scale, w, h, u.time)
    keys64, vals64 = ref64.emit_and_sort(pr)
    # same (tile, splat) instances except for rounding-distance boundary cases of the rect
    a = set(zip((fr.keys >> 16).tolist(), fr.values.tolist()))
    b = set(zip((keys64 >> 16).tolist(), vals64.tolist()))
    assert len(a ^ b) <= 0.001 * max(len(a), 1) + 2, (len(a), len(b), len(a ^ b))
    # depth codes: trunc(z^3 * 65535) evaluated in float32 vs float64 may land one bin apart (z^3*65535 ~ 6e4 has a
    # float32 ulp of 4e-3), never more
    d32 = dict(zip(fr.values.tolist(), (fr.keys & 0xFFFF).tolist()))
    d64 = dict(zip(vals64.tolist(), (keys64 & 0xFFFF).tolist()))
    diffs = np.array([abs(d32[k] - d64[k]) for k in d32 if k in d64])
    assert diffs.max() <= 1 and (diffs != 0).mean() < 0.03
    vis = np.unique(fr.values)
    np.testing.assert_allclose(fr.records["image_pos"][vis], pr["image_pos"][vis], rtol=0, atol=2e-3)
    np.testing.assert_allclose(fr.records["color"][vis, :3], pr["color"][vis], rtol=0, atol=1e-5)
    np.testing.assert_allclose(fr.records["conic"][vis], pr["conic"][vis], rtol=2e-4, atol=1e-7)
    # pixels: blend the oracle's own sorted list in float64 for a few pixels of the busiest tiles
    counts = fr.bounds[:, 1].astype(np.int64) - fr.bounds[:, 0]
    gx = (w + 15) // 16
    for tile in np.argsort(-counts)[:3]:
        if counts[tile] <= 0 or counts[tile] > 256:
            continue  # single-chunk tiles only: no tile-stop decision involved
        tx, ty = tile % gx, tile // gx
        for (dx, dy) in ((0, 0), (7, 9), (15, 15)):
            px, py = tx * 16 + dx, ty * 16 + dy
            if px >= w or py >= h:
                continue
            col, _ = ref64.render_pixels(pr, fr.values, int(fr.bounds[tile, 0]), int(counts[tile]), float(px), float(py))
            np.testing.assert_allclose(fr.rgba[py, px, :3], col, rtol=0, atol=1e-4)


# ---------------------------------------------------------------- reference fixture statistics
def test_demo_subset_statistics_match_the_reference_shaders():
    """Every 33rd splat of the original project's demo.ply (tests/golden/demo_subset.npz), 640x480, default camera: the
    oracle's ingest equals the numpy mirror bit for bit, and V, M, the occupied tiles, the last occupied tile (so Q10 "last
    occupied tile dropped" fires), the longest list and the ranges equal what the reference's own shaders give.  On the whole
    asset (271 123 splats) the same frame has V = 226 063, M = 428 272, 531 tiles, last tile 1198, longest list 7919
    (SURVEY.md Appendix B); the full file is too large to keep here."""
    ply62, s, vp, ub = demo_subset_scene()
    assert ply62.shape == (8216, 62)
    np.testing.assert_array_equal(s.view(np.uint32), swizzle_splats(ply62, 0.0).view(np.uint32))
    fr = orc.frame(s, vp, orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8)))
    ref = golden("demo_subset_640x480")
    assert fr.visible == ref["stats"]["visible"]
    assert fr.duplicates == ref["duplicates"]
    assert len(np.unique(fr.keys >> 16)) == ref["stats"]["occupied_tiles"]
    assert fr.last_tile == ref["stats"]["last_tile"] == 1198
    assert np.bincount(fr.keys >> 16).max() == ref["stats"]["longest_list"]
    assert digest(fr.bounds) == ref["bounds"]
    assert fr.bounds[1198, 1] == 0  # Q10


def test_golden_demo_subset_fixture():
    """tests/golden/demo_subset.npz: 8192 splats of the reference's demo.ply + the oracle outputs minted from them
    (tests/golden/make_golden.py).  Pins the oracle build on any box (the GPU box has no /root/reference)."""
    path = os.path.join(GOLDEN, "demo_subset.npz")
    g = np.load(path)
    s = swizzle_splats(g["ply62"], 0.0)
    np.testing.assert_array_equal(s.view(np.uint32), g["splat60"].view(np.uint32))
    fr = orc.frame(s, g["vp"], orc.uniforms_from_bytes(g["uniforms"]))
    assert fr.duplicates == int(g["duplicates"]) and fr.visible == int(g["visible"])
    np.testing.assert_array_equal(fr.keys, g["keys"])
    np.testing.assert_array_equal(fr.values, g["values"])
    np.testing.assert_array_equal(fr.bounds, g["bounds"])
    np.testing.assert_array_equal(fr.rgba.view(np.uint32), g["rgba"].view(np.uint32))
    # ref_*: minted by the reference's own shaders executed on the CPU (oracle/refshaders.py)
    assert fr.duplicates == int(g["ref_duplicates"])
    np.testing.assert_array_equal(fr.keys, g["ref_keys"])
    np.testing.assert_array_equal(fr.values, g["ref_values"])
    np.testing.assert_array_equal(fr.bounds, g["ref_bounds"])
    assert np.abs(fr.rgba - g["ref_rgba"]).max() <= 1e-4
    orc.set_blend_contraction(False)
    try:
        strict = orc.frame(s, g["vp"], orc.uniforms_from_bytes(g["uniforms"]))
    finally:
        orc.set_blend_contraction(True)
    np.testing.assert_array_equal(strict.rgba.view(np.uint32), g["ref_rgba"].view(np.uint32))
