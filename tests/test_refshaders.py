"""The pin: the reference's OWN compute shaders, executed on the CPU, against the oracle -- and against the CUDA path.

oracle/_ref/libgsr_refshaders.so is the six .glsl files of the reference compiled for the CPU (oracle/glsl_cpu:
declarations rewrapped, every statement and expression the shader author's; workgroups as fibers with real barriers and
32-wide subgroup collectives).  oracle/refshaders.py issues the dispatches of `rasterize()` (rasterizer.gd:122-160).
What those shaders computed for every case below is stored under tests/golden (tests/refgolden.py; minted by
tests/golden/make_refshaders_golden.py from the builders in this module), so the comparison needs neither the reference
nor oracle/_ref.

What is asserted
  * projection: the 48-byte records, the emitted (key, value) pairs and M are bit-identical to gsr_oracle.c;
  * the three radix-sort shaders x 4 passes are the stable LSD sort the oracle and libgsr implement;
  * tile ranges are identical, including the reference's quirks, and the uninitialised `shared` read found this way (Q20);
  * pixels: bit-identical to the oracle's uncontracted evaluation, and within the north-star 1e-4 of the gsr spec (the five
    explicit contractions the CUDA compositor uses) -- both are legal evaluations of the GLSL text;
  * (-m gpu) the CUDA frame through the C-ABI against the reference-shader frame directly.
"""
import numpy as np
import pytest

from oracle import oracle as orc
from tests.refgolden import LIBM_STEP, bits, digest, golden, libm_delta
from tests.scenes import demo_subset_scene, make_scene

RGBA_TOL = 1e-4

#        n      seed  w    h    frame time  model_scale heatmap creation scale_boost
SCENES = {
    "default_camera": (20000, 3, 320, 208, None, 10.0, 1.0, 0.0, 0.0, 1.0),
    "orbit_ragged_size": (12000, 5, 250, 130, 37, 10.0, 1.0, 0.0, 0.0, 0.5),
    "load_in_animation": (8000, 7, 192, 160, None, 0.6, 1.0, 0.0, 0.0, 1.0),       # Q14: time - splat.time = 0.6
    "scaled_heatmap": (8000, 9, 224, 128, 120, 10.0, 0.5, 1.0, 0.0, 1.5),
    "three_splats": (3, 11, 64, 48, None, 10.0, 1.0, 0.0, 0.0, 2.0),
}
RAGGED = [(1, 1), (2, 3), (15, 15), (16, 16), (17, 17), (31, 33), (257, 1), (640, 16)]
SPLAT_COUNTS = [1, 2, 33, 257]
FUZZ = [(123, 11), (321, 200)]
SORT_SIZES = [1, 2, 255, 4095, 4096, 4097, 12289, 50000]


# ---------------------------------------------------------------- inputs (shared with tests/golden/make_refshaders_golden.py)
def build(name):
    n, seed, w, h, frame, time, ms, heat, creation, boost = SCENES[name]
    splat60, vp, ub = make_scene(n, seed, w, h, frame=frame, time=time, model_scale=ms, creation_time=creation, scale_boost=boost)
    return splat60, vp, ub, w, h, heat


def ragged_scene(w, h):
    splat60, vp, ub = make_scene(3000, 50, w, h, scale_boost=1.0)
    return splat60, vp, ub, w, h, 0.0


def splat_count_scene(n):
    splat60, vp, ub = make_scene(n, 60 + n, 320, 240, scale_boost=-1.5)   # capacity is the static 10 n (Q12): keep M below it
    return splat60, vp, ub, 320, 240, 0.0


def one_splat_covering_every_tile_scene():
    w, h, n = 640, 480, 200                       # cap = 10 n = 2000 >= the 1200 tiles
    splat60, vp, ub = make_scene(n, 70, w, h)
    splat60[:, 0:3] = (0.0, 0.0, 2.5)
    splat60[:, 4:10] = 0.0
    splat60[0, 4], splat60[0, 7], splat60[0, 9] = 4.0, 4.0, 4.0
    splat60[1:, 4], splat60[1:, 7], splat60[1:, 9] = 1e-6, 1e-6, 1e-6
    splat60[:, 10] = 0.5
    return splat60, vp, ub, w, h, 0.0


def everything_culled_scene():
    w, h, n = 160, 96, 500
    splat60, vp, ub = make_scene(n, 90, w, h)
    splat60[:, 2] = -np.abs(splat60[:, 2]) - 50.0     # behind the camera / outside the frustum
    spec, _, _ = oracle_frames(splat60, vp, ub, 0.0)
    if spec.duplicates:                                  # the camera looks down the other axis: flip
        splat60[:, 2] = -splat60[:, 2]
    return splat60, vp, ub, w, h, 0.0


def degenerate_scene():
    """opacity 0 (pow(0, .2) = 0 -> radius 0), zero covariance (only the +0.3 dilation), opacity logit extremes."""
    n, w, h = 2000, 320, 240
    splat60, vp, ub = make_scene(n, 80, w, h, scale_boost=1.0)
    splat60[8, 10] = 0.0
    splat60[9, 4:10] = 0.0
    splat60[10, 10] = 1.0
    splat60[11, 10] = 1e-30
    return splat60, vp, ub, w, h, 0.0


def adversarial_splats(n, seed, w, h, frame):
    """Random splats far outside the synthetic generator's envelope: positions over four decades (also behind the camera),
    scales from 1e-5 to 6 with random orientation, opacities at the ends of [0, 1], every phase of the load-in animation,
    large SH coefficients."""
    rng = np.random.default_rng(seed)
    splat60, vp, ub = make_scene(n, seed, w, h, frame=frame)
    splat60[:, 0:3] = rng.normal(0, 1, (n, 3)).astype(np.float32) * rng.choice([0.1, 1, 3, 10, 100], size=(n, 1)).astype(np.float32)
    splat60[:, 3] = rng.choice([0.0, 9.2, 9.7, 9.99, 10.0, 12.0], size=n).astype(np.float32)     # uniforms.time is 10
    q = rng.normal(size=(n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    qw, qx, qy, qz = q.T
    R = np.stack([1 - 2 * (qy * qy + qz * qz), 2 * (qx * qy - qz * qw), 2 * (qx * qz + qy * qw),
                  2 * (qx * qy + qz * qw), 1 - 2 * (qx * qx + qz * qz), 2 * (qy * qz - qx * qw),
                  2 * (qx * qz - qy * qw), 2 * (qy * qz + qx * qw), 1 - 2 * (qx * qx + qy * qy)], axis=1).reshape(n, 3, 3)
    sc = np.exp(rng.uniform(np.log(1e-5), np.log(6), (n, 3)))
    S = np.einsum("nij,nj,nkj->nik", R, sc ** 2, R).astype(np.float32)
    splat60[:, 4], splat60[:, 5], splat60[:, 6] = S[:, 0, 0], S[:, 0, 1], S[:, 0, 2]
    splat60[:, 7], splat60[:, 8], splat60[:, 9] = S[:, 1, 1], S[:, 1, 2], S[:, 2, 2]
    splat60[:, 10] = rng.choice([0.0, 1e-6, 0.01, 0.5, 0.999, 1.0], size=n).astype(np.float32)
    splat60[:, 12:60] = rng.normal(0, 1.5, (n, 48)).astype(np.float32)
    return splat60, vp, ub


def projection_fuzz_scene(seed, frame):
    n, w, h = 100000, 640, 360
    splat60, vp, ub = adversarial_splats(n, seed, w, h, frame)
    splat60[30000:, 0:3] = 1e9        # 70 000 culled fillers: the reference sizes the pair buffers as 10 x point count (Q12)
    return splat60, vp, ub, w, h


def render_fuzz_inputs():
    """Synthetic records and ranges: indefinite conics (positive power, alpha > 1, negative transmittance -- Q8: nothing is
    clamped), ranges that run past their chunk, the heat-map term.  Returns (records, values, bounds, w, h)."""
    rng = np.random.default_rng(77)
    w, h, nrec = 96, 64, 5000
    T = ((w + 15) // 16) * ((h + 15) // 16)
    rec = np.zeros(nrec, dtype=orc.RECORD_DTYPE)
    rec["image_pos"] = rng.uniform(-20, [w + 20, h + 20], (nrec, 2)).astype(np.float32)
    rec["conic"] = np.stack([rng.uniform(-0.002, 0.05, nrec), rng.uniform(-0.03, 0.03, nrec), rng.uniform(-0.002, 0.05, nrec)], axis=1).astype(np.float32)
    rec["color"] = np.concatenate([rng.uniform(0, 1.5, (nrec, 3)), rng.choice([0.0, 0.02, 0.3, 0.9, 1.0, 1.7], size=(nrec, 1))], axis=1).astype(np.float32)
    rec["pos_xy"] = rng.normal(size=(nrec, 2)).astype(np.float32)
    rec["pos_z"] = rng.normal(size=nrec).astype(np.float32)
    lens = rng.choice([0, 1, 3, 255, 256, 257, 700], size=T)
    M = int(lens.sum())
    values = rng.integers(0, nrec, M + 300, dtype=np.uint32)           # entries past a range are read too (:72)
    bounds = np.zeros((T, 2), dtype=np.uint32)
    bounds[:, 0] = np.concatenate([[0], np.cumsum(lens)[:-1]])
    bounds[:, 1] = bounds[:, 0] + lens
    bounds[3] = (50, 10)                                                # end < start: max(0, int(y - x)) = 0 splats (:61)
    return rec, values, bounds, w, h


def boundaries_garbage_words(spec):
    """Values for the shared word gsplat_boundaries.glsl:36 reads uninitialised (Q20); the last is the first key's tile."""
    first = int(spec.keys[0] >> 16)
    return (0xFFFFFFFF, 0, first + 1, spec.bounds.shape[0] - 1, first)


def sort_inputs(n):
    rng = np.random.default_rng(n)
    keys = rng.integers(0, 2**32, n, dtype=np.uint64).astype(np.uint32)
    if n > 1000:
        keys[: n // 2] = keys[: n // 2] & np.uint32(0xFFFF00FF)       # many ties: stability is observable
    return keys, np.arange(n, dtype=np.uint32)


def pick_target_tile(spec):
    counts = spec.bounds[:, 1].astype(np.int64) - spec.bounds[:, 0].astype(np.int64)
    return int(np.argmax(counts)), counts


def demo_scene():
    _, s, vp, ub = demo_subset_scene()
    return s, vp, ub, 640, 480, 0.0


def oracle_frames(splat60, vp, ub, heat):
    u = orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8))
    spec = orc.frame(splat60, vp, u, heatmap=heat)
    orc.set_blend_contraction(False)
    try:
        strict = orc.frame(splat60, vp, u, heatmap=heat)
    finally:
        orc.set_blend_contraction(True)
    return spec, strict, u


# ---------------------------------------------------------------- checks against the stored reference outputs
def assert_stages_equal(ref, spec, strict, splat60, vp, u):
    """ref: golden record of the reference shaders' frame; spec / strict: oracle Frames with / without the spec's contractions."""
    assert not spec.overflow
    assert ref["duplicates"] == spec.duplicates
    pr = orc.project(splat60, vp, u)
    assert digest(pr.keys) == ref["keys_unsorted"], "emitted keys differ from the reference shaders"
    assert digest(pr.values) == ref["values_unsorted"], "emitted values differ from the reference shaders"
    vis = np.unique(pr.values)
    assert vis.size == spec.visible
    assert digest(pr.records[vis]) == ref["records"], "records of the visible splats differ from the reference shaders"
    assert digest(spec.keys) == ref["keys"], "sorted keys differ from the reference shaders"
    assert digest(spec.values) == ref["values"], "sorted values differ from the reference shaders"
    assert digest(spec.bounds) == ref["bounds"], "tile ranges differ from the reference shaders"
    m = spec.duplicates
    assert ref["grid_dims"][0] == max(1, -(-m // 4096)) and ref["grid_dims"][3] == max(1, -(-m // 256))   # :212-213
    # pixels: the shader text without contraction == the oracle without contraction, bit for bit ...
    assert digest(strict.rgba) == ref["rgba"], "the oracle's uncontracted frame differs from the reference shaders' frame"


def check_scene(case, splat60, vp, ub, w, h, heat=0.0):
    """Returns the oracle's (spec, strict) frames; strict.rgba is the reference shaders' frame, bit for bit."""
    spec, strict, u = oracle_frames(splat60, vp, ub, heat)
    assert_stages_equal(golden(case), spec, strict, splat60, vp, u)
    # ... and the gsr spec (explicit contractions, what libgsr computes) is inside the north-star tolerance of it
    assert np.abs(strict.rgba - spec.rgba).max() <= RGBA_TOL
    return spec, strict


@pytest.mark.parametrize("name", list(SCENES))
def test_reference_shaders_equal_oracle_bit_for_bit(name):
    splat60, vp, ub, w, h, heat = build(name)
    spec, strict = check_scene(f"scene/{name}", splat60, vp, ub, w, h, heat)
    assert spec.duplicates > 0
    assert np.all(strict.rgba[..., 3] == 1.0)


@pytest.mark.parametrize("w,h", RAGGED)
def test_ragged_resolutions(w, h):
    """Partial tiles: off-image invocations still vote in the tile-stop rule (Q9/Q17) and imageStore drops their texels."""
    check_scene(f"ragged/{w}x{h}", *ragged_scene(w, h))


@pytest.mark.parametrize("n", SPLAT_COUNTS)
def test_splat_counts_around_subgroup_and_workgroup_sizes(n):
    check_scene(f"splats/{n}", *splat_count_scene(n))


def test_one_splat_covering_every_tile_hits_the_last_grid_tile_rule():
    """A splat whose rect is the whole grid: the last occupied tile IS tile T-1, so gsplat_boundaries.glsl:47-49 stores
    M-1 as its end (Q10: the final instance of the last grid tile is dropped)."""
    spec, _ = check_scene("one_splat_covering_every_tile", *one_splat_covering_every_tile_scene())
    T = spec.bounds.shape[0]
    assert spec.duplicates >= T and int(spec.keys[-1] >> 16) == T - 1
    assert spec.bounds[T - 1, 1] == spec.duplicates - 1


def test_everything_culled():
    """M = 0: the sort runs on one empty partition, no range is written, the frame is black with alpha 1."""
    splat60, vp, ub, w, h, heat = everything_culled_scene()
    spec, _, _ = oracle_frames(splat60, vp, ub, heat)
    assert spec.duplicates == 0
    ref = golden("everything_culled")
    assert ref["duplicates"] == 0 and digest(spec.bounds) == ref["bounds"] and not spec.bounds.any()
    assert digest(spec.rgba) == ref["rgba"]
    assert not spec.rgba[..., :3].any() and np.all(spec.rgba[..., 3] == 1.0)


def test_degenerate_splats():
    spec, _ = check_scene("degenerate_splats", *degenerate_scene())
    assert (spec.values == 8).sum() <= 1          # radius 0 still rounds out to the one tile under the centre


@pytest.mark.parametrize("seed,frame", FUZZ)
def test_projection_fuzz(seed, frame):
    """gsplat_projection.glsl alone on adversarial splats: M, every emitted pair and every record bit for bit."""
    splat60, vp, ub, w, h = projection_fuzz_scene(seed, frame)
    n = splat60.shape[0]
    u = orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8))
    pr = orc.project(splat60, vp, u, cap=10 * n)
    assert 0 < pr.duplicates <= 10 * n and pr.visible > 500
    ref = golden(f"projection_fuzz/{seed}-{frame}")
    assert ref["duplicates"] == pr.duplicates
    assert digest(pr.keys) == ref["keys_unsorted"] and digest(pr.values) == ref["values_unsorted"]
    assert digest(pr.records[np.unique(pr.values)]) == ref["records"]


def test_render_fuzz():
    """gsplat_render.glsl alone on synthetic records and ranges (render_fuzz_inputs)."""
    rec, values, bounds, w, h = render_fuzz_inputs()
    orc.set_blend_contraction(False)
    try:
        want, _, _ = orc.render(rec, values, bounds, w, h, heatmap=1.0)
    finally:
        orc.set_blend_contraction(True)
    assert digest(want) == golden("render_fuzz")["rgba"]


def test_reference_demo_subset_through_the_reference_shaders():
    """Real data: every 33rd splat of the reference's own demo.ply (tests/golden/demo_subset.npz), 640x480, default camera:
    every stage of the shaders == the oracle, and Q10 fires on tile 1198 as on the whole asset (SURVEY Appendix B)."""
    spec, _ = check_scene("demo_subset_640x480", *demo_scene())
    assert spec.last_tile == 1198
    assert spec.bounds[1198, 1] == 0          # Q10: the last occupied tile never gets its end


def test_boundaries_uninitialised_shared_word():
    """Q20: invocation 0 of workgroup 0 returns before storing local[1]; invocation 1 reads it as its left neighbour."""
    splat60, vp, ub, w, h, heat = build("orbit_ragged_size")
    spec, _, _ = oracle_frames(splat60, vp, ub, heat)
    T = spec.bounds.shape[0]
    first = int(spec.keys[0] >> 16)
    for garbage in boundaries_garbage_words(spec):
        got = orc.boundaries_uninit(spec.keys, T, garbage)
        assert digest(got) == golden(f"boundaries_uninit/{garbage:#x}")["bounds"], f"garbage={garbage:#x}"
        if garbage == first:
            np.testing.assert_array_equal(got, spec.bounds)       # the defined behaviour of orc_boundaries / libgsr
        elif garbage != int(spec.keys[1] >> 16):
            assert got[int(spec.keys[1] >> 16), 0] == 1          # a range that starts at 1: instance 0 is dropped


@pytest.mark.parametrize("n", SORT_SIZES)
def test_sort_shaders_are_a_stable_lsd_sort(n):
    keys, values = sort_inputs(n)
    order = np.argsort(keys, kind="stable")
    k, v = keys[order], values[order]
    ref = golden(f"sort/{n}")
    assert digest(k) == ref["keys"] and digest(v) == ref["values"]
    ok, ov = orc.sort_pairs(keys, values)
    np.testing.assert_array_equal(k, ok)
    np.testing.assert_array_equal(v, ov)
    ek, ev = orc.sort_pairs_shader_emulation(keys, values, cap=n + 17)
    np.testing.assert_array_equal(k, ek)
    np.testing.assert_array_equal(v, ev)


def test_pick_tile():
    """gsplat_render.glsl:105-110 -> tile_splat_pos (rasterizer.gd:162-171)."""
    splat60, vp, ub, w, h, heat = build("default_camera")
    spec, _, _ = oracle_frames(splat60, vp, ub, heat)
    tile, counts = pick_target_tile(spec)
    _, _, pick = orc.render(spec.records, spec.values, spec.bounds, w, h, heatmap=heat, target_tile=tile)
    ref = golden("pick_tile")
    assert [int(x) for x in bits(pick)] == ref["pick"]
    assert pick[3] == counts[tile]


def test_libm_builtins_stay_inside_tolerance():
    """exp()/pow() are implementation-defined in GLSL: with glibc's expf/powf instead of the spec's polynomials the frame
    stays within the north-star tolerance (a 1-ulp pow() may move a tile rect; allow a vanishing fraction of pixels)."""
    splat60, vp, ub, w, h, heat = build("default_camera")
    spec, strict, _ = oracle_frames(splat60, vp, ub, heat)
    assert digest(strict.rgba) == golden("scene/default_camera")["rgba"]
    ref = golden("libm")
    assert abs(ref["duplicates"] - spec.duplicates) <= max(4, spec.duplicates // 10000)
    libm_rgba = strict.rgba.astype(np.float64)
    libm_rgba[..., :3] += libm_delta() * LIBM_STEP
    bad = (np.abs(libm_rgba - spec.rgba).max(axis=2) > RGBA_TOL).mean()
    assert bad <= 1e-3, bad


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["default_camera", "orbit_ragged_size", "load_in_animation", "scaled_heatmap"])
def test_cuda_path_against_reference_shaders(name):
    """libgsr (CUDA, through the C-ABI) against the reference's shaders themselves: integers bit-exact, pixels 1e-4."""
    from godotgaussiansplatting_b200 import _lib
    from tests.gsr_direct import Ctx

    splat60, vp, ub, w, h, heat = build(name)
    with Ctx(splat60.shape[0], w, h) as c:
        c.upload(splat60)
        c.keep_unsorted()
        rgba = c.render(vp, ub, heatmap=heat)
        t = c.taps()
        ukeys = c.copy(_lib.GSR_BUF_KEYS_UNSORTED, t["m"], np.uint32)
        uvals = c.copy(_lib.GSR_BUF_VALUES_UNSORTED, t["m"], np.uint32)
    assert t["m"] > 0
    ref = golden(f"scene/{name}")
    assert t["m"] == ref["duplicates"]
    assert digest(ukeys) == ref["keys_unsorted"] and digest(uvals) == ref["values_unsorted"]
    assert digest(t["keys"]) == ref["keys"] and digest(t["values"]) == ref["values"]
    assert digest(t["bounds"]) == ref["bounds"]
    # records and pixels against the oracle's frame, which is the reference shaders' frame (digests checked here too)
    spec, strict, u = oracle_frames(splat60, vp, ub, heat)
    assert digest(strict.rgba) == ref["rgba"]
    pr = orc.project(splat60, vp, u)
    vis = np.unique(pr.values)
    assert digest(pr.records[vis]) == ref["records"]
    for f in orc.RECORD_DTYPE.names:
        np.testing.assert_array_equal(bits(t["records"][f][vis]), bits(pr.records[f][vis]), err_msg=f"record field {f}")
    assert np.abs(rgba - strict.rgba).max() <= RGBA_TOL
