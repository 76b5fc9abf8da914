"""Mints tests/golden/refshaders.json and tests/golden/refshaders_libm.npz: what the reference's own compute shaders compute,
executed on the CPU (oracle/refshaders.py over oracle/_ref), for every case of tests/test_refshaders.py, the frame of
__graft_entry__.smoke() and the frame of tests/test_gpu_pipeline.py::test_uncontracted_blend_flag_is_bit_identical_to_the_reference_shader_text.

Needs a checkout of the original project to build oracle/_ref:
    GSR_REFERENCE_DIR=<original project> python tests/golden/make_refshaders_golden.py
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import refshaders  # noqa: E402
from tests import refgolden  # noqa: E402
from tests import test_refshaders as T  # noqa: E402
from tests.scenes import make_scene  # noqa: E402

if not refshaders.available():
    raise SystemExit("oracle/_ref is not built: set GSR_REFERENCE_DIR to a checkout of the original project")


def reference_frame(splat60, vp, ub, w, h, heat, first_tile, libm=False, target_tile=-1):
    # the shared word gsplat_boundaries.glsl:36 reads uninitialised (Q20) holds the first key's tile: the author's intent
    refshaders.set_shared_fill(first_tile, libm=libm)
    return refshaders.ReferencePipeline(splat60, w, h, libm=libm).rasterize(vp, ub, heatmap=heat, target_tile=target_tile)


def frame_case(splat60, vp, ub, w, h, heat=0.0):
    spec, _, _ = T.oracle_frames(splat60, vp, ub, heat)
    rf = reference_frame(splat60, vp, ub, w, h, heat, int(spec.keys[0] >> 16) if spec.duplicates else 0)
    return refgolden.frame_record(rf)


out = {}
for name in T.SCENES:
    out[f"scene/{name}"] = frame_case(*T.build(name))
for w, h in T.RAGGED:
    out[f"ragged/{w}x{h}"] = frame_case(*T.ragged_scene(w, h))
for n in T.SPLAT_COUNTS:
    out[f"splats/{n}"] = frame_case(*T.splat_count_scene(n))
out["one_splat_covering_every_tile"] = frame_case(*T.one_splat_covering_every_tile_scene())
out["everything_culled"] = frame_case(*T.everything_culled_scene())
out["degenerate_splats"] = frame_case(*T.degenerate_scene())

for seed, frame in T.FUZZ:
    splat60, vp, ub, w, h = T.projection_fuzz_scene(seed, frame)
    n = splat60.shape[0]
    P = refshaders.ReferencePipeline(splat60, w, h)
    P.uniforms[:] = np.frombuffer(bytes(ub), dtype=np.float32)
    P.histogram[: 1 + 4 * refshaders.RADIX] = 0
    P._dispatch("gsplat_projection", ((n + 255) // 256, 1, 1),
                [P.splats, P.culled, P.histogram, P.sort_keys, P.sort_values, P.grid_dims, P.uniforms], np.asarray(vp, dtype=np.float32).tobytes())
    m = int(P.histogram[0])
    values = P.sort_values[:m]
    out[f"projection_fuzz/{seed}-{frame}"] = {"duplicates": m, "keys_unsorted": refgolden.digest(P.sort_keys[:m]),
                                              "values_unsorted": refgolden.digest(values),
                                              "records": refgolden.digest(P.culled[np.unique(values)])}

rec, values, bounds, w, h = T.render_fuzz_inputs()
refshaders.set_shared_fill(0)
tex = np.zeros((h, w, 4), dtype=np.float32)
pick = np.zeros(4, dtype=np.float32)
P = refshaders.ReferencePipeline(np.zeros((1, 60), dtype=np.float32), w, h)
P._dispatch("gsplat_render", ((w + 15) // 16, (h + 15) // 16, 1), [rec, values, bounds, pick, tex], refshaders.create_push_constant([1.0, -1]))
out["render_fuzz"] = {"rgba": refgolden.digest(tex)}

splat60, vp, ub, w, h, heat = T.build("orbit_ragged_size")
spec, _, _ = T.oracle_frames(splat60, vp, ub, heat)
for garbage in T.boundaries_garbage_words(spec):
    out[f"boundaries_uninit/{garbage:#x}"] = {"bounds": refgolden.digest(reference_frame(splat60, vp, ub, w, h, heat, garbage).bounds)}

for n in T.SORT_SIZES:
    k, v = refshaders.sort_pairs(*T.sort_inputs(n), cap=n + 17)
    out[f"sort/{n}"] = {"keys": refgolden.digest(k), "values": refgolden.digest(v)}

splat60, vp, ub, w, h, heat = T.build("default_camera")
spec, _, _ = T.oracle_frames(splat60, vp, ub, heat)
tile, _ = T.pick_target_tile(spec)
out["pick_tile"] = {"pick": refgolden.frame_record(reference_frame(splat60, vp, ub, w, h, heat, int(spec.keys[0] >> 16), target_tile=tile))["pick"]}

base = reference_frame(splat60, vp, ub, w, h, heat, int(spec.keys[0] >> 16))
lm = reference_frame(splat60, vp, ub, w, h, heat, int(spec.keys[0] >> 16), libm=True)
assert np.array_equal(lm.rgba[..., 3], base.rgba[..., 3])
delta = np.round((lm.rgba[..., :3].astype(np.float64) - base.rgba[..., :3]) / refgolden.LIBM_STEP)
assert np.abs(delta).max() <= 127
out["libm"] = {"duplicates": int(lm.duplicates)}
np.savez_compressed(refgolden.LIBM_PATH, delta_rgb=delta.astype(np.int8))

# consumers outside tests/test_refshaders.py: __graft_entry__.smoke() and tests/test_gpu_pipeline.py
out["smoke"] = frame_case(*make_scene(20000, 1, 640, 480), 640, 480)
out["uncontracted_blend"] = frame_case(*make_scene(30000, 23, 640, 360, scale_boost=0.8), 640, 360)

# real data: the demo.ply subset; "stats" feeds tests/test_oracle.py::test_demo_subset_statistics_match_the_reference_shaders
splat60, vp, ub, w, h, heat = T.demo_scene()
spec, _, _ = T.oracle_frames(splat60, vp, ub, heat)
rf = reference_frame(splat60, vp, ub, w, h, heat, int(spec.keys[0] >> 16))
tiles = rf.keys >> 16
out["demo_subset_640x480"] = dict(refgolden.frame_record(rf), stats={
    "visible": int(np.unique(rf.values).size), "occupied_tiles": int(np.unique(tiles).size), "last_tile": int(tiles[-1]),
    "longest_list": int(np.bincount(tiles).max())})

with open(refgolden.JSON_PATH, "w") as f:
    json.dump(out, f, indent=1, sort_keys=True)
    f.write("\n")
print(refgolden.JSON_PATH, len(out), "cases;", refgolden.LIBM_PATH, os.path.getsize(refgolden.LIBM_PATH), "bytes")
