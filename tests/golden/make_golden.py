"""Mints tests/golden/demo_subset.npz from the reference's only fixture, resources/demo.ply, with a checkout of the original
project:  GSR_REFERENCE_DIR=<original project> python tests/golden/make_golden.py

Contents: every 33rd splat of demo.ply (8216 vertices, the raw 62 floats each), the default camera of
util/camera.gd:151-153 at 320x240, and for that frame
  * ref_*  -- the outputs of THE REFERENCE'S OWN SHADERS executed on the CPU (oracle/refshaders.py over
              oracle/_ref/libgsr_refshaders.so): M, sorted keys/values, tile ranges, the rgba32f texture;
  * keys/values/bounds/rgba -- the oracle's outputs under the gsr spec (identical integers; pixels differ from ref_rgba
              only by the spec's five explicit FMA contractions, <= 1e-4).
The tests need only the stored vectors, not the original project.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from godotgaussiansplatting_b200 import camera as cam  # noqa: E402
from godotgaussiansplatting_b200.ply_file import PlyFile, swizzle_splats  # noqa: E402
from oracle import oracle as orc  # noqa: E402
from tests.scenes import uniforms_bytes  # noqa: E402

ply = PlyFile(os.path.join(os.environ["GSR_REFERENCE_DIR"], "resources", "demo.ply"))
sub = np.ascontiguousarray(ply.table[::33])
W, H = 320, 240
c = cam.default_camera(aspect=W / H)
vp = cam.pack_camera_push_constants(c.get_camera_transform(), c.get_camera_projection())
ub = uniforms_bytes(c.global_position, 1.0, W, H, 10.0)
s = swizzle_splats(sub, 0.0)
fr = orc.frame(s, vp, orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8)))
from oracle import refshaders  # noqa: E402

refshaders.set_shared_fill(int(fr.keys[0] >> 16))   # Q20: the uninitialised shared word of gsplat_boundaries.glsl:36
rf = refshaders.ReferencePipeline(s, W, H).rasterize(vp, ub)
assert rf.duplicates == fr.duplicates and np.array_equal(rf.keys, fr.keys) and np.array_equal(rf.values, fr.values)
assert np.array_equal(rf.bounds, fr.bounds) and np.abs(rf.rgba - fr.rgba).max() <= 1e-4
out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "demo_subset.npz")
np.savez_compressed(out, ply62=sub, splat60=s, vp=vp, uniforms=np.frombuffer(ub, dtype=np.uint8), keys=fr.keys, values=fr.values,
                    bounds=fr.bounds, rgba=fr.rgba, duplicates=fr.duplicates, visible=fr.visible, width=W, height=H,
                    ref_keys=rf.keys, ref_values=rf.values, ref_bounds=rf.bounds, ref_rgba=rf.rgba, ref_duplicates=rf.duplicates,
                    ref_minted_by="reference shaders resources/shaders/compute/*.glsl executed by oracle/glsl_cpu")
print(out, os.path.getsize(out), "bytes; N", sub.shape[0], "V", fr.visible, "M", fr.duplicates, "C", fr.staged,
      "max|ref_rgba - rgba|", float(np.abs(rf.rgba - fr.rgba).max()))
