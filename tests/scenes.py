"""Shared scene builders for the tests (synthetic clouds -> splat60, cameras -> push constants + uniforms)."""
from __future__ import annotations

import numpy as np

from godotgaussiansplatting_b200 import camera as cam
from godotgaussiansplatting_b200.ply_file import swizzle_splats
from godotgaussiansplatting_b200.synthetic import synthetic_ply_table


def make_scene(n: int, seed: int, width: int, height: int, frame: int | None = None, time: float = 10.0, model_scale: float = 1.0,
               creation_time: float = 0.0, scale_boost: float = 0.0):
    """Returns (splat60, vp32, uniforms_bytes). frame=None -> default camera, else orbit frame."""
    table = synthetic_ply_table(n, seed)
    if scale_boost:
        table[:, 55:58] += scale_boost
    splat60 = swizzle_splats(table, creation_time)
    c = cam.default_camera(aspect=width / height) if frame is None else cam.orbit_camera(frame, aspect=width / height)
    vp = cam.pack_camera_push_constants(c.get_camera_transform(), c.get_camera_projection())
    return splat60, vp, uniforms_bytes(c.global_position, model_scale, width, height, time)


def uniforms_bytes(cam_pos, model_scale, width, height, time) -> bytes:
    buf = np.zeros(8, dtype=np.float32)
    buf[0], buf[1], buf[2], buf[3] = -cam_pos[0], -cam_pos[1], cam_pos[2], model_scale
    buf[6] = time
    raw = bytearray(buf.tobytes())
    raw[16:24] = np.array([width, height], dtype=np.int32).tobytes()
    return bytes(raw)


def demo_subset_scene():
    """Every 33rd splat of the original project's resources/demo.ply (tests/golden/demo_subset.npz, 8216 splats) through the
    ingest restatement of the oracle, at the reference's default camera, 640x480.  Returns (ply62, splat60, vp32, uniforms_bytes)."""
    import os

    from oracle import oracle as orc
    with np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "demo_subset.npz")) as g:
        ply62 = g["ply62"]
    c = cam.default_camera(aspect=640 / 480)
    vp = cam.pack_camera_push_constants(c.get_camera_transform(), c.get_camera_projection())
    return ply62, orc.preprocess_ply(ply62, 0.0), vp, uniforms_bytes([0.0, 0.0, 0.0], 1.0, 640, 480, 10.0)
