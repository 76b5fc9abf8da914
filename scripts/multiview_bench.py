"""Stereo (and 4-view) frames in one multiview context vs one single-view context per eye, on one GPU.

Scene: bench.py's c3 workload (6 M synthetic splats, seed 2), 1920x1080 per eye, the 360-step orbit of bench.py with a stereo eye pair
(ipd 0.063, asymmetric per-eye frusta as an XR runtime hands them) at every step.  Arms, alternated in the same process on one CUDA
stream, device-resident (frames stay on the GPU, like an XR compositor's swapchain images):
  (a) gsr_render_views with K = 2 in one context;
  (b) two single-view contexts, one gsr_render (asynchronous, no host copy) each per step.
Secondary: K = 4 at 1920x1080 (two stereo pairs) against four single-view frames of one context.
Prints one JSON line: ms per stereo frame of both arms and their ratio, per-stage ms (gsr_get_frame_history), the K = 4 line, a bit-for-bit
parity flag of the last stereo frame against the two mono frames, and the card's name and power limit read in the same run.

  python scripts/multiview_bench.py [--steps 360] [--warmup 20] [--rounds 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from godotgaussiansplatting_b200 import _lib  # noqa: E402
from godotgaussiansplatting_b200 import camera as cam  # noqa: E402
from godotgaussiansplatting_b200.ply_file import swizzle_splats  # noqa: E402
from godotgaussiansplatting_b200.synthetic import synthetic_ply_chunks  # noqa: E402

N, W, H, SEED = 6_000_000, 1920, 1080, 2   # bench.py WORKLOADS["c3"]
STAGES = ["Projection", "Sort", "Boundaries", "Render", "Total"]


def eye_projection(offset, aspect=W / H, near=0.05, far=4000.0, fov=75.0):
    top = near * np.tan(np.radians(fov / 2.0))
    right = top * aspect
    return cam.frustum(-right + offset * right, right + offset * right, -top, top, near, far)


def uniforms(pos):
    u = np.zeros(8, dtype=np.float32)
    u[0], u[1], u[2], u[3], u[6] = -pos[0], -pos[1], pos[2], 1.0, 10.0
    raw = bytearray(u.tobytes())
    raw[16:24] = np.array([W, H], dtype=np.int32).tobytes()
    return bytes(raw)


def eye_views(step, heads=(0,)):
    """Push constants + uniform blocks of the stereo eyes of orbit step `step` (one pair per head offset, in degrees)."""
    vps, ubs = [], []
    for off in heads:
        head = cam.orbit_camera((step + off) % 360, aspect=W / H)
        for eye, shift in zip(cam.stereo_pair(head, 0.063), (0.1, -0.1)):
            vps.append(cam.pack_camera_push_constants(eye.get_camera_transform(), eye_projection(shift)))
            ubs.append(uniforms(eye.global_position))
    return vps, ubs


class Ctx:
    def __init__(self, splat_chunks, stream, views=1):
        self.L = _lib.lib()
        self.h = C.c_void_p()
        _lib.check(self.L.gsr_create(C.byref(_lib.GsrConfig(0, 0, N, 10, 0)), C.byref(self.h)), "gsr_create")
        _lib.check(self.L.gsr_resize(self.h, W, H), "gsr_resize")
        _lib.check(self.L.gsr_set_stream(self.h, C.c_void_p(stream)), "gsr_set_stream")
        for lo, s in splat_chunks:
            _lib.check(self.L.gsr_upload_splats_aos(self.h, s.ctypes.data_as(C.POINTER(C.c_float)), lo, s.shape[0]), "upload")
        if views > 1:
            _lib.check(self.L.gsr_set_views(self.h, views), "gsr_set_views")
        self.views = views

    def render(self, vps, ubs):
        vp = np.ascontiguousarray(np.concatenate(vps), dtype=np.float32)
        fp = vp.ctypes.data_as(C.POINTER(C.c_float))
        if self.views > 1:
            _lib.check(self.L.gsr_render_views_async(self.h, fp, b"".join(ubs), 0.0, None, 0), "gsr_render_views_async")
        else:
            _lib.check(self.L.gsr_render_async(self.h, fp, ubs[0], 0.0, None), "gsr_render_async")

    def frame(self):
        out = np.empty((self.views, H, W, 4), dtype=np.float32)
        _lib.check(self.L.gsr_debug_copy(self.h, _lib.GSR_BUF_FRAMEBUFFER, C.c_void_p(out.ctypes.data), out.nbytes), "gsr_debug_copy")
        return out

    def history(self, n):
        buf = (_lib.GsrFrameRecord * n)()
        got = C.c_uint32(0)
        _lib.check(self.L.gsr_get_frame_history(self.h, n, buf, C.byref(got)), "gsr_get_frame_history")
        recs = [buf[i] for i in range(got.value)]
        out = {nm: float(np.mean([r.stage_ms[i] for r in recs])) for i, nm in enumerate(STAGES)}
        out["M"] = float(np.mean([r.duplicates for r in recs]))
        out["V"] = float(np.mean([r.visible for r in recs]))
        return out

    def close(self):
        self.L.gsr_destroy(self.h)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0], "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, plimit, clk = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": plimit, "sm_clock_max": clk}
    except Exception as e:   # the line still carries torch's device name
        return {"unavailable": f"{type(e).__name__}: {e}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=360)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the two arms (a b, b a, a b, ...)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("multiview_bench.py: no CUDA device (there is no CPU fallback)")
    stream = torch.cuda.Stream()
    chunks = [(lo, np.ascontiguousarray(swizzle_splats(blk, 0.0))) for lo, blk in synthetic_ply_chunks(N, SEED)]
    stereo = Ctx(chunks, stream.cuda_stream, views=2)
    monos = [Ctx(chunks, stream.cuda_stream), Ctx(chunks, stream.cuda_stream)]
    quad = Ctx(chunks, stream.cuda_stream, views=4)
    del chunks
    steps = [eye_views(i) for i in range(args.warmup + args.steps)]
    steps4 = [eye_views(i, heads=(0, 90)) for i in range(args.warmup + args.steps)]

    def arm_stereo(i):
        stereo.render(*steps[i])

    def arm_monos(i):
        vps, ubs = steps[i]
        monos[0].render(vps[:1], ubs[:1])
        monos[1].render(vps[1:], ubs[1:])

    def arm_quad(i):
        quad.render(*steps4[i])

    def arm_quad_mono(i):
        vps, ubs = steps4[i]
        for v in range(4):
            monos[0].render(vps[v:v + 1], ubs[v:v + 1])

    def timed(fn):
        with torch.cuda.stream(stream):
            for i in range(args.warmup):
                fn(i)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for i in range(args.warmup, args.warmup + args.steps):
                fn(i)
            e1.record(stream)
            torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    res = {"a": [], "b": [], "k4": [], "k4_mono": []}
    hist = {}
    for r in range(args.rounds):
        order = [("a", arm_stereo), ("b", arm_monos)] if r % 2 == 0 else [("b", arm_monos), ("a", arm_stereo)]
        for name, fn in order:
            res[name].append(timed(fn))
            if name == "a":
                hist["stereo_context"] = stereo.history(min(args.steps, 512))
            else:
                hist["mono_left"] = monos[0].history(min(args.steps, 512))
                hist["mono_right"] = monos[1].history(min(args.steps, 512))
    # parity of the last stereo frame (step warmup + steps - 1) against the two mono frames of the same step
    last = args.warmup + args.steps - 1
    arm_stereo(last); arm_monos(last)
    torch.cuda.synchronize()
    lay = stereo.frame()
    parity = bool(np.array_equal(lay[0].view(np.uint32), monos[0].frame()[0].view(np.uint32)) and
                  np.array_equal(lay[1].view(np.uint32), monos[1].frame()[0].view(np.uint32)))
    for r in range(args.rounds):
        order = [("k4", arm_quad), ("k4_mono", arm_quad_mono)] if r % 2 == 0 else [("k4_mono", arm_quad_mono), ("k4", arm_quad)]
        for name, fn in order:
            res[name].append(timed(fn))
    hist["quad_context"] = quad.history(min(args.steps, 512))
    for c in [stereo, quad] + monos:
        c.close()

    med = {k: float(np.median(v)) for k, v in res.items()}
    line = {
        "workload": f"c3 scene ({N} splats, seed {SEED}), {W}x{H} per eye, {args.steps}-step orbit, stereo eyes ipd 0.063, off-axis frusta; "
                    f"device-resident, {args.warmup} warm-up steps, {args.rounds} alternated rounds per arm (median)",
        "stereo_ms": {"a_render_views_k2": med["a"], "b_two_single_view_contexts": med["b"], "ratio_a_over_b": med["a"] / med["b"],
                      "rounds_a": res["a"], "rounds_b": res["b"]},
        "stage_ms": hist,
        "k4_ms": {"render_views_k4": med["k4"], "four_single_view_frames": med["k4_mono"], "ratio": med["k4"] / med["k4_mono"],
                  "rounds_k4": res["k4"], "rounds_four_single": res["k4_mono"]},
        "parity_last_stereo_frame_bitwise": parity,
        "device": torch.cuda.get_device_name(0),
        "card": card(),
    }
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
