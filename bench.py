#!/usr/bin/env python
"""bench.py -- headline benchmark of the gsr hot path (contract: see the task statement / DESIGN.md section 7).

One "step" = one frame of the hot path: projection -> key duplication -> radix sort -> tile ranges ->
alpha blend, on a synthetic splat cloud already resident in HBM.  Default workload = BASELINE.json
configs[2] ("c3"): 6 M splats, 1920x1080, 1-degree-per-frame orbit (the configuration the north-star target
">= 60 fps on a 6 M-splat scene @1080p on 1xB200" is quoted on).  N > 1 GPUs: screen-tile-row bands, one NCCL
gather of the framebuffer per frame (strong scaling: the frame is fixed, the GPUs split it).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c4] [--impl gsr|reference] [--dump-outputs DIR]

`--impl reference` times the CPU restatement of the reference pipeline (oracle/, all host threads) -- the
reference itself needs Godot 4.3 + a Vulkan device and cannot run on this box (BASELINE.md section 2).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only; nothing is cached into it

WORKLOADS = {
    # name: (N splats, W, H, seed, orbit?)      BASELINE.json configs[1..3]
    "c2": dict(n=1_000_000, w=1920, h=1080, seed=1, orbit=False, desc="1M synthetic Gaussians, SH deg 3, 1920x1080, default camera"),
    "c3": dict(n=6_000_000, w=1920, h=1080, seed=2, orbit=True, desc="6M-splat bicycle-scale synthetic scene, 1920x1080, 360-frame orbit sweep"),
    "c5": dict(n=0, w=0, h=0, seed=5, orbit=False, desc="radix-sort microbench: 2^20..2^28 32-bit tile|depth keys (+u32 values), device resident"),
    "c4": dict(n=10_000_000, w=3840, h=2160, seed=3, orbit=True, desc="10M synthetic splats, 3840x2160 orbit (multi-GPU config of BASELINE.json; sharding named in `parallelism`)"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=360, help="timed frames (default: one full 360-frame orbit)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--workload", default=os.environ.get("GSR_BENCH_WORKLOAD", "c3"), choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="gsr", choices=["gsr", "reference"])
    ap.add_argument("--splats", type=int, default=int(os.environ.get("GSR_BENCH_SPLATS", "0")), help="debug: override N (marks the line reduced)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-radix", action="store_true")
    ap.add_argument("--present", default="rows", choices=["root", "rows"],
                    help="group mode, e2e: 'root' = the frame is assembled on rank 0's device and read back over its PCIe link; 'rows' = every rank "
                         "reads its own tile rows back into one shared page-locked host frame (a PCIe link per GPU)")
    ap.add_argument("--mgpu", default="group", choices=["group", "peer", "nccl"],
                    help="N>1: 'group' (default) = NCCL-free shard group (projection sharded by splats, every rank scatters its pairs and records "
                         "into the row owners' memory over NVLink peer pointers, device-side flags); 'peer' = round-1 path: replicated cull, compositor stores bands into the root's frame over "
                         "NVLink peer memory + 4-byte NCCL sync; 'nccl' = NCCL gather of the band framebuffers")
    ap.add_argument("--overlap", type=int, default=-1, choices=[-1, 0, 1],
                    help="front/back overlap of consecutive frames (gsr_debug_pipeline): -1 = the library's default (off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame the last timed step computed to DIR/*.npy (float32), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.gpus != 1 or args.workload == "c5"):
        ap.error("--dump-outputs: only for one GPU and the frame workloads (c2, c3, c4)")
    return args


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(out_dir, rgba):
    """The RGBA32F frame a caller of the timed path receives, as DIR/rgba.npy.  A frame above 64 MB (c4) is replaced by a fixed
    sample of its pixels: DIR/rgba_sample.npy (k, 4) and their flat pixel indices y * W + x, DIR/rgba_sample_pixel.npy (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    rgba = np.ascontiguousarray(rgba, dtype=np.float32)
    if rgba.nbytes <= DUMP_LIMIT_BYTES:
        np.save(os.path.join(out_dir, "rgba.npy"), rgba)
        return
    px = rgba.reshape(-1, 4)
    k = (DUMP_LIMIT_BYTES - 4096) // (px.itemsize * 4 + 8)   # 4096: the two .npy headers
    idx = np.sort(np.random.default_rng(0).choice(px.shape[0], size=k, replace=False))
    np.save(os.path.join(out_dir, "rgba_sample.npy"), px[idx])
    np.save(os.path.join(out_dir, "rgba_sample_pixel.npy"), idx.astype(np.float64))


def frame_params(wl, n_frames, first=0):
    """Pre-pack (view_proj[32], uniforms bytes) for each frame: util/gaussian_splatting_rasterizer.gd:175-195,126."""
    from godotgaussiansplatting_b200 import camera as cam
    out = []
    aspect = wl["w"] / wl["h"]
    for f in range(first, first + n_frames):
        c = cam.orbit_camera(f % 360, aspect=aspect) if wl["orbit"] else cam.default_camera(aspect=aspect)
        vp = cam.pack_camera_push_constants(c.get_camera_transform(), c.get_camera_projection())
        p = c.global_position
        u = np.zeros(8, dtype=np.float32)
        u[0], u[1], u[2], u[3], u[6] = -p[0], -p[1], p[2], 1.0, 10.0
        raw = bytearray(u.tobytes())
        raw[16:24] = np.array([wl["w"], wl["h"]], dtype=np.int32).tobytes()
        out.append((np.ascontiguousarray(vp), bytes(raw)))
    return out


def raw_chunks(wl):
    """The scene as the 62-float vertex table a .ply of it would hold, chunk by chunk."""
    from godotgaussiansplatting_b200.synthetic import synthetic_ply_chunks
    yield from synthetic_ply_chunks(wl["n"], wl["seed"])


def scene_chunks(wl):
    """Host-side ingest (numpy mirror of util/ply_file.gd:44-69) of the same scene: 60-float Splat structs."""
    from godotgaussiansplatting_b200.ply_file import swizzle_splats
    for lo, blk in raw_chunks(wl):
        yield lo, swizzle_splats(blk, 0.0)


def oracle_scene(wl):
    """CPU-baseline legs only: the oracle's own restatement of the ingest (OpenMP) builds its input."""
    from oracle import oracle as orc
    return np.concatenate([orc.preprocess_ply(blk, 0.0) for _, blk in raw_chunks(wl)])


def make_config(args, wl):
    """`config` of the JSON line: a function of the command line only, so that both arms (--impl gsr / reference) print the
    SAME dict for the same workload and GPU count (the driver compares them).  Run-dependent facts (M, V, C, timings) live
    in `run_info`."""
    if args.gpus == 1:
        par = "single GPU"
    elif args.mgpu == "nccl":
        par = f"tile-row bands x{args.gpus} + NCCL framebuffer gather"
    else:
        par = (f"cyclic tile rows x{args.gpus} (row % {args.gpus} == rank), " +
               ("projection sharded by splats, pairs + records scattered to the row owners over NVLink peer stores, device-side flags (no NCCL on the frame path)" if args.mgpu == "group"
                else "replicated cull with early reject, 4-byte NCCL all-reduce per frame") +
               ", compositor stores into the root frame over NVLink peer memory")
    if args.gpus > 1 and args.mgpu == "group" and args.present == "rows":
        par += "; e2e: every rank reads its own rows back into one shared page-locked host frame (device-resident leg: frame assembled in rank 0's HBM)"
    return {"workload": f"{args.workload}: {wl['desc']}", "splats": wl["n"], "width": wl["w"], "height": wl["h"], "sh_degree": 3,
            "parallelism": par, "reduced": bool(args.splats),
            "l2": "inputs larger than L2 (SoA splats %.0f MB + records + pairs per frame >> 126 MB)" % (240 * wl["n"] / 1e6)}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); pw.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)), "samples": len(sm),
                "reasons": sorted(reasons)}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy, measured on this pool)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def profiled_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed ncu --set full
    capture (profiles/rNN_traffic.json, written by profiles/summarize_ncu.py from the round's .ncu-rep)."""
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")), reverse=True):
        try:
            with open(path) as f:
                d = json.load(f)
            if kernel_key in d:
                return float(d[kernel_key]), os.path.relpath(path, ROOT)
        except Exception:
            continue
    return None, None


def tune_cpu_threads(wl, splat60, frame):
    """Use 'all the host threads it can use': time one frame with every logical CPU this process may run on and with half of
    them (SMT siblings / cgroup quotas often make the full count slower for the OpenMP sort) and keep the faster setting."""
    from oracle import oracle as orc
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    best, best_ms = None, None
    for k in sorted({max(1, avail), max(1, avail // 2)}, reverse=True):
        orc.set_num_threads(k)
        ms, _, _, _ = cpu_reference_frames(wl, splat60, [frame], 1e9)
        ms2, _, _, _ = cpu_reference_frames(wl, splat60, [frame], 1e9)
        if best_ms is None or min(ms[0], ms2[0]) < best_ms:
            best, best_ms = k, min(ms[0], ms2[0])
    orc.set_num_threads(best)
    return best


def cpu_reference_frames(wl, splat60, frames, max_seconds, keep=None):
    """Times the CPU restatement (oracle) on full frames of the workload; returns (ms list, stage dict, threads).
    keep: optional list that receives the oracle's last Frame (pixels, keys, ranges) for the per-run parity check."""
    from oracle import oracle as orc
    ms, stages, info = [], [], None
    t_begin = time.perf_counter()
    for vp, ub in frames:
        u = orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8))
        t0 = time.perf_counter()
        fr = orc.frame(splat60, vp, u)
        ms.append((time.perf_counter() - t0) * 1e3)
        stages.append(fr.stage_ms)
        info = dict(duplicates=fr.duplicates, visible=fr.visible, staged=fr.staged)
        if keep is not None:
            keep[:] = [(vp, ub, fr)]
        if time.perf_counter() - t_begin > max_seconds:
            break
    return ms, stages, orc.num_threads(), info


def run_reference(args, wl, rank, world):
    """--impl reference: the reference's own pipeline on the host cores (CPU restatement; see module docstring)."""
    if rank != 0:
        return
    splat60 = oracle_scene(wl)
    frames = frame_params(wl, args.warmup + args.steps)
    # untimed warm-up (page-in, thread pool, thread-count choice), then the K timed frames
    tune_cpu_threads(wl, splat60, frames[0])
    kept = []
    ms, stages, threads, info = cpu_reference_frames(wl, splat60, frames[args.warmup:args.warmup + args.steps], math.inf, keep=kept)
    mean_ms = float(np.mean(ms))
    value = wl["n"] / 1e6 * 1000.0 / mean_ms
    ref_shaders = reference_shaders_sample(wl, splat60, frames[args.warmup])
    sample = f"{len(ms)} of {args.steps} orbit frames timed in full (all {wl['n']} splats, {wl['w']}x{wl['h']}); CPU restatement of the reference pipeline (Godot/lavapipe unavailable)"
    line = {
        "impl": "reference", "metric": "Msplats/s", "value": value, "unit": "Msplats/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": mean_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "fps": 1000.0 / mean_ms,
        "config": make_config(args, wl), "run_info": {"executed_on": "host threads (CPU restatement of the reference pipeline)"},
        "cpu_baseline": {"value": value, "unit": "Msplats/s", "cores": threads, "kind": "port", "sample": sample,
                         "stage_ms": {k: float(np.mean([s[k] for s in stages])) for k in stages[0]}, **info,
                         "reference_shaders": ref_shaders},
        "e2e": {"value": value, "unit": "Msplats/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, kept[0][2].rgba)


def reference_shaders_sample(wl, splat60, frame, every=4):
    """The reference's OWN shaders (oracle/_ref: the six .glsl files compiled for the CPU, workgroups emulated as fibers on
    one thread) timed on a bounded sample -- every 4th splat of one frame of the workload.  Reported beside the port, not
    instead of it: the port (OpenMP, all cores) is the faster, i.e. the more demanding, CPU baseline and stays `value`."""
    try:
        from oracle import oracle as orc
        from oracle import refshaders
        if not refshaders.available():
            return {"unavailable": "oracle/_ref not built (GSR_REFERENCE_DIR did not name the original project at build time)"}
        sub = np.ascontiguousarray(splat60[::every])
        vp, ub = frame
        spec = orc.frame(sub, vp, orc.uniforms_from_bytes(np.frombuffer(ub, dtype=np.uint8)))
        refshaders.set_shared_fill(int(spec.keys[0] >> 16) if spec.duplicates else 0)
        pipe = refshaders.ReferencePipeline(sub, wl["w"], wl["h"])
        t0 = time.perf_counter()
        rf = pipe.rasterize(vp, ub)
        dt = time.perf_counter() - t0
        same = bool(rf.duplicates == spec.duplicates and np.array_equal(rf.keys, spec.keys) and np.array_equal(rf.bounds, spec.bounds))
        return {"value": sub.shape[0] / 1e6 / dt, "unit": "Msplats/s", "cores": 1, "kind": "reference", "seconds": dt,
                "sample": f"every {every}th splat ({sub.shape[0]}) of one {wl['w']}x{wl['h']} frame through the reference's six compute "
                          "shaders compiled for the CPU (oracle/glsl_cpu: fibers emulate the GPU workgroups; a correctness pin, not a tuned CPU path)",
                "keys_and_ranges_identical_to_port": same, "max_abs_rgba_vs_port": float(np.abs(rf.rgba - spec.rgba).max())}
    except Exception as e:  # the extra measurement must never break the arm
        return {"unavailable": f"{type(e).__name__}: {e}"}


def run_c5(args):
    """--workload c5: the radix-sort microbench as its own JSON line (metric Gkeys/s at the largest size)."""
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- libgsr has no CPU fallback")
    torch.cuda.set_device(0)
    sizes = [20, 22, 24, 26, 28]
    res = {}
    for lg in sizes:
        res[f"2^{lg}"] = radix_microbench(torch, 0, 1 << lg, steps=args.steps, warmup=args.warmup)
    top = res[f"2^{sizes[-1]}"]
    peak, peak_src = measured_peak_gbs()
    emit({"metric": "Gkeys/s", "value": top["pairs"]["gkeys_s"], "unit": "Gpairs/s (32-bit key + 32-bit value)", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
          "ms_per_step": top["pairs"]["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
          "config": {"workload": "c5: " + WORKLOADS["c5"]["desc"], "sizes": res, "l2": "2^26 and 2^28 exceed L2; smaller sizes are L2-resident"},
          "roofline": {"kernel": "sort_hist_kernel + 4x onesweep_kernel", "bound": "hbm", "achieved": top["pairs"]["hbm_frac_of_measured"] * peak, "peak": peak,
                       "unit": "GB/s", "frac": top["pairs"]["hbm_frac_of_measured"], "traffic": None, "peak_source": peak_src,
                       "algorithmic_bytes": "68 B per pair (36 B per key keys-only), SURVEY 8d"},
          "keys_only_gkeys_s": top["keys"]["gkeys_s"], "gpu_launches": 5 * (args.warmup + args.steps) * 2 * len(sizes), "e2e": None, "cpu_baseline": None})


def radix_microbench(torch, device_index, n=1 << 26, steps=3, warmup=1):
    """config c5 point: n (tile<<16|depth16) keys + u32 values, device resident, CUDA events on the sort stream; mean of `steps`
    timed sorts after `warmup` untimed ones."""
    import ctypes as C
    from godotgaussiansplatting_b200 import _lib
    from godotgaussiansplatting_b200.synthetic import radix_keys
    L = _lib.lib()
    keys = torch.from_numpy(radix_keys(n, 5).view(np.int32)).cuda()
    vals = torch.arange(n, dtype=torch.int32, device="cuda")
    s = C.c_void_p()
    _lib.check(L.gsr_sorter_create(device_index, n, C.byref(s)), "gsr_sorter_create")
    out = {}
    try:
        for name, with_vals in (("pairs", True), ("keys", False)):
            best = []
            for it in range(warmup + steps):
                k = keys.clone()
                v = vals.clone() if with_vals else None
                torch.cuda.synchronize()
                _lib.check(L.gsr_sorter_sort_device(s, C.c_void_p(k.data_ptr()), C.c_void_p(v.data_ptr()) if with_vals else None, n,
                                                    C.c_void_p(torch.cuda.current_stream().cuda_stream)), "sort")
                torch.cuda.synchronize()
                ms = C.c_float()
                _lib.check(L.gsr_sorter_last_ms(s, C.byref(ms)), "ms")
                if it >= warmup:
                    best.append(ms.value)
            t = float(np.mean(best))
            out[name] = {"n": n, "ms": t, "gkeys_s": n / t / 1e6, "hbm_frac_of_measured": (n * (68 if with_vals else 36) / (t * 1e-3)) / 1e9 / measured_peak_gbs()[0]}
    finally:
        L.gsr_sorter_destroy(s)
    return out


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """Exactly one JSON line on the process's real stdout (library banners -- e.g. NCCL's version line -- were
    redirected to stderr in main())."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # anything a library prints to fd 1 from here on goes to stderr
    wl = dict(WORKLOADS[args.workload])
    reduced = False
    if args.splats:
        wl["n"], reduced = args.splats, True
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, wl, rank, world)
        return
    if args.workload == "c5":
        if rank == 0:
            run_c5(args)
        return

    import torch
    import torch.distributed as dist
    from godotgaussiansplatting_b200 import build as gsr_build
    from godotgaussiansplatting_b200.camera import default_camera
    from godotgaussiansplatting_b200.ply_file import PlyFile
    from godotgaussiansplatting_b200.rasterizer import GaussianSplattingRasterizer, RenderTexture

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- libgsr has no CPU fallback (use --impl reference for the CPU baseline)")
    if rank == 0:
        gsr_build.build()
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run"
    # one dedicated (non-default) stream carries libgsr's kernels, the NCCL gather and the timing events
    stream = torch.cuda.Stream(priority=-1)   # the render stream outranks libgsr's front stream (next frame's projection): freed SM slots go to the back part first
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0

    from godotgaussiansplatting_b200 import sharding
    W, H, N = wl["w"], wl["h"], wl["n"]
    tiles_y = (H + 15) // 16
    band = sharding.band_partition(tiles_y, world)[rank]
    h_pad = sharding.padded_height(H, world)

    # ---- scene: generated and uploaded chunk by chunk (PlyFile.load_gaussian_splats path, util/ply_file.gd:28-77) ----
    stub = PlyFile()
    stub.size = N
    rast = GaussianSplattingRasterizer(stub, (W, H), RenderTexture(), default_camera(aspect=W / H), device=local_rank)
    rast.init_gpu(load=False)
    rast.set_stream(stream.cuda_stream)
    if args.overlap >= 0:
        rast.debug_pipeline(args.overlap)
    keep_host = rank == 0 and not args.no_cpu_baseline   # N > 1: rank 0 keeps the scene for the one-frame parity check of the assembled frame
    host_chunks = []
    t_gen = time.perf_counter()
    for lo, blk in raw_chunks(wl):
        rast.upload_ply_raw(blk, lo, 0.0)  # device-side ingest (scope row f1): exp/sigmoid/quat->cov/SH interleave on the GPU
        if keep_host:
            host_chunks.append(blk)
    t_gen = time.perf_counter() - t_gen
    fb = None
    group = world > 1 and args.mgpu == "group"
    peer = world > 1 and args.mgpu == "peer"
    sync_flag = torch.zeros(1, dtype=torch.int32, device="cuda") if world > 1 else None
    if group:
        # NCCL-free frame path: every rank exports its arena (flag page + receive segments + record tables) and frames, the blobs are all-gathered
        # ONCE here, and from then on the ranks talk through NVLink peer memory only (include/gsr.h gsr_group_*)
        from godotgaussiansplatting_b200 import _lib as _gl
        mine = torch.frombuffer(bytearray(rast.group_export()), dtype=torch.uint8).cuda()
        blobs = torch.zeros(world * _gl.GSR_GROUP_BLOB_BYTES, dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(blobs, mine)
        rast.group_attach(rank, world, blobs.cpu().numpy().tobytes())
        dist.barrier()
    elif peer:
        # fused compositor + gather: the root exports CUDA-IPC handles of its two frames; every rank's compositor then
        # stores its band directly into the root's memory over NVLink
        handles = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            handles.copy_(torch.frombuffer(bytearray(rast.peer_export()), dtype=torch.uint8))
        dist.broadcast(handles, src=0)
        if rank != 0:
            rast.peer_import(bytes(handles.cpu().numpy().tobytes()))
        rast.set_row_interleave(rank, world)  # balanced: rank r owns tile rows r, r+G, ... ; fast sharded mode

        class _Word:  # the library's int32 "local last occupied tile + 1" word as a torch tensor (all-reduced in place)
            __cuda_array_interface__ = {"shape": (1,), "typestr": "<i4", "data": (rast.band_sync_word_ptr(), False), "version": 2}
        sync_flag = torch.as_tensor(_Word(), device="cuda")
    elif world > 1:  # NCCL gather needs a torch-visible frame
        fb = torch.zeros((h_pad, W, 4), dtype=torch.float32, device="cuda")
        rast.set_framebuffer_external(fb.data_ptr())
        rast.set_band(*band)
    # two page-locked host frames: the application consumes frame i while frame i+1 is being copied
    pinned2 = [torch.empty((H, W, 4), dtype=torch.float32).pin_memory() for _ in range(2)] if rank == 0 else None
    shared2 = None
    if group and args.present == "rows":
        # rows-local presentation: the two host frames live in shared memory, page-locked in EVERY rank's process; each rank copies
        # its own tile rows over its own PCIe link (no frame data on NVLink, one eighth of the frame per link at 8 GPUs)
        shm_names = [None, None]
        if rank == 0:
            shm_names = [f"/dev/shm/gsr_bench_{os.getpid()}_{k}" for k in range(2)]
            for nm in shm_names:
                with open(nm, "wb") as f:
                    f.truncate(H * W * 16)
        dist.broadcast_object_list(shm_names, src=0)
        shared2 = [torch.from_file(nm, shared=True, size=H * W * 4, dtype=torch.float32).view(H, W, 4) for nm in shm_names]
        for t in shared2:
            err = torch.cuda.cudart().cudaHostRegister(t.data_ptr(), t.numel() * 4, 0)
            assert int(err) == 0, f"cudaHostRegister -> {err}"
        dist.barrier()
        if rank == 0:
            for nm in shm_names:
                os.unlink(nm)
    can_pack_rgb = world == 1 or peer or group  # optional RGB32F read-back (alpha == 1.0 stays on the device), reported beside the RGBA headline
    pinned = pinned2[0] if rank == 0 else None

    frames = frame_params(wl, args.warmup + args.steps)

    def step(i, e2e):
        """e2e: False = device-resident frame; "rgba" = the RGBA32F frame the reference's texture holds (rasterizer.gd:92) lands in
        pinned host memory every step; "rgb" = the packed RGB32F variant (alpha is the constant 1.0)."""
        vp, ub = frames[i]
        rgb = e2e == "rgb"
        if world == 1:
            rast.render_raw(vp, ub, 0.0, pinned2[i & 1].data_ptr() if e2e else None, asynchronous=True, rgb_only=rgb)
        elif group:
            rast.render_raw(vp, ub, 0.0, None, asynchronous=True)  # pairs, records and rows travel over NVLink; flags order the ranks on the devices
            if e2e and shared2 is not None and not rgb:
                rast.readback_rows_async(shared2[i & 1].data_ptr())   # every rank: its own rows, its own PCIe link
            elif e2e and rank == 0:
                rast.readback_async(pinned2[i & 1].data_ptr(), rgb_only=rgb)
        elif peer:
            rast.render_raw(vp, ub, 0.0, None, asynchronous=True)  # band lands in the root's frame (slot i & 1) over NVLink
            if e2e and rank == 0:
                rast.stream_join()                                 # previous read-backs done before peers may reuse a slot
            dist.all_reduce(sync_flag, op=dist.ReduceOp.MAX)       # 4-byte sync: all rows have landed + frame-global last tile
            rast.band_fixup()                                      # reference quirk Q10 on the rank that owns that tile
            if e2e and rank == 0:
                rast.readback_async(pinned2[i & 1].data_ptr(), rgb_only=rgb)
        else:
            rast.render_raw(vp, ub, 0.0, None, asynchronous=True)
            sharding.gather_bands(fb, rank, world, dst=0)  # one NCCL gather of the band framebuffers per frame (SURVEY 8e)
            if e2e and rank == 0:
                pinned.copy_(fb[:H], non_blocking=True)

    host_enqueue_ms = {}

    def timed(e2e):
        if group and shared2 is not None:   # RGBA e2e: rows stay local and are read back by their owners; otherwise: frame on rank 0
            torch.cuda.synchronize(); dist.barrier()
            rast.group_set_present(e2e == "rgba")
            dist.barrier()
        for i in range(args.warmup):
            step(i, e2e)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        t_host = time.perf_counter()
        for i in range(args.warmup, args.warmup + args.steps):
            step(i, e2e)
        host_enqueue_ms[str(e2e)] = (time.perf_counter() - t_host) * 1e3 / args.steps   # CPU time spent enqueueing one step (a blocking call shows here)
        if e2e and (world == 1 or ((peer or group) and rank == 0) or (group and shared2 is not None)):
            rast.stream_join()  # the timed region ends when the last frame has landed in host memory
        e1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    sampler = ClockSampler(torch.cuda.current_device() if "CUDA_VISIBLE_DEVICES" not in os.environ else local_rank) if rank == 0 else None
    total_ms = timed(e2e=False)
    clocks = sampler.stop() if sampler else None
    last_frame = rast.read_framebuffer() if args.dump_outputs else None   # the frame of the last timed step (after the stream sync)
    hist = rast.frame_history(min(args.steps, 512))
    st = rast.stats()
    e2e_ms = timed(e2e="rgba")
    hist_e2e = rast.frame_history(min(args.steps, 512))   # the same per-stage GPU timestamps while frames are being read back
    e2e_rgb_ms = timed(e2e="rgb") if can_pack_rgb else None

    ms_per_step = total_ms / args.steps
    stage_total = float(np.mean([r.stage_ms[4] for r in hist]))
    if world == 1 and not (0.5 * stage_total <= ms_per_step):
        raise SystemExit(f"bench.py: loop time {ms_per_step:.3f} ms/frame is below the per-frame stage sum {stage_total:.3f} ms -- events do not bracket the work")
    fps = 1000.0 / ms_per_step
    value = N / 1e6 * fps
    e2e_value = N / 1e6 * 1000.0 / (e2e_ms / args.steps)

    # ---- per-stage means + roofline of the dominant kernel (compositor) over the timed frames ----
    names = ["Projection", "Sort", "Boundaries", "Render", "Total"]
    stage = {nm: float(np.mean([r.stage_ms[i] for r in hist])) for i, nm in enumerate(names)}
    M = float(np.mean([r.duplicates for r in hist])); V = float(np.mean([r.visible for r in hist])); Cc = float(np.mean([r.staged for r in hist]))
    T = st.tiles_x * st.tiles_y
    P = W * H
    peak, peak_src = measured_peak_gbs()
    band_frac = (band[1] - band[0]) / tiles_y
    bytes_proj = 16 * N + 224 * V + 36 * V + 8 * M
    if group:   # this rank's slice of the splats (V = its visible ones); records to one owner at least; pairs stored once (M: received ~ emitted) + packed (16 M)
        bytes_proj = 16 * N / world + 224 * V + 48 * V + 8 * M + 16 * M
    bytes_sort = 68 * M
    bytes_ranges = 4 * M + 8 * T * band_frac
    bytes_comp = 40 * Cc + 16 * P * band_frac + 8 * T * band_frac

    def gbs(b, ms):
        return b / (ms * 1e-3) / 1e9 if ms > 0 else 0.0

    dominant = max(("Projection", "Sort", "Render"), key=lambda k: stage[k])
    dom_bytes = {"Projection": bytes_proj, "Sort": bytes_sort, "Render": bytes_comp}[dominant]
    proj_name = "projection_scatter_kernel + segment wait + gather_segments_kernel" if group else "projection_kernel"
    traffic, traffic_src = profiled_traffic({"Projection": "projection_kernel", "Sort": "onesweep_kernel", "Render": "composite_kernel"}[dominant])
    if group and dominant == "Projection":
        traffic, traffic_src = None, "no single-GPU ncu capture of the scatter projection (its stores go to peer memory)"
    roofline = {"kernel": {"Projection": proj_name, "Sort": "sort_hist_kernel + 4x onesweep_kernel", "Render": "composite_kernel"}[dominant],
                "bound": "hbm", "achieved": gbs(dom_bytes, stage[dominant]), "peak": peak, "unit": "GB/s",
                "frac": gbs(dom_bytes, stage[dominant]) / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "note": ("the compositor is FP32-issue/FMA-pipe bound, not HBM bound (ncu: FMA pipe ~55-70 % of active cycles, DRAM 4 %); its HBM "
                         "fraction is reported because the contract asks for it; see per_stage for the HBM-bound kernels") if dominant == "Render" else None,
                "algorithmic_bytes_per_launch": dom_bytes, "avg_launch_ms": stage[dominant],
                "timing": "CUDA events recorded by libgsr on the render stream around every stage of every timed frame (gsr_get_frame_history)",
                "per_stage": {
                    "projection": {"ms": stage["Projection"], "GB/s": gbs(bytes_proj, stage["Projection"]), "frac": gbs(bytes_proj, stage["Projection"]) / peak, "bytes": bytes_proj},
                    "sort": {"ms": stage["Sort"], "GB/s": gbs(bytes_sort, stage["Sort"]), "frac": gbs(bytes_sort, stage["Sort"]) / peak, "bytes": bytes_sort, "gpairs_s": M / stage["Sort"] / 1e6 if stage["Sort"] > 0 else 0.0},
                    "ranges": {"ms": stage["Boundaries"], "GB/s": gbs(bytes_ranges, stage["Boundaries"]), "frac": gbs(bytes_ranges, stage["Boundaries"]) / peak, "bytes": bytes_ranges},
                    "compositor": {"ms": stage["Render"], "GB/s": gbs(bytes_comp, stage["Render"]), "frac": gbs(bytes_comp, stage["Render"]) / peak, "bytes": bytes_comp,
                                   "pair_evals_per_s": Cc * 256 / (stage["Render"] * 1e-3) if stage["Render"] > 0 else 0.0}}}

    radix = None
    if rank == 0 and not args.no_radix:
        try:
            radix = radix_microbench(torch, local_rank)
        except Exception as e:  # the headline number must survive a microbench failure
            radix = {"error": str(e)}

    cpu_baseline = None
    parity = {"checked": False, "why": "no oracle leg on this run (NCCL-gather mode or --no-cpu-baseline)"}
    if world > 1 and (group or peer):
        # ---- multi-GPU self-check: one more frame through the same path, assembled on rank 0, against the oracle ----
        vp_c, ub_c = frames[args.warmup]
        got_t = torch.zeros((H, W, 4), dtype=torch.float32).pin_memory() if rank == 0 else None
        torch.cuda.synchronize(); dist.barrier()
        if group and shared2 is not None:
            rast.group_set_present(False); dist.barrier()
        rast.render_raw(vp_c, ub_c, 0.0, None, asynchronous=True)
        if peer:
            if rank == 0:
                rast.stream_join()
            dist.all_reduce(sync_flag, op=dist.ReduceOp.MAX)
            rast.band_fixup()
        if rank == 0:
            rast.readback_async(got_t.data_ptr())
        rast.sync(); torch.cuda.synchronize(); dist.barrier()
        if keep_host:
            from oracle import oracle as orc
            splat60 = np.concatenate([orc.preprocess_ply(blk, 0.0) for blk in host_chunks])
            del host_chunks
            ref = orc.frame(splat60, vp_c, orc.uniforms_from_bytes(np.frombuffer(ub_c, dtype=np.uint8)))
            got = got_t.numpy()
            parity = {"checked": True, "against": "oracle, same camera, full workload; frame assembled on rank 0 from all ranks' rows",
                      "rgba_max_abs_err": float(np.abs(got - ref.rgba).max()),
                      "rgba_bit_identical": bool(np.array_equal(got.view(np.uint32), ref.rgba.view(np.uint32))),
                      "duplicates_M_oracle": int(ref.duplicates), "keys_equal": None, "ranges_equal": None,
                      "note": "per-rank sorted pairs vs the oracle's owned rows are checked by tests/test_gpu_multi.py and tests/test_gpu_group.py"}
            del splat60, ref
            if not parity["rgba_max_abs_err"] <= 1e-4:
                raise SystemExit(f"bench.py: PARITY FAILURE of the assembled multi-GPU frame against the oracle: {parity}")
    elif keep_host and world == 1:
        from oracle import oracle as orc
        splat60 = np.concatenate([orc.preprocess_ply(blk, 0.0) for blk in host_chunks])
        del host_chunks
        tune_cpu_threads(wl, splat60, frames[0])  # warm-up + thread-count choice
        kept = []
        ms, stages, threads, info = cpu_reference_frames(wl, splat60, frames[args.warmup:args.warmup + 3], 30.0, keep=kept)
        cpu_ms = float(np.mean(ms))
        # ---- self-check of this very run: the last oracle frame against a GPU frame of the same camera, through the C-ABI ----
        vp_c, ub_c, ref = kept[0]
        got = np.empty((H, W, 4), dtype=np.float32)
        rast.sync()
        rast.render_raw(vp_c, ub_c, 0.0, got.ctypes.data, asynchronous=False)
        stp = rast.stats()
        m = int(min(stp.duplicates, stp.capacity))
        from godotgaussiansplatting_b200 import _lib as _gl
        gk = rast.debug_copy(_gl.GSR_BUF_KEYS, m, np.uint32); gv = rast.debug_copy(_gl.GSR_BUF_VALUES, m, np.uint32)
        gb = rast.debug_copy(_gl.GSR_BUF_BOUNDS, 2 * T, np.uint32).reshape(T, 2)
        parity = {"checked": True, "against": "oracle (CPU restatement pinned to the reference's shaders), same camera, full workload",
                  "keys_equal": bool(m == ref.keys.size and np.array_equal(gk, ref.keys)),
                  "values_equal": bool(m == ref.values.size and np.array_equal(gv, ref.values)),
                  "ranges_equal": bool(np.array_equal(gb, ref.bounds)),
                  "rgba_max_abs_err": float(np.abs(got - ref.rgba).max()),
                  "rgba_bit_identical": bool(np.array_equal(got.view(np.uint32), ref.rgba.view(np.uint32))),
                  "duplicates_M": int(stp.duplicates), "staged_C": int(stp.staged)}
        del gk, gv, gb, got, kept
        if not (parity["keys_equal"] and parity["values_equal"] and parity["ranges_equal"] and parity["rgba_max_abs_err"] <= 1e-4):
            raise SystemExit(f"bench.py: PARITY FAILURE against the oracle on the benchmarked workload: {parity}")
        cpu_baseline = {"value": N / 1e6 * 1000.0 / cpu_ms, "unit": "Msplats/s", "cores": threads, "kind": "port", "ms_per_frame": cpu_ms,
                        "sample": f"{len(ms)} full orbit frame(s) of the same workload (all {N} splats, {W}x{H}); CPU restatement of the reference pipeline, Godot/lavapipe unavailable",
                        "stage_ms": {k: float(np.mean([s[k] for s in stages])) for k in stages[0]}}

    if rank == 0:
        line = {
            "metric": "Msplats/s", "value": value, "unit": "Msplats/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "fps": fps,
            "config": make_config(args, wl),
            "run_info": {"duplicates_M": M, "visible_V": V, "staged_C": Cc, "scene_build_s": t_gen,
                         "frame_overlap": ("on" if args.overlap == 1 else "off") +
                                          ": projection of frame f+1 beside the compositor of frame f (gsr_debug_pipeline; stage_ms are per-stage GPU times, their sum exceeds the frame period when on)"},
            "e2e": {"value": e2e_value, "unit": "Msplats/s", "ms_per_step": e2e_ms / args.steps, "fps": 1000.0 / (e2e_ms / args.steps),
                    "h2d_bytes_per_step": 160, "d2h_bytes_per_step": P * 16,
                    "stage_ms": {nm: float(np.mean([r.stage_ms[i] for r in hist_e2e])) for i, nm in enumerate(names)},
                    "host_enqueue_ms_per_step": host_enqueue_ms,
                    "path": "gsr_render_async(ctx, view_proj, uniforms, pinned host RGBA32F) per frame -- the frame the reference's RGBA32F texture holds (rasterizer.gd:92); 160 B of camera constants in, full frame out; read-back of frame i overlaps frame i+1 (two device + two host frames); timed region ends after the last frame landed on the host",
                    "rgb32f_packed": None if e2e_rgb_ms is None else {
                        "value": N / 1e6 * 1000.0 / (e2e_rgb_ms / args.steps), "fps": 1000.0 / (e2e_rgb_ms / args.steps), "d2h_bytes_per_step": P * 12,
                        "path": "gsr_render_async_rgb: RGB32F pack on the copy stream (alpha is the constant 1.0 of gsplat_render.glsl:101)"}},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "parity": parity, "clocks": clocks,
            "gpu_launches": int(st.kernel_launches) * args.steps, "kernel_launches_per_frame": int(st.kernel_launches),
            "stage_ms": stage, "radix": radix,
            "reference_published": {"fps": 108, "scene": "bicycle.ply ~6.1M splats @1080p", "hw": "RTX 3060 Ti", "source": "README.md:58 (other hardware; not comparable)"},
        }
        emit(line)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_frame)
    rast.cleanup_gpu()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
