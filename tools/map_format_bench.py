"""RGBA32F against RGBA16F maps (wso_set_map_format) on one GPU, in one process.

    python tools/map_format_bench.py [--reps 5] [--steps 20] [--out FILE.jsonl]

Workloads (the benchmark's configurations):
  c2   1024^2 x 100 frames of one tile per step, device-resident (wso_compute_batch)
  c3   2048^2 x 32 frames per step
  c4   64 tiles of 512^2 per step (one frame each)
  c1   one 512^2 frame per call, back to back, through the Python binding (compute_batch of one frame)
  e2e  1024^2 x 24 frames per step into pinned host memory (compute_to_host)
Each workload runs RGBA32F and RGBA16F alternately, `reps` times each, on contexts that stay alive between repetitions,
so that both formats see the same clocks and the spread is visible.  Device throughput is timed with CUDA events on the
compute stream; K1 / K2h / K2 ms come from a separate profiled pass (wso_set_profiling).  One JSON line per (workload,
format) with the device name, its power limit and max SM clock (read-only nvidia-smi query) and the design bytes per
point of the format.  Without a CUDA device the script exits with an error.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FORMATS = ("rgba32f", "rgba16f")
# design bytes per grid point and tile-frame (DESIGN.md §5): K1 32 + K2h 4 + K2 (16 of W + the two map texels: 32 bytes
# in RGBA32F, 16 in RGBA16F) = 84 / 68 for the path
DESIGN_BYTES = {"rgba32f": {"path": 84, "k2": 48}, "rgba16f": {"path": 68, "k2": 32}}
WORKLOADS = {
    "c2": dict(n=1024, frames=100, tiles=1),
    "c3": dict(n=2048, frames=32, tiles=1),
    "c4": dict(n=512, frames=64, tiles=64),
}


def gpu_info():
    import torch
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in out[-1].split(",")]
    except Exception as e:  # the numbers then carry no power limit: say so
        info["power_limit"] = info["max_sm_clock"] = f"unavailable ({e.__class__.__name__})"
    return info


def gauss(n, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))).astype(np.complex64)


def make_ctx(W, stream, n, frames, tiles, fmt):
    ws = W.WSTessendorf(n, 1000.0 * n / 512, max_tiles=tiles, max_slots=max(frames, 2))
    ws.set_map_format(fmt)
    for j in range(tiles):
        ws.SetWindSpeed(20.0 + j * 0.25, j)
        ws.PrepareWithGauss(gauss(n, 100 + j), tile=j)
    ws.set_stream(stream.cuda_stream)
    return ws


def times_of(step, frames):
    return np.float32(step * 0.5) + np.arange(frames, dtype=np.float32) * np.float32(1.0 / 60)


def bench_device(torch, ws, stream, wl, steps, warmup):
    frames, tiles = wl["frames"], wl["tiles"]
    tl = None if tiles == 1 else np.arange(frames, dtype=np.uint32)
    if tiles > 1:
        mk = lambda k: np.full(frames, np.float32(k * 0.5), np.float32)
    else:
        mk = lambda k: times_of(k, frames)
    for k in range(warmup):
        ws.compute_batch(mk(k), tiles=tl)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(steps):
        ws.compute_batch(mk(warmup + k), tiles=tl)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    ws.set_profiling(True)
    for k in range(steps):
        ws.compute_batch(mk(warmup + k), tiles=tl)
    prof = ws.profile()
    ws.set_profiling(False)
    tf = max(prof["tile_frames"], 1)
    return {"tile_frames_per_s": frames * steps / (ms * 1e-3), "us_per_tile_frame": ms * 1e3 / (frames * steps),
            "kernel_us_per_tile_frame": dict(zip(("K1", "K2h", "K2"), [m * 1e3 / tf for m in prof["ms"]]))}


def bench_c1(torch, ws, stream, calls, warmup):
    for k in range(warmup):
        ws.compute_batch([k * 0.01])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    t0 = time.perf_counter()
    for k in range(calls):
        ws.compute_batch([k * 0.01])
    e1.record(stream)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ms = e0.elapsed_time(e1)
    return {"tile_frames_per_s": calls / (ms * 1e-3), "us_per_tile_frame": ms * 1e3 / calls,
            "host_us_per_call": wall * 1e6 / calls}


def bench_e2e(W, ws, n, frames, steps, warmup, fmt):
    dt = np.float16 if fmt == "rgba16f" else np.float32
    disp = W.PinnedBuffer((frames, n, n, 4), dt)
    norm = W.PinnedBuffer((frames, n, n, 4), dt)
    try:
        for k in range(warmup):
            ws.compute_to_host(times_of(k, frames), disp.array, norm.array)
        t0 = time.perf_counter()
        for k in range(steps):
            ws.compute_to_host(times_of(warmup + k, frames), disp.array, norm.array)
        s = time.perf_counter() - t0
    finally:
        disp.close()
        norm.close()
    d2h = 2 * disp.nbytes * steps
    return {"tile_frames_per_s": frames * steps / s, "us_per_tile_frame": s * 1e6 / (frames * steps),
            "d2h_bytes_per_tile_frame": 2 * n * n * 4 * np.dtype(dt).itemsize, "d2h_gb_per_s": d2h / s / 1e9}


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--c1-calls", type=int, default=2000)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        print("map_format_bench: no CUDA device (there is no CPU fallback)", file=sys.stderr)
        return 2
    import watersurfacerendering_b200 as W
    info = gpu_info()
    stream = torch.cuda.Stream(device=0)
    torch.cuda.set_stream(stream)
    runs = {}  # (workload, fmt) -> list of result dicts
    jobs = []
    sizes = {"c1": 512, "e2e": 1024, **{k: v["n"] for k, v in WORKLOADS.items()}}
    for name, wl in WORKLOADS.items():
        ctx = {f: make_ctx(W, stream, wl["n"], wl["frames"], wl["tiles"], f) for f in FORMATS}
        jobs.append((name, wl, ctx, lambda ws, f, wl=wl: bench_device(torch, ws, stream, wl, a.steps, a.warmup)))
    ctx = {f: make_ctx(W, stream, 512, 1, 1, f) for f in FORMATS}
    jobs.append(("c1", dict(n=512, frames=1, tiles=1), ctx,
                 lambda ws, f: bench_c1(torch, ws, stream, a.c1_calls, 50)))
    ctx = {f: make_ctx(W, stream, 1024, 48, 1, f) for f in FORMATS}
    jobs.append(("e2e", dict(n=1024, frames=24, tiles=1), ctx,
                 lambda ws, f: bench_e2e(W, ws, 1024, 24, max(a.steps // 2, 5), 2, f)))
    for name, wl, ctx, fn in jobs:
        for r in range(a.reps):
            for f in (FORMATS if r % 2 == 0 else FORMATS[::-1]):   # alternate which format goes first
                runs.setdefault((name, f), []).append(fn(ctx[f], f))
        for ws in ctx.values():
            ws.close()
    lines = []
    for (name, f), rs in runs.items():
        v = [r["tile_frames_per_s"] for r in rs]
        line = {"workload": name, "format": f, "n": sizes[name],
                "tile_frames_per_s_median": statistics.median(v), "tile_frames_per_s_min": min(v),
                "tile_frames_per_s_max": max(v), "reps": rs,
                "design_bytes_per_point": DESIGN_BYTES[f], **info}
        lines.append(line)
    out = [json.dumps(x) for x in lines]
    print("\n".join(out))
    if a.out:
        with open(a.out, "w") as fh:
            fh.write("\n".join(out) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
