"""Surface-query throughput (wso_query_surface) on one GPU, in one process.

    python tools/surface_query_bench.py [--reps 5] [--calls 20] [--out FILE.jsonl]

n = 2^20 queries per call, for every combination of
  tile size N in {512, 1024};  1 cascade (L = 1000) or 3 (L = 1000, 250, 61);  I in {0, 4} inversion steps;
  map format RGBA32F / RGBA16F;  queries uniform random over a 4L x 4L area (L = 1000) or on a regular 1024 x 1024 grid
  over the same area, row by row (coherent: neighbouring threads read neighbouring texels).
Both formats run alternately, `reps` times each, on contexts that stay alive between repetitions.  Each repetition is
`calls` back-to-back calls on the context's stream between two CUDA events, after a warm-up.  For scale, the same run
times one 1024^2 wso_compute_batch frame (1 tile, RGBA32F, one frame per call, back to back).  One JSON line per
configuration with the device name, its power limit and max SM clock (read-only nvidia-smi query).  Without a CUDA
device the script exits with an error.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from map_format_bench import gpu_info  # noqa: E402

FORMATS = ("rgba32f", "rgba16f")
CASCADE_L = (1000.0, 250.0, 61.0)
NQ = 1 << 20


def make_ctx(W, stream, n, fmt):
    ws = W.WSTessendorf(n, CASCADE_L[0], max_tiles=len(CASCADE_L), max_slots=len(CASCADE_L))
    ws.set_map_format(fmt)
    for t, L in enumerate(CASCADE_L):
        ws.SetTileLength(L, t)
        ws.Prepare(seed=11 + t, tile=t)
    ws.set_stream(stream.cuda_stream)
    ws.compute_batch(np.full(len(CASCADE_L), 7.25, np.float32), tiles=np.arange(len(CASCADE_L), dtype=np.uint32))
    return ws


def query_sets(torch):
    area = 4 * CASCADE_L[0]
    rng = np.random.default_rng(1)
    rand = rng.uniform(0.0, area, (NQ, 2)).astype(np.float32)
    side = int(round(NQ ** 0.5))
    g = (np.arange(side, dtype=np.float64) + 0.5) * (area / side)
    X, Z = np.meshgrid(g, g, indexing="xy")
    grid = np.stack([X.ravel(), Z.ravel()], -1).astype(np.float32)
    return {"random": torch.from_numpy(rand).cuda(), "grid": torch.from_numpy(grid).cuda()}


def time_queries(torch, ws, stream, xz, out, slots, iters, calls, warmup):
    for _ in range(warmup):
        ws.query_surface_device(xz.data_ptr(), out.data_ptr(), NQ, slots=slots, iterations=iters)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(calls):
        ws.query_surface_device(xz.data_ptr(), out.data_ptr(), NQ, slots=slots, iterations=iters)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / calls
    return {"us_per_call": ms * 1e3, "queries_per_s": NQ / (ms * 1e-3)}


def time_compute_frame(torch, W, stream, calls=200, warmup=20):
    with W.WSTessendorf(1024, CASCADE_L[0]) as ws:
        ws.Prepare(seed=1)
        ws.set_stream(stream.cuda_stream)
        for k in range(warmup):
            ws.compute_batch([k * 0.01])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for k in range(calls):
            ws.compute_batch([k * 0.01])
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / calls


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        print("surface_query_bench: no CUDA device (there is no CPU fallback)", file=sys.stderr)
        return 2
    import watersurfacerendering_b200 as W
    info = gpu_info()
    stream = torch.cuda.Stream(device=0)
    torch.cuda.set_stream(stream)
    qs = query_sets(torch)
    out = torch.empty((NQ, 8), dtype=torch.float32, device="cuda")
    lines = []
    frame_us = time_compute_frame(torch, W, stream)
    for n in (512, 1024):
        ctx = {f: make_ctx(W, stream, n, f) for f in FORMATS}
        for ncasc in (1, 3):
            slots = tuple(range(ncasc))
            for iters in (0, 4):
                for pattern, xz in qs.items():
                    runs = {f: [] for f in FORMATS}
                    for r in range(a.reps):
                        for f in (FORMATS if r % 2 == 0 else FORMATS[::-1]):   # alternate which format goes first
                            runs[f].append(time_queries(torch, ctx[f], stream, xz, out, slots, iters, a.calls, a.warmup))
                    for f in FORMATS:
                        v = [x["queries_per_s"] for x in runs[f]]
                        med = statistics.median(v)
                        lines.append({"n": n, "cascades": ncasc, "iterations": iters, "format": f, "queries": pattern,
                                      "batch": NQ, "queries_per_s_median": med, "queries_per_s_min": min(v),
                                      "queries_per_s_max": max(v), "us_per_call_median": NQ / med * 1e6,
                                      "texel_gathers_per_query": 4 * ncasc * (iters + 2),
                                      "compute_batch_1024_us_per_frame": frame_us, "reps": runs[f], **info})
        for ws in ctx.values():
            ws.close()
    text = [json.dumps(x) for x in lines]
    print("\n".join(text))
    if a.out:
        with open(a.out, "w") as fh:
            fh.write("\n".join(text) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
