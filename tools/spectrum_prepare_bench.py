"""Wave spectra (wso_set_spectrum): device Prepare time per kind and per-frame throughput of spectrum tiles, one GPU, one
process.

    python tools/spectrum_prepare_bench.py [--reps 7] [--out-dir profiles] [--tag r7_spectrum]

1. Device Prepare (wso_prepare_counter, counter-generated xi) of one tile at N in {1024, 4096, 8192}, L = 1000 N / 512,
   U = 20 m/s, for Phillips (the existing kernel) and Pierson-Moskowitz / JONSWAP / TMA (d = 30 m) (the spectrum
   kernel).  Each call ends in a stream synchronise; the time is the host clock around the whole call (wave numbers, the
   host's table decision, the launch, the kernel).  Kinds alternate within every repetition; median and min of `reps`.
2. Per-frame throughput of a 1024^2 batch (64 tile-frames per wso_compute_batch, `calls` calls between two
   synchronisations): a Phillips tile (L = 1000), a JONSWAP tile on K1's sincos-table path (L = 1000) and a JONSWAP
   tile on K1's general body (L = 20 m: the largest |k| quantises to j > 1024).  The three contexts alternate within
   every repetition.
One JSON line per measurement plus a header line with the device name, its power limit and max SM clock (read-only
nvidia-smi query), and a Markdown table.  Without a CUDA device the script exits with an error.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from map_format_bench import gpu_info  # noqa: E402

KINDS = ("phillips", "pierson_moskowitz", "jonswap", "tma")
PREP_SIZES = (1024, 4096, 8192)
BATCH = 64


def prepare_ctx(W, n, kind):
    ws = W.WSTessendorf(n, 1000.0 * n / 512)
    ws.SetWindSpeed(20.0)
    if kind != "phillips":
        ws.set_spectrum(kind, depth=30.0 if kind == "tma" else np.inf)
    return ws


def bench_prepare(W, reps):
    rows = []
    for n in PREP_SIZES:
        ctxs = {k: prepare_ctx(W, n, k) for k in KINDS}
        for k, ws in ctxs.items():
            ws.PrepareCounterOnDevice(1)   # warm-up: module load, first allocation
        times = {k: [] for k in KINDS}
        for r in range(reps):
            for k, ws in ctxs.items():
                t0 = time.perf_counter()
                ws.PrepareCounterOnDevice(2 + r)
                times[k].append((time.perf_counter() - t0) * 1e3)
        for k in KINDS:
            rows.append(dict(part="prepare", n=n, kind=k, ms_median=round(statistics.median(times[k]), 4),
                             ms_min=round(min(times[k]), 4), reps=reps))
        for ws in ctxs.values():
            ws.close()
    return rows


def batch_ctx(W, kind, length, U):
    ws = W.WSTessendorf(1024, length, max_slots=BATCH)
    ws.SetWindSpeed(U)
    if kind != "phillips":
        ws.set_spectrum(kind)
    ws.PrepareCounterOnDevice(3)
    h0 = ws.ExportH0()
    w0 = np.float64(np.float32(2.0 * np.pi / np.float32(ws.GetAnimationPeriod())))
    jmax = int(np.max(np.rint(h0["omega"].astype(np.float64) / w0)))
    return ws, jmax


def bench_frames(W, reps, calls):
    cases = {"phillips L=1000": ("phillips", 1000.0, 30.0), "jonswap table L=1000": ("jonswap", 1000.0, 14.0),
             "jonswap general L=20": ("jonswap", 20.0, 3.0)}
    ctxs = {name: batch_ctx(W, *c) for name, c in cases.items()}
    t = (np.arange(BATCH, dtype=np.float32) * np.float32(1 / 60.0)).astype(np.float32)
    for ws, _ in ctxs.values():   # warm-up
        for _ in range(3):
            ws.compute_batch(t)
        ws.sync()
    rates = {name: [] for name in ctxs}
    for _ in range(reps):
        for name, (ws, _) in ctxs.items():
            ws.sync()
            t0 = time.perf_counter()
            for _ in range(calls):
                ws.compute_batch(t)
            ws.sync()
            rates[name].append(calls * BATCH / (time.perf_counter() - t0))
    rows = []
    for name, (ws, jmax) in ctxs.items():
        rows.append(dict(part="frames", n=1024, case=name, jmax=jmax, table=jmax < 1024,
                         tile_frames_per_s_median=round(statistics.median(rates[name]), 1),
                         tile_frames_per_s_max=round(max(rates[name]), 1), reps=reps, calls=calls, batch=BATCH))
        ws.close()
    return rows


def markdown(info, rows):
    out = [f"Device: {info['device']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}.", "",
           "Device Prepare (wso_prepare_counter), ms per call, median (min):", "",
           "| N | " + " | ".join(KINDS) + " |", "|---|" + "---|" * len(KINDS)]
    for n in PREP_SIZES:
        cells = []
        for k in KINDS:
            r = next(r for r in rows if r["part"] == "prepare" and r["n"] == n and r["kind"] == k)
            cells.append(f"{r['ms_median']:.3f} ({r['ms_min']:.3f})")
        out.append(f"| {n} | " + " | ".join(cells) + " |")
    out += ["", f"1024^2 batches of {BATCH} tile-frames, tile-frames/s, median (max):", "",
            "| tile | j max | K1 body | tile-frames/s |", "|---|---|---|---|"]
    for r in rows:
        if r["part"] == "frames":
            out.append(f"| {r['case']} | {r['jmax']} | {'table' if r['table'] else 'general'} | "
                       f"{r['tile_frames_per_s_median']:.0f} ({r['tile_frames_per_s_max']:.0f}) |")
    return "\n".join(out) + "\n"


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out-dir", default=None, help="write <tag>.jsonl and <tag>.md there")
    ap.add_argument("--tag", default="r7_spectrum")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("spectrum_prepare_bench: no CUDA device")
    import watersurfacerendering_b200 as W
    info = gpu_info()
    rows = bench_prepare(W, a.reps) + bench_frames(W, a.reps, a.calls)
    lines = [json.dumps(dict(part="header", **info))] + [json.dumps(r) for r in rows]
    md = markdown(info, rows)
    print("\n".join(lines))
    print(md)
    if a.out_dir:
        os.makedirs(a.out_dir, exist_ok=True)
        with open(os.path.join(a.out_dir, a.tag + ".jsonl"), "w") as f:
            f.write("\n".join(lines) + "\n")
        with open(os.path.join(a.out_dir, a.tag + ".md"), "w") as f:
            f.write(md)


if __name__ == "__main__":
    main()
