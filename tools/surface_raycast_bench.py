"""Ray-cast throughput (wso_raycast_surface) on one GPU, in one process.

    python tools/surface_raycast_bench.py [--reps 3] [--out FILE.jsonl]

For every combination of
  tile size N in {512, 1024};  1 cascade (L = 1000) or 3 (L = 1000, 250, 61);  I in {0, 4} inversion steps;
  map format RGBA32F / RGBA16F (alternating);  two ray sets:
    projectile: origins 5-50 m up over a 4L x 4L area (L = 1000), directions 10-80 degrees below the horizon, tmax = 500;
    grazing:    the same origins, 1-5 degrees below the horizon, tmax = 500;
  4096 rays per call (a physics step) and 2^20 (throughput),
with step = the smallest texel spacing of the cascades (L_min / N), max_steps = 1024, refine = 16.  Each repetition is
`calls` back-to-back calls on the context's stream between two CUDA events, after a warm-up; the maps stay in L2.  One
JSON line per configuration: median / min / max microseconds per call over the repetitions, rays/s, the status histogram
and the mean number of march samples per ray (from the distances of the records).

For the 4096-ray sets the same run also times the host-driven march this call replaces: one blocking
wso_query_surface_host call per march step (every still-marching ray in one call) and one per bisection step, with the
same step, budget and refinement; host clock around the whole loop.  Card name, power limit and max SM clock come from a
read-only nvidia-smi query in the same process.  Without a CUDA device the script exits with an error.
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

FORMATS = ("rgba32f", "rgba16f")
CASCADE_L = (1000.0, 250.0, 61.0)
SIZES = (4096, 1 << 20)
MAX_STEPS, REFINE, TMAX = 1024, 16, 500.0


def make_ctx(W, stream, n, fmt):
    ws = W.WSTessendorf(n, CASCADE_L[0], max_tiles=len(CASCADE_L), max_slots=len(CASCADE_L))
    ws.set_map_format(fmt)
    for t, L in enumerate(CASCADE_L):
        ws.SetTileLength(L, t)
        ws.Prepare(seed=11 + t, tile=t)
    ws.set_stream(stream.cuda_stream)
    ws.compute_batch(np.full(len(CASCADE_L), 7.25, np.float32), tiles=np.arange(len(CASCADE_L), dtype=np.uint32))
    return ws


def ray_sets(count, seed):
    rng = np.random.default_rng(seed)
    area = 4 * CASCADE_L[0]
    out = {}
    for name, (lo, hi) in (("projectile", (10.0, 80.0)), ("grazing", (1.0, 5.0))):
        r = np.zeros((count, 8), np.float32)
        r[:, 0] = rng.uniform(0, area, count)
        r[:, 1] = rng.uniform(5, 50, count)
        r[:, 2] = rng.uniform(0, area, count)
        r[:, 3] = TMAX
        el = np.radians(rng.uniform(lo, hi, count))
        az = rng.uniform(0, 2 * np.pi, count)
        r[:, 4], r[:, 5], r[:, 6] = np.cos(el) * np.cos(az), -np.sin(el), np.cos(el) * np.sin(az)
        out[name] = r
    return out


def time_raycast(torch, ws, stream, rays, out, n, slots, kw, calls, warmup):
    for _ in range(warmup):
        ws.raycast_surface_device(rays.data_ptr(), out.data_ptr(), n, slots=slots, **kw)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(calls):
        ws.raycast_surface_device(rays.data_ptr(), out.data_ptr(), n, slots=slots, **kw)
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / calls


def host_driven_march(ws, rays, slots, step, iterations):
    """The march of the contract driven from the host, one wso_query_surface_host call per march or bisection step
    over every ray still in flight (the slab clip is done on the host, without calls).  -> (seconds, calls, status)."""
    A = ws.read_heights(0, len(slots))[0]
    hb = np.float32(np.sum(np.abs(np.asarray(A, np.float32))) * np.float32(1 + 2.0 ** -10))
    o, tmax = rays[:, 0:3], rays[:, 3]
    d = rays[:, 4:7] / np.linalg.norm(rays[:, 4:7], axis=1, keepdims=True)
    t0 = time.perf_counter()
    n = rays.shape[0]
    with np.errstate(all="ignore"):
        t1, t2 = (hb - o[:, 1]) / d[:, 1], (-hb - o[:, 1]) / d[:, 1]
    s0 = np.maximum(np.minimum(t1, t2), 0)
    send = np.minimum(tmax, np.maximum(t1, t2))
    status = np.zeros(n, np.int64)
    live = s0 <= send
    lo, hi = s0.copy(), s0.copy()
    calls = 0

    def below(idx, t):
        nonlocal calls
        p = o[idx] + t[:, None] * d[idx]
        calls += 1
        return p[:, 1] <= ws.query_surface(p[:, [0, 2]], slots=slots, iterations=iterations)["height"]

    for k in range(MAX_STEPS):
        idx = np.nonzero(live)[0]
        if idx.size == 0:
            break
        t = np.minimum(s0[idx] + k * step, send[idx])
        last = t >= send[idx]
        b = below(idx, t)
        status[idx[b]] = np.where(k == 0, 2, 1)
        hi[idx[b]] = t[b]
        live[idx[b | last]] = False
        lo[idx[~b]] = t[~b]
        if k + 1 == MAX_STEPS:
            status[idx[~b & ~last]] = 3
    hit = np.nonzero(status == 1)[0]
    for _ in range(REFINE):
        if hit.size == 0:
            break
        m = lo[hit] + 0.5 * (hi[hit] - lo[hit])
        b = below(hit, m)
        hi[hit[b]] = m[b]
        lo[hit[~b]] = m[~b]
    return time.perf_counter() - t0, calls, status


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        print("surface_raycast_bench: no CUDA device (there is no CPU fallback)", file=sys.stderr)
        return 2
    import watersurfacerendering_b200 as W
    info = gpu_info()
    stream = torch.cuda.Stream(device=0)
    torch.cuda.set_stream(stream)
    sets = {n: ray_sets(n, seed=n) for n in SIZES}
    dev = {n: {k: torch.from_numpy(v).cuda() for k, v in s.items()} for n, s in sets.items()}
    out = torch.empty((SIZES[-1], 12), dtype=torch.float32, device="cuda")
    lines = []
    for n in (512, 1024):
        ctx = {f: make_ctx(W, stream, n, f) for f in FORMATS}
        for ncasc in (1, 3):
            slots = tuple(range(ncasc))
            step = min(CASCADE_L[:ncasc]) / n
            for iters in (0, 4):
                kw = dict(step=step, max_steps=MAX_STEPS, refine=REFINE, iterations=iters)
                for count in SIZES:
                    calls = 20 if count == SIZES[0] else 3
                    for name in ("projectile", "grazing"):
                        rays = dev[count][name]
                        runs = {f: [] for f in FORMATS}
                        for r in range(a.reps):
                            for f in (FORMATS if r % 2 == 0 else FORMATS[::-1]):   # alternate which format goes first
                                runs[f].append(time_raycast(torch, ctx[f], stream, rays, out, count, slots, kw, calls,
                                                            a.warmup))
                        for f in FORMATS:
                            ctx[f].raycast_surface_device(rays.data_ptr(), out.data_ptr(), count, slots=slots, **kw)
                            torch.cuda.synchronize()
                            rec = out[:count].cpu().numpy()
                            st = rec[:, 3].view(np.uint32)
                            hist = {s: int(np.sum(st == v)) for s, v in (("miss", 0), ("hit", 1), ("origin_below", 2),
                                                                          ("unresolved", 3), ("invalid", 4))}
                            med = statistics.median(runs[f])
                            line = {"n": n, "cascades": ncasc, "iterations": iters, "format": f, "rays": name,
                                    "batch": count, "step": step, "max_steps": MAX_STEPS, "refine": REFINE,
                                    "us_per_call_median": med, "us_per_call_min": min(runs[f]),
                                    "us_per_call_max": max(runs[f]), "rays_per_s_median": count / (med * 1e-6),
                                    "status": hist, "reps_us": runs[f], **info}
                            if count == SIZES[0]:
                                secs, hcalls, hst = host_driven_march(ctx[f], sets[count][name], slots, step, iters)
                                line.update({"host_march_us": secs * 1e6, "host_march_calls": hcalls,
                                             "host_march_hits": int(np.sum(hst == 1))})
                            lines.append(line)
                            print(json.dumps(line), flush=True)
        for ws in ctx.values():
            ws.close()
    if a.out:
        with open(a.out, "w") as fh:
            fh.write("\n".join(json.dumps(x) for x in lines) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
