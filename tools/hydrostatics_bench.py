"""Hydrostatics throughput (wso_hydrostatics) on one GPU, in one process.

    python tools/hydrostatics_bench.py [--reps 3] [--out FILE.jsonl] [--md FILE.md]

For every combination of
  tile size N in {512, 1024};  1 cascade (L = 1000) or 3 (L = 1000, 250, 61);  I in {0, 4} inversion steps;
  map format RGBA32F / RGBA16F (alternating);  two hulls:
    box:       a 12-triangle box, 20 x 4 x 8 m (8 vertices);
    icosphere: a 1280-triangle icosphere of radius 3 m (642 vertices);
  {16, 256, 4096} bodies per call, random headings and heels, spread over 4L x 4L (L = 1000) around the waterline,
every body of a call instancing the same vertex and triangle ranges.  Each repetition is `calls` back-to-back
wso_hydrostatics calls on the context's stream between two CUDA events, after a warm-up; the maps stay in L2.  One JSON
line per configuration: median / min / max microseconds per call over the repetitions, bodies/s and the status histogram.

For the RGBA32F context the same run also times the path this call replaces, on a host clock: every vertex of every
body transformed in NumPy (fp32), one blocking wso_query_surface_host call for all of them, the heights copied back,
then a NumPy float64 clip-and-integrate of every triangle and a per-body reduction.  Card name, power limit and max SM
clock come from a read-only nvidia-smi query in the same process.  Without a CUDA device the script exits with an error.
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
COUNTS = (16, 256, 4096)
RHO, G = 1025.0, 9.81


def box(hx, hy, hz):
    v = np.array([[x, y, z] for x in (-hx, hx) for y in (-hy, hy) for z in (-hz, hz)], np.float64)
    t = []
    for a, b, c, d in [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4), (1, 5, 7, 3)]:
        t += [(a, b, c), (a, c, d)]
    return v, orient(v, np.array(t, np.int64))


def icosphere(r, subdiv=3):
    p = (1 + 5 ** 0.5) / 2
    v = [(-1, p, 0), (1, p, 0), (-1, -p, 0), (1, -p, 0), (0, -1, p), (0, 1, p), (0, -1, -p), (0, 1, -p), (p, 0, -1),
         (p, 0, 1), (-p, 0, -1), (-p, 0, 1)]
    f = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6),
         (7, 1, 8), (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10),
         (8, 6, 7), (9, 8, 1)]
    v = [np.array(x, np.float64) / np.linalg.norm(x) for x in v]
    for _ in range(subdiv):
        mid, nf = {}, []

        def m(a, b):
            key = (min(a, b), max(a, b))
            if key not in mid:
                c = v[a] + v[b]
                v.append(c / np.linalg.norm(c))
                mid[key] = len(v) - 1
            return mid[key]

        for a, b, c in f:
            ab, bc, ca = m(a, b), m(b, c), m(c, a)
            nf += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
        f = nf
    v = np.array(v) * r
    return v, orient(v, np.array(f, np.int64))


def orient(v, t):
    n = np.cross(v[t[:, 1]] - v[t[:, 0]], v[t[:, 2]] - v[t[:, 0]])
    flip = np.einsum("ij,ij->i", n, v[t].mean(1) - v.mean(0)) < 0
    t = t.copy()
    t[flip] = t[flip][:, [0, 2, 1]]
    return t


def rotations(rng, count):
    """Random heading, heel and trim up to 20 degrees."""
    out = np.zeros((count, 3, 3))
    for i in range(count):
        yaw, roll, pitch = rng.uniform(0, 2 * np.pi), *np.radians(rng.uniform(-20, 20, 2))
        cy, sy, cr, sr, cp, sp = np.cos(yaw), np.sin(yaw), np.cos(roll), np.sin(roll), np.cos(pitch), np.sin(pitch)
        Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
        Rx = np.array([[1, 0, 0], [0, cr, -sr], [0, sr, cr]])
        Rz = np.array([[cp, -sp, 0], [sp, cp, 0], [0, 0, 1]])
        out[i] = Ry @ Rx @ Rz
    return out


def scene(W, rng, count, v, t, amp):
    b = np.zeros(count, W.BODY_DTYPE)
    b["rotation"] = rotations(rng, count).reshape(count, 9)
    area = 4 * CASCADE_L[0]
    b["position"] = np.stack([rng.uniform(0, area, count), rng.uniform(-amp, amp, count), rng.uniform(0, area, count)], 1)
    b["vertex_count"], b["triangle_count"] = len(v), len(t)
    return b


def host_path(ws, bodies, v, t, slots, iterations):
    """What a caller does without the call: transform, one blocking query for every vertex, clip and integrate in
    float64 with NumPy, reduce per body.  -> (seconds, per-body force (n, 3))."""
    t0 = time.perf_counter()
    R = bodies["rotation"].reshape(-1, 3, 3).astype(np.float32)
    pos = bodies["position"].astype(np.float32)
    cen = bodies["center"].astype(np.float32)
    arm = np.einsum("bij,bvj->bvi", R, (v.astype(np.float32)[None] - cen[:, None]))       # (n, nv, 3)
    world = arm + (pos + np.einsum("bij,bj->bi", R, cen))[:, None]
    h = ws.query_surface(world[..., [0, 2]].reshape(-1, 2), slots=slots, iterations=iterations)["height"]
    depth = h.reshape(world.shape[:2]).astype(np.float64) - world[..., 1]
    nb, nt = bodies.shape[0], t.shape[0]
    P = arm.astype(np.float64)[:, t].reshape(-1, 3, 3)
    D = depth[:, t].reshape(-1, 3)
    owner = np.repeat(np.arange(nb), nt)
    wet = D > 0
    nw = wet.sum(1)
    subs_p, subs_d, subs_o = [P[nw == 3]], [D[nw == 3]], [owner[nw == 3]]
    for lone, cnt in ((True, 1), (False, 2)):
        sel = np.nonzero(nw == cnt)[0]
        ia = np.argmax(wet[sel] == lone, axis=1)
        order = (ia[:, None] + np.arange(3)) % 3
        p = np.take_along_axis(P[sel], order[:, :, None], 1)
        d = np.take_along_axis(D[sel], order, 1)
        a, b, c = p[:, 0], p[:, 1], p[:, 2]
        da, db, dc = d[:, 0], d[:, 1], d[:, 2]
        x = lambda p0, d0, q, dq: p0 + (d0 / (d0 - dq))[:, None] * (q - p0)
        z = np.zeros_like(da)
        if lone:
            subs_p.append(np.stack([a, x(a, da, b, db), x(a, da, c, dc)], 1))
            subs_d.append(np.stack([da, z, z], 1))
            subs_o.append(owner[sel])
        else:
            xb, xc = x(b, db, a, da), x(c, dc, a, da)
            subs_p += [np.stack([xb, b, xc], 1), np.stack([b, c, xc], 1)]
            subs_d += [np.stack([z, db, z], 1), np.stack([db, dc, z], 1)]
            subs_o += [owner[sel], owner[sel]]
    P, D, O = np.concatenate(subs_p), np.concatenate(subs_d), np.concatenate(subs_o)
    S = 0.5 * np.cross(P[:, 1] - P[:, 0], P[:, 2] - P[:, 0])
    sd = D.sum(1)
    f = -(sd / 3)[:, None] * S
    g = np.einsum("ki,kij->kj", D, P) + sd[:, None] * P.sum(1)
    tau = -np.cross(g, S) / 12
    force = np.zeros((nb, 3))
    torque = np.zeros((nb, 3))
    for k in range(3):
        force[:, k] = np.bincount(O, f[:, k], nb)
        torque[:, k] = np.bincount(O, tau[:, k], nb)
    force *= RHO * G
    return time.perf_counter() - t0, force


def make_ctx(W, stream, n, fmt):
    ws = W.WSTessendorf(n, CASCADE_L[0], max_tiles=len(CASCADE_L), max_slots=len(CASCADE_L))
    ws.set_map_format(fmt)
    for t, L in enumerate(CASCADE_L):
        ws.SetTileLength(L, t)
        ws.Prepare(seed=11 + t, tile=t)
    ws.set_stream(stream.cuda_stream)
    ws.compute_batch(np.full(len(CASCADE_L), 7.25, np.float32), tiles=np.arange(len(CASCADE_L), dtype=np.uint32))
    return ws


def time_calls(torch, ws, stream, args, slots, iters, calls, warmup):
    for _ in range(warmup):
        ws.hydrostatics_device(*args, slots=slots, iterations=iters)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(calls):
        ws.hydrostatics_device(*args, slots=slots, iterations=iters)
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / calls


def write_md(path, lines, info):
    rows = ["# Hydrostatics (wso_hydrostatics): time per call", "",
            f"Card: {info['device']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}.  "
            "Produced by `tools/hydrostatics_bench.py`: device time between CUDA events over back-to-back calls after "
            "a warm-up (median over the repetitions); the host path is one blocking `wso_query_surface_host` call for "
            "every transformed vertex plus a NumPy float64 clip-and-integrate, on a host clock (RGBA32F context).", "",
            "| N | cascades | I | hull | bodies | RGBA32F us | RGBA16F us | bodies/s (RGBA32F) | host path us | "
            "host / device |", "|---|---|---|---|---|---|---|---|---|---|"]
    key = lambda x: (x["n"], x["cascades"], x["iterations"], x["hull"], x["bodies"])
    by = {}
    for x in lines:
        by.setdefault(key(x), {})[x["format"]] = x
    for k in sorted(by):
        a, b = by[k]["rgba32f"], by[k]["rgba16f"]
        hp = a.get("host_path_us")
        rows.append(f"| {k[0]} | {k[1]} | {k[2]} | {k[3]} | {k[4]} | {a['us_per_call_median']:.1f} | "
                    f"{b['us_per_call_median']:.1f} | {a['bodies_per_s_median']:.3g} | {hp:.0f} | "
                    f"{hp / a['us_per_call_median']:.0f}x |")
    with open(path, "w") as fh:
        fh.write("\n".join(rows) + "\n")


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--md", default=None, help="also write a Markdown table to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        print("hydrostatics_bench: no CUDA device (there is no CPU fallback)", file=sys.stderr)
        return 2
    import watersurfacerendering_b200 as W
    info = gpu_info()
    stream = torch.cuda.Stream(device=0)
    torch.cuda.set_stream(stream)
    hulls = {"box": box(10.0, 2.0, 4.0), "icosphere": icosphere(3.0, 3)}
    rng = np.random.default_rng(5)
    out = torch.empty((COUNTS[-1], 8), dtype=torch.float32, device="cuda")
    lines = []
    for n in (512, 1024):
        ctx = {f: make_ctx(W, stream, n, f) for f in FORMATS}
        for ncasc in (1, 3):
            slots = tuple(range(ncasc))
            amp = float(np.sum(np.abs(ctx["rgba32f"].read_heights(0, ncasc)[0])))
            for iters in (0, 4):
                for hname, (v, t) in hulls.items():
                    v4 = np.zeros((len(v), 4), np.float32)
                    v4[:, :3] = v
                    dv = torch.from_numpy(v4).cuda()
                    dt = torch.from_numpy(t.astype(np.int32)).cuda()
                    for count in COUNTS:
                        bodies = scene(W, rng, count, v, t, amp + 1.0)
                        db = torch.from_numpy(bodies.view(np.uint8).copy()).cuda()
                        args = (db.data_ptr(), count, dv.data_ptr(), len(v4), dt.data_ptr(), len(t), out.data_ptr())
                        calls = 20 if count < 4096 or hname == "box" else 5
                        runs = {f: [] for f in FORMATS}
                        for r in range(a.reps):
                            for f in (FORMATS if r % 2 == 0 else FORMATS[::-1]):   # alternate which format goes first
                                runs[f].append(time_calls(torch, ctx[f], stream, args, slots, iters, calls, a.warmup))
                        for f in FORMATS:
                            ctx[f].hydrostatics_device(*args, slots=slots, iterations=iters)
                            torch.cuda.synchronize()
                            rec = out[:count].cpu().numpy()
                            st = rec[:, 7].view(np.uint32)
                            hist = {s: int(np.sum(st == k)) for k, s in enumerate(("dry", "partial", "submerged",
                                                                                    "invalid"))}
                            med = statistics.median(runs[f])
                            line = {"n": n, "cascades": ncasc, "iterations": iters, "format": f, "hull": hname,
                                    "triangles": int(len(t)), "bodies": count, "us_per_call_median": med,
                                    "us_per_call_min": min(runs[f]), "us_per_call_max": max(runs[f]),
                                    "bodies_per_s_median": count / (med * 1e-6), "status": hist, "reps_us": runs[f],
                                    **info}
                            if f == "rgba32f":
                                ctx[f].sync()
                                secs, force = host_path(ctx[f], bodies, v, t, slots, iters)
                                dev_f = rec[:, 0:3].astype(np.float64)
                                line.update({"host_path_us": secs * 1e6, "host_path_max_rel_force_diff": float(
                                    np.abs(force - dev_f).max() / max(np.abs(dev_f).max(), 1e-30))})
                            lines.append(line)
                            print(json.dumps(line), flush=True)
        for ws in ctx.values():
            ws.close()
    if a.out:
        with open(a.out, "w") as fh:
            fh.write("\n".join(json.dumps(x) for x in lines) + "\n")
    if a.md:
        write_md(a.md, lines, info)
    return 0


if __name__ == "__main__":
    sys.exit(main())
