#!/usr/bin/env python
"""bench.py — ocean tile-frames/s of the wave-synthesis hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c1|c3|c4]

A "step" = one batch of tile-frames through ComputeWaves (K1 evolve+transform, K2h height extrema, K2 transform+pack).
Default workload = BASELINE.json configs[1]: 1024x1024 tile, animation frames t_i = i*0.05 s (1000 frames =
10 steps x 100 frames).  Under torchrun every rank owns one GPU and processes its own frames (frames are
independent: weak scaling, no data-path collective); the timed region is bracketed by barrier + synchronize and
the reported time is the max over ranks.  Rank 0 prints ONE JSON line.

  value     device-resident throughput (maps stay in HBM, 100 distinct output slots = 3.4 GB per step >> L2)
  e2e       same metric through the reference-facing C-ABI call with HOST output buffers (pinned), D2H inside
  roofline  dominant kernel: algorithmic bytes / CUDA-event duration vs the measured HBM peak
  cpu_baseline  the reference's own CPU code (oracle/_ref) or its restatement, timed on this box's host cores
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the benchmark writes nothing into the checkout, not even __pycache__ of the package it imports
sys.dont_write_bytecode = True

# algorithmic bytes per grid point per tile-frame of THIS design (DESIGN.md §5): K1 reads the 16-byte h0 record
# and writes the Hermitian-packed intermediate W (4 packed fields x 4 B); K2h re-reads packed field 0 (4 B) for the
# height extrema; K2 reads W and writes both RGBA32F maps (disp.y already normalised - no second pass).
# (SURVEY.md §8d's two-pass model of a 7-field C2R design is 40 / 8 / 60 = 108.)
KERNELS = ["K1", "K2h", "K2"]
BYTES_PER_POINT = {"K1": 32.0, "K2h": 4.0, "K2": 48.0}
SURVEY_BYTES_PER_POINT = {"K1": 40.0, "K2h": 8.0, "K2": 60.0}

WORKLOADS = {
    # name: (N, tile_length, seed, frames per step, tiles, description)
    "c1": dict(n=512, L=1000.0, seed=1234, frames=1, tiles=1, dt=1.5,
               desc="BASELINE configs[0]: default 512x512 tile, single timestep per step"),
    "c2": dict(n=1024, L=2000.0, seed=1, frames=100, tiles=1, dt=0.05,
               desc="BASELINE configs[1]: 1024x1024 tile animated, t_i = i*0.05 s, 100 frames per step"),
    "c3": dict(n=2048, L=4000.0, seed=2, frames=32, tiles=1, dt=0.05,
               desc="BASELINE configs[2]: 2048x2048 tile, all maps, frames t_i = i*0.05 s, 32 frames per step per GPU"),
    "c4": dict(n=512, L=1000.0, seed=1000, frames=64, tiles=64, dt=0.05, t0=10.0, times_per_step=16,
               desc="BASELINE configs[3]: 64 independent 512x512 tiles (wind angle 2*pi*j/64, V=5+0.5j, seed 1000+j), "
                    "tile j on GPU j mod P, every step = all tiles at 16 consecutive times t = 10 + 0.05*k"),
    # one grid over ALL ranks (strong scaling): slab-decomposed transform with one exchange step (run_slab below)
    "c5": dict(n=16384, L=32000.0, seed=7, frames=1, tiles=1, dt=0.05, t0=10.0,
               desc="BASELINE configs[4]: single 16384x16384 patch, slab-decomposed over the ranks, t = 10 + 0.05*k"),
    "c5s": dict(n=2048, L=4000.0, seed=7, frames=1, tiles=1, dt=0.05, t0=10.0,
                desc="2048x2048 patch through the slab-decomposed path (the size the slab parity tests use)"),
}


def gauss(n, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))).astype(np.complex64)


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------
def cpu_reference_model(wl, fft_fast=True):
    """The reference's CPU implementation of the path: oracle/_ref when it was compiled (kind 'reference'),
    else the C++ restatement (kind 'port').  Returns (kind, label, cores, prepare(tile)->callable(t))."""
    from oracle import port as P
    from oracle import refmodel as R
    n, L = wl["n"], wl["L"]
    # every host core this process may run on: torch.distributed.run exports OMP_NUM_THREADS=1 to its workers, which
    # would silently time the reference on one thread
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    if R.available():
        R.set_threads(ncpu)
        mode = R.FFT_FLOAT32
        label = "reference WSTessendorf.cpp verbatim + shim fp32 FFT (NOT FFTW)"
        try:
            if R.lib().wsref_set_fft_mode(R.FFT_REAL_FFTW) == 0:
                mode, label = R.FFT_REAL_FFTW, "reference WSTessendorf.cpp verbatim + libfftw3f.so.3"
        except Exception:
            pass
        cores = R.max_threads()

        def make(tile):
            m = R.RefWSTessendorf(n, L, fft_mode=mode)
            prm = tile_params(wl, tile)
            m.SetWindDirection(prm["wind"][0], prm["wind"][1])
            m.SetWindSpeed(prm["speed"])
            m.PrepareWithGauss(gauss(n, wl["seed"] + tile))
            return m.ComputeWaves
        return "reference", label, cores, make
    P.lib().wso_oracle_set_threads(ncpu)
    cores = int(P.lib().wso_oracle_max_threads())

    def make(tile):
        prm = tile_params(wl, tile)
        o = P.PortOracle(P.OceanParams(tile_size=n, tile_length=L, wind_x=prm["wind"][0], wind_y=prm["wind"][1],
                                       wind_speed=prm["speed"]))
        o.prepare(gauss(n, wl["seed"] + tile))
        return lambda t: o.compute_waves(t, fft_mode=1)[0]
    return "port", "C++ restatement oracle/ws_oracle.cpp + fp32 FFT (NOT FFTW)", cores, make


def tile_params(wl, j):
    if wl["tiles"] == 1:
        return dict(wind=(1.0, 1.0), speed=30.0)
    ang = 2.0 * np.pi * j / wl["tiles"]
    return dict(wind=(float(np.cos(ang)), float(np.sin(ang))), speed=5.0 + 0.5 * j)


def step_times(wl, step):
    f = wl["frames"]
    if wl["tiles"] > 1:
        return np.full(f, wl.get("t0", 10.0) + wl["dt"] * step, np.float32), np.arange(f, dtype=np.uint32) % wl["tiles"]
    if "t0" in wl:
        return np.array([wl["t0"] + wl["dt"] * step], np.float32), None
    i0 = step * f
    return (np.arange(i0, i0 + f, dtype=np.float32) * np.float32(wl["dt"])), None


# ----------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path computed in its last step, so that two builds can be compared output for output.
# The inputs are seeded (gauss(), tile_params(), step_times()), so the same arguments give the same inputs every run.
DUMP_TEXELS = 1 << 20      # sampled texels per map: 2 maps x 16 MB + 3 x 4 MB of coordinates
DUMP_MAX_BYTES = 64 << 20


def dump_sample(frames, rows, cols, seed=0):
    """Fixed, seeded sample of texel coordinates (frame, row, col), sorted, of `frames` maps of rows x cols."""
    total = frames * rows * cols
    rng = np.random.default_rng(seed)
    idx = np.unique(rng.integers(0, total, size=min(DUMP_TEXELS, total), dtype=np.int64))
    return np.unravel_index(idx, (frames, rows, cols))


def write_dump(out_dir, arrays):
    arrays = {k: np.ascontiguousarray(v) for k, v in arrays.items()}
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_MAX_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def dump_batch(ws, frames, out_dir):
    """Device slots 0..frames-1 after compute_batch: the height statistics of every tile-frame (amplitude, min, max),
    and both RGBA32F maps at a seeded sample of texels (sample_frame = slot, sample_row, sample_col)."""
    from watersurfacerendering_b200 import _lib as L
    n = ws.GetTileSize()
    a, mn, mx = ws.read_heights(0, frames)
    f, r, c = dump_sample(frames, n, n)
    bounds = np.searchsorted(f, np.arange(frames + 1))
    out = {"amplitude": a, "min_height": mn, "max_height": mx, "sample_frame": f.astype(np.float32),
           "sample_row": r.astype(np.float32), "sample_col": c.astype(np.float32)}
    for name, which in (("displacement", L.WSO_MAP_DISPLACEMENT), ("normal", L.WSO_MAP_NORMAL)):
        texels = np.empty((f.size, 4), np.float32)
        for s in range(frames):
            lo, hi = bounds[s], bounds[s + 1]
            if hi > lo:
                texels[lo:hi] = ws.copy_map(which, s)[r[lo:hi], c[lo:hi]]
        out[name] = texels
    write_dump(out_dir, out)


def dump_slab(b, out_dir):
    """The same for the slab path: this rank's rows of the one N x N tile-frame (sample_row = global row)."""
    from watersurfacerendering_b200 import _lib as L
    amp, mn, mx = b.read_heights()
    _, r, c = dump_sample(1, 2 * b.hl, b.n)
    out = {"amplitude": np.array([amp], np.float32), "min_height": np.array([mn], np.float32),
           "max_height": np.array([mx], np.float32), "sample_frame": np.zeros(r.size, np.float32),
           "sample_row": b.row_index()[r].astype(np.float32), "sample_col": c.astype(np.float32)}
    for name, which in (("displacement", L.WSO_MAP_DISPLACEMENT), ("normal", L.WSO_MAP_NORMAL)):
        out[name] = b.local_rows(which)[r, c]
    write_dump(out_dir, out)


def run_reference_arm(args, wl, rank, world):
    if rank != 0:
        return
    os.environ.setdefault("OMP_PROC_BIND", "close")  # read when libgomp loads (SURVEY 8d: threads pinned next to each other)
    scale = 1.0
    if wl["n"] > 4096:   # the reference needs ~33 GB and minutes per 16384^2 frame: time 4096^2 and scale by points
        scale = (wl["n"] / 4096) ** 2
        wl = dict(wl, n=4096, L=wl["L"] * 4096 / wl["n"], desc=wl["desc"] + f" [CPU arm timed at 4096^2, value / {scale:.0f}]")
    kind, label, cores, make = cpu_reference_model(wl)
    # bounded sample per step so the whole run ends within minutes
    sample = {512: 8, 1024: 3, 2048: 1}.get(wl["n"], 1)
    fns = [make(j) for j in range(min(wl["tiles"], sample))]
    def one_step(k):
        t, tl = step_times(wl, k)
        for i in range(sample):
            fns[i % len(fns)](float(t[i % len(t)]))
    for k in range(args.warmup):
        one_step(k)
    t0 = time.perf_counter()
    for k in range(args.steps):
        one_step(args.warmup + k)
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt / scale
    line = {
        "impl": "reference", "metric": "ocean tile-frames/s", "value": value, "unit": "tile-frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "tile_size": wl["n"], "frames_per_step": sample,
                   "note": "CPU arm: each step is a bounded sample of the workload's frames; rank 0 only"},
        "cpu_baseline": {"value": value, "unit": "tile-frames/s", "cores": cores, "kind": kind,
                         "sample": f"{sample} x {wl['n']}^2 tile-frames per step, {label}"},
        "e2e": {"value": value, "unit": "tile-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def measure_cpu_baseline(wl, budget_s=12.0):
    kind, label, cores, make = cpu_reference_model(wl)
    fn = make(0)
    t, _ = step_times(wl, 0)
    fn(float(t[0]))  # warm-up (first-touch, thread pool)
    t0 = time.perf_counter()
    fn(float(t[-1]))
    one = time.perf_counter() - t0
    nfr = int(max(3, min(200, budget_s / max(one, 1e-4))))
    t0 = time.perf_counter()
    for i in range(nfr):
        fn(float(t[i % len(t)]))
    dt = time.perf_counter() - t0
    out = {"value": nfr / dt, "unit": "tile-frames/s", "cores": cores, "kind": kind,
           "ms_per_tile_frame": dt / nfr * 1e3,
           "sample": f"{nfr} ComputeWaves(t) calls at {wl['n']}^2 after 1 warm-up, {label}"}
    out["cpu_fft_sanity"] = scipy_fft_sanity(wl["n"])
    return out


def scipy_fft_sanity(n, budget_s=3.0):
    """SURVEY §8(d): an independent CPU-FFT figure next to the reference arm (whose FFTW is replaced by a shim):
    seven complex64 ifft2 of N x N with every host core (pocketfft) - the FFT part of one reference ComputeWaves only."""
    try:
        import scipy.fft as sf
    except Exception as e:  # scipy absent: say so instead of failing the bench
        return {"unavailable": repr(e)}
    workers = os.cpu_count() or 1
    rng = np.random.default_rng(0)
    x = (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))).astype(np.complex64)
    sf.ifft2(x, workers=workers)
    reps, t0 = 0, time.perf_counter()
    while True:
        for _ in range(7):
            sf.ifft2(x, workers=workers)
        reps += 1
        dt = time.perf_counter() - t0
        if dt > budget_s or reps >= 50:
            break
    return {"what": "7 x scipy.fft.ifft2(complex64) per tile-frame, FFTs only", "workers": workers,
            "ms_per_tile_frame": dt / reps * 1e3, "tile_frames_per_s": reps / dt}


# ----------------------------------------------------------------------------------------------------
def run_slab(args, wl, rank, world, local_rank):
    """BASELINE configs[4]: ONE N x N tile-frame per step over all ranks (strong scaling).  Per step: K1 on the local
    column pairs -> exchange (NCCL all-to-all, or --slab-fused: peer stores inside K1 + an ordering collective) ->
    K2h -> 2-float all-reduce -> K2 on the local rows."""
    import torch
    import torch.distributed as dist
    import watersurfacerendering_b200 as W
    from watersurfacerendering_b200 import _lib as L
    from watersurfacerendering_b200.slab import SlabBackend, SlabOcean
    n = wl["n"]
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    t_prep = time.perf_counter()
    b = SlabBackend(n, wl["L"], rank, world, local_rank)
    b.set_stream(stream.cuda_stream)
    t_prep_kernel = time.perf_counter()
    b.prepare_counter_device(wl["seed"])   # Prepare() on the device: this rank's column pairs only
    t_prep_kernel = time.perf_counter() - t_prep_kernel
    t_prep = time.perf_counter() - t_prep
    ocean = SlabOcean(b, fused=bool(args.slab_fused), pipeline=(args.slab_fused == 3))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        tt = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    tk = lambda k: wl["t0"] + wl["dt"] * k
    for k in range(args.warmup):
        ocean.compute(tk(k))
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(args.warmup, args.warmup + args.steps):
        ocean.compute(tk(k))
    e1.record(stream)
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    amp, mn, mx = b.read_heights()
    if args.dump_outputs and rank == 0:
        dump_slab(b, args.dump_outputs)

    # ---- per-phase device time (events around every phase; same steps again)
    names = ["K1", "exchange", "K2h", "allreduce", "K2"]
    evs = []
    for k in range(args.warmup, args.warmup + args.steps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
        ev[0].record(stream)
        b.pass1(tk(k))
        ev[1].record(stream)
        b.exchange()   # the transposing exchange kernel: peer stores over NVLink (fused) or the local send blocks
        if world > 1 and not ocean.fused:
            dist.all_to_all_single(b.recv, b.send)
        elif world > 1:
            dist.all_reduce(ocean._scratch())
        ev[2].record(stream)
        b.heights()
        ev[3].record(stream)
        if world > 1:
            v = torch.stack((b.minmax[0], -b.minmax[1]))
            dist.all_reduce(v, op=dist.ReduceOp.MIN)
            b.minmax[0] = v[0]
            b.minmax[1] = -v[1]
        ev[4].record(stream)
        b.pass2()
        ev[5].record(stream)
        evs.append(ev)
    barrier()
    per_step = {nm: [ev[i].elapsed_time(ev[i + 1]) for ev in evs] for i, nm in enumerate(names)}
    # median over steps (a collective occasionally absorbs a host-side hiccup of the other rank), max over ranks
    phase_ms = {nm: max_over_ranks(float(np.median(per_step[nm]))) for nm in names}

    # ---- end to end: the local rows of both maps to pinned host memory inside the timed region
    rows = 2 * b.hl
    hd, hn = W.PinnedBuffer((rows, n, 4)), W.PinnedBuffer((rows, n, 4))
    import ctypes as C
    def e2e_step(k):
        ocean.compute(tk(k))
        L.check_slab(b._lib.wso_slab_copy_rows(b._h, 0, hd.array.ctypes.data_as(C.c_void_p)), b._h)
        L.check_slab(b._lib.wso_slab_copy_rows(b._h, 1, hn.array.ctypes.data_as(C.c_void_p)), b._h)
    e2e_step(0)
    barrier()
    t0 = time.perf_counter()
    ne = max(1, min(args.steps, 3))
    for k in range(ne):
        e2e_step(k + 1)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()

    peak, peak_src = measured_peak()
    pts = float(n) * n
    ms_step = ms / args.steps
    dom = max(("K1", "K2h", "K2"), key=lambda nm: phase_ms[nm])
    dom_bytes = BYTES_PER_POINT[dom] * pts / world      # per launch = this rank's share of one tile-frame
    nvl_bytes_per_gpu = 16.0 * pts / world * (world - 1) / world   # W blocks that leave each GPU
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        try:
            ns = min(n, 4096)
            wl_s = dict(wl, n=ns, L=wl["L"] * ns / n, tiles=1, frames=1)
            cb = measure_cpu_baseline(wl_s, budget_s=10.0)
            scale = (n / ns) ** 2
            cpu = {"value": cb["value"] / scale, "unit": "tile-frames/s", "cores": cb["cores"], "kind": cb["kind"],
                   "sample": f"{cb['sample']}; measured at {ns}^2 and divided by {scale:.0f} (points ratio) to stand "
                             f"for {n}^2 - the reference code needs ~33 GB and minutes per frame at 16384^2"}
        except Exception as ex:
            cpu = {"value": None, "unit": "tile-frames/s", "cores": 0, "kind": "unavailable", "sample": repr(ex)}
    if rank == 0:
        line = {
            "metric": "ocean tile-frames/s", "value": args.steps / (ms * 1e-3), "unit": "tile-frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "tile_size": n, "frames_per_step": 1,
                       "exchange": "transposing exchange kernel, peer stores over NVLink (CUDA IPC)" if ocean.fused else
                                   ("exchange kernel into send blocks + NCCL all_to_all_single" if world > 1
                                    else "exchange kernel, local (one rank)"),
                       "l2": f"one tile-frame moves {108 * pts / 1e9:.1f} GB >> 126 MB L2",
                       "parallelism": f"slab decomposition x{world}: 1 exchange + 1 two-float all-reduce per tile-frame",
                       "prepare_s": t_prep, "prepare_device_kernel_s": t_prep_kernel},
            "us_per_tile_frame": ms_step * 1e3,
            "e2e": {"value": ne / e2e_s, "unit": "tile-frames/s", "h2d_bytes_per_step": 4,
                    "d2h_bytes_per_step": int(2 * 16 * rows * n), "api": "SlabOcean.compute + wso_slab_copy_rows (pinned)"},
            "gpu_launches": int(4 * args.steps),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": dom_bytes / (phase_ms[dom] * 1e-3) / 1e9,
                         "peak": peak, "unit": "GB/s",
                         "frac": dom_bytes / (phase_ms[dom] * 1e-3) / 1e9 / peak, "peak_source": peak_src, "traffic": None,
                         "algorithmic_bytes_per_launch": dom_bytes, "avg_launch_ms": phase_ms[dom],
                         "phase_ms": phase_ms, "phase_ms_per_step_rank0": per_step,
                         "whole_path_gbs_per_gpu": sum(BYTES_PER_POINT.values()) * pts / world / (ms_step * 1e-3) / 1e9,
                         "survey_model_whole_path_gbs_per_gpu": 108.0 * pts / world / (ms_step * 1e-3) / 1e9,
                         "nvlink": None if world == 1 else {
                             "bytes_out_per_gpu": nvl_bytes_per_gpu, "exchange_ms": phase_ms["exchange"],
                             "achieved_gbs_per_dir": nvl_bytes_per_gpu / (phase_ms["exchange"] * 1e-3) / 1e9,
                             "peak_gbs_per_dir": 770.0, "peak_source": "B200_PROFILING.md measured peer copy"}},
            "heights": {"amplitude": float(amp), "min": float(mn), "max": float(mx)},
            "cpu_baseline": cpu,
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    hd.close()
    hn.close()
    b.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def bind_to_gpu_numa_node(gpu_index):
    """Run this rank (and first-touch its pinned host buffers) on the CPUs next to its GPU.  Under torchrun every rank
    otherwise starts on the same NUMA node and the end-to-end path (D2H into pinned memory) of 8 ranks funnels through one
    memory controller / one PCIe root.  Returns the CPU list, or None when NVML cannot tell."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[gpu_index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else gpu_index
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return allowed
    except Exception:
        pass
    return None


def kernel_names():
    """Which implementation of K1 / K2h / K2 a batched launch of this size runs (wso_select_kernels / WSO_WARP_CORE)."""
    return {"K1": "wso_pass1_kernel / wso_pass1w_kernel (evolve + first transform)",
            "K2h": "wso_heights_kernel / wso_heightsw_kernel (height extrema)",
            "K2": "wso_pass2_kernel / wso_pass2w_kernel (second transform + pack)"}


def load_traffic(workload):
    """Measured DRAM bytes per tile-frame and kernel (ncu --cache-control none, caches left alone between kernels:
    tools/gpu_traffic.sh -> profiles/roofline_traffic.json)."""
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        return json.load(open(tpath)).get(workload)
    except Exception:
        return None


def local_plan(wl, rank, world):
    """Tile-frames this rank processes per step: (frames F, local tile ids or None, global tile ids)."""
    if wl["tiles"] > 1:
        from watersurfacerendering_b200 import sharding
        mine = sharding.shard_indices(wl["tiles"], rank, world)   # tile j -> rank j mod P (BASELINE configs[3])
        return len(mine) * wl.get("times_per_step", 1), mine
    return wl["frames"], None


def local_step_times(wl, step, mine):
    """(times, local tile index per tile-frame) of one step on this rank."""
    if mine is not None:
        k = wl.get("times_per_step", 1)
        t = wl.get("t0", 10.0) + wl["dt"] * (step * k + np.arange(k, dtype=np.float32))
        times = np.repeat(t.astype(np.float32), len(mine))
        tiles = np.tile(np.arange(len(mine), dtype=np.uint32), k)
        return times, tiles
    return step_times(wl, step)


def bench_workload(name, wl, steps, warmup, rank, world, local_rank, *, want_e2e=True, e2e_frames=0, clocks=True,
                   dump_dir=None):
    """One workload on this rank's GPU: device-resident throughput, per-kernel times, end-to-end through host buffers.
    dump_dir: rank 0 writes the outputs of the last timed step there (dump_batch)."""
    import torch
    import torch.distributed as dist
    import watersurfacerendering_b200 as W
    from watersurfacerendering_b200 import sharding

    n = wl["n"]
    F, mine = local_plan(wl, rank, world)
    ntiles = len(mine) if mine is not None else 1
    ws = W.WSTessendorf(n, wl["L"], device=local_rank, max_tiles=ntiles, max_slots=max(F, 2))
    for jl in range(ntiles):
        j = int(mine[jl]) if mine is not None else 0
        prm = tile_params(wl, j)
        ws.SetWindDirection(prm["wind"], jl)
        ws.SetWindSpeed(prm["speed"], jl)
        # every rank owns its own realisation (its tiles / its share of the animation)
        ws.PrepareWithGauss(gauss(n, wl["seed"] + j + (7919 * rank if mine is None else 0)), tile=jl)
    # a dedicated (non-default) torch stream carries every kernel, so torch.cuda.Event brackets them
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    ws.set_stream(stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(first, count):
        for k in range(first, first + count):
            t, tl = local_step_times(wl, k, mine)
            ws.compute_batch(t, tiles=tl, first_slot=0)

    def reduce_ranks(x, op):
        if world == 1:
            return x
        tt = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=op)
        return float(tt.item())

    # ---- device-resident throughput -------------------------------------------------------------
    run_steps(0, warmup)
    barrier()
    sampler = ClockSampler(local_rank) if clocks else None
    if rank == 0 and sampler:
        sampler.start()
    l0 = ws.stats()["kernel_launches"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    run_steps(warmup, steps)
    e1.record(stream)
    barrier()
    ms = reduce_ranks(e0.elapsed_time(e1), dist.ReduceOp.MAX)
    launches = ws.stats()["kernel_launches"] - l0
    clk = sampler.stop() if (rank == 0 and sampler) else None
    frames_all = reduce_ranks(float(F), dist.ReduceOp.SUM)   # tile-frames per step over all ranks
    value = frames_all * steps / (ms * 1e-3)
    if dump_dir and rank == 0:
        dump_batch(ws, F, dump_dir)

    # ---- per-kernel timing (same steps again, CUDA events around every launch) -----------------------
    ws.set_profiling(True)
    run_steps(warmup, steps)
    prof = ws.profile()
    ws.set_profiling(False)
    names = KERNELS
    kms = prof["ms"]
    dom = int(np.argmax(kms))
    peak, peak_src = measured_peak()
    pts = float(n) * n
    tf = max(prof["tile_frames"], 1)

    def gbs(bytes_per_pt, k):
        return bytes_per_pt * pts * tf / (kms[k] * 1e-3) / 1e9 if kms[k] > 0 else None

    traffic = load_traffic(name)
    per_launch_tf = tf / max(prof["launches"], 1)
    achieved = gbs(BYTES_PER_POINT[names[dom]], dom)
    us_tf = ms * 1e3 / (F * steps)
    roofline = {
        "bound": "hbm", "kernel": kernel_names()[names[dom]],
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if achieved else None,
        "peak_source": peak_src,
        # DRAM bytes the dominant kernel really moved per launch: ncu --cache-control none (caches left alone between
        # kernels, i.e. what the running pipeline sees), per tile-frame x tile-frames per launch of THIS run
        "traffic": (traffic["bytes_per_tile_frame"][names[dom]] * per_launch_tf) if traffic else None,
        "traffic_source": (traffic or {}).get("capture"),
        "algorithmic_bytes_per_launch": BYTES_PER_POINT[names[dom]] * pts * per_launch_tf,
        "avg_launch_ms": kms[dom] / max(prof["launches"], 1),
        "timing": "cudaEvent pairs around every launch on the compute stream, separate pass over the same K steps",
        "kernel_ms": dict(zip(names, kms)),
        "kernel_share": dict(zip(names, [x / sum(kms) for x in kms])),
        "per_kernel_achieved_gbs": {nm: gbs(BYTES_PER_POINT[nm], i) for i, nm in enumerate(names)},
        "survey_model_achieved_gbs": gbs(SURVEY_BYTES_PER_POINT[names[dom]], dom),
        "whole_path_gbs": sum(BYTES_PER_POINT.values()) * pts / (us_tf * 1e-6) / 1e9,
        "whole_path_frac_survey_model": sum(SURVEY_BYTES_PER_POINT.values()) * pts / (us_tf * 1e-6) / 1e9 / peak,
        "whole_path_frac_design_bytes": sum(BYTES_PER_POINT.values()) * pts / (us_tf * 1e-6) / 1e9 / peak,
        "whole_path_frac_dram_measured": (sum(traffic["bytes_per_tile_frame"].values()) / (us_tf * 1e-6) / 1e9 / peak)
        if traffic else None,
    }
    out = {"value": value, "ms": ms, "us_per_tile_frame": us_tf, "launches": int(launches), "clocks": clk,
           "roofline": roofline, "frames_per_step_local": F, "frames_per_step_all": int(frames_all),
           "chunk": ws.stats()["chunk"], "tiles_local": ntiles}

    # ---- end to end: host output buffers, D2H inside the timed region ---------------------------------
    if want_e2e:
        Fe = e2e_frames or min(F, 24)
        disp = W.PinnedBuffer((Fe, n, n, 4))
        norm = W.PinnedBuffer((Fe, n, n, 4))

        def e2e_step(k):
            t, tl = local_step_times(wl, k, mine)
            a, mn, mx = ws.compute_to_host(t[:Fe], disp.array, norm.array, tiles=None if tl is None else tl[:Fe])
            return a

        for k in range(warmup):
            e2e_step(k)
        barrier()
        t0 = time.perf_counter()
        for k in range(warmup, warmup + steps):
            amps = e2e_step(k)
        torch.cuda.synchronize()
        e2e_s = reduce_ranks(time.perf_counter() - t0, dist.ReduceOp.MAX)
        barrier()
        fe_all = reduce_ranks(float(Fe), dist.ReduceOp.SUM)
        e2e_val = fe_all * steps / e2e_s
        d2h = int(2 * 16 * n * n * Fe + 12 * Fe)
        # the host-side ceiling of that number: the same two map copies per step, device -> the same pinned buffers,
        # with no kernels at all (PCIe / host memory system only)
        dev = torch.empty(2 * 16 * n * n * Fe, dtype=torch.uint8, device="cuda")
        hd = torch.from_numpy(disp.array.view(np.uint8).reshape(-1))
        hn = torch.from_numpy(norm.array.view(np.uint8).reshape(-1))
        half = dev.numel() // 2
        for _ in range(2):
            hd.copy_(dev[:half], non_blocking=True)
            hn.copy_(dev[half:], non_blocking=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            hd.copy_(dev[:half], non_blocking=True)
            hn.copy_(dev[half:], non_blocking=True)
        torch.cuda.synchronize()
        probe_s = reduce_ranks(time.perf_counter() - t0, dist.ReduceOp.MAX)
        barrier()
        pcie_gbs = dev.numel() * steps / probe_s / 1e9               # this rank's copies over its own link
        pcie_tfs = fe_all * steps / probe_s                          # tile-frames/s if only the copies existed
        del dev
        all_amps = sharding.gather_in_global_order(amps.tolist(), int(fe_all), rank, world) if (world > 1 and mine is None) else amps
        out["e2e"] = {"value": e2e_val, "unit": "tile-frames/s", "h2d_bytes_per_step": int(4 * Fe),
                      "d2h_bytes_per_step": d2h, "frames_per_step_per_gpu": Fe,
                      "api": "wso_compute_to_host (C ABI), pinned host maps, copies overlapped with the next chunk",
                      "last_amplitude": float(np.asarray(all_amps)[-1]),
                      "d2h_probe": {"what": "the same D2H copies with no kernels (host-side ceiling, max over ranks)",
                                    "gbs_per_gpu": pcie_gbs, "tile_frames_per_s": pcie_tfs,
                                    "e2e_frac_of_probe": e2e_val / pcie_tfs}}
        # zero-host-copy variant (SURVEY row f-2): the maps live in exportable memory a Vulkan device imports with
        # VK_KHR_external_memory_fd; the consumer reads them where K2 wrote them, so the end-to-end cost is the device
        # path itself plus the semaphore signal.  Timed with the exportable backing in place.
        try:
            ws.set_exportable(True)
            run_steps(0, 1)
            barrier()
            e0.record(stream)
            run_steps(warmup, steps)
            e1.record(stream)
            barrier()
            ms_x = reduce_ranks(e0.elapsed_time(e1), dist.ReduceOp.MAX)
            out["e2e"]["zero_copy_export"] = {"value": frames_all * steps / (ms_x * 1e-3), "unit": "tile-frames/s",
                                              "what": "maps in exportable (POSIX fd) device memory, no host copy"}
        except Exception as ex:  # no virtual-memory API on this driver: report, do not fail the bench
            out["e2e"]["zero_copy_export"] = {"unavailable": repr(ex)[:200]}
        disp.close()
        norm.close()
    ws.close()
    torch.cuda.synchronize()
    return out


def c1_latency(local_rank):
    """North-star target 'a 512^2 tile (all maps) in <= 20 us': one ComputeWaves-sized call at a time.
    isolated: CUDA events around ONE tile-frame, median; back to back: per frame of a stream of single-frame calls
    (a) through the Python binding, (b) through the C ABI with no Python in the loop (tools/lat_bench, when it builds)."""
    import torch
    import watersurfacerendering_b200 as W
    wl = WORKLOADS["c1"]
    n = wl["n"]
    ws = W.WSTessendorf(n, wl["L"], device=local_rank, max_tiles=1, max_slots=4)
    ws.PrepareWithGauss(gauss(n, wl["seed"]))
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    ws.set_stream(stream.cuda_stream)
    t = np.zeros(1, np.float32)
    for i in range(50):
        t[0] = 0.05 * i
        ws.compute_batch(t)
    torch.cuda.synchronize()
    iso = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(200):
        t[0] = 3.0 + 0.05 * i
        e0.record(stream)
        ws.compute_batch(t)
        e1.record(stream)
        e1.synchronize()
        iso.append(e0.elapsed_time(e1) * 1e3)
    frames = 2000
    e0.record(stream)
    c0 = time.perf_counter()
    for i in range(frames):
        t[0] = 20.0 + 0.05 * i
        ws.compute_batch(t, first_slot=i & 3)
    c1 = time.perf_counter()
    e1.record(stream)
    torch.cuda.synchronize()
    out = {"isolated_us_median": float(np.median(iso)), "isolated_us_min": float(np.min(iso)),
           "back_to_back_us_python_binding": e0.elapsed_time(e1) * 1e3 / frames,
           "host_enqueue_us_python_binding": (c1 - c0) * 1e6 / frames}
    ws.close()
    try:
        # built outside the tree: the benchmark leaves the checkout untouched (it may be read-only)
        with tempfile.TemporaryDirectory(prefix="wso_lat_bench_") as tmp:
            exe = os.path.join(tmp, "lat_bench")
            subprocess.run(["make", "-C", os.path.join(ROOT, "examples"), "lat_bench", f"LAT_BENCH={exe}"],
                           capture_output=True, timeout=120)
            r = subprocess.run([exe, str(n), "2000"], capture_output=True, text=True, timeout=120,
                               env=dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local_rank))))
        out["c_abi"] = json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as ex:
        out["c_abi"] = {"unavailable": repr(ex)[:200]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-targets", action="store_true", help="skip the north-star target block (c1 / c3 / c4 side runs)")
    ap.add_argument("--e2e-frames", type=int, default=0, help="tile-frames per e2e step (default: min(frames, 24))")
    ap.add_argument("--slab-fused", type=int, default=1,
                    help="c5: 1 = exchange kernel with direct peer stores over NVLink, 3 = the same issued field by field on "
                         "a second stream behind K1, 0 = exchange kernel into send blocks + NCCL all-to-all")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0: height statistics of every "
                         "tile-frame, a seeded sample of the displacement and normal maps) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    wl = dict(WORKLOADS[args.workload])

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, wl, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    if args.workload in ("c5", "c5s"):
        run_slab(args, wl, rank, world, local_rank)
        return

    n = wl["n"]
    res = bench_workload(args.workload, wl, args.steps, args.warmup, rank, world, local_rank, e2e_frames=args.e2e_frames,
                         dump_dir=args.dump_outputs)

    # ---- the north-star targets that the headline workload does not show, measured in the same run -----------
    targets = None
    if rank == 0 and world == 1 and args.workload == "c2" and not args.no_targets:
        targets = {}
        try:
            lat = c1_latency(local_rank)
            cabi = lat.get("c_abi") or {}
            # device time of ONE isolated 512^2 tile-frame: through the C ABI when tools/lat_bench built, else through
            # the Python binding (whose event records add a few microseconds around the three launches)
            targets["c1_isolated_us"] = cabi.get("isolated_us_median", lat["isolated_us_median"])
            targets["c1_isolated_us_python_binding"] = lat["isolated_us_median"]
            targets["c1_back_to_back_us"] = cabi.get("back_to_back_us_per_frame", lat["back_to_back_us_python_binding"])
            targets["c1_back_to_back_us_python_binding"] = lat["back_to_back_us_python_binding"]
            targets["c1_detail"] = lat
        except Exception as ex:
            targets["c1_error"] = repr(ex)[:300]
        try:
            r3 = bench_workload("c3", dict(WORKLOADS["c3"]), 3, 3, rank, world, local_rank, want_e2e=False, clocks=False)
            rf = r3["roofline"]
            targets.update({"c3_us_per_tile_frame": r3["us_per_tile_frame"], "c3_tile_frames_s": r3["value"],
                            "c3_frac_Balg": rf["whole_path_frac_survey_model"],
                            "c3_frac_design": rf["whole_path_frac_design_bytes"],
                            "c3_frac_dram_measured": rf["whole_path_frac_dram_measured"],
                            "c3_k1_frac_design": rf["per_kernel_achieved_gbs"]["K1"] / rf["peak"],
                            "c3_kernel_ms": rf["kernel_ms"]})
        except Exception as ex:
            targets["c3_error"] = repr(ex)[:300]
        try:
            r4 = bench_workload("c4", dict(WORKLOADS["c4"]), 5, 3, rank, world, local_rank, want_e2e=False, clocks=False)
            targets.update({"c4_tile_frames_s": r4["value"], "c4_us_per_tile_frame": r4["us_per_tile_frame"]})
        except Exception as ex:
            targets["c4_error"] = repr(ex)[:300]
        targets["north_star"] = {"c1": "<= 20 us per 512^2 tile (all maps)", "c3": ">= 0.60 of the HBM roofline at 2048^2",
                                 "c4": "near-linear 1->8 GPU scaling for batched tiles"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cpu = measure_cpu_baseline(wl)
        except Exception as ex:  # the baseline is reported, never required
            cpu = {"value": None, "unit": "tile-frames/s", "cores": 0, "kind": "unavailable", "sample": repr(ex)}

    if rank == 0:
        tiled = wl["tiles"] > 1
        line = {
            "metric": "ocean tile-frames/s", "value": res["value"], "unit": "tile-frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms"] / args.steps,
            "higher_is_better": True, "scaling": "strong" if tiled else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": wl["desc"], "tile_size": n,
                       "frames_per_step_per_gpu": res["frames_per_step_local"],
                       "frames_per_step_all_gpus": res["frames_per_step_all"],
                       "chunk_tile_frames_per_launch": res["chunk"],
                       "l2": f"outputs of one step = {res['frames_per_step_local']} slots x {32 * n * n / 1e6:.0f} MB > 126 MB L2;"
                             " h0 is resident by design (same spectrum every frame)",
                       "parallelism": (f"{wl['tiles']} tiles sharded j mod {world} ({res['tiles_local']} per GPU) x "
                                       f"{wl.get('times_per_step', 1)} time steps, no collective") if tiled
                       else f"frames sharded per GPU x{world}, no collective"},
            "us_per_tile_frame": res["us_per_tile_frame"],
            "e2e": res.get("e2e"),
            "gpu_launches": res["launches"],
            "roofline": res["roofline"],
            "targets": targets,
            "host_cpus_bound": (f"{numa[0]}-{numa[-1]} ({len(numa)} CPUs next to GPU {local_rank})" if numa else None),
            "cpu_baseline": cpu,
            "clocks": res["clocks"],
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
