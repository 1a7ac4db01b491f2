"""TEST INFRASTRUCTURE: builds and drives tests/emu/emu.cpp — the CUDA kernel bodies compiled for the CPU."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "watersurfacerendering_b200", "csrc")
LIB = os.path.join(HERE, "libwsoemu.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        deps = [os.path.join(HERE, "emu.cpp"), os.path.join(CSRC, "wso_kernels.cuh"),
                os.path.join(CSRC, "wso_device.cuh"), os.path.join(CSRC, "wso_tilings.h")]
        if not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in deps):
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            subprocess.check_call([cxx, "-std=c++17", "-O2", "-w", "-ffp-contract=off", "-fPIC", "-shared",
                                   "-I", CSRC, "-o", LIB, os.path.join(HERE, "emu.cpp")])
        L = C.CDLL(LIB)
        vp = C.c_void_p
        L.wso_emu_compute.argtypes = [C.c_int, C.c_int, vp, vp, vp, C.c_float, C.c_float, C.c_float, vp, vp, vp, vp,
                                      vp]
        L.wso_emu_compute.restype = C.c_int
        L.wso_emu_compute_slab.argtypes = [C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_float, C.c_float, C.c_float, vp,
                                           vp, vp, vp]
        L.wso_emu_compute_slab.restype = C.c_int
        L.wso_emu_slab_rank_phase.argtypes = [C.c_int] * 5 + [vp, vp, vp, C.c_float, C.c_float, C.c_float] + [vp] * 6
        L.wso_emu_slab_rank_phase.restype = C.c_int
        L.wso_emu_compute_shipped.argtypes = [C.c_int] * 4 + [vp] * 11
        L.wso_emu_compute_shipped.restype = C.c_int
        L.wso_emu_tilings.argtypes = [vp]
        L.wso_emu_tilings.restype = C.c_int
        _lib = L
    return _lib


# sizes whose first Stockham radix is 2, 4 or 8 (Plan<LOGN> in wso_device.cuh) store W in the paired layout
PAIRED_W_LOGN = {5, 6, 7, 9, 10, 11, 13, 14}


def compute(n, tile_length, lam, h0_re, h0_im, omega, t, variant=0, want_w=False, anim_period=200.0):
    """Run emulated K1+K2+K3 for one tile-frame. h0_* are (N,N) row-major [m][n] (reference layout).
    anim_period=None forces the direct sincosf path; otherwise the sincos table is used when omega allows."""
    logn = int(np.log2(n))
    amp_t = np.ascontiguousarray(np.stack([h0_re.T, h0_im.T], axis=-1).astype(np.float32))
    om_t = np.ascontiguousarray(omega.T.astype(np.float32))
    idx = np.arange(n, dtype=np.float32)
    kv = (np.pi * (np.float32(2) * idx - np.float32(n)).astype(np.float64)
          / np.float64(np.float32(tile_length))).astype(np.float32)
    disp = np.zeros((n, n, 4), np.float32)
    norm = np.zeros((n, n, 4), np.float32)
    mm = np.zeros(2, np.float32)
    a = np.zeros(1, np.float32)
    w = np.zeros((n // 2, 4, n), np.complex64) if want_w else None
    p = lambda x: None if x is None else x.ctypes.data_as(C.c_void_p)
    omega0 = 0.0 if anim_period is None else float(
        np.float32(np.float64(np.float32(2.0)) * np.pi / np.float64(np.float32(anim_period))))
    rc = lib().wso_emu_compute(logn, variant, p(amp_t), p(om_t), p(kv), omega0, float(lam), float(t), p(disp),
                               p(norm), p(mm), p(a), p(w))
    if rc != 0:
        raise ValueError(f"no emulated configuration for logn={logn} variant={variant}")
    if w is not None and logn in PAIRED_W_LOGN:
        # paired W layout (WLayout<LOGN>::paired in wso_kernels.cuh): element 2*j + half -> canonical half*N/2 + j
        w = np.concatenate([w[:, :, 0::2], w[:, :, 1::2]], axis=2)
    return a[0], disp, norm, mm[0], mm[1], w


# kinds of compute_shipped(): the tilings of wso_tilings.h as launch_all() in wso_kernels.cu runs them
KIND_LAT, KIND_BULK, KIND_PERSIST, KIND_JACOBIAN = 0, 1, 2, 3


def shipped_tilings():
    """[(logn, kind, CP, NF, RI, RH, persist)] - every tiling launch_all() can pick (kind 0 = Lat, 1 = Bulk; persist:
    bit 0 / bit 2 = Bulk's K1 / K2 have a persistent form), read from the header the library is built from."""
    out = np.zeros((64, 7), np.int32)
    n = lib().wso_emu_tilings(out.ctypes.data_as(C.c_void_p))
    return [tuple(int(v) for v in r) for r in out[:n]]


def compute_shipped(n, kind, items, half=False, want_w=False):
    """One emulated launch of len(items) tile-frames through a shipped tiling.  items: dicts with keys re, im, omega
    ((N,N) reference layout [m][n]), tile_length, lam, t and optional anim_period (None: no sincos table).
    Returns (A[k], disp[k,N,N,4], norm[k,N,N,4], min[k], max[k], W) - maps as float32 (RGBA16F maps widened)."""
    logn = int(np.log2(n))
    k = len(items)
    amp_t = np.ascontiguousarray(np.stack([np.stack([it["re"].T, it["im"].T], axis=-1) for it in items]), np.float32)
    om_t = np.ascontiguousarray(np.stack([it["omega"].T for it in items]), np.float32)
    idx = np.arange(n, dtype=np.float32)
    kv = np.ascontiguousarray(np.stack([(np.pi * (np.float32(2) * idx - np.float32(n)).astype(np.float64)
                                         / np.float64(np.float32(it["tile_length"]))).astype(np.float32)
                                        for it in items]))

    def omega0(it):
        per = it.get("anim_period", 200.0)
        return 0.0 if per is None else float(np.float32(np.float64(np.float32(2.0)) * np.pi / np.float64(np.float32(per))))

    om0 = np.array([omega0(it) for it in items], np.float32)
    lam = np.array([it["lam"] for it in items], np.float32)
    t = np.array([it["t"] for it in items], np.float32)
    tex = np.float16 if half else np.float32
    disp = np.zeros((k, n, n, 4), tex)
    norm = np.zeros((k, n, n, 4), tex)
    mm = np.zeros((k, 2), np.float32)
    a = np.zeros(k, np.float32)
    w = np.zeros((k, n // 2, 4, n), np.complex64) if want_w else None
    p = lambda x: None if x is None else x.ctypes.data_as(C.c_void_p)
    rc = lib().wso_emu_compute_shipped(logn, kind, 1 if half else 0, k, p(amp_t), p(om_t), p(kv), p(om0), p(lam), p(t),
                                       p(disp), p(norm), p(mm), p(a), p(w))
    if rc != 0:
        raise ValueError(f"no emulated launch for logn={logn} kind={kind} (rc={rc})")
    if w is not None and logn in PAIRED_W_LOGN:
        w = np.concatenate([w[..., 0::2], w[..., 1::2]], axis=-1)
    return a, disp.astype(np.float32), norm.astype(np.float32), mm[:, 0], mm[:, 1], w


def compute_slab(n, tile_length, lam, h0_re, h0_im, omega, t, world, variant=0, anim_period=200.0):
    """Same as compute(), through the slab-decomposed kernels on `world` emulated devices (fused peer stores)."""
    logn = int(np.log2(n))
    shift = int(np.log2(world))
    amp_t = np.ascontiguousarray(np.stack([h0_re.T, h0_im.T], axis=-1).astype(np.float32))
    om_t = np.ascontiguousarray(omega.T.astype(np.float32))
    idx = np.arange(n, dtype=np.float32)
    kv = (np.pi * (np.float32(2) * idx - np.float32(n)).astype(np.float64)
          / np.float64(np.float32(tile_length))).astype(np.float32)
    disp = np.zeros((n, n, 4), np.float32)
    norm = np.zeros((n, n, 4), np.float32)
    mm = np.zeros(2, np.float32)
    a = np.zeros(1, np.float32)
    p = lambda x: x.ctypes.data_as(C.c_void_p)
    omega0 = 0.0 if anim_period is None else float(
        np.float32(np.float64(np.float32(2.0)) * np.pi / np.float64(np.float32(anim_period))))
    rc = lib().wso_emu_compute_slab(logn, variant, shift, p(amp_t), p(om_t), p(kv), omega0, float(lam), float(t),
                                    p(disp), p(norm), p(mm), p(a))
    if rc != 0:
        raise ValueError(f"no emulated slab configuration for logn={logn} variant={variant} world={world} (rc={rc})")
    return a[0], disp, norm, mm[0], mm[1]


class EmuSlabBackend:
    """Drop-in for watersurfacerendering_b200.slab.SlabBackend whose phases run the emulated kernel bodies on the
    CPU (unfused exchange only): lets the gloo tests exercise the real SlabOcean orchestration without a GPU."""

    def __init__(self, n, tile_length, lam, h0_re, h0_im, omega, rank, world, variant=0, anim_period=200.0):
        import torch
        self.n, self.rank, self.world = n, rank, world
        self.logn, self.shift, self.variant = int(np.log2(n)), int(np.log2(world)), variant
        self.hl = n // 2 // world
        self.lam = float(lam)
        self.amp_t = np.ascontiguousarray(np.stack([h0_re.T, h0_im.T], axis=-1).astype(np.float32))
        self.om_t = np.ascontiguousarray(omega.T.astype(np.float32))
        idx = np.arange(n, dtype=np.float32)
        self.kv = (np.pi * (np.float32(2) * idx - np.float32(n)).astype(np.float64)
                   / np.float64(np.float32(tile_length))).astype(np.float32)
        self.omega0 = float(np.float32(np.float64(np.float32(2.0)) * np.pi / np.float64(np.float32(anim_period))))
        blk = self.hl * 4 * 2 * self.hl * 2  # floats per block
        self.send = torch.zeros(blk * world, dtype=torch.float32)
        self.recv = torch.zeros(blk * world, dtype=torch.float32)
        self.minmax = torch.zeros(2, dtype=torch.float32)
        self.ldisp = np.zeros((2 * self.hl, n, 4), np.float32)
        self.lnorm = np.zeros((2 * self.hl, n, 4), np.float32)
        self.amp = np.zeros(1, np.float32)
        self.t = 0.0
        self.fused = False

    def _phase(self, phase):
        p = lambda x: x.ctypes.data_as(C.c_void_p)
        tp = lambda x: C.c_void_p(x.data_ptr())
        rc = lib().wso_emu_slab_rank_phase(self.logn, self.variant, self.shift, self.rank, phase, p(self.amp_t),
                                           p(self.om_t), p(self.kv), self.omega0, self.lam, self.t, tp(self.send),
                                           tp(self.recv), tp(self.minmax), p(self.ldisp), p(self.lnorm), p(self.amp))
        if rc != 0:
            raise ValueError(f"emulated slab phase failed rc={rc}")

    def pass1(self, t):
        self.t = float(t)
        self.minmax[0], self.minmax[1] = 3.402823466e+38, 1.17549435e-38
        self._phase(0)

    def heights(self): self._phase(1)
    def pass2(self): self._phase(2)
    def sync(self): pass
    def read_heights(self): return self.amp[0], np.float32(self.minmax[0]), np.float32(self.minmax[1])
    def local_rows(self, which): return self.ldisp if which == 0 else self.lnorm

    def row_index(self):
        rows = np.zeros(2 * self.hl, np.uint32)
        for ml in range(self.hl):
            mp = self.rank * self.hl + ml
            rows[ml] = mp
            rows[self.hl + ml] = self.n // 2 if mp == 0 else self.n - mp
        return rows


# ---------------------------------------------------------------------------------------------------------------------
# warp-per-line kernels (wso_kernels2.cuh) on the fiber emulator (fiber_simt.h)
# ---------------------------------------------------------------------------------------------------------------------
LIB2 = os.path.join(HERE, "libwsoemu2.so")
_lib2 = None


def lib2():
    global _lib2
    if _lib2 is None:
        deps = [os.path.join(HERE, "emu2.cpp"), os.path.join(HERE, "fiber_simt.h"),
                os.path.join(CSRC, "wso_kernels2.cuh"), os.path.join(CSRC, "wso_simt.cuh"),
                os.path.join(CSRC, "wso_kernels.cuh"), os.path.join(CSRC, "wso_device.cuh")]
        if not os.path.exists(LIB2) or any(os.path.getmtime(d) > os.path.getmtime(LIB2) for d in deps):
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            subprocess.check_call([cxx, "-std=c++17", "-O3", "-w", "-ffp-contract=off", "-fPIC", "-shared",
                                   "-I", CSRC, "-I", HERE, "-o", LIB2, os.path.join(HERE, "emu2.cpp")])
        L = C.CDLL(LIB2)
        vp = C.c_void_p
        L.wso_emu2_compute.argtypes = [C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_float, C.c_float, vp, vp, vp, vp,
                                       vp, vp]
        L.wso_emu2_compute.restype = C.c_int
        _lib2 = L
    return _lib2


def compute2(n, tile_length, lam, h0_re, h0_im, omega, times, variant=0, want_w=False, anim_period=200.0):
    """Emulated warp-per-line K1 + K2h + K2 for len(times) tile-frames of one tile (one launch, several items).
    Returns (A[n_items], disp[n_items,N,N,4], norm[...], min[n_items], max[n_items], W or None)."""
    logn = int(np.log2(n))
    times = np.ascontiguousarray(np.atleast_1d(np.asarray(times, np.float32)))
    k = len(times)
    amp_t = np.ascontiguousarray(np.stack([h0_re.T, h0_im.T], axis=-1).astype(np.float32))
    om_t = np.ascontiguousarray(omega.T.astype(np.float32))
    idx = np.arange(n, dtype=np.float32)
    kv = (np.pi * (np.float32(2) * idx - np.float32(n)).astype(np.float64)
          / np.float64(np.float32(tile_length))).astype(np.float32)
    disp = np.zeros((k, n, n, 4), np.float32)
    norm = np.zeros((k, n, n, 4), np.float32)
    mm = np.zeros((k, 2), np.float32)
    a = np.zeros(k, np.float32)
    w = np.zeros((k, n // 2, 4, n), np.complex64) if want_w else None
    p = lambda x: None if x is None else x.ctypes.data_as(C.c_void_p)
    omega0 = float(np.float32(np.float64(np.float32(2.0)) * np.pi / np.float64(np.float32(anim_period))))
    rc = lib2().wso_emu2_compute(logn, variant, k, p(amp_t), p(om_t), p(kv), omega0, float(lam), p(times), p(disp),
                                 p(norm), p(mm), p(a), p(w))
    if rc != 0:
        raise ValueError(f"emu2: rc={rc} for logn={logn} variant={variant}")
    if w is not None:
        # paired W layout: element 2*j + half -> canonical half*N/2 + j
        w = np.concatenate([w[..., 0::2], w[..., 1::2]], axis=-1)
    return a, disp, norm, mm[:, 0], mm[:, 1], w
