"""RGBA16F output maps (wso_set_map_format): K2 stores every texel as four IEEE binary16 values, each the fp32 value the
RGBA32F path computes, rounded to nearest even.

CPU: the host build's float -> binary16 conversion against NumPy, and the binary16 K2 bodies on the emulator against
float16(their fp32 maps).  GPU (-m gpu): the RGBA16F maps of every compute path equal np.float16(RGBA32F maps) bit for
bit, pass an oracle gate widened by the binary16 rounding, and the format's state, host copies and interop behave.
"""
import ctypes as C
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from conftest import ROOT, SCALAR_REL_TOL, h0_struct, load_golden, rel_l2
from emu import driver as E
from oracle import port as P

HALF_ONE = 0x3C00


# ---------------------------------------------------------------------------------------------------------------------
# CPU: conversion
# ---------------------------------------------------------------------------------------------------------------------
_EMU16 = None


def _emu():
    """tests/emu/emu_f16.cpp, compiled once per session into a temporary directory (the tree may be read-only)."""
    global _EMU16
    if _EMU16 is None:
        out = os.path.join(tempfile.mkdtemp(prefix="wso_emu16_"), "libwsoemu16.so")
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-std=c++17", "-O2", "-w", "-ffp-contract=off", "-fPIC", "-shared", "-I", E.CSRC,
                               "-o", out, os.path.join(E.HERE, "emu_f16.cpp")])
        L = C.CDLL(out)
        vp = C.c_void_p
        L.wso_emu16_f32_to_f16.argtypes = [vp, vp, C.c_size_t]
        L.wso_emu16_f32_to_f16.restype = None
        L.wso_emu16_compute.argtypes = [C.c_int] * 3 + [vp, vp, vp] + [C.c_float] * 3 + [vp] * 4
        L.wso_emu16_compute.restype = C.c_int
        _EMU16 = L
    return _EMU16


def _convert(x):
    x = np.ascontiguousarray(x, np.float32)
    out = np.empty(x.shape, np.uint16)
    _emu().wso_emu16_f32_to_f16(x.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), x.size)
    return out


def _assert_same_half(x):
    got = _convert(x)
    with np.errstate(over="ignore"):
        want = np.asarray(x, np.float32).astype(np.float16)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got.view(np.float16)), nan), "NaN-ness differs"
    bad = np.flatnonzero((got != want.view(np.uint16)) & ~nan)
    assert bad.size == 0, [(hex(np.float32(x.flat[i]).view(np.uint32)), hex(got.flat[i]), hex(want.view(np.uint16).flat[i]))
                           for i in bad[:8]]


def test_f16_conversion_every_upper_pattern():
    """All 2^19 sign / exponent / upper-10-mantissa-bit patterns, each with the rounding-relevant low 13 bits exact, just
    below the tie, on the tie (the kept bit - bit 13 - runs through even and odd with the patterns) and just above it."""
    upper = np.arange(1 << 19, dtype=np.uint32) << 13
    low = np.array([0x0000, 0x0FFF, 0x1000, 0x1001, 0x1FFF], np.uint32)
    bits = (upper[:, None] | low[None, :]).ravel()
    _assert_same_half(bits.view(np.float32))


def test_f16_conversion_subnormal_range():
    """binary16 subnormals (below 2^-14): every half-unit k * 2^-25 (the ties of the subnormal grid) and its float32
    neighbours, plus random mantissas at every float32 exponent from 2^-27 to 2^-14."""
    k = np.arange(0, 2 ** 12 + 2, dtype=np.float64)
    ties = (k * 2.0 ** -25).astype(np.float32)
    x = np.concatenate([ties, np.nextafter(ties, np.float32(0)), np.nextafter(ties, np.float32(1)), -ties])
    rng = np.random.default_rng(3)
    e = rng.integers(127 - 27, 127 - 13, 1 << 16).astype(np.uint32)
    m = rng.integers(0, 1 << 23, 1 << 16).astype(np.uint32)
    s = rng.integers(0, 2, 1 << 16).astype(np.uint32)
    x = np.concatenate([x, ((s << 31) | (e << 23) | m).view(np.float32)])
    _assert_same_half(x)


def test_f16_conversion_overflow_boundary_inf_nan():
    base = np.array([65504.0, 65505.0, 65519.0, 65520.0, 65521.0, 65535.0, 65536.0, 1e5, 3.4e38], np.float32)
    x = np.concatenate([base, np.nextafter(base, np.float32(0)), np.nextafter(base, np.float32(np.inf))])
    x = np.concatenate([x, -x, np.array([np.inf, -np.inf, np.nan, -np.nan], np.float32)])
    payloads = (np.uint32(0x7F800001) + np.arange(0, 1 << 22, 4099, dtype=np.uint32)).view(np.float32)
    _assert_same_half(np.concatenate([x, payloads, -payloads]))
    got = _convert(np.array([np.inf, -np.inf, 65520.0, -65520.0, 65519.996], np.float32))
    assert got.tolist() == [0x7C00, 0xFC00, 0x7C00, 0xFC00, 0x7BFF]


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the binary16 K2 bodies on the emulator
# ---------------------------------------------------------------------------------------------------------------------
def _emu_compute(n, tile_length, lam, h0_re, h0_im, omega, t, variant, half, anim_period=200.0):
    """emu_f16.cpp wso_emu16_compute: one tile-frame -> (A, disp (N,N,4), norm, min, max); float16 maps when half."""
    logn = int(np.log2(n))
    amp_t = np.ascontiguousarray(np.stack([h0_re.T, h0_im.T], axis=-1).astype(np.float32))
    om_t = np.ascontiguousarray(omega.T.astype(np.float32))
    idx = np.arange(n, dtype=np.float32)
    kv = (np.pi * (np.float32(2) * idx - np.float32(n)).astype(np.float64)
          / np.float64(np.float32(tile_length))).astype(np.float32)
    dt = np.float16 if half else np.float32
    disp = np.zeros((n, n, 4), dt)
    norm = np.zeros((n, n, 4), dt)
    mm = np.zeros(2, np.float32)
    a = np.zeros(1, np.float32)
    p = lambda x: x.ctypes.data_as(C.c_void_p)
    omega0 = float(np.float32(np.float64(np.float32(2.0)) * np.pi / np.float64(np.float32(anim_period))))
    rc = _emu().wso_emu16_compute(logn, variant, 1 if half else 0, p(amp_t), p(om_t), p(kv), omega0, float(lam),
                                  float(t), p(disp), p(norm), p(mm), p(a))
    assert rc == 0, f"no emulated configuration for logn={logn} variant={variant}"
    return a[0], disp, norm, mm[0], mm[1]


def _emu_case(n):
    if n in (16, 64, 256):
        g, params = load_golden({16: "n16_default", 64: "n64_wind", 256: "n256_default"}[n])
        h0 = g["h0"]
        return params["tile_length"], params["lam"], h0[..., 0], h0[..., 1], h0[..., 4], params["anim_period"]
    rng = np.random.default_rng(n + 5)
    xi = (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))).astype(np.complex64)
    p = P.OceanParams(tile_size=n, tile_length=1000.0 * n / 512)
    h0 = P.PortOracle(p).prepare(xi)
    return p.tile_length, p.lam, h0["re"], h0["im"], h0["omega"], p.anim_period


# variants: 0/1 = one-CTA-per-item tilings (1024: the fused K1, paired-W K2 from registers), 200+ = the persistent K2
# (mask bit 6) and K1, 100+ = the Jacobian K2 (pack_item_jac)
@pytest.mark.parametrize("n,variants", [(16, (0, 1, 100)), (64, (0, 1, 2, 101)), (256, (0, 1, 100)),
                                        (512, (0, 1, 200, 201)), (1024, (0, 200, 201, 100))])
def test_emulated_f16_maps_are_rounded_f32_maps(n, variants):
    tl, lam, re, im, om, period = _emu_case(n)
    for v in variants:
        t = 7.625 + v * 0.5
        a, d, nm, mn, mx = _emu_compute(n, tl, lam, re, im, om, t, v, False, anim_period=period)
        a16, d16, n16, mn16, mx16 = _emu_compute(n, tl, lam, re, im, om, t, v, True, anim_period=period)
        if v == 0:  # the RGBA32F instantiation here is the kernel body emu.cpp steps
            a0, d0, n0, _, _, _ = E.compute(n, tl, lam, re, im, om, t, variant=v, anim_period=period)
            assert a0 == a and d0.tobytes() == d.tobytes() and n0.tobytes() == nm.tobytes()
        assert (a16, mn16, mx16) == (a, mn, mx)
        assert d16.view(np.uint16).tobytes() == d.astype(np.float16).view(np.uint16).tobytes(), f"N={n} v{v} disp"
        assert n16.view(np.uint16).tobytes() == nm.astype(np.float16).view(np.uint16).tobytes(), f"N={n} v{v} norm"
        if v < 100 or v >= 200:
            assert np.all(d16[..., 3].view(np.uint16) == HALF_ONE)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def wso():
    import watersurfacerendering_b200 as W
    return W


def _lib():
    from watersurfacerendering_b200 import _lib as L
    return L


def _h0_for(wso, n):
    """h0 both contexts import: the reference fixture where one exists, else what Prepare() builds from a seeded xi."""
    fixture = {16: "n16_default", 64: "n64_default", 256: "n256_default"}.get(n)
    if fixture:
        g, params = load_golden(fixture)
        return h0_struct(g["h0"]), params["tile_length"]
    L = 1000.0 * n / 512
    rng = np.random.default_rng(n)
    xi = (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))).astype(np.complex64)
    with wso.WSTessendorf(n, L) as ws:
        ws.PrepareWithGauss(xi)
        return ws.ExportH0(), L


def _pair(wso, n, h0, L, max_slots=1):
    a = wso.WSTessendorf(n, L, max_slots=max_slots)
    b = wso.WSTessendorf(n, L, max_slots=max_slots)
    b.set_map_format("rgba16f")
    for ws in (a, b):
        ws.ImportH0(h0)
    return a, b


def _same(h, f, what):
    want = f.astype(np.float16).view(np.uint16)
    got = h.view(np.uint16)
    if not np.array_equal(got, want):
        i = int(np.flatnonzero(got.ravel() != want.ravel())[0])
        raise AssertionError(f"{what}: texel value {i}: f16 {got.flat[i]:#06x} != f16(f32 {f.flat[i]!r}) {want.flat[i]:#06x}")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [16, 32, 64, 128, 256, 512, 1024, 2048, 4096])
def test_f16_bit_exact_single_frames(wso, n):
    """wso_compute (graph modes 0/1/2), wso_compute_async, several t and lambda, Jacobian on and off."""
    h0, L = _h0_for(wso, n)
    a32, a16 = _pair(wso, n, h0, L)
    with a32, a16:
        assert a16.get_map_format() == "rgba16f" and a32.get_map_format() == "rgba32f"
        for mode in (0, 1, 2):
            for ws in (a32, a16):
                ws.set_frame_graph(mode != 0, every_size=mode == 2)
            for t, lam in ((0.0, -1.0), (3.5, 0.75), (4711.25, -2.0))[: 3 if n <= 1024 else 1]:
                for ws in (a32, a16):
                    ws.SetLambda(lam)
                A = a32.ComputeWaves(t)
                assert a16.ComputeWaves(t) == A
                assert (a16.GetMinHeight(), a16.GetMaxHeight()) == (a32.GetMinHeight(), a32.GetMaxHeight())
                _same(a16.GetDisplacements().copy(), a32.GetDisplacements().copy(), f"N={n} graph={mode} t={t} disp")
                _same(a16.GetNormals().copy(), a32.GetNormals().copy(), f"N={n} graph={mode} t={t} norm")
        for ws in (a32, a16):
            ws.WaitEvent(ws.ComputeWavesAsync(9.25))
        _same(a16.copy_map(0), a32.copy_map(0), f"N={n} async disp")
        _same(a16.copy_map(1), a32.copy_map(1), f"N={n} async norm")
        assert a16.read_heights(0, 1) == a32.read_heights(0, 1)
        for ws in (a32, a16):
            ws.SetComputeJacobian(True)
            ws.ComputeWaves(5.5)
        _same(a16.GetDisplacements().copy(), a32.GetDisplacements().copy(), f"N={n} jacobian disp")
        _same(a16.GetNormals().copy(), a32.GetNormals().copy(), f"N={n} jacobian norm")


@pytest.mark.gpu
def test_f16_bit_exact_8192(wso):
    n = 8192
    h0, L = _h0_for(wso, n)
    a32, a16 = _pair(wso, n, h0, L)
    with a32, a16:
        assert a16.ComputeWaves(21.5) == a32.ComputeWaves(21.5)
        _same(a16.GetDisplacements().copy(), a32.GetDisplacements().copy(), "N=8192 disp")
        _same(a16.GetNormals().copy(), a32.GetNormals().copy(), "N=8192 norm")


# the tilings the benchmark runs: 512^2 x 64 tiles, 1024^2 x 100 frames (chunks of 4 over both lanes), 2048^2 x 8
BATCHES = [(512, 64, 64), (1024, 100, 1), (2048, 8, 1)]


def _batch(ws, n, frames, tiles):
    times = np.float32(0.125) + np.arange(frames, dtype=np.float32) * np.float32(1.0 / 60)
    ws.compute_batch(times, tiles=None if tiles == 1 else np.arange(frames, dtype=np.uint32) % tiles)
    ws.sync()
    return ws.read_heights(0, frames)


@pytest.mark.gpu
@pytest.mark.parametrize("n,frames,tiles", BATCHES)
def test_f16_bit_exact_batches_and_kernel_masks(wso, n, frames, tiles):
    """wso_compute_batch under kernel masks 0, 0x10, 0x40, 0x50 (persistent K1 / K2): RGBA16F == float16(RGBA32F) of
    the same mask; mask 0x4 (warp-per-line K2, RGBA32F only) gives the RGBA16F context the bytes of mask 0."""
    L = _lib()
    lib = L.load()
    h0, Lt = _h0_for(wso, n)
    a32 = wso.WSTessendorf(n, Lt, max_tiles=tiles, max_slots=frames)
    a16 = wso.WSTessendorf(n, Lt, max_tiles=tiles, max_slots=frames)
    a16.set_map_format("rgba16f")
    rng = np.random.default_rng(1)
    try:
        for tile in range(tiles):
            h = h0 if tile == 0 else h0.copy()
            if tile:
                f = np.float32(0.5 + rng.random())  # a different spectrum per tile, still conjugate-symmetric records
                for k in ("re", "im", "re_c", "im_c"):
                    h[k] *= f
            for ws in (a32, a16):
                ws.ImportH0(h, tile)
                ws.SetLambda(-1.0 + 0.01 * tile, tile)
        ref16 = None
        for mask in (0, 0x10, 0x40, 0x50, 0x4):
            assert lib.wso_select_kernels(mask) == 0
            h32 = _batch(a32, n, frames, tiles) if mask != 0x4 else None
            h16 = _batch(a16, n, frames, tiles)
            maps16 = [(a16.copy_map(0, s), a16.copy_map(1, s)) for s in range(frames)]
            if mask == 0x4:
                for s in range(frames):
                    assert maps16[s][0].tobytes() == ref16[s][0].tobytes() and maps16[s][1].tobytes() == ref16[s][1].tobytes()
                continue
            assert all(np.array_equal(x, y) for x, y in zip(h16, h32))
            for s in range(frames):
                _same(maps16[s][0], a32.copy_map(0, s), f"N={n} mask={mask:#x} slot {s} disp")
                _same(maps16[s][1], a32.copy_map(1, s), f"N={n} mask={mask:#x} slot {s} norm")
            if mask == 0:
                ref16 = maps16
    finally:
        lib.wso_select_kernels(0)   # the built-in choice (-1 is not accepted by wso_select_kernels)
        a32.close()
        a16.close()


_SPLIT_SCRIPT = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import watersurfacerendering_b200 as W
for n, frames in ((512, 1), (1024, 12)):
    rng = np.random.default_rng(n)
    xi = (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))).astype(np.complex64)
    a32 = W.WSTessendorf(n, 1000.0 * n / 512, max_slots=frames)
    a16 = W.WSTessendorf(n, 1000.0 * n / 512, max_slots=frames)
    a16.set_map_format("rgba16f")
    times = np.arange(frames, dtype=np.float32) * np.float32(0.25) + np.float32(2.0)
    for ws in (a32, a16):
        ws.PrepareWithGauss(xi)
        ws.compute_batch(times)
        ws.sync()
    for s in range(frames):
        for m in (0, 1):
            assert a16.copy_map(m, s).view(np.uint16).tobytes() == a32.copy_map(m, s).astype(np.float16).view(np.uint16).tobytes(), (n, s, m)
    a32.close()
    a16.close()
print("split ok")
"""


@pytest.mark.gpu
def test_f16_bit_exact_with_k2_split():
    """K2h launched with the normal map (wso_pass2nh_kernel, WSO_K2_SPLIT=1: read once per process, hence a child)."""
    env = dict(os.environ, WSO_K2_SPLIT="1")
    r = subprocess.run([sys.executable, "-c", _SPLIT_SCRIPT, ROOT], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "split ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("n", [64, 512, 1024, 2048])
def test_f16_vs_oracle(wso, n):
    """Gate widened by the binary16 rounding: per channel rel-L2 <= 2^-11 + 1e-5 and max-abs <= 2^-11 * max|ref| +
    1e-4 * range; A / min / max unchanged (they come from K2h in fp32)."""
    p = P.OceanParams(tile_size=n, tile_length=1000.0 * n / 512)
    o = P.PortOracle(p)
    rng = np.random.default_rng(n + 3)
    xi = (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))).astype(np.complex64)
    o.prepare(xi)
    with wso.WSTessendorf(n, p.tile_length) as ws:
        ws.set_map_format("rgba16f")
        ws.PrepareWithGauss(xi)
        for t in (0.0, 13.375):
            a = ws.ComputeWaves(t)
            a_ref, d_ref, n_ref = o.compute_waves(t)
            assert abs(a - a_ref) <= SCALAR_REL_TOL * a_ref
            assert abs(ws.GetMinHeight() - o.min_height) <= SCALAR_REL_TOL * a_ref
            assert abs(ws.GetMaxHeight() - o.max_height) <= SCALAR_REL_TOL * a_ref
            for name, got, ref in (("disp", ws.GetDisplacements().copy(), d_ref), ("norm", ws.GetNormals().copy(), n_ref)):
                for c in range(4):
                    g, r = got[..., c].astype(np.float64), ref[..., c].astype(np.float64)
                    if name == "disp" and c == 3:
                        assert np.all(got[..., 3].view(np.uint16) == HALF_ONE)
                        continue
                    e2 = rel_l2(g, r)
                    emax = float(np.abs(g - r).max())
                    assert e2 <= 2.0 ** -11 + 1e-5, f"N={n} {name}[{c}] rel-L2 {e2:.3e}"
                    assert emax <= 2.0 ** -11 * np.abs(r).max() + 1e-4 * (r.max() - r.min()), f"N={n} {name}[{c}] max {emax:.3e}"


@pytest.mark.gpu
def test_f16_state_and_lifecycle(wso):
    L = _lib()
    lib = L.load()
    n = 128
    h0, Lt = _h0_for(wso, n)
    with wso.WSTessendorf(n, Lt, max_slots=3) as ref, wso.WSTessendorf(n, Lt, max_slots=3) as ws:
        ref.ImportH0(h0)
        h = ws._h
        # invalid formats: refused, state unchanged
        for bad in (-1, 2, 16):
            assert lib.wso_set_map_format(h, bad) == L.WSO_ERR_INVALID_ARG
        assert ws.get_map_format() == "rgba32f"
        with pytest.raises(ValueError):
            ws.set_map_format("rgb565")
        ws.set_map_format("rgba16f")
        # reset contents before the first compute: binary16 zeros and (0, 1, 0, 0), on the host mirror and every slot
        for s in range(3):
            assert not ws.copy_map(0, s).view(np.uint16).any()
            nm = ws.copy_map(1, s).view(np.uint16)
            assert np.all(nm[..., 1] == HALF_ONE) and not nm[..., [0, 2, 3]].any()
        assert not ws.GetDisplacements().view(np.uint16).any()
        assert np.all(ws.GetNormals().view(np.uint16)[..., 1] == HALF_ONE)
        # the float-typed calls refuse RGBA16F and leave the context usable
        fbuf = np.zeros((n, n, 4), np.float32)
        p, cnt = C.c_void_p(), C.c_size_t()
        assert lib.wso_map_host(h, 0, C.byref(p), C.byref(cnt)) == L.WSO_ERR_INVALID_ARG
        assert b"wso_map_host_bytes" in lib.wso_last_error(h)
        assert lib.wso_copy_map(h, 0, 0, fbuf.ctypes.data_as(C.c_void_p)) == L.WSO_ERR_INVALID_ARG
        assert b"wso_copy_map_bytes" in lib.wso_last_error(h)
        t1 = np.array([1.0], np.float32)
        assert lib.wso_compute_to_host(h, 1, None, t1.ctypes.data_as(C.c_void_p), fbuf.ctypes.data_as(C.c_void_p),
                                       fbuf.ctypes.data_as(C.c_void_p), None, None, None) == L.WSO_ERR_INVALID_ARG
        assert b"wso_compute_to_host_bytes" in lib.wso_last_error(h)
        # byte-typed calls reject buffers that are too small
        small = np.zeros(n * n * 8 - 1, np.uint8)
        assert lib.wso_copy_map_bytes(h, 0, 0, small.ctypes.data_as(C.c_void_p), small.nbytes) == L.WSO_ERR_INVALID_ARG
        assert lib.wso_compute_to_host_bytes(h, 1, None, t1.ctypes.data_as(C.c_void_p), small.ctypes.data_as(C.c_void_p),
                                             small.ctypes.data_as(C.c_void_p), small.nbytes, None, None, None) \
            == L.WSO_ERR_INVALID_ARG
        nb = C.c_size_t()
        assert lib.wso_map_host_bytes(h, 1, C.byref(p), C.byref(nb)) == 0 and nb.value == n * n * 8
        # slot pointers 8*N*N bytes apart
        ptrs = [ws.map_device(0, s) for s in range(3)]
        assert ptrs[1] - ptrs[0] == 8 * n * n and ptrs[2] - ptrs[1] == 8 * n * n
        ws.ImportH0(h0)
        # RGBA32F -> RGBA16F -> RGBA32F: correct maps each time, one recapture per switch (graph mode 2: every size)
        for x in (ref, ws):
            x.set_frame_graph(True, every_size=True)
        ref.ComputeWaves(2.5)
        want_d, want_n = ref.GetDisplacements().copy(), ref.GetNormals().copy()
        ws.set_map_format("rgba32f")
        ws.ComputeWaves(2.5)
        ws.ComputeWaves(2.5)   # the first frame of a shape is a plain launch; the second captures
        caps = ws.stats()["frame_graph_captures"]
        assert ws.GetDisplacements().tobytes() == want_d.tobytes() and ws.GetNormals().tobytes() == want_n.tobytes()
        for fmt in ("rgba16f", "rgba32f", "rgba16f"):
            ws.set_map_format(fmt)
            ws.ComputeWaves(2.5)
            ws.ComputeWaves(2.5)
            got_d, got_n = ws.GetDisplacements().copy(), ws.GetNormals().copy()
            if fmt == "rgba16f":
                _same(got_d, want_d, "switch disp")
                _same(got_n, want_n, "switch norm")
            else:
                assert got_d.tobytes() == want_d.tobytes() and got_n.tobytes() == want_n.tobytes()
            caps += 1
            assert ws.stats()["frame_graph_captures"] == caps, fmt
        # the format survives Prepare() and a tile-size change
        ws.ImportH0(h0)
        assert ws.get_map_format() == "rgba16f"
        ws.SetTileSize(64)
        ws.Prepare(seed=3)
        assert ws.get_map_format() == "rgba16f" and ws.GetDisplacements().shape == (64, 64, 4)
        assert ws.GetDisplacements().dtype == np.float16
        ws.ComputeWaves(1.0)
        with wso.WSTessendorf(64, Lt) as r64:
            r64.Prepare(seed=3)
            r64.ComputeWaves(1.0)
            _same(ws.GetDisplacements().copy(), r64.GetDisplacements().copy(), "after size change")


@pytest.mark.gpu
def test_f16_compute_to_host_matches_copy_map(wso):
    n, frames = 512, 11
    h0, Lt = _h0_for(wso, n)
    with wso.WSTessendorf(n, Lt, max_slots=64) as ws, wso.WSTessendorf(n, Lt, max_slots=64) as ref:
        ws.set_map_format("rgba16f")
        for x in (ws, ref):
            x.ImportH0(h0)
        times = np.float32(0.5) + np.arange(frames, dtype=np.float32)
        d = wso.PinnedBuffer((frames, n, n, 4), np.float16)
        nm = wso.PinnedBuffer((frames, n, n, 4), np.float16)
        try:
            a, mn, mx = ws.compute_to_host(times, d.array, nm.array)
            host_d, host_n = d.array.copy(), nm.array.copy()
        finally:
            d.close()
            nm.close()
        ws.compute_batch(times)
        ref.compute_batch(times)
        assert np.array_equal(a, ws.read_heights(0, frames)[0])
        for s in range(frames):
            assert host_d[s].tobytes() == ws.copy_map(0, s).tobytes()
            assert host_n[s].tobytes() == ws.copy_map(1, s).tobytes()
            _same(host_d[s], ref.copy_map(0, s), f"to_host disp {s}")


@pytest.mark.gpu
def test_f16_export_and_import(wso):
    from test_interop import _read_through_fd
    L = _lib()
    n, slots = 256, 3
    h0, Lt = _h0_for(wso, n)
    with wso.WSTessendorf(n, Lt, max_slots=slots) as ws:
        ws.ImportH0(h0)
        ws.set_exportable(True)
        ws.set_map_format("rgba16f")
        ws.compute_batch([0.5, 1.5, 2.5])
        ws.sync()
        for which in (0, 1):
            fd, nbytes = ws.export_fd(which)
            try:
                assert nbytes >= slots * 8 * n * n
                raw = _read_through_fd(fd, nbytes)
            finally:
                os.close(fd)
            seen = raw[: slots * n * n * 8].view(np.float16).reshape(slots, n, n, 4)
            for s in range(slots):
                assert seen[s].tobytes() == ws.copy_map(which, s).tobytes()
    with wso.WSTessendorf(n, Lt, max_slots=slots) as owner, wso.WSTessendorf(n, Lt, max_slots=slots) as ws:
        ws.set_map_format("rgba16f")
        owner.set_exportable(True)
        owner.set_map_format("rgba16f")   # the owner's array: exactly max_slots * 8 * N*N, granularity-rounded
        fd, nbytes = owner.export_fd(0)
        try:
            with pytest.raises(L.WsoError):
                ws.import_external_fd(0, fd, slots * 8 * n * n - 16, 0)   # smaller than max_slots * 8 * N*N
        finally:
            os.close(fd)
