"""Surface queries (wso_query_surface): height, normal and undisplaced origin of the surface at arbitrary world points,
sampled from the maps of 1..4 slots (cascades) with a fixed-point inversion of the choppy displacement.

`query_oracle` below is a NumPy float64 statement of the contract in include/wsocean.h ("Surface queries").  With
pos32=True it rounds the sample positions where the contract does (x mod L in float64 rounded to fp32, then fp32 position
sums and scaling); the blends, sums and the normal stay float64.

CPU: the host build of the kernel body (tests/emu/emu_query.cpp, the same wso_query.cuh the sm_100a kernel compiles)
against the oracle, its exactness properties, and the oracle itself against an analytic wave.  GPU (-m gpu): device
records equal the host build's bit for bit on the library's own maps, agree with the oracle, pin the world-space
convention with a one-hot spectrum, follow computes in stream order, and the C ABI validates and keeps its state.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT
from emu import driver as E

FIELDS = ("height", "normal_x", "normal_y", "normal_z", "offset_x", "offset_z", "residual", "w")
F32 = np.float32


# ---------------------------------------------------------------------------------------------------------------------
# host build of the query body
# ---------------------------------------------------------------------------------------------------------------------
_SHIM = None


def _shim():
    """tests/emu/emu_query.cpp, compiled once per session into a temporary directory (the tree may be read-only)."""
    global _SHIM
    if _SHIM is None:
        out = os.path.join(tempfile.mkdtemp(prefix="wso_emuq_"), "libwsoemuq.so")
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-std=c++17", "-O2", "-w", "-ffp-contract=off", "-fPIC", "-shared", "-I", E.CSRC,
                               "-o", out, os.path.join(E.HERE, "emu_query.cpp")])
        L = C.CDLL(out)
        vp = C.c_void_p
        L.wso_emuq_query.argtypes = [C.c_int, C.c_uint32, C.c_int, vp, vp, vp, vp, vp, C.c_int, C.c_uint32, vp, vp]
        L.wso_emuq_query.restype = C.c_int
        _SHIM = L
    return _SHIM


def host_query(disp, norm, A, L, lam, q, iterations):
    """Host build: disp / norm = lists of (N,N,4) maps (float32, or float16 = RGBA16F), one per cascade -> (n, 8) float32."""
    half = disp[0].dtype == np.float16
    dt = np.float16 if half else np.float32
    disp = [np.ascontiguousarray(d, dt) for d in disp]
    norm = [np.ascontiguousarray(g, dt) for g in norm]
    ns = len(disp)
    pd = (C.c_void_p * ns)(*[d.ctypes.data for d in disp])
    pn = (C.c_void_p * ns)(*[g.ctypes.data for g in norm])
    a = np.ascontiguousarray(A, F32)
    lt = np.ascontiguousarray(L, F32)
    lm = np.ascontiguousarray(lam, F32)
    q = np.ascontiguousarray(q, F32).reshape(-1, 2)
    out = np.zeros((q.shape[0], 8), F32)
    p = lambda x: x.ctypes.data_as(C.c_void_p)
    rc = _shim().wso_emuq_query(1 if half else 0, disp[0].shape[0], ns, C.cast(pd, C.c_void_p), C.cast(pn, C.c_void_p),
                                p(a), p(lt), p(lm), int(iterations), q.shape[0], p(q), p(out))
    assert rc == 0
    return out


# ---------------------------------------------------------------------------------------------------------------------
# the float64 oracle
# ---------------------------------------------------------------------------------------------------------------------
def _positions(x, L, n, pos32, delta):
    """u (float64) of world coordinate x (+ offset delta) in texels of a tile of length L."""
    if not pos32:
        return (np.asarray(x, np.float64) + delta) * n / L
    xd = np.asarray(x, F32).astype(np.float64)
    Ld = np.float64(F32(L))
    xr = (xd - np.floor(xd / Ld) * Ld).astype(F32)
    p = (xr + np.asarray(delta, F32)).astype(F32)
    nl = F32(np.float64(n) / Ld)
    return (p * nl).astype(F32).astype(np.float64)


def sample(m, u, v):
    """Bilinear blend of the (N,N,C) map m at texel coordinates (u, v) (u along columns = x), REPEAT wrap, float64."""
    n = m.shape[0]
    n0, m0 = np.floor(u), np.floor(v)
    fu, fv = (u - n0)[:, None], (v - m0)[:, None]
    c0 = n0.astype(np.int64) % n
    r0 = m0.astype(np.int64) % n
    c1, r1 = (c0 + 1) % n, (r0 + 1) % n
    m = np.asarray(m, np.float64)
    top = m[r0, c0] * (1 - fu) + m[r0, c1] * fu
    bot = m[r1, c0] * (1 - fu) + m[r1, c1] * fu
    return top * (1 - fv) + bot * fv


def _dh(disp, L, q, delta, pos32):
    n = disp[0].shape[0]
    hx = np.zeros(q.shape[0])
    hz = np.zeros(q.shape[0])
    for d, l in zip(disp, L):
        s = sample(d, _positions(q[:, 0], l, n, pos32, delta[0]), _positions(q[:, 1], l, n, pos32, delta[1]))
        hx += s[:, 0]
        hz += s[:, 2]
    return hx, hz


def query_oracle(maps, A, L, lam, q, I, pos32=True, offset=None):
    """The contract in float64.  maps = [(disp, norm), ...] per cascade; q = (n, 2) world points; I iterations.
    offset: evaluate at p = q + offset instead of iterating (the recomputation of a reported record).  -> dict of fields."""
    disp = [d for d, _ in maps]
    norm = [g for _, g in maps]
    n = disp[0].shape[0]
    q = np.asarray(q, np.float64).reshape(-1, 2)
    rnd = (lambda x: np.asarray(x, F32).astype(np.float64)) if pos32 else (lambda x: x)
    if offset is None:
        dx = np.zeros(q.shape[0])
        dz = np.zeros(q.shape[0])
        for _ in range(I):
            hx, hz = _dh(disp, L, q, (dx, dz), pos32)
            dx, dz = rnd(-hx), rnd(-hz)
    else:
        dx, dz = (np.asarray(offset[0], np.float64), np.asarray(offset[1], np.float64))
    h = np.zeros(q.shape[0])
    hx = np.zeros(q.shape[0])
    hz = np.zeros(q.shape[0])
    sx = np.zeros(q.shape[0])
    sz = np.zeros(q.shape[0])
    ex = np.ones(q.shape[0])
    ez = np.ones(q.shape[0])
    w = None
    for d, g, a, l, lm in zip(disp, norm, A, L, lam):
        u = _positions(q[:, 0], l, n, pos32, dx)
        v = _positions(q[:, 1], l, n, pos32, dz)
        sd, sg = sample(d, u, v), sample(g, u, v)
        h += np.float64(F32(a)) * sd[:, 1]
        hx += sd[:, 0]
        hz += sd[:, 2]
        sx += sg[:, 0]
        sz += sg[:, 1]
        ex += np.float64(F32(lm)) * sg[:, 2]
        ez += np.float64(F32(lm)) * sg[:, 3]
        w = sd[:, 3] if w is None else w
    nx, nz = -sx / ex, -sz / ez
    ln = np.sqrt(nx * nx + 1.0 + nz * nz)
    return {"height": h, "normal_x": nx / ln, "normal_y": 1.0 / ln, "normal_z": nz / ln, "offset_x": dx, "offset_z": dz,
            "residual": np.hypot(dx + hx, dz + hz), "w": w}


def _scales(maps, A):
    """What each field is compared relative to: height to sum A_s max|D.y|, offsets and residual to sum max|D.x, D.z|."""
    hs = sum(abs(float(a)) * float(np.abs(np.asarray(d[..., 1], np.float64)).max()) for (d, _), a in zip(maps, A))
    ds = sum(float(np.abs(np.asarray(d[..., [0, 2]], np.float64)).max()) for d, _ in maps)
    return {"height": hs, "normal_x": 1.0, "normal_y": 1.0, "normal_z": 1.0, "offset_x": ds, "offset_z": ds,
            "residual": ds, "w": 1.0}


def _assert_close(got, ref, scales, tol, where=None, what="", fields=FIELDS):
    for k, f in enumerate(FIELDS):
        if f not in fields:
            continue
        g = np.asarray(got[:, k], np.float64)
        r = ref[f]
        err = np.abs(g - r)
        if where is not None:
            err = err[where]
        worst = float(err.max()) if err.size else 0.0
        assert worst <= tol * scales[f], f"{what} {f}: max error {worst:.3e} > {tol} * {scales[f]:.3e}"


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def _smooth_random_map(rng, n, amp, waves=6, noise=0.01):
    """(N,N) field: a few random low-order periodic waves plus `noise` white noise, max |value| about amp."""
    idx = np.arange(n) / n
    f = np.zeros((n, n))
    for _ in range(waves):
        kx, kz = rng.integers(-4, 5, 2)
        f += rng.standard_normal() * np.cos(2 * np.pi * (kx * idx[None, :] + kz * idx[:, None]) + rng.uniform(0, 6.3))
    f += noise * rng.standard_normal((n, n)) * np.abs(f).max()
    return f * (amp / np.abs(f).max())


def _random_cascades(rng, n, lengths, half, lip=0.45):
    """Maps per cascade, D.x / D.z scaled so that Dh is a contraction with Lipschitz constant < lip (summed bound over
    the cascades of sqrt(2) * the steepest texel-to-texel step of either channel over the texel spacing)."""
    maps, A, lam = [], [], []
    raw = []
    for s, l in enumerate(lengths):
        d = np.stack([_smooth_random_map(rng, n, 1.0) for _ in range(4)], -1)
        d[..., 3] = 1.0 if s % 2 == 0 else d[..., 3]
        g = np.stack([_smooth_random_map(rng, n, 0.5) for _ in range(4)], -1)
        raw.append((d, g, l))
    steep = []
    for d, _, l in raw:
        st = max(np.abs(np.diff(d[..., c], axis=a, append=d[..., c].take([0], axis=a))).max() for c in (0, 2)
                 for a in (0, 1))
        steep.append(2.0 * st / (l / n))
    scale = lip / sum(steep)
    dt = np.float16 if half else F32
    for (d, g, l), s in zip(raw, range(len(raw))):
        d = d.copy()
        d[..., [0, 2]] *= scale
        maps.append((d.astype(dt), g.astype(dt)))
        A.append(F32(rng.uniform(0.5, 3.0)))
        lam.append(F32(rng.uniform(-1.2, 1.2)))
    return maps, A, lam


def _queries(rng, lengths, n, count=600):
    """Random points over several tiles of every cascade (negative and far out), texel coordinates and tile edges."""
    lmax, lmin = max(lengths), min(lengths)
    q = [rng.uniform(-3 * lmax, 4 * lmax, (count, 2))]
    k = rng.integers(-3 * n, 4 * n, (64, 2)).astype(np.float64)
    q.append(k * (lmin / n))                                              # texel positions of the finest cascade
    e = rng.integers(-4, 5, (32, 2)).astype(np.float64) * lmax
    q.append(e)                                                           # tile corners
    q.append(np.stack([rng.integers(-4, 5, 32) * lmin, rng.uniform(-lmax, lmax, 32)], -1))  # tile edges
    return np.concatenate(q).astype(F32)


@pytest.mark.parametrize("half", [False, True], ids=["rgba32f", "rgba16f"])
@pytest.mark.parametrize("n", [16, 64, 512])
def test_host_body_matches_oracle(n, half):
    rng = np.random.default_rng(n * 10 + half)
    all_lengths = [F32(1000.0), F32(250.0), F32(61.0), F32(17.3)]
    for ns in (1, 2, 3, 4):
        lengths = all_lengths[:ns]
        maps, A, lam = _random_cascades(rng, n, lengths, half)
        q = _queries(rng, lengths, n)
        sc = _scales(maps, A)
        for I in (0, 1, 4, 16):
            got = host_query([d for d, _ in maps], [g for _, g in maps], A, lengths, lam, q, I)
            ref = query_oracle(maps, A, lengths, lam, q, I)
            _assert_close(got, ref, sc, 1e-5, what=f"N={n} cascades={ns} I={I}")
            if I == 16:  # contraction < 0.45: converged far below the tolerance
                assert float(got[:, 6].max()) <= 1e-5 * sc["residual"]


@pytest.mark.parametrize("half", [False, True], ids=["rgba32f", "rgba16f"])
def test_host_body_exactness(half):
    """L = N * 2^k, queries on a 1/64-texel grid: texel positions give fl(A * D.y) exactly at I = 0, q and q +- 3L give
    the same records bit for bit, and q = 10^6 m agrees with q mod L."""
    n, rng = 64, np.random.default_rng(11 + half)
    lengths = [F32(n * 8), F32(n * 2), F32(n / 4)]
    maps, A, lam = _random_cascades(rng, n, lengths, half)
    disp, norm = [d for d, _ in maps], [g for _, g in maps]
    # I = 0 at texel positions of one cascade
    k = rng.integers(-2 * n, 3 * n, (256, 2))
    q = (k * (lengths[0] / n)).astype(F32)
    got = host_query(disp[:1], norm[:1], A[:1], lengths[:1], lam[:1], q, 0)
    dy = disp[0][..., 1].astype(F32)[k[:, 1] % n, k[:, 0] % n]
    assert np.array_equal(got[:, 0].view(np.uint32), (A[0] * dy).astype(F32).view(np.uint32))
    assert np.array_equal(got[:, 4:6], np.zeros((256, 2), F32))
    # periodicity, bit for bit: q on a 1/64-texel grid of the finest cascade, shifted by 3 L of the coarsest
    q = (rng.integers(-64 * n, 64 * n, (512, 2)) * (lengths[2] / n / 64)).astype(F32)
    for I in (0, 4):
        base = host_query(disp, norm, A, lengths, lam, q, I)
        for sh in (3.0, -3.0):
            qs = (q.astype(np.float64) + sh * np.float64(lengths[0])).astype(F32)
            assert np.array_equal(qs.astype(np.float64) - q, np.full(q.shape, sh * np.float64(lengths[0])))
            other = host_query(disp, norm, A, lengths, lam, qs, I)
            assert np.array_equal(base.view(np.uint32), other.view(np.uint32)), (I, sh)
    # far away: 10^6 m against the same point reduced mod L
    far = np.full((256, 2), 1.0e6) + (rng.integers(0, 64 * n, (256, 2)) * (lengths[2] / n / 64))
    far = far.astype(F32)
    near = np.mod(far.astype(np.float64), np.float64(lengths[0])).astype(F32)
    for I in (0, 4):
        a = host_query(disp, norm, A, lengths, lam, far, I)
        b = host_query(disp, norm, A, lengths, lam, near, I)
        sc = _scales(maps, A)
        for k_, f in enumerate(FIELDS):
            assert np.abs(a[:, k_].astype(np.float64) - b[:, k_]).max() <= 1e-6 * sc[f], f


def _analytic_wave(n, L, lam, H=1.3, a=(3, 5), t_phase=0.4):
    """One wave: h = H cos(kx x + kz z + t_phase), D = lam * k^ * H sin(...), slopes -k H sin, dDx/dx = kx k^x H cos.
    -> (disp, norm) sampled at the texels (float64), A = H, the closed form, k."""
    kx, kz = 2 * np.pi * a[0] / L, 2 * np.pi * a[1] / L
    kk = np.hypot(kx, kz)
    ux, uz = kx / kk, kz / kk
    x = np.arange(n) * L / n

    def fields(x, z):
        th = kx * x + kz * z + t_phase
        c, s = np.cos(th), np.sin(th)
        return (lam * ux * H * s, c, lam * uz * H * s, np.ones_like(c)), (-kx * H * s, -kz * H * s, kx * ux * H * c,
                                                                          kz * uz * H * c), H * c
    X, Z = np.meshgrid(x, x, indexing="xy")
    d, g, _ = fields(X, Z)
    return np.stack(d, -1), np.stack(g, -1), fields, (kx, kz)


def test_oracle_against_analytic_wave():
    """The oracle itself: I = 0 samples against the closed form within the bilinear bound, the inversion against a float64
    Newton solution of p + Dh(p) = q on the closed form."""
    n, L, lam, H = 64, 200.0, -0.8, 1.3
    disp, norm, fields, (kx, kz) = _analytic_wave(n, L, lam, H)
    rng = np.random.default_rng(5)
    q = rng.uniform(-2 * L, 3 * L, (400, 2))
    delta = L / n
    bound = ((kx * delta) ** 2 + (kz * delta) ** 2) / 8
    r = query_oracle([(disp, norm)], [H], [L], [lam], q, 0, pos32=False)
    (dxf, _, dzf, _), (gx, gz, gzz, gww), h = fields(q[:, 0], q[:, 1])
    assert np.abs(r["height"] - h).max() <= bound * H * 1.0001
    s = sample(disp, q[:, 0] * n / L, q[:, 1] * n / L)
    assert np.abs(s[:, 0] - dxf).max() <= bound * abs(lam) * H * 1.0001
    sg = sample(norm, q[:, 0] * n / L, q[:, 1] * n / L)
    assert np.abs(sg[:, 0] - gx).max() <= bound * kx * H * 1.0001
    # inversion: Newton on the continuous field
    p = q.copy()
    for _ in range(50):
        (fx, _, fz, _), _, _ = fields(p[:, 0], p[:, 1])
        th = kx * p[:, 0] + kz * p[:, 1] + 0.4
        c = np.cos(th)
        # Jacobian of F(p) = p + Dh(p) - q
        j11 = 1 + lam * (kx / np.hypot(kx, kz)) * H * c * kx
        j12 = lam * (kx / np.hypot(kx, kz)) * H * c * kz
        j21 = lam * (kz / np.hypot(kx, kz)) * H * c * kx
        j22 = 1 + lam * (kz / np.hypot(kx, kz)) * H * c * kz
        fxv, fzv = p[:, 0] + fx - q[:, 0], p[:, 1] + fz - q[:, 1]
        det = j11 * j22 - j12 * j21
        p = p - np.stack([(j22 * fxv - j12 * fzv) / det, (-j21 * fxv + j11 * fzv) / det], -1)
    lip = abs(lam) * H * np.hypot(kx, kz)
    assert lip < 0.5
    r = query_oracle([(disp, norm)], [H], [L], [lam], q, 16, pos32=False)
    err = np.hypot(q[:, 0] + r["offset_x"] - p[:, 0], q[:, 1] + r["offset_z"] - p[:, 1])
    assert err.max() <= (bound * abs(lam) * H * np.sqrt(2) + lip ** 16 * abs(lam) * H) / (1 - lip)


def test_adaptor_query_surface_compiles(tmp_path):
    src = tmp_path / "q.cpp"
    src.write_text(r'''
#include <vector>
#include "wso_tessendorf_adaptor.hpp"
static_assert(sizeof(wso_surface_sample) == 32, "one 32-byte record per query");
float use(WSTessendorf& m) {
    std::vector<float> xz = {0.0f, 0.0f, 12.5f, -300.0f};
    std::vector<wso_surface_sample> out(2);
    m.QuerySurface(xz.data(), 2, out.data());
    m.QuerySurface(xz.data(), 2, out.data(), 0);
    return out[0].height + out[1].normal_y + out[1].offset_x + out[1].residual + out[0].w;
}
''')
    gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([gxx, "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)])


def test_record_dtype_matches_the_c_struct():
    import watersurfacerendering_b200 as W
    assert W.SURFACE_SAMPLE_DTYPE.itemsize == 32
    assert W.SURFACE_SAMPLE_DTYPE.names == FIELDS


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
CASCADE_L = (1000.0, 250.0, 61.0)


def _ocean(W, n, ncasc, fmt, seed=3, jacobian=False):
    ws = W.WSTessendorf(n, CASCADE_L[0], max_tiles=ncasc, max_slots=ncasc)
    ws.set_map_format(fmt)
    if jacobian:
        ws.SetComputeJacobian(True)
    for t in range(ncasc):
        ws.SetTileLength(CASCADE_L[t], t)
        ws.Prepare(seed=seed + t, tile=t)
    ws.compute_batch(np.full(ncasc, 7.25, F32), tiles=np.arange(ncasc, dtype=np.uint32))
    return ws


def _maps_of(ws, ncasc):
    A = ws.read_heights(0, ncasc)[0]
    maps = [(ws.copy_map(0, s), ws.copy_map(1, s)) for s in range(ncasc)]
    return maps, [F32(a) for a in A]


def _as_rows(rec):
    return np.ascontiguousarray(rec).view(F32).reshape(-1, 8)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["rgba32f", "rgba16f"])
@pytest.mark.parametrize("n", [512, 1024])
def test_device_equals_host_build_and_oracle(n, fmt):
    import watersurfacerendering_b200 as W
    rng = np.random.default_rng(n)
    for ncasc in (1, 3):
        ws = _ocean(W, n, ncasc, fmt)
        try:
            maps, A = _maps_of(ws, ncasc)
            lengths = [F32(l) for l in CASCADE_L[:ncasc]]
            lam = [F32(ws.GetDisplacementLambda(t)) for t in range(ncasc)]
            q = rng.uniform(-2 * CASCADE_L[0], 2 * CASCADE_L[0], (1 << 16, 2)).astype(F32)
            sc = _scales(maps, A)
            for I in (0, 4):
                dev = _as_rows(ws.query_surface(q, slots=tuple(range(ncasc)), iterations=I))
                host = host_query([d for d, _ in maps], [g for _, g in maps], A, lengths, lam, q, I)
                assert np.array_equal(dev.view(np.uint32), host.view(np.uint32)), \
                    f"N={n} {fmt} cascades={ncasc} I={I}: device and host build differ"
                # the offset against the oracle's iteration where that has converged (I = 0: everywhere)
                ref = query_oracle(maps, A, lengths, lam, q, I)
                ok = (ref["residual"] < 1e-3 * float(min(lengths)) / n) if I else np.ones(q.shape[0], bool)
                assert ok.sum() >= 500
                _assert_close(dev, ref, sc, 1e-5, where=ok, what=f"N={n} {fmt} cascades={ncasc} I={I}",
                              fields=("offset_x", "offset_z"))
                # every other field - the residual |offset + Dh(q + offset)| included - at the reported point, at every
                # query, folded or not.  (Against the oracle's own p the normal is ill-conditioned next to folds, where
                # 1 + lambda*dDx/dx nears 0: a last-bit difference of p moves it by more than the tolerance.)
                again = query_oracle(maps, A, lengths, lam, q, I, offset=(dev[:, 4], dev[:, 5]))
                again["offset_x"], again["offset_z"] = dev[:, 4], dev[:, 5]
                _assert_close(dev, again, sc, 1e-5, what=f"N={n} {fmt} cascades={ncasc} I={I} at the reported p")
        finally:
            ws.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["rgba32f", "rgba16f"])
def test_convention_pin_one_hot(fmt):
    """One wave vector off both axes, (m, n) = (N/2+3, N/2+5): h = 2 Re(h0) cos(kx x + kz z) at t = 0 with kx = 2 pi 5 / L,
    kz = 2 pi 3 / L.  Off-grid queries against the closed form within the bilinear bound: catches swapped m / n, a
    half-texel shift or a sign error that a comparison against an oracle sharing the convention could not."""
    import watersurfacerendering_b200 as W
    n, L, lam = 256, 400.0, -0.7
    m0, n0 = n // 2 + 3, n // 2 + 5
    h0 = np.zeros((n, n, 5), F32)
    re, im = 0.75, -0.4
    h0[m0, n0] = (re, im, re, -im, 0.0)
    kx, kz = 2 * np.pi * 5 / L, 2 * np.pi * 3 / L
    kk = np.hypot(kx, kz)
    H = 2 * re
    with W.WSTessendorf(n, L) as ws:
        ws.set_map_format(fmt)
        ws.SetLambda(lam)
        ws.ImportH0(h0)
        ws.compute_batch([0.0])
        rng = np.random.default_rng(9)
        q = rng.uniform(-1.5 * L, 2.5 * L, (4096, 2)).astype(F32)
        th = kx * q[:, 0].astype(np.float64) + kz * q[:, 1]
        delta = L / n
        bound = ((kx * delta) ** 2 + (kz * delta) ** 2) / 8
        slack = 2e-3 if fmt == "rgba16f" else 2e-5   # binary16 texels: 2^-11 relative
        r0 = ws.query_surface(q, iterations=0)
        assert np.abs(r0["height"] - H * np.cos(th)).max() <= (bound + slack) * H
        sx, sz = -kx * H * np.sin(th), -kz * H * np.sin(th)
        ex = 1 + lam * kx * (kx / kk) * H * np.cos(th)
        ez = 1 + lam * kz * (kz / kk) * H * np.cos(th)
        nv = np.stack([-sx / ex, np.ones_like(sx), -sz / ez], -1)
        nv /= np.linalg.norm(nv, axis=-1, keepdims=True)
        got = np.stack([r0["normal_x"], r0["normal_y"], r0["normal_z"]], -1)
        assert np.abs(got - nv).max() <= (bound + slack) * 4 * kk * H
        # one inversion step: offset = -Dh(q) = -(lam k^ H sin)
        r1 = ws.query_surface(q, iterations=1)
        dx, dz = lam * (kx / kk) * H * np.sin(th), lam * (kz / kk) * H * np.sin(th)
        assert np.abs(r1["offset_x"] + dx).max() <= (bound + slack) * abs(lam) * H
        assert np.abs(r1["offset_z"] + dz).max() <= (bound + slack) * abs(lam) * H
        assert np.all(r0["w"] == 1.0)


def _torch():
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available()
    return torch


@pytest.mark.gpu
@pytest.mark.parametrize("caller_stream", [False, True])
def test_stream_order_without_host_sync(caller_stream):
    torch = _torch()
    import watersurfacerendering_b200 as W
    n, t1, t2 = 512, 3.5, 41.0
    rng = np.random.default_rng(2)
    q = torch.from_numpy(rng.uniform(-1500, 1500, (8192, 2)).astype(F32)).cuda()
    with W.WSTessendorf(n, 1000.0) as ws:
        ws.Prepare(seed=17)
        stream = torch.cuda.Stream() if caller_stream else None
        if stream is not None:
            ws.set_stream(stream.cuda_stream)
        # synchronised references
        ws.compute_batch([t1])
        ws.sync()
        ref1 = ws.query_surface(q.cpu().numpy(), iterations=4)
        ws.compute_batch([t2])
        ws.sync()
        ref2 = ws.query_surface(q.cpu().numpy(), iterations=4)
        torch.cuda.synchronize()
        o1 = torch.empty((q.shape[0], 8), dtype=torch.float32, device="cuda")
        o2 = torch.empty_like(o1)
        # everything enqueued back to back on the context's stream
        ws.compute_batch([t1])
        ws.query_surface_device(q.data_ptr(), o1.data_ptr(), q.shape[0], iterations=4)
        ws.compute_batch([t2])
        ws.query_surface_device(q.data_ptr(), o2.data_ptr(), q.shape[0], iterations=4)
        ws.sync()
        assert np.array_equal(o1.cpu().numpy().view(np.uint32), _as_rows(ref1).view(np.uint32))
        assert np.array_equal(o2.cpu().numpy().view(np.uint32), _as_rows(ref2).view(np.uint32))
        assert not np.array_equal(_as_rows(ref1), _as_rows(ref2))
        if stream is not None:
            ws.set_stream(None)


@pytest.mark.gpu
def test_jacobian_channel_in_w():
    import watersurfacerendering_b200 as W
    n = 512
    rng = np.random.default_rng(4)
    q = rng.uniform(-800, 800, (4096, 2)).astype(F32)
    ws = _ocean(W, n, 1, "rgba32f", jacobian=True)
    try:
        maps, A = _maps_of(ws, 1)
        assert np.any(maps[0][0][..., 3] != 1.0)
        for I in (0, 4):
            r = _as_rows(ws.query_surface(q, iterations=I))
            ref = query_oracle(maps, A, [F32(CASCADE_L[0])], [F32(-1.0)], q, 0, offset=(r[:, 4], r[:, 5]))
            assert np.abs(r[:, 7] - ref["w"]).max() <= 1e-5 * float(np.abs(maps[0][0][..., 3]).max())
        ws.SetComputeJacobian(False)
        ws.compute_batch([7.25])
        r = ws.query_surface(q, iterations=4)
        assert np.all(r["w"] == 1.0)
    finally:
        ws.close()


@pytest.mark.gpu
def test_errors_state_and_launch_count():
    torch = _torch()
    import watersurfacerendering_b200 as W
    from watersurfacerendering_b200 import _lib as L
    lib = L.load()
    q = np.zeros((4, 2), F32)
    with W.WSTessendorf(256, 500.0, max_slots=3) as ws:
        ws.Prepare(seed=1)

        def expect_invalid(fn, *a, **k):
            with pytest.raises(L.WsoError) as e:
                fn(*a, **k)
            assert e.value.status == L.WSO_ERR_INVALID_ARG
            assert lib.wso_last_error(ws._h)

        expect_invalid(ws.query_surface, q)                    # slot 0 holds no frame yet
        ws.compute_batch([1.0])                                # slot 0 only
        ws.query_surface(q)
        expect_invalid(ws.query_surface, q, slots=(1,))        # never written
        expect_invalid(ws.query_surface, q, slots=(3,))        # >= max_slots
        expect_invalid(ws.query_surface, q, slots=())          # n_slots 0
        ws.compute_batch([1.0, 2.0, 3.0])
        expect_invalid(ws.query_surface, q, slots=(0, 1, 2, 0, 1))   # n_slots 5
        ws.query_surface(q, slots=(0, 1, 2, 0))
        expect_invalid(ws.query_surface, q, iterations=17)
        ws.query_surface(q, iterations=16)
        xz = torch.zeros((4, 2), dtype=torch.float32, device="cuda")
        out = torch.zeros((4 * 8 + 4,), dtype=torch.float32, device="cuda")
        expect_invalid(ws.query_surface_device, 0, out.data_ptr(), 4)
        expect_invalid(ws.query_surface_device, xz.data_ptr(), 0, 4)
        expect_invalid(ws.query_surface_device, xz.data_ptr(), out.data_ptr() + 4, 4)   # misaligned
        sl = np.zeros(1, np.uint32)
        assert lib.wso_query_surface(ws._h, 1, None, 0, 4, C.c_void_p(xz.data_ptr()), C.c_void_p(out.data_ptr())) \
            == L.WSO_ERR_INVALID_ARG
        assert lib.wso_query_surface(None, 1, sl.ctypes.data_as(C.c_void_p), 0, 4, None, None) == L.WSO_ERR_INVALID_ARG
        # a query launches exactly one kernel; n == 0 launches nothing
        k0 = ws.stats()["kernel_launches"]
        ws.query_surface_device(xz.data_ptr(), out.data_ptr(), 4, slots=(0, 1, 2))
        ws.query_surface(q, slots=(2,))
        ws.query_surface_device(0, 0, 0)
        assert ws.query_surface(np.zeros((0, 2), F32)).size == 0
        assert ws.stats()["kernel_launches"] == k0 + 2
        # non-finite coordinates: NaN records, no error
        r = ws.query_surface(np.array([[np.nan, 0.0], [np.inf, 1.0]], F32))
        assert np.all(np.isnan(r["height"]))
        # map resets make every slot unqueryable until a compute writes it again
        ws.set_map_format("rgba16f")
        expect_invalid(ws.query_surface, q)
        ws.compute_batch([1.0])
        ws.query_surface(q)
        expect_invalid(ws.query_surface, q, slots=(1,))
        ws.set_exportable(True)
        expect_invalid(ws.query_surface, q)
        ws.compute_batch([1.0])
        ws.query_surface(q)
        ws.SetTileSize(128)
        ws.Prepare(seed=1)
        expect_invalid(ws.query_surface, q)
        ws.ComputeWaves(2.0)
        r = ws.query_surface(q)
        assert np.all(np.isfinite(r["height"]))
