"""Ray casts (wso_raycast_surface): the first point of a segment at or under the displaced surface, marched over the maps
of 1..4 slots (cascades) with the surface-query sampling (tests/test_surface_query.py).

`raycast_oracle` below is a NumPy statement of the contract in include/wsocean.h ("Ray casts").  It rounds the unit
direction, the slab, the sample parameters and the march positions where the contract does (fp32), and evaluates the
heights in float64 through the query oracle's bilinear sampling.  It also returns, per ray, the smallest |f| = |y - H| of
every sample whose sign decided the ray's path, so that rays whose path hangs on a near-tie can be set aside.

CPU: the host build of the kernel body (tests/emu/emu_raycast.cpp, the same wso_query.cuh the sm_100a kernel compiles)
against the oracle, the oracle against closed forms, properties of the host build, and the slab bound on the library's
golden maps.  GPU (-m gpu): device records equal the host build's bit for bit on the library's own maps and their
surfaces equal wso_query_surface's, a one-hot spectrum pins the world-space convention, calls follow computes in stream
order, and the C ABI validates its arguments and keeps its state.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import test_surface_query as Q
from conftest import ROOT, load_golden
from emu import driver as E

F32 = np.float32
MISS, HIT, BELOW, UNRESOLVED, INVALID = 0, 1, 2, 3, 4
MARGIN = F32(1.0 + 2.0 ** -10)
RAY_FIELDS = ("distance", "x", "z", "status") + Q.FIELDS


# ---------------------------------------------------------------------------------------------------------------------
# host build of the ray-cast body
# ---------------------------------------------------------------------------------------------------------------------
_SHIM = None


def _shim():
    """tests/emu/emu_raycast.cpp, compiled once per session into a temporary directory (the tree may be read-only)."""
    global _SHIM
    if _SHIM is None:
        out = os.path.join(tempfile.mkdtemp(prefix="wso_emur_"), "libwsoemur.so")
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-std=c++17", "-O2", "-w", "-ffp-contract=off", "-fPIC", "-shared", "-I", E.CSRC,
                               "-o", out, os.path.join(E.HERE, "emu_raycast.cpp")])
        L = C.CDLL(out)
        vp = C.c_void_p
        L.wso_emur_raycast.argtypes = [C.c_int, C.c_uint32, C.c_int, vp, vp, vp, vp, vp, C.c_int, C.c_float, C.c_uint32,
                                       C.c_uint32, C.c_uint32, vp, vp]
        L.wso_emur_raycast.restype = C.c_int
        _SHIM = L
    return _SHIM


def host_raycast(maps, A, L, lam, rays, I, step, max_steps, refine):
    """Host build: maps = [(disp, norm), ...] (float32, or float16 = RGBA16F); rays (n, 8) -> (n, 12) float32 records
    (distance, x, z, status bits, the 8 sample fields)."""
    half = maps[0][0].dtype == np.float16
    dt = np.float16 if half else F32
    disp = [np.ascontiguousarray(d, dt) for d, _ in maps]
    norm = [np.ascontiguousarray(g, dt) for _, g in maps]
    ns = len(disp)
    pd = (C.c_void_p * ns)(*[d.ctypes.data for d in disp])
    pn = (C.c_void_p * ns)(*[g.ctypes.data for g in norm])
    a = np.ascontiguousarray(A, F32)
    lt = np.ascontiguousarray(L, F32)
    lm = np.ascontiguousarray(lam, F32)
    rays = np.ascontiguousarray(rays, F32).reshape(-1, 8)
    out = np.zeros((rays.shape[0], 12), F32)
    p = lambda x: x.ctypes.data_as(C.c_void_p)
    rc = _shim().wso_emur_raycast(1 if half else 0, disp[0].shape[0], ns, C.cast(pd, C.c_void_p), C.cast(pn, C.c_void_p),
                                  p(a), p(lt), p(lm), int(I), float(step), int(max_steps), int(refine), rays.shape[0],
                                  p(rays), p(out))
    assert rc == 0
    return out


def status_of(rec):
    return np.ascontiguousarray(rec[:, 3]).view(np.uint32)


def make_rays(o, d, tmax=np.inf):
    o, d = np.broadcast_arrays(np.atleast_2d(np.asarray(o, F32)), np.atleast_2d(np.asarray(d, F32)))
    r = np.zeros((o.shape[0], 8), F32)
    r[:, 0:3] = o
    r[:, 3] = np.broadcast_to(np.asarray(tmax, F32), (o.shape[0],))
    r[:, 4:7] = d
    return r


# ---------------------------------------------------------------------------------------------------------------------
# the oracle
# ---------------------------------------------------------------------------------------------------------------------
def slab_height(A):
    hb = F32(0.0)
    for s, a in enumerate(A):
        hb = abs(F32(a)) if s == 0 else F32(hb + abs(F32(a)))
    return F32(hb * MARGIN)


def unit_directions(d):
    """d^ as the contract rounds it (fp32), and the rays whose direction is INVALID."""
    d = np.asarray(d, F32)
    with np.errstate(all="ignore"):
        m = np.abs(d).max(axis=1)
        bad = ~np.isfinite(d).all(axis=1) | ~(m > 0)
        v = d / np.where(bad, F32(1), m)[:, None]
        ln = np.sqrt((v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1]) + v[:, 2] * v[:, 2])
        return v / ln[:, None], bad


def _reduce(x, L):
    xd = np.asarray(x, F32).astype(np.float64)
    Ld = np.float64(F32(L))
    return (xd - np.floor(xd / Ld) * Ld).astype(F32)


class _Heights:
    """H at march positions (p_s + t d^) in float64 with fp32 positions and offsets, as query_oracle(pos32=True)."""

    def __init__(self, maps, A, L, I):
        self.disp = [np.asarray(d, np.float64) for d, _ in maps]
        self.A = [np.float64(F32(a)) for a in A]
        n = self.disp[0].shape[0]
        self.nl = [F32(np.float64(n) / np.float64(F32(l))) for l in L]
        self.I = I

    def _pos(self, q, delta, nl):
        return ((q + delta.astype(F32)).astype(F32) * nl).astype(F32).astype(np.float64)

    def __call__(self, px, pz, ux, uz, t):
        sx, sz = (t * ux).astype(F32), (t * uz).astype(F32)
        qx = [(p + sx).astype(F32) for p in px]
        qz = [(p + sz).astype(F32) for p in pz]
        dx = np.zeros(t.shape[0])
        dz = np.zeros(t.shape[0])
        for _ in range(self.I):
            hx = np.zeros(t.shape[0])
            hz = np.zeros(t.shape[0])
            for s, d in enumerate(self.disp):
                v = Q.sample(d, self._pos(qx[s], dx, self.nl[s]), self._pos(qz[s], dz, self.nl[s]))
                hx += v[:, 0]
                hz += v[:, 2]
            dx, dz = (-hx).astype(F32).astype(np.float64), (-hz).astype(F32).astype(np.float64)
        h = np.zeros(t.shape[0])
        for s, d in enumerate(self.disp):
            h += self.A[s] * Q.sample(d, self._pos(qx[s], dx, self.nl[s]), self._pos(qz[s], dz, self.nl[s]))[:, 1]
        return h


def raycast_oracle(maps, A, L, rays, I, step, max_steps, refine, tol=0.0):
    """The contract with float64 heights.  -> status, distance (float32), the smallest |f| over the march samples, and
    per HIT the width of the bisection bracket at the first bisection sample with |f| < tol (0 if none): from there a
    height that differs by tol may choose the other half, so an fp32 build can end anywhere in that bracket."""
    rays = np.asarray(rays, F32).reshape(-1, 8)
    n = rays.shape[0]
    o, tmax = rays[:, 0:3], rays[:, 3]
    u, bad_d = unit_directions(rays[:, 4:7])
    invalid = bad_d | ~np.isfinite(o).all(axis=1) | ~(tmax >= 0)
    hb = slab_height(A)
    H = _Heights(maps, A, L, I)
    status = np.full(n, -1)
    dist = np.full(n, np.nan, F32)
    tight = np.full(n, np.inf)
    wtie = np.zeros(n)
    status[invalid] = INVALID
    below = ~invalid & (o[:, 1] < -hb)
    status[below] = BELOW
    dist[below] = 0
    live = status < 0
    oy = o[:, 1]
    with np.errstate(all="ignore"):
        t1 = ((hb - oy) / u[:, 1]).astype(F32)
        t2 = ((-hb - oy) / u[:, 1]).astype(F32)
    flat = u[:, 1] == 0
    entry = np.where(flat, F32(-np.inf), np.minimum(t1, t2))
    exit_ = np.where(flat, np.where(oy <= hb, F32(np.inf), F32(-np.inf)), np.maximum(t1, t2))
    s0 = np.where(entry > 0, entry, F32(0)).astype(F32)
    send = np.where(tmax < exit_, tmax, exit_).astype(F32)
    with np.errstate(invalid="ignore"):
        nomeet = live & ~(s0 <= send)
    status[nomeet] = MISS
    dist[nomeet] = np.inf
    live &= ~nomeet
    px = [_reduce(o[:, 0], l) for l in L]
    pz = [_reduce(o[:, 2], l) for l in L]

    def f(idx, t):
        y = (oy[idx] + (t * u[idx, 1]).astype(F32)).astype(F32).astype(np.float64)
        return y - H([p[idx] for p in px], [p[idx] for p in pz], u[idx, 0], u[idx, 2], t)

    lo = s0.copy()
    hi = s0.copy()
    for k in range(max_steps):
        idx = np.nonzero(live)[0]
        if idx.size == 0:
            break
        t = (s0[idx] + F32(F32(k) * F32(step))).astype(F32)
        last = ~(t < send[idx])
        t = np.where(last, send[idx], t).astype(F32)
        fv = f(idx, t)
        tight[idx] = np.minimum(tight[idx], np.abs(fv))
        under = fv <= 0
        h_idx = idx[under]
        hi[h_idx] = t[under]
        status[h_idx] = np.where((k == 0) & (s0[h_idx] == 0), BELOW, HIT)
        m_idx = idx[~under & last]
        status[m_idx] = MISS
        dist[m_idx] = np.inf
        rest = idx[~under & ~last]
        lo[rest] = t[~under & ~last]
        if k + 1 == max_steps:
            status[rest] = UNRESOLVED
            dist[rest] = lo[rest]
        live[h_idx] = False
        live[m_idx] = False
    hit = np.nonzero(status == HIT)[0]
    for _ in range(refine):
        if hit.size == 0:
            break
        mid = (lo[hit] + (F32(0.5) * (hi[hit] - lo[hit]).astype(F32)).astype(F32)).astype(F32)
        fv = f(hit, mid)
        first = (np.abs(fv) < tol) & (wtie[hit] == 0)
        wtie[hit[first]] = (hi[hit] - lo[hit])[first]
        under = fv <= 0
        hi[hit[under]] = mid[under]
        lo[hit[~under]] = mid[~under]
    sel = (status == HIT) | ((status == BELOW) & ~below)
    dist[sel] = hi[sel]
    assert not np.any(status < 0)
    return status, dist, tight, wtie


# ---------------------------------------------------------------------------------------------------------------------
# rays
# ---------------------------------------------------------------------------------------------------------------------
def _dirs(rng, n, lo_deg, hi_deg, up=False):
    el = np.radians(rng.uniform(lo_deg, hi_deg, n))
    az = rng.uniform(0, 2 * np.pi, n)
    s = 1.0 if up else -1.0
    # lengths other than 1: the contract normalises
    return np.stack([np.cos(el) * np.cos(az), s * np.sin(el), np.cos(el) * np.sin(az)], -1) * rng.uniform(0.3, 7.0, (n, 1))


def ray_mix(rng, hb, lengths, n=64):
    """Steep, grazing, upward, vertical and horizontal rays; origins near the origin, many tiles away and negative."""
    lmax = float(max(lengths))
    parts = []

    def org(k, y_lo, y_hi, far=False):
        span = 40 * lmax if far else 2 * lmax
        xz = rng.uniform(-span, span, (k, 2))
        return np.stack([xz[:, 0], rng.uniform(y_lo, y_hi, k), xz[:, 1]], -1)

    for far in (False, True):
        parts.append(make_rays(org(n, 1.2 * hb, 6 * hb, far), _dirs(rng, n, 30, 89)))         # steep
        parts.append(make_rays(org(n, 0.2 * hb, 1.5 * hb, far), _dirs(rng, n, 3, 12)))        # grazing
        parts.append(make_rays(org(n // 2, -0.5 * hb, 3 * hb, far), _dirs(rng, n // 2, 5, 80, up=True)))  # upward
        parts.append(make_rays(org(n // 2, -0.5 * hb, 3 * hb, far), [0.0, -2.5, 0.0]))        # vertical
        ho = org(n // 2, -0.9 * hb, 0.9 * hb, far)
        hd = _dirs(rng, n // 2, 0, 0)
        parts.append(make_rays(ho, hd, rng.uniform(0, 3 * lmax / 64, n // 2)))                 # horizontal, short
        parts.append(make_rays(org(n // 2, 1.2 * hb, 4 * hb, far), _dirs(rng, n // 2, 20, 60),
                               rng.uniform(0, 4 * hb, n // 2)))                                 # short range
    return np.concatenate(parts).astype(F32)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: host build against the oracle
# ---------------------------------------------------------------------------------------------------------------------
ALL_L = [F32(1000.0), F32(250.0), F32(61.0), F32(17.3)]


def _tol(A):
    """|f| below which a sample's sign may differ between fp32 and float64 heights."""
    return 2e-5 * float(slab_height(A))


@pytest.mark.parametrize("half", [False, True], ids=["rgba32f", "rgba16f"])
@pytest.mark.parametrize("ns", [1, 2, 3, 4])
def test_host_body_matches_oracle(ns, half):
    n = 64
    rng = np.random.default_rng(100 + 10 * ns + half)
    lengths = ALL_L[:ns]
    maps, A, lam = Q._random_cascades(rng, n, lengths, half)
    hb = float(slab_height(A))
    step = float(min(lengths)) / n / 8
    rays = ray_mix(rng, hb, lengths)
    for I in (0, 4):
        for max_steps, refine in ((8, 16), (3000, 10)):
            got = host_raycast(maps, A, lengths, lam, rays, I, step, max_steps, refine)
            st, dist, tight, wtie = raycast_oracle(maps, A, lengths, rays, I, step, max_steps, refine, _tol(A))
            sure = tight >= _tol(A)
            what = f"cascades={ns} I={I} max_steps={max_steps}"
            assert (~sure).sum() <= 0.02 * rays.shape[0], f"{what}: {(~sure).sum()} near-tie rays"
            assert np.array_equal(status_of(got)[sure], st[sure]), what
            assert np.any(st[sure] == MISS), what
            assert np.any(st[sure] == (HIT if max_steps > 8 else UNRESOLVED)), what
            g = got[:, 0].astype(np.float64)
            ok = sure & (st != INVALID)
            allow = np.maximum(step * 2.0 ** -refine, wtie[ok]) + 4 * np.spacing(np.abs(dist[ok]).astype(F32))
            fin = np.isfinite(dist[ok])
            assert np.all(np.abs(g[ok][fin] - dist[ok][fin]) <= allow[fin]), what
            assert np.array_equal(g[ok][~fin], dist[ok][~fin].astype(np.float64)), what


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the oracle against closed forms
# ---------------------------------------------------------------------------------------------------------------------
def test_oracle_constant_height():
    """H = A*c everywhere: the crossing of a ray is (oy - A c) / -d^y."""
    n, L, A, c = 32, 100.0, F32(2.0), F32(0.37)
    disp = np.zeros((n, n, 4), F32)
    disp[..., 1] = c
    disp[..., 3] = 1
    maps = [(disp, np.zeros((n, n, 4), F32))]
    rng = np.random.default_rng(3)
    o = np.stack([rng.uniform(-300, 300, 300), rng.uniform(1, 8, 300), rng.uniform(-300, 300, 300)], -1)
    rays = make_rays(o, _dirs(rng, 300, 5, 90))
    step, refine = L / n, 16
    st, dist, _, _ = raycast_oracle(maps, [A], [F32(L)], rays, 0, step, 4096, refine)
    assert np.all(st == HIT)
    u, _ = unit_directions(rays[:, 4:7])
    exact = (rays[:, 1].astype(np.float64) - np.float64(A) * np.float64(c)) / -u[:, 1].astype(np.float64)
    err = dist.astype(np.float64) - exact
    # at or under the surface, at most one refined interval past it; fp32 y and t*d^y: a few ulp of oy over d^y
    allow = 8 * np.spacing(rays[:, 1]).astype(np.float64) / -u[:, 1]
    assert np.all(err >= -allow) and np.all(err <= step * 2.0 ** -refine + allow)


def test_oracle_cosine_bilinear_brentq():
    """One cosine, lambda = 0: the bilinear surface's first crossing, solved with brentq between the march samples."""
    from scipy.optimize import brentq
    n, L, lam, Hamp = 64, 200.0, 0.0, 1.3
    disp, norm, _, _ = Q._analytic_wave(n, L, lam, 1.0)
    maps = [(disp.astype(F32), norm.astype(F32))]
    A = [F32(Hamp)]
    rng = np.random.default_rng(8)
    o = np.stack([rng.uniform(-2 * L, 2 * L, 300), rng.uniform(0.5, 6, 300), rng.uniform(-2 * L, 2 * L, 300)], -1)
    rays = make_rays(o, _dirs(rng, 300, 25, 90))
    step, refine = L / n, 18
    st, dist, tight, _ = raycast_oracle(maps, A, [F32(L)], rays, 0, step, 4096, refine)
    u, _ = unit_directions(rays[:, 4:7])
    hb = float(slab_height(A))
    d64 = np.asarray(maps[0][0], np.float64)
    checked = 0
    for i in np.nonzero((st == HIT) & (tight >= 1e-6))[0]:
        ox, oy, oz = rays[i, :3].astype(np.float64)
        ux, uy, uz = u[i].astype(np.float64)

        def g(t):
            t = np.atleast_1d(t)
            h = Q.sample(d64, (ox + t * ux) * n / L, (oz + t * uz) * n / L)[:, 1]
            return float((oy + t * uy - float(A[0]) * h)[0])

        s0 = max(0.0, (hb - oy) / uy)
        t_prev = s0
        k = 0
        while True:
            t = s0 + k * step
            if g(t) <= 0:
                break
            t_prev = t
            k += 1
        root = brentq(g, t_prev, t, xtol=1e-12) if t > t_prev else t
        assert -1e-4 <= float(dist[i]) - root <= step * 2.0 ** -refine + 1e-4, (i, float(dist[i]), root)
        checked += 1
    assert checked >= 250


# ---------------------------------------------------------------------------------------------------------------------
# CPU: properties of the host build
# ---------------------------------------------------------------------------------------------------------------------
def _property_setup(half, ns=3, seed=21):
    """Cascades long enough that origins in [150, 300] and the samples of the rays below stay inside [0, L_s) of every
    cascade: there the march positions equal the query's reduced positions, so the host query body re-evaluates f."""
    n = 64
    lengths = [F32(2000.0), F32(700.0), F32(450.0)][:ns]
    rng = np.random.default_rng(seed + half)
    maps, A, lam = Q._random_cascades(rng, n, lengths, half)
    return n, lengths, maps, A, lam, rng


def _host_height(maps, A, lengths, lam, x, z, I):
    return Q.host_query([d for d, _ in maps], [g for _, g in maps], A, lengths, lam,
                        np.stack([x, z], -1).astype(F32), I)


@pytest.mark.parametrize("half", [False, True], ids=["rgba32f", "rgba16f"])
def test_host_hits_properties(half):
    n, lengths, maps, A, lam, rng = _property_setup(half)
    hb = float(slab_height(A))
    step = 450.0 / n / 2
    refine, I = 14, 4
    k = 300
    o = np.stack([rng.uniform(150, 300, k), rng.uniform(0.3 * hb, 3 * hb, k), rng.uniform(150, 300, k)], -1)
    d = _dirs(rng, k, 15, 89)
    rays = make_rays(o, d, 140.0)
    rec = host_raycast(maps, A, lengths, lam, rays, I, step, 4096, refine)
    st = status_of(rec)
    hit = np.nonzero(st == HIT)[0]
    assert hit.size >= 200
    u, _ = unit_directions(rays[:, 4:7])
    # the surface record is the host query body at (x, z), bit for bit
    q = _host_height(maps, A, lengths, lam, rec[hit, 1], rec[hit, 2], I)
    assert np.array_equal(q.view(np.uint32), rec[hit, 4:].view(np.uint32))
    # x, z as the contract rounds them
    b = rec[hit, 0]
    assert np.array_equal(rec[hit, 1], (rays[hit, 0] + (b * u[hit, 0]).astype(F32)).astype(F32))
    assert np.array_equal(rec[hit, 2], (rays[hit, 2] + (b * u[hit, 2]).astype(F32)).astype(F32))
    # no march sample before the bracket is at or under the surface (re-evaluated with the query body)
    for i in hit:
        ox, oy, oz = rays[i, :3]
        s0 = max(F32(0), F32((slab_height(A) - oy) / u[i, 1]))
        ts = (s0 + (np.arange(4096, dtype=F32) * F32(step)).astype(F32)).astype(F32)
        ts = ts[ts < rec[i, 0]]
        if ts.size == 0:
            continue
        x = (ox + (ts * u[i, 0]).astype(F32)).astype(F32)
        z = (oz + (ts * u[i, 2]).astype(F32)).astype(F32)
        y = (oy + (ts * u[i, 1]).astype(F32)).astype(F32)
        h = _host_height(maps, A, lengths, lam, x, z, I)[:, 0]
        assert np.all(y > h), i
    # the hit's y is within the refine bound of the surface height there
    slope = 0.0
    for (dm, _), a, l in zip(maps, A, lengths):
        dy = np.asarray(dm[..., 1], np.float64)
        st_ = max(np.abs(np.diff(dy, axis=ax, append=dy.take([0], axis=ax))).max() for ax in (0, 1))
        slope += abs(float(a)) * 2 * st_ / (float(l) / n)
    slope /= 1 - 0.45        # the inversion is a contraction with Lipschitz constant < 0.45
    y_hit = (rays[hit, 1] + (b * u[hit, 1]).astype(F32)).astype(np.float64)
    bound = step * 2.0 ** -refine * (1 + slope) + 1e-5 * hb
    assert np.all(np.abs(y_hit - rec[hit, 4]) <= bound)
    assert np.all(y_hit <= rec[hit, 4] + 1e-5 * hb)


@pytest.mark.parametrize("half", [False, True], ids=["rgba32f", "rgba16f"])
def test_host_special_rays(half):
    n, lengths, maps, A, lam, rng = _property_setup(half, ns=2)
    hb = float(slab_height(A))
    step = float(min(lengths)) / n
    I = 4
    cast = lambda r, ms=4096, rf=16, st=step: host_raycast(maps, A, lengths, lam, r, I, st, ms, rf)
    k = 64
    xz = rng.uniform(-5000, 5000, (k, 2)).astype(F32)
    # vertical, downward from above the slab: x = ox, z = oz, the query record there
    r = cast(make_rays(np.stack([xz[:, 0], np.full(k, 2 * hb), xz[:, 1]], -1), [0.0, -1.0, 0.0]))
    assert np.all(status_of(r) == HIT)
    assert np.array_equal(r[:, 1], xz[:, 0]) and np.array_equal(r[:, 2], xz[:, 1])
    qr = _host_height(maps, A, lengths, lam, xz[:, 0], xz[:, 1], I)
    assert np.array_equal(r[:, 4:].view(np.uint32), qr.view(np.uint32))
    # origin under the surface: ORIGIN_BELOW, distance 0, the record at the origin
    h = qr[:, 0]
    for y in ((h - F32(0.05) * F32(hb)).astype(F32), np.full(k, -2 * hb, F32)):
        r = cast(make_rays(np.stack([xz[:, 0], y, xz[:, 1]], -1), _dirs(rng, k, -80, 80)))
        assert np.all(status_of(r) == BELOW) and np.all(r[:, 0] == 0)
        assert np.array_equal(r[:, 4:].view(np.uint32), qr.view(np.uint32))
    # upward from above the slab: MISS without a sample
    r = cast(make_rays(np.stack([xz[:, 0], np.full(k, 1.5 * hb), xz[:, 1]], -1), _dirs(rng, k, 1, 90, up=True)))
    assert np.all(status_of(r) == MISS) and np.all(r[:, 0] == np.inf) and np.all(np.isnan(r[:, 1:3]))
    assert np.all(np.isnan(r[:, 4:]))
    # a tiny budget: UNRESOLVED at the last sample; continuing from there finds what an unlimited cast finds, within a
    # step (the continued march samples a shifted grid)
    o = np.stack([xz[:, 0], np.full(k, 1.2 * hb), xz[:, 1]], -1)
    d = _dirs(rng, k, 20, 50)
    rays = make_rays(o, d)
    step = step / 16
    full = cast(rays, st=step)
    assert np.all(status_of(full) == HIT)
    part = cast(rays, ms=3, st=step)
    assert np.all(status_of(part) == UNRESOLVED) and np.all(np.isnan(part[:, 4:]))
    u, _ = unit_directions(rays[:, 4:7])
    s0 = ((F32(hb) - rays[:, 1]) / u[:, 1]).astype(F32)
    s0 = np.where(s0 > 0, s0, F32(0))
    assert np.array_equal(part[:, 0], (s0 + F32(2) * F32(step)).astype(F32))
    t = part[:, 0]
    rays2 = make_rays((o + t[:, None] * u).astype(F32), d)
    more = cast(rays2, st=step)
    assert np.all(status_of(more) == HIT)
    assert np.all(np.abs((t.astype(np.float64) + more[:, 0]) - full[:, 0]) <= step * 1.001)
    # INVALID rays leave their neighbours alone
    mixed = rays.copy()
    mixed[1::4, 4:7] = 0                    # zero direction
    mixed[2::4, 0] = np.nan                 # NaN origin
    mixed[3::4, 3] = -1                     # negative tmax
    r = cast(mixed, st=step)
    bad = np.zeros(k, bool)
    bad[1::4] = bad[2::4] = bad[3::4] = True
    assert np.all(status_of(r)[bad] == INVALID) and np.all(np.isnan(r[bad][:, [0, 1, 2] + list(range(4, 12))]))
    assert np.array_equal(r[~bad].view(np.uint32), full[~bad].view(np.uint32))
    for bad_ray in ([np.inf, 1, 0, 1, 0, -1, 0, 0], [0, 1, 0, np.nan, 0, -1, 0, 0], [0, 1, 0, 1, np.inf, -1, 0, 0],
                    [0, 1, 0, 1, np.nan, -1, 0, 0]):
        assert status_of(cast(np.array([bad_ray], F32)))[0] == INVALID
    # tmax = 0 inside the slab above the surface: one sample at 0, MISS
    r = cast(make_rays(np.stack([xz[:, 0], h + F32(0.05 * hb), xz[:, 1]], -1), [0, -1, 0], 0.0))
    assert np.all(status_of(r) == MISS)


@pytest.mark.parametrize("half", [False, True], ids=["rgba32f", "rgba16f"])
def test_host_tile_shift(half):
    """One cascade with L = 2N: origins on a 1/64-texel grid shifted by whole tile lengths march the same samples."""
    n = 64
    L = F32(2 * n)
    rng = np.random.default_rng(31 + half)
    maps, A, lam = Q._random_cascades(rng, n, [L], half)
    hb = float(slab_height(A))
    k = 200
    xz = (rng.integers(0, 64 * n, (k, 2)) * (float(L) / n / 64)).astype(F32)
    o = np.stack([xz[:, 0], np.full(k, 1.5 * hb), xz[:, 1]], -1).astype(F32)
    d = _dirs(rng, k, 5, 85)
    base = host_raycast(maps, A, [L], lam, make_rays(o, d), 4, float(L) / n, 4096, 16)
    assert np.sum(status_of(base) == HIT) >= 150
    for sh in (3, -7, 40):
        o2 = o.copy()
        o2[:, 0] += F32(sh * float(L))
        o2[:, 2] -= F32(sh * float(L))
        assert np.array_equal(o2[:, 0].astype(np.float64) - o[:, 0], np.full(k, sh * float(L)))
        other = host_raycast(maps, A, [L], lam, make_rays(o2, d), 4, float(L) / n, 4096, 16)
        assert np.array_equal(status_of(other), status_of(base))
        assert np.array_equal(other[:, 0], base[:, 0])


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the slab bound, the adaptor, the record layout
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["n64_default", "n256_default"])
def test_slab_bound_on_golden_maps(name):
    g, params = load_golden(name)
    rng = np.random.default_rng(5)
    n = g["disp"].shape[1]
    L = F32(params["tile_length"])
    for half in (False, True):
        dt = np.float16 if half else F32
        nf = g["disp"].shape[0]
        for frames in ([0], [0, nf - 1], [k % nf for k in range(4)], [nf - 1] * 4):
            maps = [(g["disp"][f].astype(dt), g["norm"][f].astype(dt)) for f in frames]
            A = [F32(g["A"][f]) for f in frames]
            assert max(float(np.abs(m[..., 1].astype(np.float64)).max()) for m, _ in maps) <= 1.0
            lengths = [F32(float(L) / (1 + 0.37 * s)) for s in range(len(frames))]
            lam = [F32(params["lam"])] * len(frames)
            q = rng.uniform(-3 * float(L), 3 * float(L), (20000, 2)).astype(F32)
            hb = slab_height(A)
            for I in (0, 4):
                h = Q.host_query([m for m, _ in maps], [g_ for _, g_ in maps], A, lengths, lam, q, I)[:, 0]
                assert np.all(np.abs(h) <= hb), (name, half, frames, I)
            # the sampled heights come close to the bound: the margin is small
            top = max(float(np.abs(g["disp"][f][..., 1]).max()) for f in frames)
            assert top == 1.0


def test_adaptor_raycast_surface_compiles(tmp_path):
    src = tmp_path / "r.cpp"
    src.write_text(r'''
#include <vector>
#include "wso_tessendorf_adaptor.hpp"
static_assert(sizeof(wso_ray_hit) == 48, "one 48-byte record per ray");
float use(WSTessendorf& m) {
    std::vector<float> rays = {0.0f, 10.0f, 0.0f, 500.0f, 0.3f, -1.0f, 0.1f, 0.0f};
    std::vector<wso_ray_hit> out(1);
    wso_ray_params p = {0.5f, 1024u, 16u, 4u};
    m.RaycastSurface(rays.data(), 1, out.data(), p);
    return out[0].distance + out[0].x + out[0].z + (out[0].status == WSO_RAY_HIT ? out[0].surface.height : 0.0f);
}
''')
    gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([gxx, "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)])


def test_record_dtype_matches_the_c_struct():
    import watersurfacerendering_b200 as W
    from watersurfacerendering_b200 import _lib as L
    assert W.RAY_HIT_DTYPE.itemsize == 48
    assert W.RAY_HIT_DTYPE.names == RAY_FIELDS
    assert (L.WSO_RAY_MISS, L.WSO_RAY_HIT, L.WSO_RAY_ORIGIN_BELOW, L.WSO_RAY_UNRESOLVED, L.WSO_RAY_INVALID) == \
        (MISS, HIT, BELOW, UNRESOLVED, INVALID)
    assert C.sizeof(L.WsoRayParams) == 16


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
CASCADE_L = (1000.0, 250.0, 61.0, 17.3)


def _ocean(W, n, ncasc, fmt, seed=3):
    ws = W.WSTessendorf(n, CASCADE_L[0], max_tiles=ncasc, max_slots=ncasc)
    ws.set_map_format(fmt)
    for t in range(ncasc):
        ws.SetTileLength(CASCADE_L[t], t)
        ws.Prepare(seed=seed + t, tile=t)
    ws.compute_batch(np.full(ncasc, 7.25, F32), tiles=np.arange(ncasc, dtype=np.uint32))
    return ws


def _rows(rec):
    return np.ascontiguousarray(rec).view(F32).reshape(-1, 12)


def _gpu_rays(rng, hb, k=2048):
    """Projectiles (5-50 m up, 10-80 degrees down), near-grazing rays (1-5 degrees down) and the CPU mix."""
    xz = rng.uniform(-3000, 3000, (k, 2))
    o = np.stack([xz[:, 0], rng.uniform(5, 50, k), xz[:, 1]], -1)
    proj = make_rays(o, _dirs(rng, k, 10, 80), 500.0)
    o = np.stack([xz[:, 1], rng.uniform(0.5 * hb, 2 * hb, k), xz[:, 0]], -1)
    graze = make_rays(o, _dirs(rng, k, 1, 5), 500.0)
    return np.concatenate([proj, graze, ray_mix(rng, hb, CASCADE_L[:1], 32)]).astype(F32)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["rgba32f", "rgba16f"])
@pytest.mark.parametrize("n", [512, 1024])
def test_device_equals_host_build_and_query(n, fmt):
    import watersurfacerendering_b200 as W
    rng = np.random.default_rng(n + 7)
    for ncasc in (1, 2, 3, 4):
        ws = _ocean(W, n, ncasc, fmt)
        try:
            slots = tuple(range(ncasc))
            maps, A = Q._maps_of(ws, ncasc)
            lengths = [F32(l) for l in CASCADE_L[:ncasc]]
            lam = [F32(ws.GetDisplacementLambda(t)) for t in range(ncasc)]
            rays = _gpu_rays(rng, float(slab_height(A)))
            step = float(min(lengths)) / n
            for I in (0, 4):
                kw = dict(step=step, max_steps=1024, refine=16, iterations=I)
                dev = _rows(ws.raycast_surface(rays[:, 0:3], rays[:, 4:7], rays[:, 3], slots=slots, **kw))
                host = host_raycast(maps, A, lengths, lam, rays, I, step, 1024, 16)
                what = f"N={n} {fmt} cascades={ncasc} I={I}"
                assert np.array_equal(dev.view(np.uint32), host.view(np.uint32)), what + ": device and host build differ"
                st = status_of(dev)
                # the statuses the comparison covers; with four cascades the finest step is 1.7-3.4 cm and many rays
                # spend the 1024-sample budget before they reach the surface, so the HIT count is modest there
                assert np.sum(st == HIT) >= 100 and np.any(st == MISS), what
                # the finest step of three or more cascades is short enough for grazing rays to spend the budget
                assert np.any(st == UNRESOLVED) or ncasc < 3, what
                hit = np.nonzero((st == HIT) | (st == BELOW))[0]
                q = Q._as_rows(ws.query_surface(dev[hit, 1:3], slots=slots, iterations=I))
                assert np.array_equal(q.view(np.uint32), dev[hit, 4:].view(np.uint32)), what
        finally:
            ws.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["rgba32f", "rgba16f"])
def test_convention_pin_one_hot(fmt):
    """The one-hot spectrum of test_surface_query: h = H cos(kx x + kz z) with kx = 2 pi 5 / L, kz = 2 pi 3 / L.
    Downward rays hit the closed-form surface within the bilinear bound (I = 0: the height field at the hit's x, z)."""
    from scipy.optimize import brentq
    import watersurfacerendering_b200 as W
    n, L, lam = 256, 400.0, -0.7
    m0, n0 = n // 2 + 3, n // 2 + 5
    h0 = np.zeros((n, n, 5), F32)
    re, im = 0.75, -0.4
    h0[m0, n0] = (re, im, re, -im, 0.0)
    kx, kz = 2 * np.pi * 5 / L, 2 * np.pi * 3 / L
    H = 2 * re
    delta = L / n
    bound = ((kx * delta) ** 2 + (kz * delta) ** 2) / 8
    slack = 2e-3 if fmt == "rgba16f" else 2e-5
    with W.WSTessendorf(n, L) as ws:
        ws.set_map_format(fmt)
        ws.SetLambda(lam)
        ws.ImportH0(h0)
        ws.compute_batch([0.0])
        rng = np.random.default_rng(12)
        k = 2048
        o = np.stack([rng.uniform(-1.5 * L, 2.5 * L, k), rng.uniform(2, 10, k), rng.uniform(-1.5 * L, 2.5 * L, k)], -1)
        d = _dirs(rng, k, 40, 90)
        step, refine = delta, 20
        r = ws.raycast_surface(o, d, slots=(0,), step=step, refine=refine, iterations=0)
        assert np.all(r["status"] == HIT)
        u, _ = unit_directions(np.asarray(d, F32))
        u = u.astype(np.float64)
        o = o.astype(F32).astype(np.float64)
        slope = H * np.hypot(kx, kz)
        err = []
        for i in range(k):
            g = lambda t: o[i, 1] + t * u[i, 1] - H * np.cos(kx * (o[i, 0] + t * u[i, 0]) + kz * (o[i, 2] + t * u[i, 2]))
            t = float(r["distance"][i])
            lo, hi = t - 2 * step, t + 2 * step
            if g(lo) > 0 > g(hi):
                err.append(abs(brentq(g, lo, hi, xtol=1e-10) - t) * (-u[i, 1] - slope * np.hypot(u[i, 0], u[i, 2])))
        assert len(err) >= 0.9 * k
        # a height error e moves the crossing by e / (-d^y - slope |d^h|) along the ray
        assert max(err) <= (bound + slack) * H + step * 2.0 ** -refine + 1e-4
        th = kx * r["x"].astype(np.float64) + kz * r["z"]
        assert np.abs(r["height"] - H * np.cos(th)).max() <= (bound + slack) * H


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
    rays_np = _gpu_rays(rng, 3.0, 2048)
    rays = torch.from_numpy(rays_np).cuda()
    kw = dict(step=61.0 / 512, max_steps=1024, refine=16, iterations=4)
    with W.WSTessendorf(n, 1000.0, max_tiles=2, max_slots=2) as ws:
        ws.SetTileLength(61.0, 1)
        ws.Prepare(seed=17)
        ws.Prepare(seed=18, tile=1)
        stream = torch.cuda.Stream() if caller_stream else None
        if stream is not None:
            ws.set_stream(stream.cuda_stream)
        tiles = np.array([0, 1], np.uint32)
        refs = []
        for t in (t1, t2):
            ws.compute_batch([t, t], tiles=tiles)
            ws.sync()
            refs.append(_rows(ws.raycast_surface(rays_np[:, 0:3], rays_np[:, 4:7], rays_np[:, 3], slots=(0, 1), **kw)))
        torch.cuda.synchronize()
        o1 = torch.empty((rays.shape[0], 12), dtype=torch.float32, device="cuda")
        o2 = torch.empty_like(o1)
        k0 = ws.stats()["kernel_launches"]
        ws.compute_batch([t1, t1], tiles=tiles)
        k1 = ws.stats()["kernel_launches"]
        ws.raycast_surface_device(rays.data_ptr(), o1.data_ptr(), rays.shape[0], slots=(0, 1), **kw)
        assert ws.stats()["kernel_launches"] == k1 + 1
        ws.compute_batch([t2, t2], tiles=tiles)
        ws.raycast_surface_device(rays.data_ptr(), o2.data_ptr(), rays.shape[0], slots=(0, 1), **kw)
        assert ws.stats()["kernel_launches"] == 2 * (k1 - k0) + k0 + 2
        ws.sync()
        assert np.array_equal(o1.cpu().numpy().view(np.uint32), refs[0].view(np.uint32))
        assert np.array_equal(o2.cpu().numpy().view(np.uint32), refs[1].view(np.uint32))
        assert not np.array_equal(refs[0], refs[1])
        if stream is not None:
            ws.set_stream(None)


@pytest.mark.gpu
def test_after_compute_async():
    """wso_compute_async, then a ray cast on the same stream with no host sync in between, sees the new frame."""
    torch = _torch()
    import watersurfacerendering_b200 as W
    rng = np.random.default_rng(6)
    rays_np = _gpu_rays(rng, 3.0, 1024)
    rays = torch.from_numpy(rays_np).cuda()
    kw = dict(step=1000.0 / 512, refine=12, iterations=2)
    with W.WSTessendorf(512, 1000.0) as ws:
        ws.Prepare(seed=5)
        refs = []
        for t in (2.0, 9.0):
            ws.compute_batch([t])
            refs.append(_rows(ws.raycast_surface(rays_np[:, 0:3], rays_np[:, 4:7], rays_np[:, 3], **kw)))
        out = torch.empty((rays.shape[0], 12), dtype=torch.float32, device="cuda")
        for t, ref in zip((2.0, 9.0), refs):
            ws.ComputeWavesAsync(t)
            ws.raycast_surface_device(rays.data_ptr(), out.data_ptr(), rays.shape[0], **kw)
            ws.sync()
            assert np.array_equal(out.cpu().numpy().view(np.uint32), ref.view(np.uint32))


@pytest.mark.gpu
def test_errors_state_and_launch_count():
    torch = _torch()
    import watersurfacerendering_b200 as W
    from watersurfacerendering_b200 import _lib as L
    lib = L.load()
    o = np.array([[0.0, 5.0, 0.0], [10.0, 5.0, -3.0]], F32)
    d = np.array([[0.2, -1.0, 0.1]], F32)
    with W.WSTessendorf(256, 500.0, max_slots=3) as ws:
        ws.Prepare(seed=1)
        kw = dict(step=1.0)

        def expect_invalid(fn, *a, **k):
            k0 = ws.stats()["kernel_launches"]
            with pytest.raises(L.WsoError) as e:
                fn(*a, **k)
            assert e.value.status == L.WSO_ERR_INVALID_ARG
            assert lib.wso_last_error(ws._h)
            assert ws.stats()["kernel_launches"] == k0

        expect_invalid(ws.raycast_surface, o, d, **kw)                      # slot 0 holds no frame yet
        ws.compute_batch([1.0])
        good = ws.raycast_surface(o, d, **kw)
        assert np.all(good["status"] == HIT)
        expect_invalid(ws.raycast_surface, o, d, slots=(1,), **kw)          # never written
        expect_invalid(ws.raycast_surface, o, d, slots=(3,), **kw)          # >= max_slots
        expect_invalid(ws.raycast_surface, o, d, slots=(), **kw)            # n_slots 0
        ws.compute_batch([1.0, 2.0, 3.0])
        expect_invalid(ws.raycast_surface, o, d, slots=(0, 1, 2, 0, 1), **kw)
        ws.raycast_surface(o, d, slots=(0, 1, 2, 0), **kw)
        for bad in (dict(step=0.0), dict(step=-1.0), dict(step=np.inf), dict(step=np.nan), dict(step=1.0, max_steps=0),
                    dict(step=1.0, max_steps=4097), dict(step=1.0, refine=25), dict(step=1.0, iterations=17)):
            expect_invalid(ws.raycast_surface, o, d, **bad)
        ws.raycast_surface(o, d, step=1e-30, max_steps=4096, refine=24, iterations=16)
        rays = torch.zeros((4, 8), dtype=torch.float32, device="cuda")
        rays[:, 1] = 5.0
        rays[:, 5] = -1.0
        out = torch.zeros((4 * 12 + 4,), dtype=torch.float32, device="cuda")
        expect_invalid(ws.raycast_surface_device, 0, out.data_ptr(), 4, **kw)
        expect_invalid(ws.raycast_surface_device, rays.data_ptr(), 0, 4, **kw)
        expect_invalid(ws.raycast_surface_device, rays.data_ptr(), out.data_ptr() + 4, 4, **kw)      # misaligned out
        expect_invalid(ws.raycast_surface_device, rays.data_ptr() + 8, out.data_ptr(), 3, **kw)      # misaligned rays
        sl = np.zeros(1, np.uint32)
        pr = L.WsoRayParams(1.0, 16, 4, 0)
        slp = sl.ctypes.data_as(C.c_void_p)
        rp, op = C.c_void_p(rays.data_ptr()), C.c_void_p(out.data_ptr())
        assert lib.wso_raycast_surface(ws._h, 1, slp, None, 4, rp, op) == L.WSO_ERR_INVALID_ARG
        assert lib.wso_raycast_surface(ws._h, 1, None, C.byref(pr), 4, rp, op) == L.WSO_ERR_INVALID_ARG
        assert lib.wso_raycast_surface(None, 1, slp, C.byref(pr), 4, rp, op) == L.WSO_ERR_INVALID_ARG
        assert lib.wso_raycast_surface_host(ws._h, 1, slp, C.byref(pr), 4, None, None) == L.WSO_ERR_INVALID_ARG
        # one launch per call; n == 0 launches nothing (and still checks its arguments)
        k0 = ws.stats()["kernel_launches"]
        ws.raycast_surface_device(rays.data_ptr(), out.data_ptr(), 4, slots=(0, 1, 2), **kw)
        ws.raycast_surface(o, d, slots=(2,), **kw)
        ws.raycast_surface_device(0, 0, 0, **kw)
        assert ws.raycast_surface(np.zeros((0, 3), F32), d, **kw).size == 0
        expect_invalid(ws.raycast_surface_device, 0, 0, 0, step=0.0)
        assert ws.stats()["kernel_launches"] == k0 + 2
        torch.cuda.synchronize()
        ref = ws.raycast_surface(rays[:, 0:3].cpu().numpy(), rays[:, 4:7].cpu().numpy(), slots=(0, 1, 2), **kw)
        assert np.array_equal(out[:48].view(4, 12).cpu().numpy(), _rows(ref), equal_nan=True)
        # bad rays are records, not errors
        r = ws.raycast_surface(np.array([[np.nan, 1, 0], [0, 1, 0]], F32), np.array([[0, -1, 0], [0, 0, 0]], F32), **kw)
        assert np.all(r["status"] == INVALID) and np.all(np.isnan(r["distance"]))
        # map resets make every slot unusable until a compute writes it again
        ws.set_map_format("rgba16f")
        expect_invalid(ws.raycast_surface, o, d, **kw)
        ws.compute_batch([1.0])
        ws.raycast_surface(o, d, **kw)
        expect_invalid(ws.raycast_surface, o, d, slots=(1,), **kw)
        ws.SetTileSize(128)
        ws.Prepare(seed=1)
        expect_invalid(ws.raycast_surface, o, d, **kw)
        ws.ComputeWaves(2.0)
        r = ws.raycast_surface(o, d, **kw)
        assert np.all(r["status"] == HIT)
