"""Wave spectra (include/wsocean.h, "Wave spectra"): Pierson-Moskowitz, JONSWAP and TMA with finite depth, directional
spreading and wave-number bands, built at Prepare time.

CPU: the host build (wso_spectrum_h0) against the float64 restatement in tests/spectrum_ref.py, that restatement against
closed forms, statistics of the counter generator, record properties and band partitions of cascades.
GPU: the device Prepare kernel against the host build, maps of device-prepared tiles against tests/spectral_ref.py,
export / import round trips, the default spectrum leaving every Prepare entry point unchanged, a banded three-cascade
context and argument validation.
"""
import ctypes as C
import math

import numpy as np
import pytest
import scipy.integrate
import scipy.optimize

import spectrum_ref as S
from watersurfacerendering_b200 import _lib as L

PHILLIPS, PM, JONSWAP, TMA = 0, 1, 2, 3
KIND_NAMES = {PM: "pierson_moskowitz", JONSWAP: "jonswap", TMA: "tma"}


def _params(n, tile_length, wind=(1.0, 1.0), speed=30.0, period=200.0):
    p = L.WsoParams()
    L.load().wso_default_params(C.byref(p))
    p.tile_size, p.tile_length = n, tile_length
    p.wind_dir_x, p.wind_dir_y, p.wind_speed, p.anim_period = wind[0], wind[1], speed, period
    return p


def _spec(kind=PHILLIPS, **kw):
    from watersurfacerendering_b200.surface import make_spectrum
    return make_spectrum(kind, **kw)


def _ref_spec(s):
    return S.spectrum(s.kind, s.fetch, s.depth, s.gamma, s.spread, (s.k_min, s.k_max), s.scale)


def _host(p, s, xi=None, seed=0):
    from watersurfacerendering_b200 import spectrum_h0
    return spectrum_h0(p, s, xi, seed)


def _xi(n, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))).astype(np.complex64)


def _ulp(a, b):
    ia = np.ascontiguousarray(a, np.float32).view(np.int32).astype(np.int64)
    ib = np.ascontiguousarray(b, np.float32).view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, np.int64(-2 ** 31) - ia, ia)
    ib = np.where(ib < 0, np.int64(-2 ** 31) - ib, ib)
    return np.abs(ia - ib)


def _assert_records(got, ref, what, max_ulp=1):
    assert got["omega"].tobytes() == ref["omega"].tobytes(), f"{what}: dispersion must be bit-exact"
    assert np.array_equal(got["re_c"], got["re"]) and np.array_equal(got["im_c"], -got["im"]), f"{what}: conj"
    n_diff = 0
    for f in ("re", "im"):
        d = _ulp(got[f], ref[f])
        assert d.max() <= max_ulp, f"{what}: {f} differs by {d.max()} ulp"
        n_diff += int(np.count_nonzero(d))
    return n_diff


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the host build against the float64 restatement
# ---------------------------------------------------------------------------------------------------------------------
# (kind, N, L, wind dir, U, depth, spread, band, fetch, gamma)
HOST_CASES = [
    (PM, 128, 1000.0, (1.0, 1.0), 30.0, np.inf, 0.0, (0.0, np.inf), 1e5, 3.3),
    (PM, 64, 250.0, (0.3, -1.0), 8.0, 20.0, 4.0, (0.05, 1.2), 1e5, 3.3),
    (JONSWAP, 128, 500.0, (-1.0, 0.2), 12.0, np.inf, 0.0, (0.0, np.inf), 4e4, 3.3),
    (JONSWAP, 64, 120.0, (0.0, 1.0), 20.0, 5.0, 10.0, (0.2, 3.0), 1e5, 5.0),
    (JONSWAP, 128, 60.0, (1.0, 0.0), 3.0, np.inf, 0.0, (1.0, np.inf), 2e3, 1.0),
    (TMA, 128, 800.0, (1.0, 1.0), 15.0, 20.0, 0.0, (0.0, np.inf), 1e5, 3.3),
    (TMA, 64, 200.0, (-0.6, -0.8), 10.0, 5.0, 2.0, (0.0, 1.0), 3e4, 3.3),
    (TMA, 64, 300.0, (0.7, 0.7), 25.0, np.inf, 0.0, (0.0, np.inf), 1e5, 3.3),
]


@pytest.mark.parametrize("case", range(len(HOST_CASES)))
@pytest.mark.parametrize("source", ["xi", "counter"])
def test_host_build_matches_float64_restatement(case, source):
    kind, n, length, wind, U, depth, spread, band, fetch, gamma = HOST_CASES[case]
    p = _params(n, length, wind, U)
    s = _spec(kind, fetch=fetch, depth=depth, gamma=gamma, spread=spread, k_band=band)
    if source == "xi":
        xi = _xi(n, case)
        got = _host(p, s, xi)
    else:
        got = _host(p, s, None, seed=11)
        xi = _counter_xi(n, 11)
    ref, P = S.records(n, length, wind, U, 200.0, _ref_spec(s), xi)
    _assert_records(got, ref, f"case {case} {source}")
    assert np.count_nonzero(got["re"]) > n  # the case lights part of the grid


def _counter_xi(n, seed):
    """The counter generator's Gaussian array (wso::counter_gauss in wso_host_prepare.cpp), restated: a 64-bit mix of
    (seed, m*N+n), then Box-Muller in float64."""
    M = (1 << 64) - 1

    def mix(x):
        x = (x + 0x9E3779B97F4A7C15) & M
        x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & M
        x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & M
        return x ^ (x >> 31)
    sm = mix(seed)
    out = np.zeros((n, n), np.complex64)
    for idx in range(n * n):
        u = mix(sm ^ mix((idx + 0x632BE59BD9B4E019) & M))
        u1 = ((u >> 40) + 1.0) * (1.0 / 16777216.0)
        u2 = ((u >> 8) & 0xFFFFFF) * (1.0 / 16777216.0)
        r = math.sqrt(-2.0 * math.log(u1))
        a = 2.0 * math.pi * u2
        out.flat[idx] = complex(np.float32(r * math.cos(a)), np.float32(r * math.sin(a)))
    return out


def test_phillips_through_spectrum_h0_equals_counter_h0():
    from watersurfacerendering_b200.slab import counter_h0
    for n, length, wind in ((64, 1000.0, (1.0, 1.0)), (128, 300.0, (0.2, -0.9))):
        p = _params(n, length, wind, 17.0)
        assert _host(p, _spec(PHILLIPS), None, seed=5).tobytes() == counter_h0(p, 5, 0, n).tobytes()
        xi = _xi(n, 3)
        ph = _host(p, _spec(PHILLIPS), xi)
        assert np.isfinite(ph["re"]).all() and np.count_nonzero(ph["re"]) > 0


def test_spectrum_h0_rows_are_a_slice_of_the_grid():
    from watersurfacerendering_b200 import spectrum_h0
    p = _params(64, 400.0, (1.0, 0.3), 11.0)
    s = _spec(JONSWAP, depth=30.0)
    full = spectrum_h0(p, s, None, 9)
    assert spectrum_h0(p, s, None, 9, m0=10, rows=7).tobytes() == full[10:17].tobytes()


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the restatement against closed forms
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("s", [0.05, 1.0, 4.0, 10.0, 40.0])
def test_directional_spreading_integrates_to_one(s):
    q = S.spreading_norm(s)
    # D depends on cos(theta) only: twice the integral over [0, pi] (quad copes with the |cos|^2s cusps at the ends)
    half, err = scipy.integrate.quad(lambda t: S.directional(math.cos(t), s, q), 0.0, math.pi, epsabs=1e-13, limit=400)
    assert abs(2.0 * half - 1.0) < 1e-9
    th = np.linspace(0.0, 2.0 * np.pi, 1001)
    assert np.allclose(S.directional(np.cos(th), s, q), S.directional(np.cos(th + np.pi), s, q))  # even in k


def test_pierson_moskowitz_grid_sum_is_m0():
    """Grid: N = 1024, L = 2000 m, U = 10 m/s: dk = 2 pi / L = kp / 23 resolves the peak (kp = omega_p^2 / g =
    0.072 rad/m) and the grid reaches |k| = 1.6 rad/m = 22 kp per axis, where the omega^-5 tail has left < 0.3 % of m0."""
    n, length, U = 1024, 2000.0, 10.0
    spec = S.spectrum(PM)
    _, _, k = S.grid(n, length)
    kx, kz, _ = S.grid(n, length)
    valid = k > np.float32(1e-5)
    inv = np.where(valid, np.float32(1) / np.where(valid, k, 1), 0).astype(np.float32)
    P, _ = S.energy(k[valid].astype(np.float64), (kx * inv)[valid], (kz * inv)[valid], (1.0, 0.0), U, spec, length)
    wp = 0.855 * S.G / U
    m0 = 0.0081 * S.G ** 2 / (5 * wp ** 4)
    assert abs(P.sum() / m0 - 1.0) < 0.01, P.sum() / m0


def test_tma_in_deep_water_equals_jonswap():
    k = np.geomspace(1e-3, 20.0, 4000)
    ux = np.cos(np.linspace(0, 7, k.size)).astype(np.float32)
    uz = np.sqrt(1 - ux.astype(np.float64) ** 2).astype(np.float32)
    pj, wj = S.energy(k, ux, uz, (1.0, 0.0), 12.0, S.spectrum(JONSWAP), 500.0)
    pt, wt = S.energy(k, ux, uz, (1.0, 0.0), 12.0, S.spectrum(TMA, depth=1e6), 500.0)
    assert np.array_equal(pj, pt) and np.array_equal(wj, wt)
    # and through the library: TMA at depth +inf builds the JONSWAP records
    p = _params(64, 500.0, (1.0, 0.0), 12.0)
    assert _host(p, _spec(TMA), None, 1).tobytes() == _host(p, _spec(JONSWAP), None, 1).tobytes()


@pytest.mark.parametrize("depth", [20.0, 5.0, 0.5])
def test_finite_depth_dispersion_relation(depth):
    """omega(k) solves omega^2 = g k tanh(k d): invert it with brentq and recover k."""
    for k in (0.01, 0.1, 0.5, 2.0, 10.0):
        w, cg = S.dispersion(np.float64(k), depth)
        kk = scipy.optimize.brentq(lambda x: S.G * x * math.tanh(x * depth) - w * w, 1e-9, 1e3, xtol=1e-15)
        assert abs(kk - k) <= 1e-10 * k
        h = 1e-6 * k
        num = (S.dispersion(np.float64(k + h), depth)[0] - S.dispersion(np.float64(k - h), depth)[0]) / (2 * h)
        assert abs(cg - num) <= 1e-6 * cg


# ---------------------------------------------------------------------------------------------------------------------
# CPU: statistics and record properties of the host build
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", [PM, JONSWAP, TMA])
def test_counter_generator_energy_within_5_sigma(kind):
    n, length, U = 256, 800.0, 14.0
    p = _params(n, length, (1.0, 0.4), U)
    s = _spec(kind, depth=25.0 if kind == TMA else np.inf)
    h = _host(p, s, None, seed=2024)
    _, P = S.records(n, length, (1.0, 0.4), U, 200.0, _ref_spec(s), np.ones((n, n), np.complex64))
    e = float(np.sum(h["re"].astype(np.float64) ** 2 + h["im"].astype(np.float64) ** 2))
    sigma = math.sqrt(float(np.sum(P * P)))
    assert abs(e - P.sum()) <= 5 * sigma, (e, P.sum(), sigma)


@pytest.mark.parametrize("kind", [PM, JONSWAP, TMA])
def test_deep_water_j_equals_phillips_j_in_band(kind):
    n, length = 128, 700.0
    p = _params(n, length, (0.5, 1.0), 9.0)
    from watersurfacerendering_b200.slab import counter_h0
    ph = counter_h0(p, 3, 0, n)
    sp = _host(p, _spec(kind, k_band=(0.02, 0.5)), None, 3)
    lit = sp["re"] != 0
    assert lit.sum() > 100
    assert np.array_equal(sp["omega"][lit], ph["omega"][lit])


@pytest.mark.parametrize("kind", [PM, JONSWAP, TMA])
def test_records_are_point_symmetric_and_banded(kind):
    n, length = 128, 400.0
    band = (0.05, 0.9)
    p = _params(n, length, (0.8, -0.3), 11.0)
    s = _spec(kind, depth=15.0 if kind == TMA else np.inf, k_band=band)
    h = _host(p, s, np.full((n, n), 1 + 1j, np.complex64))
    assert np.array_equal(h["re_c"], h["re"]) and np.array_equal(h["im_c"], -h["im"])
    # P(k) == P(-k): record (m, c) and (N-m, N-c) carry the same amplitude bit for bit (xi = 1 + i everywhere)
    inner = h[1:, 1:]
    assert inner["re"].tobytes() == inner[::-1, ::-1]["re"].tobytes()
    assert inner["omega"].tobytes() == inner[::-1, ::-1]["omega"].tobytes()
    _, _, k = S.grid(n, length)
    out = ~((k >= np.float32(band[0])) & (k < np.float32(band[1])))
    assert np.all(h["re"][out] == 0) and np.all(h["im"][out] == 0) and np.all(h["omega"][out] == 0)
    assert np.all(h["omega"][h["re"] == 0] == 0)


EXTREMES = [
    dict(speed=1e-4, length=1e6), dict(speed=1e-4, length=0.01), dict(speed=3e4, length=1e6),
    dict(speed=3e4, length=0.01), dict(speed=10.0, length=1000.0, fetch=1e-3), dict(speed=10.0, length=1000.0, fetch=1e12),
    dict(speed=1e3, length=5.0, depth=1e-3), dict(speed=10.0, length=1e5, depth=1e-30), dict(speed=10.0, spread=1e6),
    dict(speed=10.0, spread=1e-6), dict(speed=10.0, gamma=1e6), dict(speed=10.0, scale=3.4e38),
    dict(speed=3e4, length=1e-3, scale=3.4e38, fetch=1e-30), dict(speed=1e-4, length=1e9, scale=0.0, fetch=1e30),
]


@pytest.mark.parametrize("kind", [PM, JONSWAP, TMA])
@pytest.mark.parametrize("ext", range(len(EXTREMES)))
def test_no_nan_or_inf_at_extreme_inputs(kind, ext):
    e = dict(EXTREMES[ext])
    p = _params(64, e.pop("length", 500.0), (0.3, 0.7), e.pop("speed"), period=e.pop("period", 200.0))
    h = _host(p, _spec(kind, **e), None, 7)
    for f in ("re", "im", "re_c", "im_c", "omega"):
        assert np.isfinite(h[f]).all(), f


def test_bands_partition_the_energy_of_cascades():
    """Three cascades (L = 1000, 250, 62.5) at one N with adjoining bands [0, c1), [c1, c2), [c2, inf): every wave vector
    that two grids share carries energy in at most one of them, and in exactly the one whose band holds it."""
    n, U = 256, 12.0
    lengths = (1000.0, 250.0, 62.5)
    cuts = (0.0, 0.4, 1.6, np.inf)
    recs = []
    for i, length in enumerate(lengths):
        p = _params(n, length, (1.0, 0.5), U)
        recs.append(_host(p, _spec(JONSWAP, k_band=(cuts[i], cuts[i + 1])), None, 100 + i))
    shared_lit = 0
    for a in range(3):
        for b in range(a + 1, 3):
            ratio = int(round(lengths[a] / lengths[b]))   # grid b's index step is `ratio` steps of grid a
            # integer wave-vector index q (kx = 2 pi q / L) <-> array index q + N/2 on both grids
            qb = np.arange(-n // 2, n // 2)
            qa = qb * ratio
            ok = (qa >= -n // 2) & (qa < n // 2)
            ia, ib = qa[ok] + n // 2, qb[ok] + n // 2
            ea = recs[a]["re"][np.ix_(ia, ia)] != 0
            eb = recs[b]["re"][np.ix_(ib, ib)] != 0
            assert not np.any(ea & eb), f"cascades {a} and {b} both carry energy at a shared wave vector"
            shared_lit += int(np.count_nonzero(ea | eb))
    assert shared_lit > 100


def test_spectrum_h0_rejects_invalid_arguments():
    lib = L.load()
    p = _params(64, 500.0)
    out = np.zeros(64 * 64 * 5, np.float32)

    def call(s, m0=0, rows=64, pp=p):
        return lib.wso_spectrum_h0(C.byref(pp), C.byref(s), None, 1, m0, rows, out.ctypes.data_as(C.c_void_p))

    assert call(_spec(JONSWAP)) == L.WSO_OK
    for s in _invalid_spectra():
        assert call(s) == L.WSO_ERR_INVALID_ARG, _fields(s)
    assert call(_spec(JONSWAP), m0=60, rows=5) == L.WSO_ERR_INVALID_ARG
    bad = _params(64, -1.0)
    assert call(_spec(JONSWAP), pp=bad) == L.WSO_ERR_INVALID_ARG
    assert lib.wso_spectrum_h0(None, C.byref(_spec(JONSWAP)), None, 1, 0, 64, out.ctypes.data_as(C.c_void_p)) \
        == L.WSO_ERR_INVALID_ARG
    d = L.WsoSpectrum()
    assert lib.wso_default_spectrum(C.byref(d)) == L.WSO_OK
    assert _fields(d) == _fields(_spec(PHILLIPS))
    assert lib.wso_default_spectrum(None) == L.WSO_ERR_INVALID_ARG


def _fields(s):
    return tuple(getattr(s, f) for f, _ in L.WsoSpectrum._fields_)


def _invalid_spectra():
    nan, inf = float("nan"), float("inf")
    bad = [dict(kind=4), dict(kind=99)]
    bad += [dict(kind=JONSWAP, fetch=v) for v in (0.0, -1.0, nan, inf)]
    bad += [dict(kind=TMA, depth=v) for v in (0.0, -5.0, nan, -inf)]
    bad += [dict(kind=JONSWAP, gamma=v) for v in (0.99, nan, inf)]
    bad += [dict(kind=PM, spread=v) for v in (-1.0, nan, inf)]
    bad += [dict(kind=PM, k_band=v) for v in ((-0.1, 1.0), (nan, 1.0), (inf, inf), (1.0, 1.0), (2.0, 1.0), (0.0, nan))]
    bad += [dict(kind=PM, scale=v) for v in (-1.0, nan, inf)]
    bad += [dict(kind=PHILLIPS, depth=10.0), dict(kind=PHILLIPS, scale=2.0), dict(kind=PHILLIPS, k_band=(0.1, inf)),
            dict(kind=PHILLIPS, fetch=5e4), dict(kind=PHILLIPS, gamma=2.0), dict(kind=PHILLIPS, spread=3.0)]
    out = []
    for b in bad:
        b = dict(b)
        kind = b.pop("kind")
        s = _spec(PM if kind > TMA else kind, **b)
        s.kind = kind
        out.append(s)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _ws(W, n, length, kind, tiles=1, slots=1, wind=(1.0, 0.6), U=11.0, **kw):
    ws = W.WSTessendorf(n, length, max_tiles=tiles, max_slots=slots)
    for t in range(tiles):
        ws.SetWindDirection(wind, t)
        ws.SetWindSpeed(U, t)
        ws.SetLambda(-0.9, t)
        if kind != PHILLIPS:
            ws.set_spectrum(KIND_NAMES[kind], t, **kw)
    return ws


def _ctx_params(ws, tile=0):
    return ws._get(tile)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [PM, JONSWAP, TMA])
@pytest.mark.parametrize("n", [64, 512, 1024])
@pytest.mark.parametrize("entry", ["gauss_device", "counter"])
def test_gpu_device_prepare_equals_host_build(kind, n, entry):
    import watersurfacerendering_b200 as W
    length = 1000.0 * n / 512
    kw = dict(depth=30.0 if kind == TMA else np.inf, k_band=(0.0, 2.0) if kind == JONSWAP else (0.0, np.inf))
    with _ws(W, n, length, kind, **kw) as ws:
        s = L.WsoSpectrum()
        L.check(ws._lib.wso_get_spectrum(ws._h, 0, C.byref(s)))
        if entry == "gauss_device":
            xi = _xi(n, n + kind)
            ws.PrepareWithGaussOnDevice(xi)
            want = _host(_ctx_params(ws), s, xi)
            # the host Prepare entry point builds the same records through the same arithmetic
            with _ws(W, n, length, kind, **kw) as wh:
                wh.PrepareWithGauss(xi)
                assert wh.ExportH0().tobytes() == want.tobytes()
        else:
            ws.PrepareCounterOnDevice(77)
            want = _host(_ctx_params(ws), s, None, 77)
        got = ws.ExportH0()
    n_diff = _assert_records(got, want, f"{KIND_NAMES[kind]} N={n} {entry}")
    print(f"{KIND_NAMES[kind]} N={n} {entry}: {n_diff} of {2 * n * n} amplitude components differ by 1 ulp")


def _frame_check(ws, h0, length, lam, t, what):
    import spectral_ref as R
    from test_spectral_coverage import check_maps
    a = ws.ComputeWaves(t)
    ref = R.Frame(h0["re"], h0["im"], h0["omega"], length, lam, t, dense=True)
    check_maps(ws.GetDisplacements(), ws.GetNormals(), a, ws.GetMinHeight(), ws.GetMaxHeight(), ref, what,
               path="spectrum")
    return a


# (kind, N, L, U, depth, table path?)
MAP_CASES = [(JONSWAP, 512, 1000.0, 14.0, np.inf, True), (TMA, 512, 400.0, 10.0, 12.0, True),
             (JONSWAP, 1024, 20.0, 3.0, np.inf, False), (TMA, 1024, 20.0, 3.0, 4.0, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(MAP_CASES)))
def test_gpu_maps_of_device_prepared_spectrum_vs_float64_reference(case):
    import watersurfacerendering_b200 as W
    kind, n, length, U, depth, table = MAP_CASES[case]
    with _ws(W, n, length, kind, U=U, depth=depth) as ws:
        ws.PrepareCounterOnDevice(5 + case)
        h0 = ws.ExportH0()
        w0 = S.omega0(200.0)
        jmax = int(np.max(np.rint(h0["omega"].astype(np.float64) / np.float64(w0))))
        assert (jmax < 1024) == table, f"jmax = {jmax}"
        for t in (0.0, 37.25):
            _frame_check(ws, h0, length, -0.9, t, f"{KIND_NAMES[kind]} N={n} L={length} t={t}")
        # round trip: the exported records, imported into a fresh context, give the same maps bit for bit
        a = ws.ComputeWaves(37.25)
        d, nm = ws.GetDisplacements().copy(), ws.GetNormals().copy()
        with _ws(W, n, length, PHILLIPS, U=U) as wi:
            wi.ImportH0(h0)
            assert wi.ExportH0().tobytes() == h0.tobytes()
            assert wi.ComputeWaves(37.25) == a
            assert np.array_equal(wi.GetDisplacements(), d) and np.array_equal(wi.GetNormals(), nm)


@pytest.mark.gpu
def test_gpu_default_spectrum_leaves_every_prepare_unchanged():
    import watersurfacerendering_b200 as W
    n, length = 256, 500.0
    xi = _xi(n, 42)
    entries = [lambda ws: ws.Prepare(seed=9), lambda ws: ws.PrepareWithGauss(xi),
               lambda ws: ws.PrepareWithGaussOnDevice(xi), lambda ws: ws.PrepareCounterOnDevice(9)]
    for i, prep in enumerate(entries):
        outs = []
        for set_default in (False, True):
            with W.WSTessendorf(n, length) as ws:
                if set_default:
                    ws.set_spectrum("jonswap", depth=10.0)
                    ws.set_spectrum("phillips")
                    assert ws.get_spectrum() == W.surface.spectrum_dict(_spec(PHILLIPS))
                prep(ws)
                ws.ComputeWaves(3.5)
                outs.append((ws.ExportH0().tobytes(), ws.GetDisplacements().tobytes(), ws.GetNormals().tobytes()))
        assert outs[0] == outs[1], f"entry point {i}"


@pytest.mark.gpu
def test_gpu_banded_cascades_compute_and_query():
    import watersurfacerendering_b200 as W
    n = 512
    lengths = (1000.0, 250.0, 62.5)
    cuts = (0.0, 0.4, 1.6, np.inf)
    ws = W.WSTessendorf(n, lengths[0], max_tiles=3, max_slots=3)
    with ws:
        for t, length in enumerate(lengths):
            ws.SetTileLength(length, t)
            ws.SetWindSpeed(12.0, t)
            ws.set_spectrum("tma", t, depth=40.0, k_band=(cuts[t], cuts[t + 1]))
            ws.PrepareCounterOnDevice(300 + t, tile=t)
        ws.compute_batch([4.0, 4.0, 4.0], tiles=[0, 1, 2], first_slot=0)
        ws.sync()
        a, mn, mx = ws.read_heights(0, 3)
        assert np.all(np.isfinite(a)) and np.all(np.asarray(a) > 0)
        xz = np.random.default_rng(1).uniform(-3000, 3000, (4096, 2)).astype(np.float32)
        q = ws.query_surface(xz, slots=(0, 1, 2), iterations=4)
        assert np.isfinite(q["height"]).all()
        # Hs of the sum lies near 4 sqrt(sum P) of the three bands (one realisation: within a factor 2)
        energy = 0.0
        for t, length in enumerate(lengths):
            h0 = ws.ExportH0(t)
            energy += float(np.sum(h0["re"].astype(np.float64) ** 2 + h0["im"].astype(np.float64) ** 2))
        hs_q = 4.0 * float(np.std(q["height"]))
        assert 0.5 < hs_q / (4.0 * math.sqrt(energy)) < 2.0


@pytest.mark.gpu
def test_gpu_set_spectrum_validation_leaves_state_unchanged():
    import watersurfacerendering_b200 as W
    with W.WSTessendorf(64, 200.0, max_tiles=2) as ws:
        ws.set_spectrum("tma", 1, depth=8.0, k_band=(0.1, 5.0), spread=3.0)
        before = [ws.get_spectrum(0), ws.get_spectrum(1)]
        for s in _invalid_spectra():
            for tile in (0, 1):
                assert ws._lib.wso_set_spectrum(ws._h, tile, C.byref(s)) == L.WSO_ERR_INVALID_ARG, _fields(s)
        assert ws._lib.wso_set_spectrum(ws._h, 2, C.byref(_spec(PM))) == L.WSO_ERR_INVALID_ARG
        assert ws._lib.wso_set_spectrum(ws._h, 0, None) == L.WSO_ERR_INVALID_ARG
        assert ws._lib.wso_get_spectrum(ws._h, 2, C.byref(L.WsoSpectrum())) == L.WSO_ERR_INVALID_ARG
        assert [ws.get_spectrum(0), ws.get_spectrum(1)] == before
