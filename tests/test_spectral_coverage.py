"""Every K1 -> K2h -> K2 path the library ships, against the float64 spectral reference (tests/spectral_ref.py).

Spectra:
  * white: every record - the Nyquist row and column (index 0), the DC lines (N/2) and the DC record included - has a
    magnitude of about 1/N and a random phase, so every wave vector carries about 1/N of the signal;
  * sparse: the indices {0, 1, N/2-1, N/2, N/2+1, N-1} crossed on both axes, points on the kx = -kz anti-diagonal (where
    every Prepare()-built spectrum with the default wind is zero) and random interior points; "mirrored" sets light k
    and -k, "one-sided" sets only one of them.
Dispersion classes (upload_h0() in wso_api.cu sorts an imported spectrum by them):
  (a) table + even: omega = fl(j omega0), j = f(|k|) - the FAST K1 bodies, warp-per-line set and persistent kernels;
  (b) table, odd: j(k) != j(-k);   (c) off the table, even: omega = 1.37 f(|k|);   (d) off the table, odd: random omega.
(b)-(d) run the general K1 body, and one such item demotes every other item of its launch to it.

Gates, from an fp32 error model (eps(N) = log2(N) 2^-24):
  * white spectra: per channel rel-L2 <= C_WHITE eps(N) (the Jacobian: rel-L2 of J - 1);
  * sparse spectra: per texel |err| <= C_SPARSE eps(N) sum_k |X_k|, X_k the channel's coefficient of wave vector k;
  * RGBA16F maps: the same, widened by the binary16 rounding (2^-11 relative, 2^-25 absolute).
Observed worst ratios err / (eps(N) scale) over every channel and A / min / max (the gate sits at about 4x the worst):
  CPU emulator of the kernel bodies (g++ -ffp-contract=off), N = 16 ... 2048, every shipped launch:
    white  0.73 (16)  2.00 (32)  1.47 (64)  1.19 (128)  1.16 (256)  1.57 (512)  1.25 (1024)  1.10 (2048)
    sparse 0.48 (16)  1.30 (32)  1.55 (64)  1.07 (128)  1.36 (256)  2.03 (512)  1.54 (1024)  0.89 (2048)
  B200 (1000 W power limit), every GPU test below (single frames, Bulk batches under every mask, c4, the Jacobian,
  the K2 split, the slab path):
    white  0.74 (16)  1.48 (32)  1.09 (64)  0.87 (128)  0.90 (256)  1.64 (512)  0.93 (1024)  0.94 (2048)  0.97 (4096)
    sparse 0.39 (64)  0.71 (256)  1.67 (512, c4)  0.83 (2048)  1.17 (8192)
  WSO_SPECTRAL_RATIOS=<file> appends every observation as a JSON line.
"""
import json
import math
import os
import subprocess
import sys
from functools import lru_cache

import numpy as np
import pytest

import spectral_ref as R
from oracle import port as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C_WHITE = 8.0
C_SPARSE = 8.0
F16_REL = 2.0 ** -11
F16_ABS = 2.0 ** -25
ANIM_PERIOD = 200.0   # the default animation period: omega0 of the table classes
CLASSES = "abcd"


def eps(n):
    return math.log2(n) * 2.0 ** -24


# ---------------------------------------------------------------------------------------------------------------------
# spectra
# ---------------------------------------------------------------------------------------------------------------------
def white_records(n, rng):
    mag = (0.5 + rng.random((n, n))) / n
    ph = rng.random((n, n)) * 2 * np.pi
    return (mag * np.cos(ph)).astype(np.float32), (mag * np.sin(ph)).astype(np.float32)


def sparse_records(n, rng, mirrored):
    """A few lit records; mirrored: the set is closed under k -> -k (index i -> (N - i) mod N)."""
    special = sorted({0, 1, n // 2 - 1, n // 2, n // 2 + 1, n - 1})
    pts = {(m, c) for m in special for c in special}
    pts |= {(m, (n - m) % n) for m in (1, n // 4, n // 2 - 1, n // 2 + 1, 3 * n // 4 + 1)}  # kx = -kz
    pts |= {(int(a), int(b)) for a, b in rng.integers(1, n, (6, 2))}
    mirror = lambda p: ((n - p[0]) % n, (n - p[1]) % n)
    if mirrored:
        pts |= {mirror(p) for p in pts}
    else:
        pts = {p for p in pts if p <= mirror(p)}
    re = np.zeros((n, n), np.float32)
    im = np.zeros((n, n), np.float32)
    for m, c in sorted(pts):
        mag, ph = 0.5 + rng.random(), 2 * np.pi * rng.random()
        re[m, c], im[m, c] = mag * np.cos(ph), mag * np.sin(ph)
    return re, im


def omega0():
    return np.float32(np.float64(np.float32(2.0)) * np.pi / np.float64(np.float32(ANIM_PERIOD)))


def dispersion(cls, n, tile_length, rng):
    kv = R.wave_numbers(n, tile_length)
    k = np.sqrt(kv[None, :] * kv[None, :] + kv[:, None] * kv[:, None]).astype(np.float32)
    w0 = omega0()
    j = np.minimum(np.floor(np.sqrt(np.float32(9.81) * k) / w0), 1000).astype(np.int32)
    if cls == "b":
        j = np.minimum(j + rng.integers(0, 24, (n, n)), 1023).astype(np.int32)
    om = (j.astype(np.float32) * w0).astype(np.float32)
    if cls == "c":
        om = (om * np.float32(1.37)).astype(np.float32)
    elif cls == "d":
        om = rng.uniform(0.0, 6.0, (n, n)).astype(np.float32)
    return om


# (tile length / N, lambda, t) of the two items every emulated launch carries
ITEM_PARAMS = [(1.0, -0.8, 13.7), (0.75, 1.3, 2.25)]


@lru_cache(maxsize=64)
def item(n, spec, cls, which=0, seed=0):
    """spec: 'white', 'sparse' (mirrored) or 'sparse1' (one-sided).  -> dict for emu.driver.compute_shipped / the GPU."""
    rng = np.random.default_rng([n, "wsS".find(spec[0]) + 7 * len(spec), CLASSES.index(cls), which, seed])
    lf, lam, t = ITEM_PARAMS[which]
    tile_length = lf * n
    re, im = white_records(n, rng) if spec == "white" else sparse_records(n, rng, spec == "sparse")
    om = dispersion(cls, n, tile_length, rng)
    return dict(re=re, im=im, omega=om, tile_length=tile_length, lam=lam, t=t, anim_period=ANIM_PERIOD)


@lru_cache(maxsize=32)
def reference(n, spec, cls, which=0, seed=0, t=None, lam=None, jacobian=False):
    it = item(n, spec, cls, which, seed)
    return R.Frame(it["re"], it["im"], it["omega"], it["tile_length"], it["lam"] if lam is None else lam,
                   it["t"] if t is None else t, jacobian=jacobian, dense=spec == "white")


def h0_records(it):
    h0 = np.zeros(it["re"].shape, P.H0_DTYPE)
    h0["re"], h0["im"], h0["re_c"], h0["im_c"], h0["omega"] = it["re"], it["im"], it["re"], -it["im"], it["omega"]
    return h0


# ---------------------------------------------------------------------------------------------------------------------
# the gate
# ---------------------------------------------------------------------------------------------------------------------
_RATIOS = []


def _log_ratio(**kw):
    _RATIOS.append(kw)
    path = os.environ.get("WSO_SPECTRAL_RATIOS")
    if path:
        with open(path, "a") as f:
            f.write(json.dumps(kw) + "\n")


def check_maps(disp, norm, a, mn, mx, ref, what, path, half=False):
    """disp / norm: the kernel's maps of one tile-frame ([N, N, 4], float32 or float16); a, mn, mx: its A, min, max."""
    n = ref.n
    e = eps(n)
    jac = ref.jacobian
    acc = np.zeros((8, 5))   # per channel (disp 0..3, norm 0..3): sum err^2, sum sig^2, sum ref^2, max err, max excess
    for r0, d_ref, n_ref in ref.blocks():
        rows = slice(r0, r0 + d_ref.shape[0])
        for ci, (got, rf) in enumerate(((disp, d_ref), (norm, n_ref))):
            g = np.asarray(got[rows], np.float64)
            for c in range(4):
                k = 4 * ci + c
                if ci == 0 and c == 3 and not jac:
                    assert np.all(g[..., 3] == 1.0), f"{what}: disp.w must be exactly 1.0"
                    continue
                err = np.abs(g[..., c] - rf[..., c])
                sig = rf[..., c] - 1.0 if k == 3 else rf[..., c]
                acc[k, 0] += float(np.sum(err * err))
                acc[k, 1] += float(np.sum(sig * sig))
                acc[k, 2] += float(np.sum(rf[..., c] ** 2))
                acc[k, 3] = max(acc[k, 3], float(err.max()))
                excess = err - F16_REL * np.abs(rf[..., c]) - F16_ABS if half else err
                acc[k, 4] = max(acc[k, 4], float(excess.max()))
    names = ["disp.x", "disp.y", "disp.z", "disp.w(J)", "norm.x", "norm.y", "norm.z", "norm.w"]
    worst = 0.0
    if ref.dense:
        for k in range(8):
            if k == 3 and not jac:
                continue
            rel = math.sqrt(acc[k, 0] / acc[k, 1])
            tol = C_WHITE * e + (F16_REL * math.sqrt(acc[k, 2] / acc[k, 1]) if half else 0.0)
            assert rel <= tol, f"{what}: {names[k]} rel-L2 {rel:.3e} > {tol:.3e} ({rel / e:.2f} eps)"
            worst = max(worst, rel / e)
        a_scale = ref.A
    else:
        ds, ns = ref.texel_scale()
        scale = np.concatenate([ds, ns])
        for k in range(8):
            if k == 3 and not jac:
                continue
            got_err = acc[k, 4]
            if scale[k] == 0.0:
                assert acc[k, 3] <= 1e-30, f"{what}: {names[k]} must be zero, max |x| = {acc[k, 3]:.3e}"
                continue
            tol = C_SPARSE * e * scale[k]
            assert got_err <= tol, f"{what}: {names[k]} max err {got_err:.3e} > {tol:.3e} ({got_err / (e * scale[k]):.3f})"
            worst = max(worst, acc[k, 3] / (e * scale[k]))
        a_scale = ref.sparse.abs_sum(0)
    c = C_WHITE if ref.dense else C_SPARSE
    for name, got, want in (("A", a, ref.A), ("min", mn, ref.hmin), ("max", mx, ref.hmax)):
        err = abs(float(got) - want)
        assert err <= c * e * a_scale, f"{what}: {name} {float(got)!r} vs {want!r} ({err / (e * a_scale):.2f})"
        worst = max(worst, err / (e * a_scale))
    if not half:
        _log_ratio(n=n, path=path, spectrum="white" if ref.dense else "sparse", what=what, ratio=round(worst, 4))
    return worst


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference itself
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [16, 64, 128])
@pytest.mark.parametrize("mirrored", [False, True])
def test_reference_dense_equals_sparse(n, mirrored):
    it = item(n, "sparse" if mirrored else "sparse1", "d")
    H = R.heights_spectrum(it["re"], it["im"], it["omega"], it["t"])
    dense = R.fields_dense(H, it["tile_length"])
    sparse = R.SparseTerms(H, it["tile_length"]).fields(np.arange(n))
    for f in range(R.N_FIELDS):
        scale = max(np.abs(dense[f]).max(), 1e-300)
        assert np.abs(dense[f] - sparse[f]).max() <= 1e-12 * scale, f


def test_reference_one_hot_closed_form():
    """One record h0 at (m0, c0): h(r, c) = (-1)^(r+c) H cos(2 pi (m0 r + c0 c) / N), slopes and displacements with their
    multipliers c(k), H = 2 Re(h0 e^{i phi})."""
    n, L, t = 32, 40.0, 3.0
    r, c = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    sign = np.where((r + c) & 1, -1.0, 1.0)
    kv = R.wave_numbers(n, L).astype(np.float64)
    for m0, c0 in [(3, 5), (0, 7), (n // 2, 1), (n - 1, n // 2), (0, 0)]:
        re = np.zeros((n, n), np.float32)
        im = np.zeros((n, n), np.float32)
        om = np.zeros((n, n), np.float32)
        re[m0, c0], im[m0, c0], om[m0, c0] = 0.7, -0.3, 0.31415927
        ph = float(np.float32(np.float32(0.31415927) * np.float32(t)))
        H = 2.0 * (float(np.float32(0.7)) * np.cos(ph) - float(np.float32(-0.3)) * np.sin(ph))
        theta = 2 * np.pi * ((m0 * r + c0 * c) % n) / n
        kx, kz = kv[c0], kv[m0]
        inv = float(R.inv_length(np.float32(kx), np.float32(kz)))
        fr = R.Frame(re, im, om, L, -1.0, t)
        d, nm = fr.whole()
        h = sign * H * np.cos(theta)
        assert np.abs(d[..., 1] * fr.A - h).max() <= 1e-12 * abs(H)
        assert np.abs(nm[..., 0] - sign * (-kx * H) * np.sin(theta)).max() <= 1e-12 * abs(H) * (abs(kx) + 1)
        assert np.abs(d[..., 0] - (-1.0) * sign * (kx * inv * H) * np.sin(theta)).max() <= 1e-12 * abs(H)
        assert np.abs(nm[..., 3] - sign * kz * kz * inv * H * np.cos(theta)).max() <= 1e-12 * abs(H) * (kz * kz + 1)


@pytest.mark.parametrize("name", ["n64_default", "n256_default"])
def test_reference_matches_oracle(name):
    """The float64 reference against the C++ restatement of the reference code (fp32 spectra, float64 FFT) on the
    fixture spectra: they differ by the fp32 rounding of the spectra only."""
    from conftest import load_golden
    g, params = load_golden(name)
    h0 = g["h0"]
    n = params["tile_size"]
    o = P.PortOracle(P.OceanParams(tile_size=n, tile_length=params["tile_length"], lam=params["lam"]))
    o.import_h0(h0.view(P.H0_DTYPE).reshape(n, n))
    for t in g["t"][:2]:
        a_ref, d_ref, n_ref = o.compute_waves(float(t))
        fr = R.Frame(h0[..., 0], h0[..., 1], h0[..., 4], params["tile_length"], params["lam"], float(t))
        d, nm = fr.whole()
        assert abs(fr.A - a_ref) <= 1e-6 * a_ref
        for got, want in ((d, d_ref), (nm, n_ref)):
            for ch in range(4):
                w = want[..., ch].astype(np.float64)
                assert np.linalg.norm(got[..., ch] - w) <= 4 * 2.0 ** -24 * math.log2(n) * max(np.linalg.norm(w), 1e-30)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the emulated kernel bodies at every shipped tiling
# ---------------------------------------------------------------------------------------------------------------------
def _emu():
    from emu import driver as E
    return E


EMU_LOGN = range(4, 12)


def _emulated_launches():
    """(logn, kind) of every launch the emulator can run: Lat, Bulk, Bulk with its persistent forms, Jacobian."""
    out = []
    for logn in EMU_LOGN:
        out += [(logn, 0), (logn, 1), (logn, 3)]
        if logn in (9, 10, 11):
            out.append((logn, 2))
    return out


def test_emulator_covers_every_shipped_tiling():
    """Every (size, tiling) launch_all() can pick up to 2048^2 - Lat and Bulk from wso_tilings.h, Bulk's persistent K1 / K2
    where PersistOk allows them - is one of the emulated launches below, and the emulator runs it through that header."""
    E = _emu()
    rows = E.shipped_tilings()
    assert sorted({r[0] for r in rows}) == list(range(4, 14))
    launches = set(_emulated_launches())
    for logn, kind, cp, nf, ri, rh, persist in rows:
        assert cp >= 1 and nf in (1, 2, 4) and ri >= 1 and rh >= 1
        if logn > 11:
            continue   # 4096^2 / 8192^2: GPU tests only
        assert (logn, kind) in launches
        if kind == 1:
            assert (logn, 3) in launches   # the Jacobian launch runs Bulk's K1 / K2h
            assert ((logn, 2) in launches) == (persist != 0), (logn, persist)


def _emu_cases():
    cases = []
    for logn, kind in _emulated_launches():
        combos = [(s, c) for s in ("white", "sparse1") for c in CLASSES]
        if logn == 11:   # the largest size on a subset of the classes
            combos = [("white", "a"), ("white", "d"), ("sparse1", "b")]
        cases += [(1 << logn, kind, s, c) for s, c in combos]
    return cases


@pytest.mark.parametrize("n,kind,spec,cls", _emu_cases())
def test_emulated_launch_vs_float64_reference(n, kind, spec, cls):
    """One launch of two items: item 0 of the given spectrum and class, item 1 a white class-(a) spectrum with another
    tile length, lambda and time - a class (b)-(d) item 0 demotes item 1 to the general K1 body as well."""
    E = _emu()
    jac = kind == E.KIND_JACOBIAN
    items = [item(n, spec, cls, 0), item(n, "white", "a", 1)]
    a, disp, norm, mn, mx, _ = E.compute_shipped(n, kind, items)
    for i, (s, c) in enumerate(((spec, cls), ("white", "a"))):
        ref = reference(n, s, c, i, jacobian=jac)
        check_maps(disp[i], norm[i], a[i], mn[i], mx[i], ref, f"emu N={n} kind={kind} {s}/{c} item {i}",
                   path=f"emu kind {kind}")


@pytest.mark.parametrize("logn,kind", [(l, k) for l, k in _emulated_launches() if l in (4, 6, 8, 9, 10)])
def test_emulated_f16_launch_vs_float64_reference(logn, kind):
    """RGBA16F maps (K2 with TEX = Half4) of every emulated launch, gate widened by the binary16 rounding."""
    E = _emu()
    n = 1 << logn
    jac = kind == E.KIND_JACOBIAN
    items = [item(n, "white", "d", 0), item(n, "sparse1", "a", 1)]
    a, disp, norm, mn, mx, _ = E.compute_shipped(n, kind, items, half=True)
    for i, (s, c) in enumerate((("white", "d"), ("sparse1", "a"))):
        check_maps(disp[i], norm[i], a[i], mn[i], mx[i], reference(n, s, c, i, jacobian=jac),
                   f"emu f16 N={n} kind={kind} item {i}", path=f"emu f16 kind {kind}", half=True)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _ws(W, n, its, max_slots=1, jacobian=False, fmt="rgba32f"):
    ws = W.WSTessendorf(n, its[0]["tile_length"], max_tiles=len(its), max_slots=max_slots)
    ws.set_map_format(fmt)
    for j, it in enumerate(its):
        ws.SetTileLength(it["tile_length"], j)
        ws.SetAnimationPeriod(ANIM_PERIOD, j)
        ws.SetLambda(it["lam"], j)
        ws.ImportH0(h0_records(it), tile=j)
    if jacobian:
        ws.SetComputeJacobian(True)
    return ws


def _single_frame_cases():
    return [(1 << l, c) for l in range(4, 14) for c in CLASSES]


@pytest.mark.gpu
@pytest.mark.parametrize("n,cls", _single_frame_cases())
def test_gpu_single_frame_vs_float64_reference(n, cls):
    """ComputeWaves(t) - the Lat tilings, one item per launch - with the frame graph off (0), up to 512^2 (1) and at every
    size (2), over the whole map: white spectra up to 4096^2, a one-sided sparse spectrum at 8192^2."""
    import watersurfacerendering_b200 as W
    spec = "white" if n <= 4096 else "sparse1"
    it = item(n, spec, cls)
    ref = reference(n, spec, cls)
    with _ws(W, n, [it]) as ws:
        first = None
        for mode in (0, 1, 2):
            ws.set_frame_graph(mode != 0, every_size=mode == 2)
            for rep in range(2):   # the first frame of a shape is a plain launch, the second one a graph launch
                a = ws.ComputeWaves(it["t"])
                d, nm = ws.GetDisplacements(), ws.GetNormals()
                if first is None:
                    check_maps(d, nm, a, ws.GetMinHeight(), ws.GetMaxHeight(), ref, f"N={n} {spec}/{cls}",
                               path="single frame")
                    first = (a, d.copy(), nm.copy())
                else:   # the same kernels with the same arguments: the same bits, graph launch or not
                    assert a == first[0] and np.array_equal(d, first[1]) and np.array_equal(nm, first[2]), \
                        f"N={n} {spec}/{cls} graph mode {mode} call {rep}"


# class (a) under every kernel-set mask; the other classes run the general K1 body whatever the mask says
_MASKS_A = [0, 1, 2, 4, 7, 0x10, 0x40, 0x50]
_MASKS_OTHER = [0, 7, 0x50]


def _bulk_cases():
    return [(n, "a", m) for n in (512, 1024, 2048) for m in _MASKS_A] + \
           [(n, c, m) for n in (512, 1024, 2048) for c in "bcd" for m in _MASKS_OTHER]


@pytest.mark.gpu
@pytest.mark.parametrize("n,cls,mask", _bulk_cases())
def test_gpu_bulk_batch_vs_float64_reference(n, cls, mask):
    """Batches of more than kSmallChunk (4) frames at distinct times - the Bulk tilings; at 1024^2 several chunks on both
    compute lanes - under the kernel-set masks of wso_select_kernels."""
    import watersurfacerendering_b200 as W
    from watersurfacerendering_b200 import _lib
    nframes = 9 if n <= 1024 else 5
    it = item(n, "white", cls)
    times = [it["t"] + 0.75 * i for i in range(nframes)]
    L = _lib.load()
    assert L.wso_select_kernels(mask) == 0
    try:
        with _ws(W, n, [it], max_slots=nframes) as ws:
            if n == 1024:
                assert ws.stats()["chunk"] < nframes
            ws.compute_batch(np.array(times, np.float32))
            a, mn, mx = ws.read_heights(0, nframes)
            for i in (0, nframes // 2, nframes - 1):
                ref = reference(n, "white", cls, t=float(np.float32(times[i])))
                check_maps(ws.copy_map(0, i), ws.copy_map(1, i), a[i], mn[i], mx[i], ref,
                           f"N={n} class {cls} mask {mask:#x} frame {i}", path=f"bulk mask {mask:#x}")
    finally:
        L.wso_select_kernels(-1)


@pytest.mark.gpu
def test_gpu_c4_sixty_four_tiles_vs_float64_reference():
    """The multi-tile workload at full size: 64 tiles of 512^2, each with its own white or sparse spectrum, lambda and
    tile length; two launches of 128 tile-frames with interleaved tile indices and distinct times.  The second launch
    carries one class-(d) tile among table tiles (every item on the general K1 body).  Every slot against the reference
    of its own tile, time and lambda."""
    import watersurfacerendering_b200 as W
    n, ntiles, nslots = 512, 64, 128
    specs = [("white" if j % 3 else "sparse1", "a", j) for j in range(ntiles)]
    its = [item(n, s, c, which=j % 2, seed=j) for s, c, j in specs]
    rng = np.random.default_rng(4)
    with _ws(W, n, its, max_slots=nslots) as ws:
        for launch in range(2):
            if launch == 1:
                specs[37] = ("white", "d", 37)
                its[37] = item(n, "white", "d", which=1, seed=37)
                ws.ImportH0(h0_records(its[37]), tile=37)
            tiles = np.concatenate([rng.permutation(ntiles), rng.permutation(ntiles)]).astype(np.uint32)
            times = (np.arange(nslots, dtype=np.float32) * np.float32(0.37) + np.float32(1.0 + 50 * launch))
            ws.compute_batch(times, tiles=tiles)
            a, mn, mx = ws.read_heights(0, nslots)
            for s in range(nslots):
                j = int(tiles[s])
                spec, cls, _ = specs[j]
                it = its[j]
                ref = R.Frame(it["re"], it["im"], it["omega"], it["tile_length"], it["lam"], float(times[s]),
                              dense=spec == "white")
                check_maps(ws.copy_map(0, s), ws.copy_map(1, s), a[s], mn[s], mx[s], ref,
                           f"c4 launch {launch} slot {s} tile {j} ({spec}/{cls})", path=f"c4 launch {launch}")


@pytest.mark.gpu
@pytest.mark.parametrize("n,cls", [(1 << l, c) for l in range(4, 13) for c in CLASSES])
def test_gpu_jacobian_vs_float64_reference(n, cls):
    """The Jacobian channel (disp.w = J) at 16^2 ... 4096^2: one frame and a batch of three."""
    import watersurfacerendering_b200 as W
    it = item(n, "white", cls)
    with _ws(W, n, [it], max_slots=3, jacobian=True) as ws:
        a = ws.ComputeWaves(it["t"])
        ref = reference(n, "white", cls, jacobian=True)
        check_maps(ws.GetDisplacements(), ws.GetNormals(), a, ws.GetMinHeight(), ws.GetMaxHeight(), ref,
                   f"N={n} class {cls} jacobian frame", path="jacobian frame")
        times = np.array([it["t"], 0.5, 7.25], np.float32)
        ws.compute_batch(times)
        a, mn, mx = ws.read_heights(0, 3)
        for i in (1, 2):
            ref = reference(n, "white", cls, t=float(times[i]), jacobian=True)
            check_maps(ws.copy_map(0, i), ws.copy_map(1, i), a[i], mn[i], mx[i], ref,
                       f"N={n} class {cls} jacobian batch frame {i}", path="jacobian batch")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [16, 64, 256, 512, 1024, 2048, 4096])
def test_gpu_f16_vs_float64_reference(n):
    """RGBA16F maps, one pass per path: a single frame (Lat), a batch (Bulk) and the Jacobian launch."""
    import watersurfacerendering_b200 as W
    for cls in "ad":
        it = item(n, "white", cls)
        with _ws(W, n, [it], max_slots=6, fmt="rgba16f") as ws:
            a = ws.ComputeWaves(it["t"])
            ref = reference(n, "white", cls)
            check_maps(ws.GetDisplacements(), ws.GetNormals(), a, ws.GetMinHeight(), ws.GetMaxHeight(), ref,
                       f"f16 N={n} class {cls} frame", path="f16 frame", half=True)
            times = np.array([it["t"]] * 6, np.float32)
            ws.compute_batch(times)
            a, mn, mx = ws.read_heights(0, 6)
            check_maps(ws.copy_map(0, 5), ws.copy_map(1, 5), a[5], mn[5], mx[5], ref, f"f16 N={n} class {cls} batch",
                       path="f16 batch", half=True)
            ws.SetComputeJacobian(True)
            a = ws.ComputeWaves(it["t"])
            check_maps(ws.GetDisplacements(), ws.GetNormals(), a, ws.GetMinHeight(), ws.GetMaxHeight(),
                       reference(n, "white", cls, jacobian=True), f"f16 N={n} class {cls} jacobian",
                       path="f16 jacobian", half=True)


def k2_split_child():
    """Run in a child process with WSO_K2_SPLIT=1 (read once per process): K2h launched together with the normal map."""
    import watersurfacerendering_b200 as W
    for n in (64, 256, 512, 1024):
        for cls in "ad":
            it = item(n, "white", cls)
            ref = reference(n, "white", cls)
            with _ws(W, n, [it], max_slots=6) as ws:
                a = ws.ComputeWaves(it["t"])
                check_maps(ws.GetDisplacements(), ws.GetNormals(), a, ws.GetMinHeight(), ws.GetMaxHeight(), ref,
                           f"split N={n} class {cls} frame", path="k2 split frame")
                ws.compute_batch(np.full(6, it["t"], np.float32))
                a, mn, mx = ws.read_heights(0, 6)
                check_maps(ws.copy_map(0, 5), ws.copy_map(1, 5), a[5], mn[5], mx[5], ref,
                           f"split N={n} class {cls} batch", path="k2 split batch")
    print("split ok")


@pytest.mark.gpu
def test_gpu_k2_split_vs_float64_reference():
    env = dict(os.environ, WSO_K2_SPLIT="1")
    code = ("import sys; sys.path[:0] = [sys.argv[1], sys.argv[2]]; import test_spectral_coverage as T; "
            "T.k2_split_child()")
    r = subprocess.run([sys.executable, "-c", code, ROOT, os.path.join(ROOT, "tests")], env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0 and "split ok" in r.stdout, r.stdout[-4000:] + r.stderr[-4000:]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [64, 256, 2048])   # the sizes the slab path supports (wso::slab_size_supported)
def test_gpu_slab_world1_vs_float64_reference(n):
    """The slab kernels on one device: class (a) white and sparse spectra against the reference; classes (b)-(d) are
    refused (the slab path needs the table and even dispersion)."""
    from watersurfacerendering_b200 import _lib
    from watersurfacerendering_b200.slab import SlabBackend, SlabOcean
    for spec in ("white", "sparse"):
        it = item(n, spec, "a")
        b = SlabBackend(n, it["tile_length"], 0, 1, 0, lambda_=it["lam"], anim_period=ANIM_PERIOD)
        try:
            b.import_h0(h0_records(it))
            ocean = SlabOcean(b)
            ocean.compute(it["t"])
            b.sync()
            disp, norm = ocean.gather_maps()
            a, mn, mx = b.read_heights()
            check_maps(disp, norm, a, mn, mx, reference(n, spec, "a"), f"slab N={n} {spec}", path="slab world 1")
            for cls in "bcd":
                with pytest.raises(_lib.WsoError) as e:
                    b.import_h0(h0_records(item(n, "white", cls)))
                assert e.value.status == _lib.WSO_ERR_INVALID_ARG
        finally:
            b.close()
