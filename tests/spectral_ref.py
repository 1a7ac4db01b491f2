"""TEST INFRASTRUCTURE: a float64 reference of the frame contract the K1 -> K2h -> K2 kernels implement.

Input: the fp32 spectrum records (re, im, omega) in the reference layout [m][n] (m: row, kz; n: column, kx), the tile
length, lambda and t.  What stays fp32 because the contract fixes it:
  * the wave numbers kv and 1/|k|, computed as upload_h0() does (wso_api.cu);
  * the phase phi = fl32(omega * t).
Everything after that is float64:
  * H(k) = 2 Re(h0(k) e^{i phi}) (h0_conj = conj(h0), the only records wso_import_h0 accepts);
  * the seven spectra of oracle.port.numpy_spectra (and dxDz = kx uz H for the Jacobian), inverse-transformed and
    multiplied by (-1)^(m+n);
  * A = max(|min h|, |max h|) (min / max start at FLT_MAX / FLT_MIN as in the reference);
  * disp = (lambda Dx, h / A, lambda Dz, 1 or J), norm = (fld1, fld2, fld5, fld6),
    J = (1 + l dxDx)(1 + l dzDz) - (l dxDz)(l dzDx) (wsocean.h, wso_set_compute_jacobian).

Two evaluators of the inverse transform:
  * dense: complex128 ifft2 (scipy.fft), for N <= 4096;
  * sparse: a sum of K plane waves with exact integer phases (m r mod N), each an outer product of a column and a row
    vector, O(K N^2), evaluated in row blocks so that 8192^2 fits in a few GB.
"""
from __future__ import annotations

import numpy as np
import scipy.fft

F32 = np.float32
FLT_MAX = float(np.finfo(np.float32).max)
FLT_MIN = float(np.finfo(np.float32).tiny)
# field index -> multiplier c(k) of H(k): spectra 0..6 of numpy_spectra, 7 = dxDz (== dzDx) of the Jacobian
#   0: H   1: i kx H   2: i kz H   3: -i ux H   4: -i uz H   5: kx ux H   6: kz uz H   7: kx uz H
N_FIELDS = 8


def wave_numbers(n: int, tile_length: float) -> np.ndarray:
    """kv as the library computes it (wso::host_wave_numbers, the reference's WSTessendorf.cpp:75-80): fp32."""
    idx = np.arange(n, dtype=np.float32)
    return (np.pi * (F32(2) * idx - F32(n)).astype(np.float64) / np.float64(F32(tile_length))).astype(np.float32)


def inv_length(kx: np.ndarray, kz: np.ndarray) -> np.ndarray:
    """1/|k| as upload_h0() stores it in the records: fp32, 0 where |k| <= 1e-5."""
    d = (kx * kx + kz * kz).astype(np.float32)
    ln = np.sqrt(d)
    with np.errstate(divide="ignore"):
        inv = (F32(1) / ln).astype(np.float32)
    return np.where(ln > F32(1e-5), inv, F32(0)).astype(np.float32)


def heights_spectrum(re, im, omega, t) -> np.ndarray:
    """H(k) = h0 e^{i phi} + conj(h0) e^{-i phi} = 2 Re(h0 e^{i phi}), phi = fl32(omega t): float64, real."""
    ph = (np.asarray(omega, np.float32) * F32(t)).astype(np.float32).astype(np.float64)
    return 2.0 * (np.asarray(re, np.float64) * np.cos(ph) - np.asarray(im, np.float64) * np.sin(ph))


def _multiplier(f, kx, kz, inv):
    """(real part, imaginary part) of c_f(k), broadcast over [m][n]; kx = kv[n], kz = kv[m] (float64 of fp32)."""
    ux, uz = kx * inv, kz * inv
    zero = 0.0
    return {0: (1.0, zero), 1: (zero, kx), 2: (zero, kz), 3: (zero, -ux), 4: (zero, -uz),
            5: (kx * ux, zero), 6: (kz * uz, zero), 7: (kx * uz, zero)}[f]


def _axes(n, tile_length):
    kv = wave_numbers(n, tile_length)
    inv = inv_length(kv[None, :], kv[:, None]).astype(np.float64)
    kv = kv.astype(np.float64)
    return kv[None, :], kv[:, None], inv


def _sign(rows, n):
    r = np.asarray(rows)[:, None]
    c = np.arange(n)[None, :]
    return np.where((r + c) & 1, -1.0, 1.0)


# ---------------------------------------------------------------------------------------------------------------------
# evaluators: signed fields fld_f[r, c] = (-1)^(r+c) Re sum_k c_f(k) H(k) exp(2 pi i (m r + n c) / N)
# ---------------------------------------------------------------------------------------------------------------------
def fields_dense(H, tile_length, which=range(N_FIELDS)) -> dict:
    n = H.shape[0]
    kx, kz, inv = _axes(n, tile_length)
    sign = _sign(np.arange(n), n)
    out = {}
    for f in which:
        cr, ci = _multiplier(f, kx, kz, inv)
        x = np.empty((n, n), np.complex128)
        x.real = cr * H
        x.imag = ci * H
        out[f] = sign * (scipy.fft.ifft2(x, workers=-1).real * (float(n) * n))
    return out


class SparseTerms:
    """The lit records of a spectrum: K plane waves with their complex amplitudes per field."""

    def __init__(self, H, tile_length):
        n = H.shape[0]
        self.n = n
        self.m, self.c = np.nonzero(H)
        h = H[self.m, self.c]
        kx, kz, inv = _axes(n, tile_length)
        kxk = np.broadcast_to(kx, (n, n))[self.m, self.c]
        kzk = np.broadcast_to(kz, (n, n))[self.m, self.c]
        ik = inv[self.m, self.c]
        self.coef = {}
        for f in range(N_FIELDS):
            cr, ci = _multiplier(f, kxk, kzk, ik)
            self.coef[f] = (np.broadcast_to(cr, h.shape) + 1j * np.broadcast_to(ci, h.shape)) * h

    def abs_sum(self, f) -> float:
        """sum_k |X_k| of field f: the scale of its per-texel error bound."""
        return float(np.abs(self.coef[f]).sum())

    def fields(self, rows, which=range(N_FIELDS)) -> dict:
        """Signed fields on the given rows, exact integer phases: (m r mod N) and (n c mod N)."""
        n = self.n
        rows = np.asarray(rows)
        two_pi_n = 2.0 * np.pi / n
        u = np.exp(1j * two_pi_n * ((self.m[None, :] * rows[:, None]) % n))    # [R, K]
        v = np.exp(1j * two_pi_n * ((self.c[:, None] * np.arange(n)[None, :]) % n))  # [K, N]
        sign = _sign(rows, n)
        out = {}
        for f in which:
            cu = u * self.coef[f][None, :]
            out[f] = sign * (cu.real @ v.real - cu.imag @ v.imag)
        return out


# ---------------------------------------------------------------------------------------------------------------------
# the maps
# ---------------------------------------------------------------------------------------------------------------------
def amplitude(h_min, h_max):
    """A, min, max as the kernels reduce them (start values FLT_MAX / FLT_MIN, WSTessendorf.cpp:288-289)."""
    mx = max(FLT_MIN, float(h_max))
    mn = min(FLT_MAX, float(h_min))
    return max(abs(mn), abs(mx)), mn, mx


def maps(fld, a, lam, jacobian=False):
    """disp[..., 4], norm[..., 4] (float64) from the signed fields and the amplitude A."""
    lam = float(F32(lam))
    h = fld[0]
    if jacobian:
        w = (1.0 + lam * fld[5]) * (1.0 + lam * fld[6]) - (lam * fld[7]) ** 2
    else:
        w = np.ones_like(h)
    disp = np.stack([lam * fld[3], h / a, lam * fld[4], w], axis=-1)
    norm = np.stack([fld[1], fld[2], fld[5], fld[6]], axis=-1)
    return disp, norm


class Frame:
    """The reference of one tile-frame.  dense=None picks the sparse evaluator when at most 1 % of the records are lit."""

    def __init__(self, re, im, omega, tile_length, lam, t, jacobian=False, dense=None):
        self.n = np.asarray(re).shape[0]
        self.lam, self.jacobian = float(F32(lam)), jacobian
        H = heights_spectrum(re, im, omega, t)
        if dense is None:
            dense = np.count_nonzero(H) > 0.01 * self.n * self.n
        self.dense = dense
        self.sparse = None if dense else SparseTerms(H, tile_length)
        self._fld = fields_dense(H, tile_length) if dense else None
        if dense:
            h = self._fld[0]
            self.A, self.hmin, self.hmax = amplitude(h.min(), h.max())
        else:
            lo, hi = np.inf, -np.inf
            for r0, blk in self._blocks(which=(0,)):
                lo, hi = min(lo, blk[0].min()), max(hi, blk[0].max())
            self.A, self.hmin, self.hmax = amplitude(lo, hi)

    def _blocks(self, rows_per_block=None, which=range(N_FIELDS)):
        n = self.n
        rb = rows_per_block or max(1, min(n, (1 << 22) // n))
        for r0 in range(0, n, rb):
            yield r0, self.sparse.fields(np.arange(r0, min(n, r0 + rb)), which)

    def blocks(self, rows_per_block=None):
        """(first row, disp[R, N, 4], norm[R, N, 4]) over the whole map."""
        if self.dense:
            d, nm = maps(self._fld, self.A, self.lam, self.jacobian)
            yield 0, d, nm
            return
        for r0, fld in self._blocks(rows_per_block):
            d, nm = maps(fld, self.A, self.lam, self.jacobian)
            yield r0, d, nm

    def whole(self):
        """disp, norm over the whole map (float64)."""
        parts = list(self.blocks())
        return np.concatenate([p[1] for p in parts]), np.concatenate([p[2] for p in parts])

    def texel_scale(self):
        """Per-channel sum_k |X_k| of the sparse error model: disp (4,), norm (4,) and the J channel."""
        s = [self.sparse.abs_sum(f) for f in range(N_FIELDS)]
        lam = abs(self.lam)
        ds = np.array([lam * s[3], s[0] / self.A, lam * s[4],
                       lam * s[5] * (1 + lam * s[6]) + lam * s[6] * (1 + lam * s[5]) + 2 * lam * lam * s[7] * s[7]])
        ns = np.array([s[1], s[2], s[5], s[6]])
        return ds, ns
