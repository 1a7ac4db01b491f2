"""TEST INFRASTRUCTURE: a float64 NumPy restatement of the wave-spectrum contract (include/wsocean.h, "Wave spectra").

records() builds the N*N h0 records of a non-Phillips tile from the same inputs as wso_spectrum_h0: the fp32 part (k,
1/|k|, unit direction, deep-water j, the two amplitude products) with float32 arrays, everything else in float64 in the
order the header states.  lgamma comes from scipy (the library calls the C library's), so amplitudes may differ from the
library's by an ulp where the two round differently; the quantised dispersion does not depend on it.
"""
from __future__ import annotations

import numpy as np
import scipy.special

import spectral_ref as R

F32 = np.float32
G = 9.81
LN2 = 0.69314718055994530942
LNPI = 1.14472988584940017414
AMP_CAP = 2.0 ** 64
MAX_R4 = 1400.0
PM, JONSWAP, TMA = 1, 2, 3


def spectrum(kind, fetch=1e5, depth=np.inf, gamma=3.3, spread=0.0, k_band=(0.0, np.inf), scale=1.0) -> dict:
    return dict(kind=int(kind), fetch=float(F32(fetch)), depth=float(F32(depth)), gamma=float(F32(gamma)),
                spread=float(F32(spread)), k_min=F32(k_band[0]), k_max=F32(k_band[1]), scale=float(F32(scale)))


def normalised_wind(wx, wy, speed):
    """What the setters store (wso::normalise_like_setters): fp32."""
    wx, wy = F32(wx), F32(wy)
    inv = F32(1) / np.sqrt(F32(wx * wx) + F32(wy * wy), dtype=np.float32)
    return F32(wx * inv), F32(wy * inv), max(F32(speed), F32(1e-4))


def omega0(anim_period):
    return F32(np.float64(F32(2.0)) * np.pi / np.float64(F32(anim_period)))


def spreading_norm(s):
    s = np.asarray(s, np.float64)
    return np.exp((((2.0 * s - 1.0) * LN2 + 2.0 * scipy.special.gammaln(s + 1.0)) - scipy.special.gammaln(2.0 * s + 1.0))
                  - LNPI)


def directional(cs, s, q):
    """D(c, s) = (Q(s)/2) (((1+c)/2)^s + ((1-c)/2)^s)."""
    return (0.5 * q) * ((0.5 * (1.0 + cs)) ** s + (0.5 * (1.0 - cs)) ** s)


def consts(wind_speed, spec, tile_length):
    U, F = float(wind_speed), spec["fetch"]
    if spec["kind"] == PM:
        alpha, wp = 0.0081, 0.855 * G / U
    else:
        alpha, wp = 0.076 * (U * U / (F * G)) ** 0.22, 22.0 * np.cbrt(G * G / (U * F))
    dk = 2.0 * np.pi / float(F32(tile_length))
    return dict(alpha_g2=alpha * G * G, omega_p=wp, mu=-2.33 - 1.45 * (U * wp / G - 1.17), split=1.05 * wp,
                amp_scale=spec["scale"] * (dk * dk), deep=bool(np.isinf(spec["depth"])))


def dispersion(k, depth):
    """omega(k) and d omega / dk, float64 (k: float64 of the fp32 |k|)."""
    if np.isinf(depth):
        w = np.sqrt(G * k)
        return w, G / (2.0 * w)
    kd = k * depth
    th = np.tanh(kd)
    w = np.sqrt((G * k) * th)
    return w, (G * (th + kd * (1.0 - th * th))) / (2.0 * w)


def energy(k, ux, uz, wind, wind_speed, spec, tile_length):
    """P(k) for in-band wave vectors: k float64 of fp32 |k|, (ux, uz) fp32 unit direction, wind = normalised (x, y)."""
    c = consts(wind_speed, spec, tile_length)
    w, cg = dispersion(k, spec["depth"])
    wp = c["omega_p"]
    r = wp / w
    r2 = r * r
    r4 = r2 * r2
    iw = 1.0 / w
    iw2 = iw * iw
    with np.errstate(over="ignore", under="ignore", invalid="ignore"):
        S = (c["alpha_g2"] * ((iw2 * iw2) * iw)) * np.exp(-1.25 * r4)
        if spec["kind"] != PM:
            sigma = np.where(w <= wp, 0.07, 0.09)
            dw = w - wp
            so = sigma * wp
            S = S * spec["gamma"] ** np.exp(-(dw * dw) / (2.0 * (so * so)))
            if spec["kind"] == TMA and not c["deep"]:
                wh = w * np.sqrt(spec["depth"] / G)
                phi = np.where(wh <= 1.0, 0.5 * (wh * wh), np.where(wh < 2.0, 1.0 - 0.5 * ((2.0 - wh) * (2.0 - wh)), 1.0))
                S = S * phi
        S = np.where(r4 < MAX_R4, S, 0.0)
        cs = np.clip(ux.astype(np.float64) * float(wind[0]) + uz.astype(np.float64) * float(wind[1]), -1.0, 1.0)
        if spec["spread"] > 0:
            s = np.full_like(w, spec["spread"])
        else:
            x = w / wp
            s = np.where(w <= c["split"], 6.97 * x ** 4.06, 9.77 * x ** c["mu"])
        D = directional(cs, s, spreading_norm(s))
        P = c["amp_scale"] * (((S * D) * cg) / k)
    return P, w


def grid(n, tile_length):
    kv = R.wave_numbers(n, tile_length)
    kx, kz = np.broadcast_to(kv[None, :], (n, n)), np.broadcast_to(kv[:, None], (n, n))
    k = np.sqrt((kx * kx).astype(F32) + (kz * kz).astype(F32), dtype=np.float32)
    return kx, kz, k


def records(n, tile_length, wind_dir, wind_speed, anim_period, spec, xi):
    """h0 records [m][n] (oracle.port.H0_DTYPE layout) and P [m][n] (0 outside the band)."""
    from oracle.port import H0_DTYPE
    wx, wy, U = normalised_wind(wind_dir[0], wind_dir[1], wind_speed)
    kx, kz, k = grid(n, tile_length)
    valid = k > F32(1e-5)
    with np.errstate(divide="ignore", invalid="ignore"):
        inv = np.where(valid, F32(1) / k, F32(0)).astype(F32)
    ux, uz = (kx * inv).astype(F32), (kz * inv).astype(F32)
    band = valid & (k >= spec["k_min"]) & (k < spec["k_max"])
    P = np.zeros((n, n))
    W = np.zeros((n, n))
    kb = k[band].astype(np.float64)
    P[band], W[band] = energy(kb, ux[band], uz[band], (wx, wy), U, spec, tile_length)
    P = np.where(P > 0, P, 0.0)
    s_amp = np.minimum(np.sqrt(P), AMP_CAP).astype(F32)
    xi = np.asarray(xi, np.complex64)
    c = F32(1) / np.sqrt(F32(2), dtype=np.float32)
    re = ((c * xi.real.astype(F32)).astype(F32) * s_amp).astype(F32)
    im = ((c * xi.imag.astype(F32)).astype(F32) * s_amp).astype(F32)
    w0 = omega0(anim_period)
    if np.isinf(spec["depth"]):
        jf = np.floor((np.sqrt((F32(9.81) * k).astype(F32), dtype=np.float32) / w0).astype(F32)).astype(F32)
    else:
        jf = np.floor(W / np.float64(w0)).astype(F32)
    disp = np.where(s_amp == 0, F32(0), (jf * w0).astype(F32)).astype(F32)
    h0 = np.zeros((n, n), H0_DTYPE)
    h0["re"], h0["im"], h0["re_c"], h0["im_c"], h0["omega"] = re, im, re, -im, disp
    return h0, P
