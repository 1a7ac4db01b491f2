// wso_spectrum.cuh — empirical wave spectra (Pierson-Moskowitz, JONSWAP, TMA) with directional spreading, finite depth
// and a wave-number band: the per-wave-vector record arithmetic of include/wsocean.h, "Wave spectra".
//
// Written once for the device Prepare kernel (wso_prepare_kernels.cu) and for the host build (wso_spectrum_h0, wso_prepare /
// wso_prepare_gauss of a non-Phillips tile).  Every fp32 and float64 add, multiply, divide and square root is an explicit
// round-to-nearest operation (rmul / radd / rdiv / sqrt_ieee; mul64 / add64 / sub64 / div64 / sqrt64 below), so nvcc cannot
// contract anything into an FMA and the two builds agree bit for bit except where the float64 library functions (exp,
// pow, tanh, lgamma) of the device and of the host C library round differently: amplitudes may then differ by 1 ulp.
// The quantised dispersion of a deep-water tile uses fp32 operations only, so it is always bit-identical.
#pragma once

#include "wso_device.cuh"

namespace wso {

namespace spec {
#if defined(__CUDA_ARCH__)
WSO_HD double mul64(double a, double b) { return __dmul_rn(a, b); }
WSO_HD double add64(double a, double b) { return __dadd_rn(a, b); }
WSO_HD double sub64(double a, double b) { return __dsub_rn(a, b); }
WSO_HD double div64(double a, double b) { return __ddiv_rn(a, b); }
WSO_HD double sqrt64(double a) { return __dsqrt_rn(a); }
#else
WSO_HD double mul64(double a, double b) { return a * b; }
WSO_HD double add64(double a, double b) { return a + b; }
WSO_HD double sub64(double a, double b) { return a - b; }
WSO_HD double div64(double a, double b) { return a / b; }
WSO_HD double sqrt64(double a) { return std::sqrt(a); }
#endif

static constexpr double kG = 9.81;
static constexpr double kLn2 = 0.69314718055994530942;
static constexpr double kLnPi = 1.14472988584940017414;
static constexpr double kAmpCap = 18446744073709551616.0;  // 2^64: s_amp saturates here (no inf for any valid input)
// (omega_p / omega)^4 at or above this: S(omega) = 0 (exp(-1.25 * 1400) underflows float64 anyway; the guard keeps
// omega^-5 from overflowing into inf * 0 for tiny winds and huge tiles)
static constexpr double kMaxR4 = 1400.0;
}  // namespace spec

enum SpectrumKind { kSpecPhillips = 0, kSpecPM = 1, kSpecJonswap = 2, kSpecTMA = 3 };

// Per-tile constants of a non-Phillips spectrum, derived once on the host (spectrum_consts) and used unchanged by both
// builds, so the per-kind float64 constants never differ between device and host.
struct SpectrumConsts {
    int kind;            // kSpecPM / kSpecJonswap / kSpecTMA
    int deep;            // depth == +inf
    float wind_x, wind_y;  // normalised wind direction, as the setters store it
    float inv_sqrt2;     // 1/sqrt(2), rounded as the Phillips build rounds it
    float omega0;        // base frequency fl(2*pi/T)
    float k_min, k_max;  // band, compared in fp32 against fp32 |k|
    double depth;        // d (finite only when !deep)
    double sqrt_d_over_g;  // sqrt(d/g) (TMA)
    double omega_p;      // peak frequency
    double alpha_g2;     // alpha * g * g
    double gamma;        // peak enhancement (JONSWAP / TMA)
    double spread;       // 0: Hasselmann s(omega); > 0: constant s
    double q_const;      // Q(spread) when spread > 0
    double split;        // 1.05 * omega_p
    double mu;           // Hasselmann exponent above 1.05 omega_p
    double amp_scale;    // scale * (2*pi/L)^2
};

// Q(s) = 2^(2s-1) Gamma(s+1)^2 / (pi Gamma(2s+1)), through lgamma
WSO_HD double spreading_norm(double s) {
    using namespace spec;
    const double l = sub64(sub64(add64(mul64(sub64(mul64(2.0, s), 1.0), kLn2), mul64(2.0, lgamma(add64(s, 1.0)))),
                               lgamma(add64(mul64(2.0, s), 1.0))),
                          kLnPi);
    return exp(l);
}

// Continuous dispersion omega(k) and its derivative d omega / dk, float64.
WSO_HD void spectrum_dispersion(const SpectrumConsts& c, double k, double* omega, double* cg) {
    using namespace spec;
    if (c.deep) {
        *omega = sqrt64(mul64(kG, k));
        *cg = div64(kG, mul64(2.0, *omega));
    } else {
        const double kd = mul64(k, c.depth);
        const double th = tanh(kd);
        *omega = sqrt64(mul64(mul64(kG, k), th));
        *cg = div64(mul64(kG, add64(th, mul64(kd, sub64(1.0, mul64(th, th))))), mul64(2.0, *omega));
    }
}

// P(k) = scale * S(k) * (2 pi / L)^2 for an in-band wave vector of fp32 length k and unit direction (ux, uz); float64.
WSO_HD double spectrum_energy(const SpectrumConsts& c, double k, float ux, float uz, double omega, double cg) {
    using namespace spec;
    // S(omega): Pierson-Moskowitz shape alpha g^2 omega^-5 exp(-5/4 (omega_p/omega)^4)
    const double r = div64(c.omega_p, omega);
    const double r2 = mul64(r, r);
    const double r4 = mul64(r2, r2);
    if (!(r4 < kMaxR4)) return 0.0;
    const double iw = div64(1.0, omega);
    const double iw2 = mul64(iw, iw);
    double S = mul64(mul64(c.alpha_g2, mul64(mul64(iw2, iw2), iw)), exp(mul64(-1.25, r4)));
    if (c.kind != kSpecPM) {
        // JONSWAP peak enhancement gamma^exp(-(omega - omega_p)^2 / (2 sigma^2 omega_p^2))
        const double sigma = omega <= c.omega_p ? 0.07 : 0.09;
        const double dw = sub64(omega, c.omega_p);
        const double so = mul64(sigma, c.omega_p);
        const double e = exp(div64(-mul64(dw, dw), mul64(2.0, mul64(so, so))));
        S = mul64(S, pow(c.gamma, e));
        if (c.kind == kSpecTMA && !c.deep) {
            // Kitaigorodskii depth attenuation Phi(omega_h), omega_h = omega sqrt(d/g)
            const double wh = mul64(omega, c.sqrt_d_over_g);
            double phi = 1.0;
            if (wh <= 1.0) phi = mul64(0.5, mul64(wh, wh));
            else if (wh < 2.0) {
                const double t = sub64(2.0, wh);
                phi = sub64(1.0, mul64(0.5, mul64(t, t)));
            }
            S = mul64(S, phi);
        }
    }
    // D = 1/2 Q(s) [((1+c)/2)^s + ((1-c)/2)^s]: Hasselmann's Q(s)|cos(theta/2)|^2s made even in k
    double cs = add64(mul64((double)ux, (double)c.wind_x), mul64((double)uz, (double)c.wind_y));
    cs = cs > 1.0 ? 1.0 : (cs < -1.0 ? -1.0 : cs);
    double s = c.spread, q = c.q_const;
    if (!(s > 0.0)) {
        const double x = div64(omega, c.omega_p);
        s = omega <= c.split ? mul64(6.97, pow(x, 4.06)) : mul64(9.77, pow(x, c.mu));
        q = spreading_norm(s);
    }
    const double D = mul64(mul64(0.5, q), add64(pow(mul64(0.5, add64(1.0, cs)), s), pow(mul64(0.5, sub64(1.0, cs)), s)));
    // S(k) = S(omega) D (d omega / dk) / k, times the wave-number cell area and the caller's scale
    return mul64(c.amp_scale, div64(mul64(mul64(S, D), cg), k));
}

// The record of one wave vector: amplitude (re, im), 1/|k| and the quantised dispersion as the multiple j of omega0
// (jf, a float holding an integer; 0 where the amplitude is zero).  The stored dispersion is fl(jf * omega0).
WSO_HD void spectrum_record(const SpectrumConsts& c, float kx, float kz, float xr, float xi, float* re, float* im,
                            float* inv_out, float* jf_out) {
    using namespace spec;
    const float dot = radd(rmul(kx, kx), rmul(kz, kz));
    const float k = sqrt_ieee(dot);
    *re = 0.0f;
    *im = 0.0f;
    *inv_out = 0.0f;
    *jf_out = 0.0f;
    if (!(k > 0.00001f)) return;
    const float inv = rdiv(1.0f, k);
    *inv_out = inv;
    const float ux = rmul(kx, inv), uz = rmul(kz, inv);
    float s_amp = 0.0f;
    double omega = 0.0;
    if (k >= c.k_min && k < c.k_max) {
        double cg;
        spectrum_dispersion(c, (double)k, &omega, &cg);
        const double P = spectrum_energy(c, (double)k, ux, uz, omega, cg);
        // P not > 0 (scale 0 against an overflowed S at absurd inputs: 0 * inf) carries no energy
        if (P > 0.0) {
            const double sq = sqrt64(P);
            s_amp = (float)(sq < kAmpCap ? sq : kAmpCap);
        }
    }
    *re = rmul(rmul(c.inv_sqrt2, xr), s_amp);
    *im = rmul(rmul(c.inv_sqrt2, xi), s_amp);
    if (s_amp == 0.0f) return;
    // quantised as the Phillips build quantises: deep water from the same fp32 operations, so j matches it bit for bit
    *jf_out = c.deep ? floorf(rdiv(sqrt_ieee(rmul(9.81f, k)), c.omega0)) : (float)floor(div64(omega, (double)c.omega0));
}

#if defined(__CUDACC__)
// Device Prepare of a non-Phillips tile (wso_prepare_kernels.cu): same thread-to-work mapping and output arrays as
// launch_prepare (PrepareArgs), the records from spectrum_record.
struct SpectrumPrepareArgs {
    float4* h0;
    float4* hs;
    const float* kv;      // [n] wave numbers (device)
    const float2* xi;     // [n][n] Gaussian array (device), or NULL: counter-based
    uint64_t seed_mixed;  // counter_seed_mix(seed)
    int n;
    int table;            // 1: w holds the integer j (K1's sincos table, table_len = j_cap + 1); 0: w = omega
    int j_cap;            // largest j the host found in the band (table only)
    SpectrumConsts c;
};
cudaError_t launch_prepare_spectrum(const SpectrumPrepareArgs& a, cudaStream_t stream);
#endif

}  // namespace wso
