// wso_host_prepare.cpp — see wso_host_prepare.h.  Compiled with -ffp-contract=off: every product below is
// a separately rounded fp32 operation, as in the reference's x86 build, so that a given Gaussian array
// yields bit-identical h0 (tests/test_parity_gpu.py::test_prepare_matches_reference).
#include "wso_host_prepare.h"

#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <limits>

#include "wso_spectrum.cuh"

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

namespace wso {

namespace {
constexpr float kGravity = 9.81f;  // reference: WSTessendorf.h:230

inline float wave_number(uint32_t i, uint32_t n, float tile_length) {
    const float centred = 2.0f * (float)(int32_t)i - (float)(int32_t)n;
    return (float)(M_PI * centred / tile_length);
}

// Uniform float in [-1,1] assembled from four rand()%255 bytes: glm::linearRand<float>
// (libs/glm/glm/gtc/random.inl:13-86,177-183).  GCC evaluates the right operand of the vec `|` first,
// so within each 16/32-bit word the LOW part is drawn before the HIGH part.
inline uint32_t draw_byte() { return (uint32_t)(std::rand() % 255); }
inline uint32_t draw_u16() {
    const uint32_t lo = draw_byte();
    const uint32_t hi = draw_byte();
    return (hi << 8) | lo;
}
inline uint32_t draw_u32() {
    const uint32_t lo = draw_u16();
    const uint32_t hi = draw_u16();
    return (hi << 16) | lo;
}
inline float uniform_pm1() { return (float)draw_u32() / (float)UINT32_MAX * 2.0f + -1.0f; }

// Marsaglia polar, mean 0 deviation 1 (random.inl:218-232)
inline float gauss01() {
    float w, x1, x2;
    do {
        x1 = uniform_pm1();
        x2 = uniform_pm1();
        w = x1 * x1 + x2 * x2;
    } while (w > 1.0f);
    return x2 * 1.0f * 1.0f * std::sqrt((-2.0f * std::log(w)) / w) + 0.0f;
}
}  // namespace

DerivedParams derive_params(const wso_params& p) {
    // p holds the setter-normalised state (see normalise_like_setters)
    DerivedParams d;
    d.wind_x = p.wind_dir_x;
    d.wind_y = p.wind_dir_y;
    d.wind_speed = p.wind_speed;
    d.base_freq = (float)(2.0f * M_PI / p.anim_period);
    return d;
}

void normalise_like_setters(wso_params& p, const wso_params* current) {
    // SetWindDirection: m_WindDir = glm::normalize(w) = w * (1/sqrt(dot(w,w)))   (WSTessendorf.cpp:476-479)
    // A direction bit-identical to the stored (already normalised) one is kept as is, so that
    // get -> modify another field -> set round trips do not re-normalise.
    if (!(current && current->wind_dir_x == p.wind_dir_x && current->wind_dir_y == p.wind_dir_y)) {
        const float inv = 1.0f / std::sqrt(p.wind_dir_x * p.wind_dir_x + p.wind_dir_y * p.wind_dir_y);
        p.wind_dir_x = p.wind_dir_x * inv;
        p.wind_dir_y = p.wind_dir_y * inv;
    }
    // SetWindSpeed: glm::max(0.0001f, v)                                           (WSTessendorf.cpp:481-484)
    p.wind_speed = p.wind_speed > 0.0001f ? p.wind_speed : 0.0001f;
}

void host_wave_numbers(uint32_t n, float tile_length, std::vector<float>& kv) {
    kv.resize(n);
    for (uint32_t i = 0; i < n; ++i) kv[i] = wave_number(i, n, tile_length);
}

void host_gauss_array_from_rand(uint32_t n, std::vector<float>& xi) {
    xi.resize((size_t)2 * n * n);
    for (size_t i = 0; i < (size_t)n * n; ++i) {
        // Complex(gaussRand(), gaussRand()): constructor arguments are evaluated right-to-left by GCC
        xi[2 * i + 1] = gauss01();
        xi[2 * i] = gauss01();
    }
}

H0Builder::H0Builder(const wso_params& p) {
    const DerivedParams d = derive_params(p);
    wind_x = d.wind_x;
    wind_y = d.wind_y;
    base_freq = d.base_freq;
    phillips_const = p.phillips_const;
    damping = p.damping;
    inv_sqrt2 = 1.0f / std::sqrt(2.0f);   // reference: WSTessendorf.h:231
    const float Lw = d.wind_speed * d.wind_speed / kGravity;
    Lw2 = Lw * Lw;
}

wso_h0_record H0Builder::at(float kx, float kz, float xi_re, float xi_im) const {
    const float dot = kx * kx + kz * kz;
    const float k = std::sqrt(dot);
    wso_h0_record r;
    if (k > 0.00001f) {
        const float inv = 1.0f / std::sqrt(dot);
        const float ux = kx * inv, uz = kz * inv;
        // Phillips spectrum (reference: WSTessendorf.h:249-263); (k^.w)^2 is even in k^, so the
        // "conjugate" amplitude built from -k^ equals conj(amplitude) exactly.
        const float k2 = k * k;
        const float k4 = k2 * k2;
        float cf = ux * wind_x + uz * wind_y;
        cf = cf * cf;
        const float ph = phillips_const * std::exp(-1.0f / (k2 * Lw2)) / k4 * cf * std::exp(-k2 * damping * damping);
        const float s = std::sqrt(ph);
        r.amp_re = inv_sqrt2 * xi_re * s;       // reference: WSTessendorf.h:237-243
        r.amp_im = inv_sqrt2 * xi_im * s;
        r.amp_conj_re = r.amp_re;
        r.amp_conj_im = -r.amp_im;
        // reference: QDispersion, WSTessendorf.h:284-297
        r.dispersion = std::floor(std::sqrt(kGravity * k) / base_freq) * base_freq;
    } else {
        r.amp_re = r.amp_im = r.amp_conj_re = 0.0f;
        r.amp_conj_im = -0.0f;
        r.dispersion = 0.0f;
    }
    return r;
}

void host_base_wave_heights(const wso_params& p, const float* xi, std::vector<wso_h0_record>& h0) {
    const uint32_t n = p.tile_size;
    const H0Builder hb(p);
    h0.resize((size_t)n * n);
    std::vector<float> kv;
    host_wave_numbers(n, p.tile_length, kv);
    for (uint32_t m = 0; m < n; ++m)
        for (uint32_t c = 0; c < n; ++c) {
            const size_t i = (size_t)m * n + c;
            h0[i] = hb.at(kv[c], kv[m], xi[2 * i], xi[2 * i + 1]);
        }
}

// Counter-based Gaussian pair for wave vector index idx = m*N + n: a 64-bit mix of (seed, idx) -> two uniforms ->
// Box-Muller.  Used where the reference's serial rand() stream is impractical (a 16384^2 grid generated in slabs on
// several devices); the same function serves the product and, through wso_counter_gauss(), its checkers.
static inline uint64_t mix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

void counter_gauss(uint64_t seed, uint64_t idx, float* re, float* im) {
    const uint64_t u = mix64(mix64(seed) ^ mix64(idx + 0x632BE59BD9B4E019ull));
    const double u1 = ((double)(u >> 40) + 1.0) * (1.0 / 16777216.0);        // (0, 1]
    const double u2 = (double)((u >> 8) & 0xFFFFFFull) * (1.0 / 16777216.0);  // [0, 1)
    const double r = std::sqrt(-2.0 * std::log(u1));
    const double a = 2.0 * M_PI * u2;
    *re = (float)(r * std::cos(a));
    *im = (float)(r * std::sin(a));
}

wso_spectrum default_spectrum() {
    wso_spectrum s;
    s.kind = WSO_SPECTRUM_PHILLIPS;
    s.fetch = 1.0e5f;
    s.depth = std::numeric_limits<float>::infinity();
    s.gamma = 3.3f;
    s.spread = 0.0f;
    s.k_min = 0.0f;
    s.k_max = std::numeric_limits<float>::infinity();
    s.scale = 1.0f;
    return s;
}

bool spectrum_is_phillips(const wso_spectrum& s) { return s.kind == WSO_SPECTRUM_PHILLIPS; }

bool spectrum_valid(const wso_spectrum& s) {
    if (s.kind > WSO_SPECTRUM_TMA) return false;
    if (s.kind == WSO_SPECTRUM_PHILLIPS) {
        // the Phillips kind is today's Prepare, which reads none of these fields: only the defaults are accepted
        const wso_spectrum d = default_spectrum();
        return std::memcmp(&s, &d, sizeof(s)) == 0;
    }
    const auto finite = [](float x) { return std::isfinite(x); };
    return finite(s.fetch) && s.fetch > 0.0f && s.depth > 0.0f && !std::isnan(s.depth) && finite(s.gamma) &&
           s.gamma >= 1.0f && finite(s.spread) && s.spread >= 0.0f && finite(s.k_min) && s.k_min >= 0.0f &&
           !std::isnan(s.k_max) && s.k_max > s.k_min && finite(s.scale) && s.scale >= 0.0f;
}

SpectrumConsts spectrum_consts(const wso_params& p, const wso_spectrum& s) {
    const double g = spec::kG;
    const double U = (double)p.wind_speed;
    const double F = (double)s.fetch;
    SpectrumConsts c;
    c.kind = (int)s.kind;
    c.deep = std::isinf(s.depth) ? 1 : 0;
    c.wind_x = p.wind_dir_x;
    c.wind_y = p.wind_dir_y;
    c.inv_sqrt2 = 1.0f / std::sqrt(2.0f);
    c.omega0 = derive_params(p).base_freq;
    c.k_min = s.k_min;
    c.k_max = s.k_max;
    c.depth = c.deep ? 0.0 : (double)s.depth;
    c.sqrt_d_over_g = c.deep ? 0.0 : std::sqrt(c.depth / g);
    double alpha;
    if (s.kind == WSO_SPECTRUM_PIERSON_MOSKOWITZ) {
        alpha = 0.0081;
        c.omega_p = 0.855 * g / U;                        // U: wind speed at 19.5 m
    } else {
        alpha = 0.076 * std::pow(U * U / (F * g), 0.22);  // U: wind speed at 10 m, F: fetch
        c.omega_p = 22.0 * std::cbrt(g * g / (U * F));
    }
    c.alpha_g2 = alpha * g * g;
    c.gamma = (double)s.gamma;
    c.spread = (double)s.spread;
    c.q_const = s.spread > 0.0f ? spreading_norm(c.spread) : 0.0;
    c.split = 1.05 * c.omega_p;
    c.mu = -2.33 - 1.45 * (U * c.omega_p / g - 1.17);
    const double dk = 2.0 * M_PI / (double)p.tile_length;
    c.amp_scale = (double)s.scale * (dk * dk);
    return c;
}

double spectrum_max_j(const SpectrumConsts& c, const std::vector<float>& kv) {
    // |kx| in ascending order: kv[N/2 + t] for t = 0 .. N/2-1 (>= 0), then |kv[0]| (kv[N-i] == -kv[i] exactly).  For a
    // fixed kz the fp32 |k| is non-decreasing along this order, so the largest |kx| with |k| < k_max is a binary search.
    const size_t n = kv.size(), h = n / 2;
    std::vector<float> ax(h + 1);
    for (size_t t = 0; t < h; ++t) ax[t] = kv[h + t];
    ax[h] = -kv[0];
    const auto klen = [](float kx, float kz) { return std::sqrt(kx * kx + kz * kz); };
    float kbest = 0.0f;
    for (size_t m = 0; m < n; ++m) {
        const float kz = kv[m];
        size_t lo = 0, hi = h + 1;  // first index with |k| >= k_max
        while (lo < hi) {
            const size_t mid = (lo + hi) / 2;
            if (klen(ax[mid], kz) < c.k_max) lo = mid + 1;
            else hi = mid;
        }
        if (lo == 0) continue;
        const float k = klen(ax[lo - 1], kz);
        if (k >= c.k_min && k > 0.00001f && k > kbest) kbest = k;
    }
    if (!(kbest > 0.0f)) return 0.0;
    if (c.deep) return (double)std::floor(std::sqrt(9.81f * kbest) / c.omega0);
    double omega, cg;
    spectrum_dispersion(c, (double)kbest, &omega, &cg);
    return std::floor(omega / (double)c.omega0);
}

void host_spectrum_rows(const wso_params& p, const wso_spectrum& s, const float* xi, uint64_t seed, uint32_t m0,
                        uint32_t rows, wso_h0_record* out) {
    const uint32_t n = p.tile_size;
    std::vector<float> kv;
    host_wave_numbers(n, p.tile_length, kv);
    const bool phillips = spectrum_is_phillips(s);
    const H0Builder hb(p);
    const SpectrumConsts c = phillips ? SpectrumConsts{} : spectrum_consts(p, s);
    for (uint32_t m = m0; m < m0 + rows; ++m)
        for (uint32_t col = 0; col < n; ++col) {
            const size_t idx = (size_t)m * n + col;
            float xr, xim;
            if (xi) {
                xr = xi[2 * idx];
                xim = xi[2 * idx + 1];
            } else {
                counter_gauss(seed, idx, &xr, &xim);
            }
            wso_h0_record& r = out[(size_t)(m - m0) * n + col];
            if (phillips) {
                r = hb.at(kv[col], kv[m], xr, xim);
                continue;
            }
            float re, im, inv, jf;
            spectrum_record(c, kv[col], kv[m], xr, xim, &re, &im, &inv, &jf);
            r.amp_re = re;
            r.amp_im = im;
            r.amp_conj_re = re;
            r.amp_conj_im = -im;
            r.dispersion = jf * c.omega0;
        }
}

}  // namespace wso
