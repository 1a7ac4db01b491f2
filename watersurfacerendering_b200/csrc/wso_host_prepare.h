// wso_host_prepare.h — host side of Prepare(): wave numbers, Gaussian array, Phillips h0(k), dispersion.
// Product code (one-off per Prepare, stays on the CPU like the reference's; device Prepare is row f-3).
#pragma once
#include <cstdint>
#include <vector>

#include "wsocean.h"

namespace wso {

// reference: WSTessendorf::SetWindDirection / SetWindSpeed / SetAnimationPeriod (WSTessendorf.cpp:476-490)
struct DerivedParams {
    float wind_x, wind_y;  // normalised
    float wind_speed;      // clamped
    float base_freq;       // (float)(2.0f * M_PI / T)
};
DerivedParams derive_params(const wso_params& p);
// Apply what the reference setters do on assignment (normalise wind direction, clamp wind speed).
void normalise_like_setters(wso_params& p, const wso_params* current);

// kv[i] = (float)(M_PI * (2.0f*i - N) / L)                       reference: WSTessendorf.cpp:60-85
void host_wave_numbers(uint32_t n, float tile_length, std::vector<float>& kv);
// N*N complex<float> drawn from rand() in glm::gaussRand order      reference: WSTessendorf.cpp:87-103
void host_gauss_array_from_rand(uint32_t n, std::vector<float>& xi);
// h0 records, row-major [m][n]                                      reference: WSTessendorf.cpp:105-148
void host_base_wave_heights(const wso_params& p, const float* xi, std::vector<wso_h0_record>& h0);
// the same arithmetic for one wave vector (slab-decomposed grids build only their own columns)
struct H0Builder {
    explicit H0Builder(const wso_params& p);
    wso_h0_record at(float kx, float kz, float xi_re, float xi_im) const;
    float wind_x, wind_y, base_freq, phillips_const, damping, inv_sqrt2, Lw2;
};
// counter-based standard-normal pair for wave vector index idx (see wso_host_prepare.cpp)
void counter_gauss(uint64_t seed, uint64_t idx, float* re, float* im);

// Wave spectra (include/wsocean.h, "Wave spectra"; per-wave-vector arithmetic in wso_spectrum.cuh).
struct SpectrumConsts;
wso_spectrum default_spectrum();
bool spectrum_valid(const wso_spectrum& s);
bool spectrum_is_phillips(const wso_spectrum& s);
// p: setter-normalised parameters; s: a valid non-Phillips spectrum
SpectrumConsts spectrum_consts(const wso_params& p, const wso_spectrum& s);
// largest multiple j of omega0 any in-band wave vector of the grid kv x kv can be quantised to (0: none in band);
// j is monotone in |k|, so this is j of the largest in-band |k|
double spectrum_max_j(const SpectrumConsts& c, const std::vector<float>& kv);
// records of rows [m0, m0+rows) of the N*N grid: xi = full N*N complex array, or NULL = counter_gauss(seed, m*N+n);
// the Phillips kind goes through H0Builder (bit for bit what wso_prepare_gauss / wso_counter_h0 build)
void host_spectrum_rows(const wso_params& p, const wso_spectrum& s, const float* xi, uint64_t seed, uint32_t m0,
                        uint32_t rows, wso_h0_record* out);

}  // namespace wso
