// wso_counter_gauss.cuh — device build of the counter-based Gaussian generator (wso::counter_gauss in
// wso_host_prepare.cpp), shared by the device Prepare kernels of wso_prepare_kernels.cu and wso_spectrum.cu.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace wso {

namespace {

__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// device build of wso::counter_gauss (wso_host_prepare.cpp): same integer mix, Box-Muller in float64
__device__ __forceinline__ float2 counter_gauss_dev(uint64_t seed_mixed, uint64_t idx) {
    const uint64_t u = mix64(seed_mixed ^ mix64(idx + 0x632BE59BD9B4E019ull));
    const double u1 = ((double)(u >> 40) + 1.0) * (1.0 / 16777216.0);
    const double u2 = (double)((u >> 8) & 0xFFFFFFull) * (1.0 / 16777216.0);
    const double r = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincos(2.0 * 3.14159265358979323846 * u2, &sn, &cs);
    return make_float2((float)(r * cs), (float)(r * sn));
}

}  // namespace

}  // namespace wso
