// wso_prepare_kernels.cu — Prepare() on the device (SURVEY §8 row f-3): wave vectors, Phillips spectrum h0(k),
// quantised dispersion and the compact record arrays K1 reads, built in one pass from either an uploaded Gaussian
// array or a counter-based one generated in the kernel.
//
// Replaces (device build of) reference WSTessendorf::ComputeWaveVectors (src/scene/WSTessendorf.cpp:60-85),
// ComputeBaseWaveHeightField (cpp:105-148) with PhillipsSpectrum / BaseWaveHeightFT / QDispersion
// (WSTessendorf.h:237-263, 284-297).  The host build of the same arithmetic is wso_host_prepare.cpp (H0Builder::at):
// every fp32 product, quotient and square root below is the same single IEEE operation in the same order (no FMA
// contraction); the two exp() calls are evaluated in float64 and rounded once, which agrees with the host's expf
// except where that (<= 0.502 ulp) function rounds the other way - amplitudes may differ from the host build by 1 ulp
// in rare wave vectors, dispersion, 1/|k| and the layout are bit-identical (tests/test_prepare_device.py).
#include <cuda_runtime.h>
#include <stdint.h>

#include "wso_counter_gauss.cuh"
#include "wso_kernels.cuh"
#include "wso_launch.h"

namespace wso {

namespace {

__device__ __forceinline__ float exp_f32(float x) { return (float)exp((double)x); }

// the record of one wave vector: (amp.re, amp.im, 1/|k|, j) with omega = fl(float(j) * omega0)
__device__ __forceinline__ float4 record_at(const PrepareArgs& a, float kx, float kz, float2 xi) {
    const float dot = __fadd_rn(__fmul_rn(kx, kx), __fmul_rn(kz, kz));
    const float k = __fsqrt_rn(dot);
    if (!(k > 0.00001f)) return make_float4(0.0f, 0.0f, 0.0f, __int_as_float(0));
    const float inv = __fdiv_rn(1.0f, k);
    const float ux = __fmul_rn(kx, inv), uz = __fmul_rn(kz, inv);
    const float k2 = __fmul_rn(k, k);
    const float k4 = __fmul_rn(k2, k2);
    float cf = __fadd_rn(__fmul_rn(ux, a.wind_x), __fmul_rn(uz, a.wind_y));
    cf = __fmul_rn(cf, cf);
    // A * exp(-1/(k^2 L^2)) / k^4 * (k^.w)^2 * exp(-k^2 l^2)        reference: WSTessendorf.h:249-263
    float ph = __fmul_rn(a.phillips_const, exp_f32(__fdiv_rn(-1.0f, __fmul_rn(k2, a.Lw2))));
    ph = __fdiv_rn(ph, k4);
    ph = __fmul_rn(ph, cf);
    ph = __fmul_rn(ph, exp_f32(__fmul_rn(__fmul_rn(-k2, a.damping), a.damping)));
    const float s = __fsqrt_rn(ph);
    // (1/sqrt 2) * xi * sqrt(P)                                        reference: WSTessendorf.h:237-243
    const float re = __fmul_rn(__fmul_rn(a.inv_sqrt2, xi.x), s);
    const float im = __fmul_rn(__fmul_rn(a.inv_sqrt2, xi.y), s);
    // floor(sqrt(g k) / omega0) * omega0: the integer multiple is what K1's per-frame table is indexed by
    const float jf = floorf(__fdiv_rn(__fsqrt_rn(__fmul_rn(9.81f, k)), a.omega0));
    return make_float4(re, im, inv, __int_as_float((int)jf));
}

// One thread = one evolve work item of K1: rows (i, N-i) x columns (j, N-j) (the partners of index 0 are N/2),
// i.e. four wave vectors, their four records and - away from the index-0 lines - the two pair-summed records.
__global__ void __launch_bounds__(256) wso_prepare_kernel(const PrepareArgs a) {
    const int N = a.n, H = N >> 1;
    const int i = blockIdx.y * blockDim.x + threadIdx.x;
    const int jl = blockIdx.x;
    if (i >= H) return;
    const int j = a.j0 + jl;
    const int mA = i, mB = (i == 0) ? H : N - i;
    const int nA = j, nB = (j == 0) ? H : N - j;
    const float kxA = a.kv[nA], kxB = a.kv[nB], kzA = a.kv[mA], kzB = a.kv[mB];
    float2 x0, x1, x2, x3;
    if (a.xi != nullptr) {
        x0 = a.xi[(size_t)mA * N + nA];
        x1 = a.xi[(size_t)mA * N + nB];
        x2 = a.xi[(size_t)mB * N + nA];
        x3 = a.xi[(size_t)mB * N + nB];
    } else {
        x0 = counter_gauss_dev(a.seed_mixed, (uint64_t)mA * N + nA);
        x1 = counter_gauss_dev(a.seed_mixed, (uint64_t)mA * N + nB);
        x2 = counter_gauss_dev(a.seed_mixed, (uint64_t)mB * N + nA);
        x3 = counter_gauss_dev(a.seed_mixed, (uint64_t)mB * N + nB);
    }
    const float4 q0 = record_at(a, kxA, kzA, x0), q1 = record_at(a, kxB, kzA, x1);
    const float4 q2 = record_at(a, kxA, kzB, x2), q3 = record_at(a, kxB, kzB, x3);
    float4* colA = a.h0 + (size_t)jl * 2 * N;
    float4* colB = colA + N;
    colA[mA] = q0;
    colB[mA] = q1;
    colA[mB] = q2;
    colB[mB] = q3;
    float4* rec0 = a.hs + hs_index(jl, i, 0, H);
    float4* rec1 = a.hs + hs_index(jl, i, 1, H);
    if (i != 0 && j != 0) {
        // h0(k) + h0(-k): (m,n) mirrors into (N-m, N-n); 1/|k| and the dispersion are even in k
        *rec0 = make_float4(__fadd_rn(q0.x, q3.x), __fadd_rn(q0.y, q3.y), q0.z, q0.w);
        *rec1 = make_float4(__fadd_rn(q1.x, q2.x), __fadd_rn(q1.y, q2.y), q1.z, q1.w);
    } else {
        *rec0 = make_float4(0.f, 0.f, 0.f, 0.f);
        *rec1 = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

// Device records -> the reference's 20-byte BaseWaveHeight records, row-major [m][n] (export / checkpoint).
__global__ void __launch_bounds__(256) wso_export_records_kernel(const float4* __restrict__ h0, float* __restrict__ out,
                                                                 int N, float omega0, int table) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    const int m = blockIdx.y;
    if (n >= N) return;
    const float4 q = h0[h0_index(n, m, N, 0)];
    const float w = table ? __fmul_rn((float)__float_as_int(q.w), omega0) : q.w;
    float* o = out + ((size_t)m * N + n) * 5;
    o[0] = q.x;
    o[1] = q.y;
    o[2] = q.x;
    o[3] = -q.y;
    o[4] = w;
}

}  // namespace

cudaError_t launch_prepare(const PrepareArgs& a, int n_pairs, cudaStream_t stream) {
    const int H = a.n / 2;
    const int threads = H < 256 ? H : 256;
    const dim3 grid((unsigned)n_pairs, (unsigned)((H + threads - 1) / threads), 1);
    wso_prepare_kernel<<<grid, threads, 0, stream>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_export_records(const float4* h0, float* out20, int n, float omega0, bool table, cudaStream_t stream) {
    const int threads = n < 256 ? n : 256;
    const dim3 grid((unsigned)((n + threads - 1) / threads), (unsigned)n, 1);
    wso_export_records_kernel<<<grid, threads, 0, stream>>>(h0, out20, n, omega0, table ? 1 : 0);
    return cudaGetLastError();
}

uint64_t counter_seed_mix(uint64_t seed) {
    uint64_t x = seed + 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

}  // namespace wso
