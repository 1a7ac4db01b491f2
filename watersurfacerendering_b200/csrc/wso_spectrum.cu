// wso_spectrum.cu — device Prepare of the empirical wave spectra (include/wsocean.h, "Wave spectra"): the records of a
// Pierson-Moskowitz / JONSWAP / TMA tile, built with the thread-to-work mapping and the output arrays of
// wso_prepare_kernel (wso_prepare_kernels.cu).  The per-wave-vector arithmetic is wso_spectrum.cuh, shared with the host
// build (wso_host_prepare.cpp).  A translation unit of its own: its float64 library calls would otherwise move the
// constants the existing Prepare kernels read.
#include <cuda_runtime.h>
#include <stdint.h>

#include "wso_counter_gauss.cuh"
#include "wso_kernels.cuh"
#include "wso_spectrum.cuh"

namespace wso {

namespace {

// One record of a non-Phillips spectrum: (amp.re, amp.im, 1/|k|, j or omega)
__device__ __forceinline__ float4 spectrum_record_at(const SpectrumPrepareArgs& a, float kx, float kz, float2 xi) {
    float re, im, inv, jf;
    spectrum_record(a.c, kx, kz, xi.x, xi.y, &re, &im, &inv, &jf);
    if (a.table) {
        // j is monotone in |k|: the host's j of the largest in-band |k| bounds every record (the cap only matters should
        // the device tanh round across an integer where the host's does not)
        const int j = (int)jf;
        return make_float4(re, im, inv, __int_as_float(j < a.j_cap ? j : a.j_cap));
    }
    return make_float4(re, im, inv, __fmul_rn(jf, a.c.omega0));
}

// The mapping of wso_prepare_kernel: one thread = rows (i, N-i) x columns (j, N-j), four records and the two pair sums.
__global__ void __launch_bounds__(256) wso_prepare_spectrum_kernel(const SpectrumPrepareArgs a) {
    const int N = a.n, H = N >> 1;
    const int i = blockIdx.y * blockDim.x + threadIdx.x;
    const int j = blockIdx.x;
    if (i >= H) return;
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
    const float4 q0 = spectrum_record_at(a, kxA, kzA, x0), q1 = spectrum_record_at(a, kxB, kzA, x1);
    const float4 q2 = spectrum_record_at(a, kxA, kzB, x2), q3 = spectrum_record_at(a, kxB, kzB, x3);
    float4* colA = a.h0 + (size_t)j * 2 * N;
    float4* colB = colA + N;
    colA[mA] = q0;
    colB[mA] = q1;
    colA[mB] = q2;
    colB[mB] = q3;
    float4* rec0 = a.hs + hs_index(j, i, 0, H);
    float4* rec1 = a.hs + hs_index(j, i, 1, H);
    if (i != 0 && j != 0) {
        *rec0 = make_float4(__fadd_rn(q0.x, q3.x), __fadd_rn(q0.y, q3.y), q0.z, q0.w);
        *rec1 = make_float4(__fadd_rn(q1.x, q2.x), __fadd_rn(q1.y, q2.y), q1.z, q1.w);
    } else {
        *rec0 = make_float4(0.f, 0.f, 0.f, 0.f);
        *rec1 = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

}  // namespace

cudaError_t launch_prepare_spectrum(const SpectrumPrepareArgs& a, cudaStream_t stream) {
    const int H = a.n / 2;
    const int threads = H < 256 ? H : 256;
    const dim3 grid((unsigned)H, (unsigned)((H + threads - 1) / threads), 1);
    wso_prepare_spectrum_kernel<<<grid, threads, 0, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace wso
