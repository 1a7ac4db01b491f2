// wso_hydro.cu — the hydrostatics kernel (wso_hydrostatics): one 256-thread CTA per body.
//   phase 1: the threads stride over the body's vertices (transform, surface height, depth) into shared memory as
//            (arm xyz, depth) float4s; one barrier also ORs the invalid / wet / dry flags;
//   phase 2: thread t adds triangles t, t + 256, ... in increasing order into seven float64 sums in registers;
//   combine: the lanes' sums go to shared memory (over the vertex array) and a fixed pairwise tree (strides 128 ... 1)
//            adds them; thread 0 stores the record as two float4s.
// The per-vertex, per-triangle and combine steps are wso_hydro.cuh's, shared with the host build.  Its own translation
// unit, so the query and ray-cast kernels compile exactly as before.
#include <atomic>

#include <cuda_runtime.h>
#include <stdint.h>

#include "wso_hydro.cuh"

namespace wso {

namespace {

constexpr size_t kHydroSmemBytes = sizeof(float4) * kMaxHullVertices;   // 64 KB (opt-in above 48 KB)
static_assert(sizeof(double) * kHydroSums * kHydroLanes <= kHydroSmemBytes, "the tree reuses the vertex array");

template <class Texel, int NS>
__global__ void __launch_bounds__(256) wso_hydro_kernel(const __grid_constant__ HydroArgs a) {
    extern __shared__ float4 sv[];
    const uint32_t tid = threadIdx.x;
    const HydroBody b = a.bodies[blockIdx.x];
    float4* o = a.out + 2 * (size_t)blockIdx.x;
    if (!hydro_ranges_ok(a, b)) {   // uniform over the CTA
        if (tid == 0) hydro_invalid(o);
        return;
    }
    const HydroPose p = hydro_pose(b);
    int bad = !p.ok, wet = 0, dry = 0;
    for (uint32_t v = tid; v < b.vertex_count; v += kHydroLanes) {
        bool ok;
        const float4 w = hydro_vertex<Texel, NS>(a.q, p, __ldg(a.vertices + b.vertex_first + v), ok);
        bad |= !ok;
        wet |= w.w > 0.0f;
        dry |= !(w.w > 0.0f);
        sv[v] = w;
    }
    bad = __syncthreads_or(bad);
    wet = __syncthreads_or(wet);
    dry = __syncthreads_or(dry);
    if (bad) {
        if (tid == 0) hydro_invalid(o);
        return;
    }
    double acc[kHydroSums];
#pragma unroll
    for (int k = 0; k < kHydroSums; ++k) acc[k] = 0.0;
    int bad_index = 0;
    for (uint32_t i = tid; i < b.triangle_count; i += kHydroLanes) {
        const uint32_t* tri = a.triangles + 3 * ((size_t)b.triangle_first + i);
        const uint32_t i0 = __ldg(tri), i1 = __ldg(tri + 1), i2 = __ldg(tri + 2);
        if (i0 >= b.vertex_count || i1 >= b.vertex_count || i2 >= b.vertex_count) {
            bad_index = 1;
            continue;
        }
        hydro_triangle(sv[i0], sv[i1], sv[i2], acc);
    }
    if (__syncthreads_or(bad_index)) {   // also the barrier before the vertex array is reused
        if (tid == 0) hydro_invalid(o);
        return;
    }
    double* sums = reinterpret_cast<double*>(sv);   // [k][lane]
#pragma unroll
    for (int k = 0; k < kHydroSums; ++k) sums[k * kHydroLanes + tid] = acc[k];
    __syncthreads();
#pragma unroll
    for (uint32_t stride = kHydroLanes / 2; stride >= 1; stride /= 2) {
        if (tid < stride) {
            double x[kHydroSums], y[kHydroSums];
#pragma unroll
            for (int k = 0; k < kHydroSums; ++k) {
                x[k] = sums[k * kHydroLanes + tid];
                y[k] = sums[k * kHydroLanes + tid + stride];
            }
            hydro_combine(x, y);
#pragma unroll
            for (int k = 0; k < kHydroSums; ++k) sums[k * kHydroLanes + tid] = x[k];
        }
        __syncthreads();
    }
    if (tid == 0) {
        double s[kHydroSums];
#pragma unroll
        for (int k = 0; k < kHydroSums; ++k) s[k] = sums[k * kHydroLanes];
        float4 r[2];
        hydro_record(a.k, s, hydro_status(wet != 0, dry != 0), r);
        o[0] = r[0];
        o[1] = r[1];
    }
}

template <class Texel, int NS>
cudaError_t launch_hydro_ns(const HydroArgs& a, cudaStream_t stream) {
    static std::atomic<bool> configured[16];   // per device: opt in to 64 KB of dynamic shared memory once
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 16 || !configured[dev].load(std::memory_order_acquire)) {
        const cudaError_t e = cudaFuncSetAttribute(wso_hydro_kernel<Texel, NS>,
                                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kHydroSmemBytes);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 16) configured[dev].store(true, std::memory_order_release);
    }
    wso_hydro_kernel<Texel, NS><<<a.n, kHydroLanes, kHydroSmemBytes, stream>>>(a);
    return cudaGetLastError();
}

template <class Texel>
cudaError_t launch_hydro_texel(const HydroArgs& a, int n_slots, cudaStream_t stream) {
    switch (n_slots) {
        case 1: return launch_hydro_ns<Texel, 1>(a, stream);
        case 2: return launch_hydro_ns<Texel, 2>(a, stream);
        case 3: return launch_hydro_ns<Texel, 3>(a, stream);
        case 4: return launch_hydro_ns<Texel, 4>(a, stream);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace

cudaError_t launch_hydrostatics(const HydroArgs& a, int n_slots, bool half, cudaStream_t stream) {
    return half ? launch_hydro_texel<Half4>(a, n_slots, stream) : launch_hydro_texel<float4>(a, n_slots, stream);
}

}  // namespace wso
