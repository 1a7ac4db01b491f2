// wso_query_kernels.cu — the surface-query kernel (wso_query_surface) and the ray-cast kernel (wso_raycast_surface,
// one thread per ray, three 16-byte stores per record).  Query kernel: one thread per query, the per-query body of
// wso_query.cuh, the cascade constants in a __grid_constant__ parameter block.  Texel loads go through the read-only
// non-coherent path (the maps of every cascade together are a few MB at 512^2 / 1024^2 and stay L2-resident across
// queries); each record leaves as two 16-byte stores.
#include <cuda_runtime.h>
#include <stdint.h>

#include "wso_query.cuh"

namespace wso {

namespace {

template <class Texel, int NS>
__global__ void __launch_bounds__(256) wso_query_kernel(const __grid_constant__ QueryArgs a) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const float qx = __ldg(a.xz + 2 * (size_t)i), qz = __ldg(a.xz + 2 * (size_t)i + 1);
    float4 o[2];
    query_point<Texel, NS>(a, qx, qz, o);
    a.out[2 * (size_t)i] = o[0];
    a.out[2 * (size_t)i + 1] = o[1];
}

// One thread per ray; rays of a warp march different numbers of samples and leave the loop independently.
template <class Texel, int NS>
__global__ void __launch_bounds__(256) wso_raycast_kernel(const __grid_constant__ RayArgs a) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const float4 ro = __ldg(a.rays + 2 * (size_t)i), rd = __ldg(a.rays + 2 * (size_t)i + 1);
    float4 o[3];
    raycast_ray<Texel, NS>(a, ro, rd, o);
    a.out[3 * (size_t)i] = o[0];
    a.out[3 * (size_t)i + 1] = o[1];
    a.out[3 * (size_t)i + 2] = o[2];
}

template <class Texel>
cudaError_t launch_raycast_texel(const RayArgs& a, int n_slots, cudaStream_t stream) {
    const unsigned threads = 256;
    const unsigned blocks = (unsigned)((a.n + threads - 1) / threads);
    switch (n_slots) {
        case 1: wso_raycast_kernel<Texel, 1><<<blocks, threads, 0, stream>>>(a); break;
        case 2: wso_raycast_kernel<Texel, 2><<<blocks, threads, 0, stream>>>(a); break;
        case 3: wso_raycast_kernel<Texel, 3><<<blocks, threads, 0, stream>>>(a); break;
        case 4: wso_raycast_kernel<Texel, 4><<<blocks, threads, 0, stream>>>(a); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

template <class Texel>
cudaError_t launch_texel(const QueryArgs& a, int n_slots, cudaStream_t stream) {
    const unsigned threads = 256;
    const unsigned blocks = (unsigned)((a.n + threads - 1) / threads);
    switch (n_slots) {
        case 1: wso_query_kernel<Texel, 1><<<blocks, threads, 0, stream>>>(a); break;
        case 2: wso_query_kernel<Texel, 2><<<blocks, threads, 0, stream>>>(a); break;
        case 3: wso_query_kernel<Texel, 3><<<blocks, threads, 0, stream>>>(a); break;
        case 4: wso_query_kernel<Texel, 4><<<blocks, threads, 0, stream>>>(a); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_query_surface(const QueryArgs& a, int n_slots, bool half, cudaStream_t stream) {
    return half ? launch_texel<Half4>(a, n_slots, stream) : launch_texel<float4>(a, n_slots, stream);
}

cudaError_t launch_raycast_surface(const RayArgs& a, int n_slots, bool half, cudaStream_t stream) {
    return half ? launch_raycast_texel<Half4>(a, n_slots, stream) : launch_raycast_texel<float4>(a, n_slots, stream);
}

}  // namespace wso
