// TEST INFRASTRUCTURE — host build of the surface-query body (wso_query.cuh, wso_query_surface).
//
// The same per-query code the sm_100a kernel runs, compiled by g++ with -ffp-contract=off: every fp32 / float64 operation
// in it is an explicit round-to-nearest one, so its records equal the device's bit for bit on the same maps.  Built and
// loaded by tests/test_surface_query.py; never linked into the product library.
#include <cstdint>

#include "wso_query.cuh"

using namespace wso;

extern "C" {

// half: the maps hold RGBA16F texels.  disp[s] / norm[s]: N*N texels of cascade s, ampl[s] = A_s, length[s] = L_s,
// lambda[s] = lambda_s.  xz: n (x, z) pairs; out: n x 8 floats.  Returns 0, or -1 for an unsupported argument.
int wso_emuq_query(int half, uint32_t tile_n, int n_slots, const void* const* disp, const void* const* norm,
                   const float* ampl, const float* length, const float* lambda, int iterations, uint32_t n,
                   const float* xz, float* out) {
    if (n_slots < 1 || n_slots > kMaxQueryCascades || tile_n == 0 || (tile_n & (tile_n - 1)) != 0) return -1;
    QueryArgs a{};
    for (int s = 0; s < n_slots; ++s) a.c[s] = make_query_cascade(disp[s], norm[s], ampl + s, tile_n, length[s], lambda[s]);
    a.mask = tile_n - 1;
    int logn = 0;
    while ((1u << logn) < tile_n) ++logn;
    a.logn = logn;
    a.iterations = iterations;
    a.n = n;
    for (uint32_t i = 0; i < n; ++i) {
        float4 o[2];
        const float x = xz[2 * (size_t)i], z = xz[2 * (size_t)i + 1];
        switch (n_slots * 2 + (half ? 1 : 0)) {
            case 2: query_point<float4, 1>(a, x, z, o); break;
            case 3: query_point<Half4, 1>(a, x, z, o); break;
            case 4: query_point<float4, 2>(a, x, z, o); break;
            case 5: query_point<Half4, 2>(a, x, z, o); break;
            case 6: query_point<float4, 3>(a, x, z, o); break;
            case 7: query_point<Half4, 3>(a, x, z, o); break;
            case 8: query_point<float4, 4>(a, x, z, o); break;
            default: query_point<Half4, 4>(a, x, z, o); break;
        }
        float* r = out + 8 * (size_t)i;
        r[0] = o[0].x; r[1] = o[0].y; r[2] = o[0].z; r[3] = o[0].w;
        r[4] = o[1].x; r[5] = o[1].y; r[6] = o[1].z; r[7] = o[1].w;
    }
    return 0;
}

}  // extern "C"
