// TEST INFRASTRUCTURE — host build of the ray-cast body (wso_query.cuh, wso_raycast_surface).
//
// The same per-ray code the sm_100a kernel runs, compiled by g++ with -ffp-contract=off: every fp32 / float64 operation
// in it is an explicit round-to-nearest one, so its records equal the device's bit for bit on the same maps.  Built and
// loaded by tests/test_surface_raycast.py; never linked into the product library.
#include <cstdint>

#include "wso_query.cuh"

using namespace wso;

extern "C" {

// half: the maps hold RGBA16F texels.  disp[s] / norm[s]: N*N texels of cascade s, ampl[s] = A_s, length[s] = L_s,
// lambda[s] = lambda_s.  rays: n x 8 floats (ox, oy, oz, tmax, dx, dy, dz, -); out: n x 12 floats (the 48-byte
// wso_ray_hit).  The march parameters are not range-checked here.  Returns 0, or -1 for an unsupported argument.
int wso_emur_raycast(int half, uint32_t tile_n, int n_slots, const void* const* disp, const void* const* norm,
                     const float* ampl, const float* length, const float* lambda, int iterations, float step,
                     uint32_t max_steps, uint32_t refine, uint32_t n, const float* rays, float* out) {
    if (n_slots < 1 || n_slots > kMaxQueryCascades || tile_n == 0 || (tile_n & (tile_n - 1)) != 0 || max_steps == 0)
        return -1;
    RayArgs a{};
    for (int s = 0; s < n_slots; ++s)
        a.q.c[s] = make_query_cascade(disp[s], norm[s], ampl + s, tile_n, length[s], lambda[s]);
    a.q.mask = tile_n - 1;
    int logn = 0;
    while ((1u << logn) < tile_n) ++logn;
    a.q.logn = logn;
    a.q.iterations = iterations;
    a.step = step;
    a.max_steps = max_steps;
    a.refine = refine;
    a.n = n;
    for (uint32_t i = 0; i < n; ++i) {
        const float* r = rays + 8 * (size_t)i;
        const float4 ro = make_float4(r[0], r[1], r[2], r[3]), rd = make_float4(r[4], r[5], r[6], r[7]);
        float4 o[3];
        switch (n_slots * 2 + (half ? 1 : 0)) {
            case 2: raycast_ray<float4, 1>(a, ro, rd, o); break;
            case 3: raycast_ray<Half4, 1>(a, ro, rd, o); break;
            case 4: raycast_ray<float4, 2>(a, ro, rd, o); break;
            case 5: raycast_ray<Half4, 2>(a, ro, rd, o); break;
            case 6: raycast_ray<float4, 3>(a, ro, rd, o); break;
            case 7: raycast_ray<Half4, 3>(a, ro, rd, o); break;
            case 8: raycast_ray<float4, 4>(a, ro, rd, o); break;
            default: raycast_ray<Half4, 4>(a, ro, rd, o); break;
        }
        float* w = out + 12 * (size_t)i;
        for (int k = 0; k < 3; ++k) {
            w[4 * k] = o[k].x;
            w[4 * k + 1] = o[k].y;
            w[4 * k + 2] = o[k].z;
            w[4 * k + 3] = o[k].w;
        }
    }
    return 0;
}

}  // extern "C"
