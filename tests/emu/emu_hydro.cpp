// TEST INFRASTRUCTURE — host build of the hydrostatics body (wso_hydro.cuh, wso_hydrostatics).
//
// The same per-vertex, per-triangle and combine code the sm_100a kernel runs, its 256 lanes stepped one after the other
// in the kernel's order, compiled by g++ with -ffp-contract=off: every fp32 / float64 operation in it is an explicit
// round-to-nearest one, so its records equal the device's bit for bit on the same maps.  Built and loaded by
// tests/test_hydrostatics.py; never linked into the product library.
#include <cstdint>
#include <vector>

#include "wso_hydro.cuh"

using namespace wso;

extern "C" {

// half: the maps hold RGBA16F texels.  disp[s] / norm[s]: N*N texels of cascade s, ampl[s] = A_s, length[s] = L_s.
// bodies: n x 80-byte wso_body; vertices: n_vertices x 4 floats; triangles: n_triangles x 3 uint32; out: n x 8 floats
// (the 32-byte wso_hydro_result).  k = density * gravity.  Returns 0, or -1 for an unsupported argument.
int wso_emuh_hydro(int half, uint32_t tile_n, int n_slots, const void* const* disp, const void* const* norm,
                   const float* ampl, const float* length, int iterations, double k, uint32_t n, const void* bodies,
                   uint32_t n_vertices, const float* vertices, uint32_t n_triangles, const uint32_t* triangles,
                   float* out) {
    if (n_slots < 1 || n_slots > kMaxQueryCascades || tile_n == 0 || (tile_n & (tile_n - 1)) != 0) return -1;
    HydroArgs a{};
    for (int s = 0; s < n_slots; ++s) a.q.c[s] = make_query_cascade(disp[s], norm[s], ampl + s, tile_n, length[s], 0.0f);
    a.q.mask = tile_n - 1;
    int logn = 0;
    while ((1u << logn) < tile_n) ++logn;
    a.q.logn = logn;
    a.q.iterations = iterations;
    a.bodies = static_cast<const HydroBody*>(bodies);
    a.vertices = reinterpret_cast<const float4*>(vertices);
    a.triangles = triangles;
    a.n = n;
    a.n_vertices = n_vertices;
    a.n_triangles = n_triangles;
    a.k = k;
    std::vector<float4> sv(kMaxHullVertices);
    for (uint32_t i = 0; i < n; ++i) {
        float4 o[2];
        switch (n_slots * 2 + (half ? 1 : 0)) {
            case 2: hydro_body_host<float4, 1>(a, i, sv.data(), o); break;
            case 3: hydro_body_host<Half4, 1>(a, i, sv.data(), o); break;
            case 4: hydro_body_host<float4, 2>(a, i, sv.data(), o); break;
            case 5: hydro_body_host<Half4, 2>(a, i, sv.data(), o); break;
            case 6: hydro_body_host<float4, 3>(a, i, sv.data(), o); break;
            case 7: hydro_body_host<Half4, 3>(a, i, sv.data(), o); break;
            case 8: hydro_body_host<float4, 4>(a, i, sv.data(), o); break;
            default: hydro_body_host<Half4, 4>(a, i, sv.data(), o); break;
        }
        float* w = out + 8 * (size_t)i;
        for (int j = 0; j < 2; ++j) {
            w[4 * j] = o[j].x;
            w[4 * j + 1] = o[j].y;
            w[4 * j + 2] = o[j].z;
            w[4 * j + 3] = o[j].w;
        }
    }
    return 0;
}

}  // extern "C"
