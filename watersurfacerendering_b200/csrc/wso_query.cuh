// wso_query.cuh — surface queries (wso_query_surface): height, normal and undisplaced origin of the ocean surface at
// arbitrary world positions, sampled from the displacement and normal maps of up to four slots (cascades).
//
// The per-query body is written once, for the device (wso_query_kernels.cu) and for the host build the tests step
// (tests/emu/emu_query.cpp).  Every fp32 operation is an explicit round-to-nearest one (rmul / radd / rsub / rdiv /
// sqrt_ieee; double: dmul / dsub / ddiv below), so that nvcc cannot contract anything into an FMA and the two builds give
// bit-identical records.  The contract (include/wsocean.h, "Surface queries"):
//   texel [m][n] of a slot is the field at world (x, z) = (n*L/N, m*L/N), L-periodic;
//   S[F](x, z): u = x*N/L, v = z*N/L, bilinear blend of texels [m0|m0+1][n0|n0+1] (n0 = floor(u), m0 = floor(v)),
//              indices wrapped mod N; x and z are reduced mod L once per cascade in float64, the rest is fp32;
//   p = q + d_I with d_0 = 0, d_{k+1} = -Dh(q + d_k), Dh = sum over cascades of (S[D.x], S[D.z]).
#pragma once

#include "wso_device.cuh"

namespace wso {

static constexpr int kMaxQueryCascades = 4;
static constexpr int kMaxQueryIterations = 16;

// One cascade (slot) of a query: where its maps are and how its texels map to world space.
struct QueryCascade {
    const void* disp;    // N*N texels of the slot's displacement map (float4 or Half4)
    const void* norm;    // N*N texels of its normal map
    const float* ampl;   // the slot's A (d_ampl[slot] on the device)
    double length;       // L_s, the tile_length the slot's tile was prepared with
    float n_over_l;      // N / L_s, rounded once to fp32
    float lambda;        // lambda of the compute that wrote the slot
};

struct QueryArgs {
    QueryCascade c[kMaxQueryCascades];
    const float* xz;     // n x (x, z)
    float4* out;         // n x 2 float4: (height, normal xyz), (offset x, offset z, residual, w)
    uint32_t n;          // queries
    uint32_t mask;       // N - 1
    int logn;            // log2 N
    int iterations;      // I
};

WSO_HD QueryCascade make_query_cascade(const void* disp, const void* norm, const float* ampl, uint32_t n,
                                       float tile_length, float lambda) {
    QueryCascade c;
    c.disp = disp;
    c.norm = norm;
    c.ampl = ampl;
    c.length = (double)tile_length;
    c.n_over_l = (float)((double)n / (double)tile_length);
    c.lambda = lambda;
    return c;
}

#if defined(__CUDA_ARCH__)
WSO_HD double dmul(double a, double b) { return __dmul_rn(a, b); }
WSO_HD double dsub(double a, double b) { return __dsub_rn(a, b); }
WSO_HD double ddiv(double a, double b) { return __ddiv_rn(a, b); }
// read-only, non-coherent texel loads: 16 bytes (RGBA32F), or 8 bytes and cvt f16x2 -> f32 (RGBA16F)
WSO_HD float4 ld_texel(const float4* p) { return __ldg(p); }
WSO_HD float4 ld_texel(const Half4* p) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
    __half2 xy, zw;
    memcpy(&xy, &u.x, 4);
    memcpy(&zw, &u.y, 4);
    const float2 a = __half22float2(xy), b = __half22float2(zw);
    return make_float4(a.x, a.y, b.x, b.y);
}
WSO_HD int floor_to_int(float f) { return __float2int_rd(f); }
#else
WSO_HD double dmul(double a, double b) { return a * b; }
WSO_HD double dsub(double a, double b) { return a - b; }
WSO_HD double ddiv(double a, double b) { return a / b; }
WSO_HD float4 ld_texel(const float4* p) { return *p; }
WSO_HD float4 ld_texel(const Half4* p) {
    return make_float4(f16_to_f32((uint16_t)(p->xy & 0xffffu)), f16_to_f32((uint16_t)(p->xy >> 16)),
                       f16_to_f32((uint16_t)(p->zw & 0xffffu)), f16_to_f32((uint16_t)(p->zw >> 16)));
}
// cvt.rmi.s32.f32 semantics where the value fits (non-finite coordinates only feed NaN into the weights)
WSO_HD int floor_to_int(float f) { return (f == f && std::fabs(f) < 2147483520.0f) ? (int)std::floor(f) : 0; }
#endif

// x mod L in float64 (x - floor(x/L)*L; the product and difference are exact for every |x| a float64 quotient resolves),
// rounded once to fp32.  Rounding can land on L itself or a hair below 0: the index wrap absorbs both.
WSO_HD float reduce_mod(float x, double length) {
    const double k = floor(ddiv((double)x, length));
    return (float)dsub((double)x, dmul(k, length));
}

// lerp a + f*(b - a) channel by channel
WSO_HD float4 lerp4(float4 a, float4 b, float f) {
    return make_float4(radd(a.x, rmul(f, rsub(b.x, a.x))), radd(a.y, rmul(f, rsub(b.y, a.y))),
                       radd(a.z, rmul(f, rsub(b.z, a.z))), radd(a.w, rmul(f, rsub(b.w, a.w))));
}

// Bilinear sample S[F] of one map at slot-local position (x, z) (x, z already reduced mod L, offsets added).
template <class Texel>
WSO_HD float4 sample_map(const Texel* map, float n_over_l, uint32_t mask, int logn, float x, float z) {
    const float u = rmul(x, n_over_l), v = rmul(z, n_over_l);
    const int n0 = floor_to_int(u), m0 = floor_to_int(v);
    const float fu = rsub(u, (float)n0), fv = rsub(v, (float)m0);
    const uint32_t c0 = (uint32_t)n0 & mask, c1 = (uint32_t)(n0 + 1) & mask;
    const uint32_t r0 = ((uint32_t)m0 & mask) << logn, r1 = ((uint32_t)(m0 + 1) & mask) << logn;
    const float4 t00 = ld_texel(map + (r0 | c0)), t01 = ld_texel(map + (r0 | c1));
    const float4 t10 = ld_texel(map + (r1 | c0)), t11 = ld_texel(map + (r1 | c1));
    return lerp4(lerp4(t00, t01, fu), lerp4(t10, t11, fu), fv);
}

// One query.  NS cascades (1..4), a.iterations fixed-point steps.  o[0] = (height, normal x, y, z),
// o[1] = (offset x, offset z, residual, w).
template <class Texel, int NS>
WSO_HD void query_point(const QueryArgs& a, float qx, float qz, float4* o) {
    float xr[NS], zr[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        xr[s] = reduce_mod(qx, a.c[s].length);
        zr[s] = reduce_mod(qz, a.c[s].length);
    }
    // d_{k+1} = -Dh(q + d_k), held as offsets from q
    float dx = 0.0f, dz = 0.0f;
    for (int k = 0; k < a.iterations; ++k) {
        float hx = 0.0f, hz = 0.0f;
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            const float4 d = sample_map(static_cast<const Texel*>(a.c[s].disp), a.c[s].n_over_l, a.mask, a.logn,
                                        radd(xr[s], dx), radd(zr[s], dz));
            hx = s == 0 ? d.x : radd(hx, d.x);
            hz = s == 0 ? d.z : radd(hz, d.z);
        }
        dx = -hx;
        dz = -hz;
    }
    // everything at p = q + d_I
    float h = 0.0f, hx = 0.0f, hz = 0.0f, w = 1.0f, sx = 0.0f, sz = 0.0f, ex = 1.0f, ez = 1.0f;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const float px = radd(xr[s], dx), pz = radd(zr[s], dz);
        const float4 d = sample_map(static_cast<const Texel*>(a.c[s].disp), a.c[s].n_over_l, a.mask, a.logn, px, pz);
        const float4 g = sample_map(static_cast<const Texel*>(a.c[s].norm), a.c[s].n_over_l, a.mask, a.logn, px, pz);
        const float amp = *a.c[s].ampl;
        const float lam = a.c[s].lambda;
        if (s == 0) {
            h = rmul(amp, d.y);
            hx = d.x;
            hz = d.z;
            w = d.w;
            sx = g.x;
            sz = g.y;
        } else {
            h = radd(h, rmul(amp, d.y));
            hx = radd(hx, d.x);
            hz = radd(hz, d.z);
            sx = radd(sx, g.x);
            sz = radd(sz, g.y);
        }
        ex = radd(ex, rmul(lam, g.z));
        ez = radd(ez, rmul(lam, g.w));
    }
    // normalize(-sx/ex, 1, -sz/ez)
    const float nx = -rdiv(sx, ex), nz = -rdiv(sz, ez);
    const float len = sqrt_ieee(radd(radd(rmul(nx, nx), 1.0f), rmul(nz, nz)));
    const float rx = radd(dx, hx), rz = radd(dz, hz);
    o[0] = make_float4(h, rdiv(nx, len), rdiv(1.0f, len), rdiv(nz, len));
    o[1] = make_float4(dx, dz, sqrt_ieee(radd(rmul(rx, rx), rmul(rz, rz))), w);
}

}  // namespace wso
