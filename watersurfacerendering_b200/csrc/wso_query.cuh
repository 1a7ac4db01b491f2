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

// The a.iterations fixed-point steps d_{k+1} = -Dh(q + d_k) from d_0 = 0, held as offsets (dx, dz) from the slot-local
// positions (xr[s], zr[s]) of q: query_point's loop, for the ray march.
template <class Texel, int NS>
WSO_HD void invert_offsets(const QueryArgs& a, const float* xr, const float* zr, float& dx, float& dz) {
    dx = 0.0f;
    dz = 0.0f;
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
    // d_{k+1} = -Dh(q + d_k), held as offsets from q.  (The same loop as invert_offsets: calling it here changes the
    // instruction schedule of the one-cascade query kernels, so the query keeps its own copy.)
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

// ---------------------------------------------------------------------------------------------------------------------
// Ray casts (wso_raycast_surface): the first point of a segment at or under the displaced surface.  Contract and
// operation order: include/wsocean.h, "Ray casts".
// ---------------------------------------------------------------------------------------------------------------------
static constexpr uint32_t kMaxRaySteps = 4096;
static constexpr uint32_t kMaxRayRefine = 24;
enum : uint32_t { kRayMiss = 0, kRayHit = 1, kRayOriginBelow = 2, kRayUnresolved = 3, kRayInvalid = 4 };

// Height slab: Hb = fl(fl(sum_s |A_s|) * kSlabMargin) bounds every H the march or a query can return.  Proof, with
// u = 2^-24 the fp32 unit roundoff:
//   texels: K2 writes disp.y = fl(fl(h) * fl(1/A)) with |fl(h)| <= A, so |D.y| <= (1 + u)^2 < 1 + 3u; binary16 rounds
//           such a value to at most 1 (rounding is monotone and 1 is a binary16 value); decoding is exact.
//   lerp:   a + f*(b - a) with |a|, |b| <= M and 0 <= f < 1 lies in [-M, M] exactly; its three roundings add at most
//           (2M * 2u + M * u)(1 + O(u)), so |lerp| <= M (1 + 5u + O(u^2)).  Two levels: |S[D.y]| <= 1 + 13u + O(u^2).
//   height: fl(A_s * S_s) and up to three fp32 sums: |H| <= sum_s |A_s| * (1 + 17u + O(u^2)).
//   Hb:     up to three roundings in the sum of |A_s| and one in the product: Hb >= sum_s |A_s| (1 + 2^-10)(1 - u)^4.
// 2^-10 = 16384u, so |H| < Hb with a wide margin (it also absorbs a normalisation a few ulp looser than K2's).
static constexpr float kSlabMargin = 1.0f + 1.0f / 1024.0f;

struct RayArgs {
    QueryArgs q;          // cascades, mask, logn, iterations (q.xz, q.out, q.n unused)
    const float4* rays;   // n x 2 float4: (ox, oy, oz, tmax), (dx, dy, dz, unused)
    float4* out;          // n x 3 float4: (distance, x, z, status bits), then the query record at (x, z)
    uint32_t n;           // rays
    float step;           // march spacing along d^, world units
    uint32_t max_steps;   // march samples per ray, 1..kMaxRaySteps
    uint32_t refine;      // bisection steps, 0..kMaxRayRefine
};

WSO_HD float bits_to_float(uint32_t u) {
    float f;
    memcpy(&f, &u, 4);
    return f;
}
WSO_HD uint32_t float_to_bits(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    return u;
}
WSO_HD bool is_finite(float f) { return (float_to_bits(f) & 0x7f800000u) != 0x7f800000u; }
WSO_HD float abs_f(float f) { return bits_to_float(float_to_bits(f) & 0x7fffffffu); }

// The per-ray state of the march: the origin reduced per cascade, the unit direction, the amplitudes.
template <int NS>
struct RayMarch {
    float px[NS], pz[NS];   // reduce_mod(ox, L_s), reduce_mod(oz, L_s)
    float amp[NS];          // A_s
    float oy, ux, uy, uz;   // origin height, d^
};

// f(t) <= 0: the point at parameter t is at or under the surface.  Only the displacement maps are read:
// H = sum_s A_s * S_s[D.y](q_s + d_I) at the march positions q_s = (px[s] + t*ux, pz[s] + t*uz).
template <class Texel, int NS>
WSO_HD bool ray_below(const QueryArgs& a, const RayMarch<NS>& m, float t) {
    const float sx = rmul(t, m.ux), sz = rmul(t, m.uz);
    float qx[NS], qz[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        qx[s] = radd(m.px[s], sx);
        qz[s] = radd(m.pz[s], sz);
    }
    float dx, dz;
    invert_offsets<Texel, NS>(a, qx, qz, dx, dz);
    float h = 0.0f;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const float4 d = sample_map(static_cast<const Texel*>(a.c[s].disp), a.c[s].n_over_l, a.mask, a.logn,
                                    radd(qx[s], dx), radd(qz[s], dz));
        h = s == 0 ? rmul(m.amp[s], d.y) : radd(h, rmul(m.amp[s], d.y));
    }
    return radd(m.oy, rmul(t, m.uy)) <= h;
}

// One ray: ro = (ox, oy, oz, tmax), rd = (dx, dy, dz, -).  o[0] = (distance, x, z, status bits), o[1], o[2] = the
// query record at (x, z) (query_point: bit for bit what wso_query_surface returns there).
template <class Texel, int NS>
WSO_HD void raycast_ray(const RayArgs& r, float4 ro, float4 rd, float4* o) {
    const QueryArgs& a = r.q;
    const float nan = bits_to_float(0x7fc00000u), inf = bits_to_float(0x7f800000u);
    // direction: scaled by its largest component first, so that the squares neither overflow nor underflow
    const float mx = abs_f(rd.x), my = abs_f(rd.y), mz = abs_f(rd.z);
    const float mxy = mx > my ? mx : my;
    const float dm = mxy > mz ? mxy : mz;
    if (!is_finite(ro.x) || !is_finite(ro.y) || !is_finite(ro.z) || !is_finite(rd.x) || !is_finite(rd.y) ||
        !is_finite(rd.z) || !(dm > 0.0f) || !(ro.w >= 0.0f)) {
        o[0] = make_float4(nan, nan, nan, bits_to_float(kRayInvalid));
        o[1] = o[2] = make_float4(nan, nan, nan, nan);
        return;
    }
    RayMarch<NS> m;
    const float vx = rdiv(rd.x, dm), vy = rdiv(rd.y, dm), vz = rdiv(rd.z, dm);
    const float len = sqrt_ieee(radd(radd(rmul(vx, vx), rmul(vy, vy)), rmul(vz, vz)));
    m.ux = rdiv(vx, len);
    m.uy = rdiv(vy, len);
    m.uz = rdiv(vz, len);
    m.oy = ro.y;
    float hb = 0.0f;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        m.px[s] = reduce_mod(ro.x, a.c[s].length);
        m.pz[s] = reduce_mod(ro.z, a.c[s].length);
        m.amp[s] = *a.c[s].ampl;
        hb = s == 0 ? abs_f(m.amp[s]) : radd(hb, abs_f(m.amp[s]));
    }
    hb = rmul(hb, kSlabMargin);
    uint32_t status;
    float lo = 0.0f, hi = 0.0f;   // bracket [a, b]; hi = the reported distance
    if (ro.y < -hb) {
        status = kRayOriginBelow;
    } else {
        // [s0, s_end] = [0, tmax] clipped to the slab |y| <= Hb
        float entry = -inf, exit = ro.y <= hb ? inf : -inf;
        if (m.uy != 0.0f) {
            const float t1 = rdiv(rsub(hb, ro.y), m.uy), t2 = rdiv(rsub(-hb, ro.y), m.uy);
            entry = t1 < t2 ? t1 : t2;
            exit = t1 < t2 ? t2 : t1;
        }
        const float s0 = entry > 0.0f ? entry : 0.0f;
        const float send = ro.w < exit ? ro.w : exit;
        status = kRayMiss;
        if (s0 <= send) {
            lo = hi = s0;
            for (uint32_t k = 0;; ++k) {
                float t = radd(s0, rmul((float)k, r.step));
                const bool last = !(t < send);
                if (last) t = send;
                if (ray_below<Texel, NS>(a, m, t)) {
                    hi = t;   // lo = the sample before (k = 0: t itself)
                    status = (k == 0 && s0 == 0.0f) ? kRayOriginBelow : kRayHit;
                    break;
                }
                if (last) break;
                lo = t;
                if (k + 1 == r.max_steps) {
                    status = kRayUnresolved;
                    break;
                }
            }
        }
        if (status == kRayHit) {
            for (uint32_t i = 0; i < r.refine; ++i) {
                const float mid = radd(lo, rmul(0.5f, rsub(hi, lo)));
                if (ray_below<Texel, NS>(a, m, mid))
                    hi = mid;
                else
                    lo = mid;
            }
        }
    }
    if (status == kRayHit || status == kRayOriginBelow) {
        const float x = radd(ro.x, rmul(hi, m.ux)), z = radd(ro.z, rmul(hi, m.uz));
        o[0] = make_float4(hi, x, z, bits_to_float(status));
        query_point<Texel, NS>(a, x, z, o + 1);
    } else {
        o[0] = make_float4(status == kRayMiss ? inf : lo, nan, nan, bits_to_float(status));
        o[1] = o[2] = make_float4(nan, nan, nan, nan);
    }
}

}  // namespace wso
