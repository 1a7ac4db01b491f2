// wso_hydro.cuh — hydrostatic force and torque on triangle-mesh hulls (wso_hydrostatics), over the maps of 1..4 slots.
// Contract and operation order: include/wsocean.h, "Hydrostatic forces".
//
// The per-vertex, per-triangle and combine steps are written once here.  The sm_100a kernel (wso_hydro.cu) runs them
// with one 256-thread CTA per body; hydro_body_host below runs the same 256 lanes one after the other, in the same order,
// for the host build the tests step (tests/emu/emu_hydro.cpp).  Every fp32 operation is an explicit round-to-nearest one
// (rmul / radd / rsub), every float64 one too (dadd / dsub / dmul / ddiv / dsqrt), so that nvcc contracts nothing into
// an FMA and the two builds give bit-identical records.
#pragma once

#include "wso_query.cuh"

namespace wso {

static constexpr uint32_t kHydroLanes = 256;          // threads per body (kernel) = lanes of the fixed-order sum
static constexpr uint32_t kMaxHullVertices = 4096;    // per body: 64 KB of (arm, depth) float4s in shared memory
static constexpr uint32_t kMaxHullTriangles = 65536;  // per body
static constexpr int kHydroSums = 7;                  // F' xyz, tau' xyz, wetted area
enum : uint32_t { kHydroDry = 0, kHydroPartial = 1, kHydroSubmerged = 2, kHydroInvalid = 3 };

// struct wso_body of the C ABI (80 bytes, checked in wso_api.cu)
struct HydroBody {
    float rotation[9];   // row-major R, body -> world
    float position[3];   // t
    float center[3];     // c, body coordinates
    uint32_t vertex_first, vertex_count, triangle_first, triangle_count;
    uint32_t unused;
};

struct HydroArgs {
    QueryArgs q;                 // cascades, mask, logn, iterations (q.xz, q.out, q.n unused)
    const HydroBody* bodies;     // n bodies
    const float4* vertices;      // n_vertices x (x, y, z, -), body coordinates
    const uint32_t* triangles;   // n_triangles x 3 indices, relative to the body's vertex_first
    float4* out;                 // n x 2 float4: (force xyz, wetted area), (torque xyz, status bits)
    uint32_t n;                  // bodies
    uint32_t n_vertices, n_triangles;
    double k;                    // density * gravity (exact in float64)
};

#if defined(__CUDA_ARCH__)
WSO_HD double dadd(double a, double b) { return __dadd_rn(a, b); }
WSO_HD double dsqrt(double a) { return __dsqrt_rn(a); }
#else
WSO_HD double dadd(double a, double b) { return a + b; }
WSO_HD double dsqrt(double a) { return std::sqrt(a); }
#endif

// The pose of one body: R, c, and c_w = t + R c (fp32).  ok: R, t and c are finite.
struct HydroPose {
    float r[9];
    float c[3];
    float cw[3];
    bool ok;
};

// R v, row by row: fl(fl(fl(R_i0 v0) + fl(R_i1 v1)) + fl(R_i2 v2))
WSO_HD float rot_row(const float* r, float x, float y, float z) {
    return radd(radd(rmul(r[0], x), rmul(r[1], y)), rmul(r[2], z));
}

WSO_HD HydroPose hydro_pose(const HydroBody& b) {
    HydroPose p;
    bool ok = true;
    for (int i = 0; i < 9; ++i) {
        p.r[i] = b.rotation[i];
        ok = ok && is_finite(p.r[i]);
    }
    for (int i = 0; i < 3; ++i) {
        p.c[i] = b.center[i];
        ok = ok && is_finite(p.c[i]) && is_finite(b.position[i]);
    }
    for (int i = 0; i < 3; ++i) p.cw[i] = radd(b.position[i], rot_row(p.r + 3 * i, p.c[0], p.c[1], p.c[2]));
    p.ok = ok;
    return p;
}

// The counts of a body fit the limits and its ranges lie inside the arrays.
WSO_HD bool hydro_ranges_ok(const HydroArgs& a, const HydroBody& b) {
    return b.vertex_count >= 1 && b.vertex_count <= kMaxHullVertices && b.triangle_count <= kMaxHullTriangles &&
           (uint64_t)b.vertex_first + b.vertex_count <= a.n_vertices &&
           (uint64_t)b.triangle_first + b.triangle_count <= a.n_triangles;
}

// One vertex v (body coordinates): -> (arm xyz, depth).  e = v - c, arm = R e, world = c_w + arm, H = the height
// wso_query_surface returns at (world.x, world.z) (the same reduction, inversion and height sum, so the same bits),
// depth = H - world.y.  ok: v, the arm and the depth are finite.
template <class Texel, int NS>
WSO_HD float4 hydro_vertex(const QueryArgs& a, const HydroPose& p, float4 v, bool& ok) {
    const float ex = rsub(v.x, p.c[0]), ey = rsub(v.y, p.c[1]), ez = rsub(v.z, p.c[2]);
    const float ax = rot_row(p.r, ex, ey, ez), ay = rot_row(p.r + 3, ex, ey, ez), az = rot_row(p.r + 6, ex, ey, ez);
    const float wx = radd(p.cw[0], ax), wy = radd(p.cw[1], ay), wz = radd(p.cw[2], az);
    float xr[NS], zr[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        xr[s] = reduce_mod(wx, a.c[s].length);
        zr[s] = reduce_mod(wz, a.c[s].length);
    }
    float dx, dz;
    invert_offsets<Texel, NS>(a, xr, zr, dx, dz);
    float h = 0.0f;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const float4 d = sample_map(static_cast<const Texel*>(a.c[s].disp), a.c[s].n_over_l, a.mask, a.logn,
                                    radd(xr[s], dx), radd(zr[s], dz));
        const float amp = *a.c[s].ampl;
        h = s == 0 ? rmul(amp, d.y) : radd(h, rmul(amp, d.y));
    }
    const float depth = rsub(h, wy);
    ok = is_finite(v.x) && is_finite(v.y) && is_finite(v.z) && is_finite(ax) && is_finite(ay) && is_finite(az) &&
         is_finite(depth);
    return make_float4(ax, ay, az, depth);
}

struct HydroPoint {
    double x, y, z, d;   // arm, depth
};

WSO_HD HydroPoint hydro_point(float4 v) { return HydroPoint{(double)v.x, (double)v.y, (double)v.z, (double)v.w}; }

// The point where the depth, linear along the edge p -> q, is zero (p wet, q dry): u = d_p / (d_p - d_q),
// x = p + u (q - p) per component.
WSO_HD HydroPoint hydro_cross(const HydroPoint& p, const HydroPoint& q) {
    const double u = ddiv(p.d, dsub(p.d, q.d));
    return HydroPoint{dadd(p.x, dmul(u, dsub(q.x, p.x))), dadd(p.y, dmul(u, dsub(q.y, p.y))),
                      dadd(p.z, dmul(u, dsub(q.z, p.z))), 0.0};
}

// One wet sub-triangle, added to acc[7] in the order F' xyz, tau' xyz, |S|:
//   S = 1/2 (y1 - y0) x (y2 - y0), sd = (d0 + d1) + d2, F' = -(sd / 3) S,
//   g = ((d0 y0 + d1 y1) + d2 y2) + sd ((y0 + y1) + y2), tau' = -((g x S) / 12), |S| = sqrt((Sx^2 + Sy^2) + Sz^2).
WSO_HD void hydro_sub(const HydroPoint& p0, const HydroPoint& p1, const HydroPoint& p2, double* acc) {
    const double ax = dsub(p1.x, p0.x), ay = dsub(p1.y, p0.y), az = dsub(p1.z, p0.z);
    const double bx = dsub(p2.x, p0.x), by = dsub(p2.y, p0.y), bz = dsub(p2.z, p0.z);
    const double sx = dmul(0.5, dsub(dmul(ay, bz), dmul(az, by)));
    const double sy = dmul(0.5, dsub(dmul(az, bx), dmul(ax, bz)));
    const double sz = dmul(0.5, dsub(dmul(ax, by), dmul(ay, bx)));
    const double sd = dadd(dadd(p0.d, p1.d), p2.d);
    const double m = ddiv(sd, 3.0);
    const double gx = dadd(dadd(dadd(dmul(p0.d, p0.x), dmul(p1.d, p1.x)), dmul(p2.d, p2.x)),
                           dmul(sd, dadd(dadd(p0.x, p1.x), p2.x)));
    const double gy = dadd(dadd(dadd(dmul(p0.d, p0.y), dmul(p1.d, p1.y)), dmul(p2.d, p2.y)),
                           dmul(sd, dadd(dadd(p0.y, p1.y), p2.y)));
    const double gz = dadd(dadd(dadd(dmul(p0.d, p0.z), dmul(p1.d, p1.z)), dmul(p2.d, p2.z)),
                           dmul(sd, dadd(dadd(p0.z, p1.z), p2.z)));
    acc[0] = dadd(acc[0], -dmul(m, sx));
    acc[1] = dadd(acc[1], -dmul(m, sy));
    acc[2] = dadd(acc[2], -dmul(m, sz));
    acc[3] = dadd(acc[3], -ddiv(dsub(dmul(gy, sz), dmul(gz, sy)), 12.0));
    acc[4] = dadd(acc[4], -ddiv(dsub(dmul(gz, sx), dmul(gx, sz)), 12.0));
    acc[5] = dadd(acc[5], -ddiv(dsub(dmul(gx, sy), dmul(gy, sx)), 12.0));
    acc[6] = dadd(acc[6], dsqrt(dadd(dadd(dmul(sx, sx), dmul(sy, sy)), dmul(sz, sz))));
}

// One triangle (v0, v1, v2) = (arm, depth) of its vertices, clipped at depth 0 and added to acc.  The vertices are
// rotated cyclically (keeping the winding) so that the one vertex on its own side of the waterline comes first, a:
//   one wet vertex a:  (a, X_ab, X_ac);
//   two wet b, c:      the quad (X_ba, b, c, X_ca), split along the diagonal b - X_ca: (X_ba, b, X_ca), (b, c, X_ca);
//   all wet:           (v0, v1, v2).  No wet vertex: nothing.
WSO_HD void hydro_triangle(float4 v0, float4 v1, float4 v2, double* acc) {
    const bool w0 = v0.w > 0.0f, w1 = v1.w > 0.0f, w2 = v2.w > 0.0f;
    const int nw = (int)w0 + (int)w1 + (int)w2;
    if (nw == 0) return;
    const HydroPoint p0 = hydro_point(v0), p1 = hydro_point(v1), p2 = hydro_point(v2);
    if (nw == 3) {
        hydro_sub(p0, p1, p2, acc);
        return;
    }
    // a: the vertex whose wetness differs from the other two
    const bool lone_wet = nw == 1;
    const int ia = (w0 == lone_wet) ? 0 : (w1 == lone_wet) ? 1 : 2;
    const HydroPoint a = ia == 0 ? p0 : ia == 1 ? p1 : p2;
    const HydroPoint b = ia == 0 ? p1 : ia == 1 ? p2 : p0;
    const HydroPoint c = ia == 0 ? p2 : ia == 1 ? p0 : p1;
    if (lone_wet) {
        hydro_sub(a, hydro_cross(a, b), hydro_cross(a, c), acc);
    } else {
        const HydroPoint xba = hydro_cross(b, a), xca = hydro_cross(c, a);
        hydro_sub(xba, b, xca, acc);
        hydro_sub(b, c, xca, acc);
    }
}

WSO_HD void hydro_combine(double* a, const double* b) {
    for (int k = 0; k < kHydroSums; ++k) a[k] = dadd(a[k], b[k]);
}

// The record: force = fl32(k * sum F'), wetted area = fl32(sum |S|), torque = fl32(k * sum tau') (about c_w, world axes).
WSO_HD void hydro_record(double k, const double* sum, uint32_t status, float4* o) {
    o[0] = make_float4((float)dmul(k, sum[0]), (float)dmul(k, sum[1]), (float)dmul(k, sum[2]), (float)sum[6]);
    o[1] = make_float4((float)dmul(k, sum[3]), (float)dmul(k, sum[4]), (float)dmul(k, sum[5]), bits_to_float(status));
}

WSO_HD void hydro_invalid(float4* o) {
    const float nan = bits_to_float(0x7fc00000u);
    o[0] = make_float4(nan, nan, nan, nan);
    o[1] = make_float4(nan, nan, nan, bits_to_float(kHydroInvalid));
}

WSO_HD uint32_t hydro_status(bool any_wet, bool any_dry) {
    return !any_wet ? kHydroDry : any_dry ? kHydroPartial : kHydroSubmerged;
}

#if !defined(__CUDA_ARCH__)
// Host build of one body: the kernel's 256 lanes run one after the other, each over the same vertices and triangles
// and in the same order, then the same pairwise tree.  sv: kMaxHullVertices float4s of scratch.
template <class Texel, int NS>
void hydro_body_host(const HydroArgs& a, uint32_t body, float4* sv, float4* o) {
    const HydroBody& b = a.bodies[body];
    if (!hydro_ranges_ok(a, b)) {
        hydro_invalid(o);
        return;
    }
    const HydroPose p = hydro_pose(b);
    bool bad = !p.ok, wet = false, dry = false;
    for (uint32_t t = 0; t < kHydroLanes; ++t) {
        for (uint32_t v = t; v < b.vertex_count; v += kHydroLanes) {
            bool ok;
            const float4 w = hydro_vertex<Texel, NS>(a.q, p, a.vertices[b.vertex_first + v], ok);
            bad = bad || !ok;
            wet = wet || w.w > 0.0f;
            dry = dry || !(w.w > 0.0f);
            sv[v] = w;
        }
    }
    if (bad) {
        hydro_invalid(o);
        return;
    }
    static thread_local double lanes[kHydroLanes][kHydroSums];
    bool bad_index = false;
    for (uint32_t t = 0; t < kHydroLanes; ++t) {
        double* acc = lanes[t];
        for (int k = 0; k < kHydroSums; ++k) acc[k] = 0.0;
        for (uint32_t i = t; i < b.triangle_count; i += kHydroLanes) {
            const uint32_t* tri = a.triangles + 3 * ((size_t)b.triangle_first + i);
            const uint32_t i0 = tri[0], i1 = tri[1], i2 = tri[2];
            if (i0 >= b.vertex_count || i1 >= b.vertex_count || i2 >= b.vertex_count) {
                bad_index = true;
                continue;
            }
            hydro_triangle(sv[i0], sv[i1], sv[i2], acc);
        }
    }
    if (bad_index) {
        hydro_invalid(o);
        return;
    }
    for (uint32_t stride = kHydroLanes / 2; stride >= 1; stride /= 2)
        for (uint32_t t = 0; t < stride; ++t) hydro_combine(lanes[t], lanes[t + stride]);
    hydro_record(a.k, lanes[0], hydro_status(wet, dry), o);
}
#endif

}  // namespace wso
