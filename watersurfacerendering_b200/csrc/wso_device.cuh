// wso_device.cuh — building blocks shared by the sm_100a kernels.
//
// Everything here is written as plain "per-thread body" code behind two tiny executor types
// (DeviceExec / HostExec) so that the SAME kernel bodies can also be compiled by g++ and stepped
// thread-by-thread on the CPU by tests/emu (index/layout debugging without a GPU).  The host build
// is test infrastructure only; the product library contains the CUDA build exclusively.
#pragma once

#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#define WSO_HD __host__ __device__ __forceinline__
#else
#include <cmath>
#define WSO_HD inline
struct float2 {
    float x, y;
};
struct alignas(16) float4 {
    float x, y, z, w;
};
static inline float2 make_float2(float x, float y) { return float2{x, y}; }
static inline float4 make_float4(float x, float y, float z, float w) { return float4{x, y, z, w}; }
#endif

namespace wso {

// ---------------------------------------------------------------------------------------------
// fp32 helpers.  wso_mul/add/sub are NEVER contracted into FMAs: the spectrum-evolve step mirrors
// the reference's x86 (non-FMA) rounding order (reference: WSTessendorf.h:265-275, cpp:303-336).
// ---------------------------------------------------------------------------------------------
#if defined(__CUDA_ARCH__)
WSO_HD float rmul(float a, float b) { return __fmul_rn(a, b); }
WSO_HD float radd(float a, float b) { return __fadd_rn(a, b); }
WSO_HD float rsub(float a, float b) { return __fsub_rn(a, b); }
WSO_HD float rdiv(float a, float b) { return __fdiv_rn(a, b); }
WSO_HD float rsqrt_ieee(float a) { return __fdiv_rn(1.0f, __fsqrt_rn(a)); }
WSO_HD float sqrt_ieee(float a) { return __fsqrt_rn(a); }
WSO_HD void sincos_acc(float x, float* s, float* c) { sincosf(x, s, c); }
#else
WSO_HD float rmul(float a, float b) { return a * b; }
WSO_HD float radd(float a, float b) { return a + b; }
WSO_HD float rsub(float a, float b) { return a - b; }
WSO_HD float rdiv(float a, float b) { return a / b; }
WSO_HD float rsqrt_ieee(float a) { return 1.0f / std::sqrt(a); }
WSO_HD float sqrt_ieee(float a) { return std::sqrt(a); }
WSO_HD void sincos_acc(float x, float* s, float* c) {
    *s = std::sin(x);
    *c = std::cos(x);
}
#endif

// Complex arithmetic on float2.  sm_100a has packed-fp32 instructions (FADD2 / FMUL2 / FFMA2: add|mul|fma.rn.f32x2 on a
// 64-bit register pair, each half an IEEE round-to-nearest operation) whose source operands take a half swap, a
// per-half negation and a scalar broadcast for free.  A complex add is ONE instruction, "a + i*b" is ONE instruction,
// a complex multiply is TWO (a.x*w + a.y*(i*w)) - half the issue slots of the scalar forms.  The transform stages are
// add/multiply dominated and the kernels are instruction-issue bound, not FP-pipe bound (DESIGN.md §6).
// The operand order inside cmul (swapped operand first) is the one ptxas folds into operand modifiers.
#if defined(__CUDA_ARCH__) && !defined(WSO_NO_F32X2)
WSO_HD float2 cadd(float2 a, float2 b) { return __fadd2_rn(a, b); }
WSO_HD float2 csub(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
WSO_HD float2 cadd_i(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.y, b.x)); }  // a + i*b
WSO_HD float2 csub_i(float2 a, float2 b) { return __fadd2_rn(a, make_float2(b.y, -b.x)); }  // a - i*b
WSO_HD float2 cadd_conj(float2 a, float2 b) { return __fadd2_rn(a, make_float2(b.x, -b.y)); }  // a + conj(b)
WSO_HD float2 csub_conj(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, b.y)); }  // a - conj(b)
WSO_HD float2 cscale(float s, float2 a) { return __fmul2_rn(a, make_float2(s, s)); }
WSO_HD float2 cmul(float2 a, float2 b) {
    return __ffma2_rn(make_float2(a.x, a.x), b, __fmul2_rn(make_float2(-b.y, b.x), make_float2(a.y, a.y)));
}
#else
WSO_HD float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
WSO_HD float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
WSO_HD float2 cadd_i(float2 a, float2 b) { return make_float2(a.x - b.y, a.y + b.x); }
WSO_HD float2 csub_i(float2 a, float2 b) { return make_float2(a.x + b.y, a.y - b.x); }
WSO_HD float2 cadd_conj(float2 a, float2 b) { return make_float2(a.x + b.x, a.y - b.y); }
WSO_HD float2 csub_conj(float2 a, float2 b) { return make_float2(a.x - b.x, a.y + b.y); }
WSO_HD float2 cscale(float s, float2 a) { return make_float2(s * a.x, s * a.y); }
WSO_HD float2 cmul(float2 a, float2 b) {
    return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
#endif
WSO_HD float2 cconj(float2 a) { return make_float2(a.x, -a.y); }

// Cache policy of the two big streams (measured with `ncu --cache-control none`, profiles/r1n_traffic.md and
// r1o_traffic.md: with plain stores the 32 B/pt of map output pushed 60 % of the intermediate W out of the 126 MB L2
// before K2 re-read it; with evict-first map stores 32 %).
//   st_stream: the output maps are written once and not read again by this library -> evict-first (st.global.cs)
//   ld_last  : K2 is the last reader of W -> the line may go as soon as it has been read (ld.global.lu); +3 % at 1024^2
#if defined(__CUDA_ARCH__) && !defined(WSO_EXP_NO_STREAM_STORES)
WSO_HD void st_stream(float4* p, float4 v) { __stcs(p, v); }
#else
WSO_HD void st_stream(float4* p, float4 v) { *p = v; }
#endif

// ---------------------------------------------------------------------------------------------
// RGBA16F output texel (wso_set_map_format): (x, y, z, w) as four IEEE binary16 values, little-endian, tightly packed
// - 8 bytes, VK_FORMAT_R16G16B16A16_SFLOAT.  xy holds x in bits 0..15 and y in bits 16..31, zw likewise.
// Conversion: the fp32 value the RGBA32F path stores, rounded to nearest even (cvt.rn.f16x2.f32 on the device, one
// instruction per two channels).  As with any IEEE conversion, magnitudes >= 65520 become +-inf, values below 2^-24
// go to subnormals / signed zero, and NaN stays NaN.
// ---------------------------------------------------------------------------------------------
struct alignas(8) Half4 {
    uint32_t xy, zw;
};

#if !defined(__CUDA_ARCH__)
// Portable float -> binary16 bits, IEEE round to nearest even (the host build of the kernel bodies, tests/emu).
WSO_HD uint16_t f32_to_f16_rn(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    const uint32_t sign = (u >> 16) & 0x8000u;
    const uint32_t a = u & 0x7fffffffu;
    if (a > 0x7f800000u) return (uint16_t)(sign | 0x7e00u | ((a >> 13) & 0x3ffu));  // NaN (quiet)
    if (a >= 0x47800000u) return (uint16_t)(sign | 0x7c00u);                         // >= 2^16 and inf
    if (a >= 0x38800000u) {
        // normal binary16 range (>= 2^-14): rebias the exponent by 127 - 15, round the 13 dropped mantissa bits to
        // nearest even; a carry out of the mantissa steps the exponent (65520 and up -> 0x7c00 = inf)
        return (uint16_t)(sign | ((a - 0x38000000u + 0xfffu + ((a >> 13) & 1u)) >> 13));
    }
    const uint32_t e = a >> 23;
    if (e < 102u) return (uint16_t)sign;  // below 2^-25: rounds to zero (2^-25 itself is the tie 0 | 2^-24 -> even 0)
    // subnormal binary16: the value in units of 2^-24 is mant * 2^(e - 126), 14 <= 126 - e <= 24
    const uint32_t mant = (a & 0x7fffffu) | 0x800000u;
    const uint32_t s = 126u - e;
    uint32_t r = mant >> s;
    const uint32_t rem = mant & ((1u << s) - 1u), half = 1u << (s - 1u);
    if (rem > half || (rem == half && (r & 1u))) ++r;  // may carry into the smallest normal, 0x0400: still right
    return (uint16_t)(sign | r);
}

// Portable binary16 bits -> float (exact: every binary16 value is a float), for the host build of the query body
// (wso_query.cuh) reading RGBA16F maps.
WSO_HD float f16_to_f32(uint16_t h) {
    const uint32_t sign = (uint32_t)(h & 0x8000u) << 16;
    const uint32_t e = (h >> 10) & 0x1fu, m = h & 0x3ffu;
    uint32_t u;
    if (e == 0x1fu) {
        u = sign | 0x7f800000u | (m << 13);  // inf, NaN (payload kept)
    } else if (e != 0u) {
        u = sign | ((e + 112u) << 23) | (m << 13);  // normal: rebias 15 -> 127
    } else if (m == 0u) {
        u = sign;  // signed zero
    } else {
        // subnormal m * 2^-24: shift the leading one up to bit 10, lowering the exponent of 2^-14 once per step
        uint32_t ex = 113u;
        uint32_t mm = m;
        while ((mm & 0x400u) == 0u) {
            mm <<= 1;
            --ex;
        }
        u = sign | (ex << 23) | ((mm & 0x3ffu) << 13);
    }
    float f;
    memcpy(&f, &u, 4);
    return f;
}
#endif

// binary16 bits of (lo, hi) in one 32-bit word, lo in bits 0..15
#if defined(__CUDA_ARCH__)
WSO_HD uint32_t half2_bits(float lo, float hi) {
    const __half2 h = __floats2half2_rn(lo, hi);  // cvt.rn.f16x2.f32
    uint32_t u;
    memcpy(&u, &h, 4);
    return u;
}
#else
WSO_HD uint32_t half2_bits(float lo, float hi) { return (uint32_t)f32_to_f16_rn(lo) | ((uint32_t)f32_to_f16_rn(hi) << 16); }
#endif

// one 8-byte evict-first store (st.global.cs.v2.b32): same cache policy as the RGBA32F maps
#if defined(__CUDA_ARCH__) && !defined(WSO_EXP_NO_STREAM_STORES)
WSO_HD void st_stream(Half4* p, Half4 v) {
    asm volatile("st.global.cs.v2.b32 [%0], {%1, %2};" ::"l"(p), "r"(v.xy), "r"(v.zw) : "memory");
}
#else
WSO_HD void st_stream(Half4* p, Half4 v) { *p = v; }
#endif

// Store one output texel in the map's format (the kernels compute fp32 either way).
WSO_HD void st_texel(float4* p, float x, float y, float z, float w) { st_stream(p, make_float4(x, y, z, w)); }
WSO_HD void st_texel(Half4* p, float x, float y, float z, float w) { st_stream(p, Half4{half2_bits(x, y), half2_bits(z, w)}); }
// ld_ro: spectrum records are read-only for the lifetime of a launch (experiment hook: the non-coherent path)
#if defined(__CUDA_ARCH__) && defined(WSO_EXP_LDG_RECORDS)
WSO_HD float4 ld_ro(const float4* p) { return __ldg(p); }
#else
WSO_HD float4 ld_ro(const float4* p) { return *p; }
#endif
#if defined(__CUDA_ARCH__) && !defined(WSO_EXP_NO_LAST_USE_LOADS)
WSO_HD float4 ld_last(const float4* p) { return __ldlu(p); }
WSO_HD float2 ld_last(const float2* p) { return __ldlu(p); }
#else
WSO_HD float4 ld_last(const float4* p) { return *p; }
WSO_HD float2 ld_last(const float2* p) { return *p; }
#endif

// st_keep: K1's stores of the intermediate W, which K2h / K2 read back within the same chunk.  Experiment hook
// (-DWSO_EXP_W_EVICT_LAST): an L2 evict-last cache hint on the store (createpolicy + st.global.L2::cache_hint).
#if defined(__CUDA_ARCH__) && defined(WSO_EXP_W_EVICT_LAST)
WSO_HD void st_keep(float4* p, float4 v) {
    asm volatile(
        "{\n\t.reg .b64 pol;\n\t"
        "createpolicy.fractional.L2::evict_last.b64 pol, 1.0;\n\t"
        "st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, pol;\n\t}"
        ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
        : "memory");
}
#else
WSO_HD void st_keep(float4* p, float4 v) { *p = v; }
#endif

// ---------------------------------------------------------------------------------------------
// Shared-memory line layout: logical element i of an FFT line lives at pad_idx(i).
// One float2 of padding per 16 elements makes every access pattern of the Stockham stages below
// (unit stride, stride R0 after the first stage, 16-element groups afterwards) bank-conflict free
// for 64-bit accesses (tools/bank_conflicts.py).
// ---------------------------------------------------------------------------------------------
WSO_HD int pad_idx(int i) { return i + (i >> 4); }
template <int N>
struct LineStride {
    // +4 keeps consecutive lines 4 (64-bit) banks apart: the pass-1 store phase reads the same
    // element of 4 adjacent lines in one request.
    static constexpr int value = N + (N >> 4) + 4;
};

// ---------------------------------------------------------------------------------------------
// Radix plans (Stockham autosort, decimation in time).  Product of radices == N.
// First radix <= 8 or 16 with second radix 16 keeps all smem traffic conflict free.
// ---------------------------------------------------------------------------------------------
template <int LOGN>
struct Plan;
template <> struct Plan<4>  { static constexpr int S = 1; static constexpr int R[4] = {16, 1, 1, 1}; };
template <> struct Plan<5>  { static constexpr int S = 2; static constexpr int R[4] = {2, 16, 1, 1}; };
template <> struct Plan<6>  { static constexpr int S = 2; static constexpr int R[4] = {4, 16, 1, 1}; };
template <> struct Plan<7>  { static constexpr int S = 2; static constexpr int R[4] = {8, 16, 1, 1}; };
template <> struct Plan<8>  { static constexpr int S = 2; static constexpr int R[4] = {16, 16, 1, 1}; };
template <> struct Plan<9>  { static constexpr int S = 3; static constexpr int R[4] = {2, 16, 16, 1}; };
template <> struct Plan<10> { static constexpr int S = 3; static constexpr int R[4] = {4, 16, 16, 1}; };
template <> struct Plan<11> { static constexpr int S = 3; static constexpr int R[4] = {8, 16, 16, 1}; };
template <> struct Plan<12> { static constexpr int S = 3; static constexpr int R[4] = {16, 16, 16, 1}; };
template <> struct Plan<13> { static constexpr int S = 4; static constexpr int R[4] = {2, 16, 16, 16}; };
template <> struct Plan<14> { static constexpr int S = 4; static constexpr int R[4] = {4, 16, 16, 16}; };

// ---------------------------------------------------------------------------------------------
// Small in-register DFTs, backward sign: X[k] = sum_n x[n] exp(+2*pi*i*n*k/R), natural order.
// ---------------------------------------------------------------------------------------------
// multiply by exp(+2*pi*i*E/16), E compile-time
template <int E>
WSO_HD float2 mul_w16(float2 a) {
    constexpr int e = E & 15;
    if (e == 0) return a;
    if (e == 4) return make_float2(-a.y, a.x);
    if (e == 8) return make_float2(-a.x, -a.y);
    if (e == 12) return make_float2(a.y, -a.x);
    constexpr float h = 0.70710678118654752440f;
    constexpr float c1 = 0.92387953251128675613f;  // cos(pi/8)
    constexpr float s1 = 0.38268343236508977173f;  // sin(pi/8)
    // (cos, sin) of e*pi/8
    constexpr float wc = (e == 1) ? c1 : (e == 2) ? h : (e == 3) ? s1 : (e == 5) ? -s1 : (e == 6) ? -h : (e == 7) ? -c1
                       : (e == 9) ? -c1 : (e == 10) ? -h : (e == 11) ? -s1 : (e == 13) ? s1 : (e == 14) ? h : c1;
    constexpr float ws = (e == 1) ? s1 : (e == 2) ? h : (e == 3) ? c1 : (e == 5) ? c1 : (e == 6) ? h : (e == 7) ? s1
                       : (e == 9) ? -s1 : (e == 10) ? -h : (e == 11) ? -c1 : (e == 13) ? -c1 : (e == 14) ? -h : -s1;
    return cmul(a, make_float2(wc, ws));
}

WSO_HD void dft2(float2& a, float2& b) {
    const float2 t = a;
    a = cadd(t, b);
    b = csub(t, b);
}
// in-place on 4 named values, natural order out
WSO_HD void dft4(float2& x0, float2& x1, float2& x2, float2& x3) {
    const float2 s0 = cadd(x0, x2), d0 = csub(x0, x2);
    const float2 s1 = cadd(x1, x3), d1 = csub(x1, x3);
    x0 = cadd(s0, s1);
    x1 = cadd_i(d0, d1);
    x2 = csub(s0, s1);
    x3 = csub_i(d0, d1);
}

template <int R>
struct Dft;
template <> struct Dft<1> { static WSO_HD void run(float2*) {} };
template <> struct Dft<2> { static WSO_HD void run(float2* v) { dft2(v[0], v[1]); } };
template <> struct Dft<4> { static WSO_HD void run(float2* v) { dft4(v[0], v[1], v[2], v[3]); } };
template <> struct Dft<8> {
    static WSO_HD void run(float2* v) {
        // radix-2 x radix-4 (DIT): E = DFT4(even), O = DFT4(odd), X[k] = E[k] + w8^k O[k]
        dft4(v[0], v[2], v[4], v[6]);
        dft4(v[1], v[3], v[5], v[7]);
        const float2 o0 = v[1], o1 = mul_w16<2>(v[3]), o2 = mul_w16<4>(v[5]), o3 = mul_w16<6>(v[7]);
        const float2 e0 = v[0], e1 = v[2], e2 = v[4], e3 = v[6];
        v[0] = cadd(e0, o0); v[4] = csub(e0, o0);
        v[1] = cadd(e1, o1); v[5] = csub(e1, o1);
        v[2] = cadd(e2, o2); v[6] = csub(e2, o2);
        v[3] = cadd(e3, o3); v[7] = csub(e3, o3);
    }
};
template <> struct Dft<16> {
    static WSO_HD void run(float2* v) {
        // radix-4 x radix-4 (DIT): Y_a = DFT4 over b of x[a+4b]; X[k1+4k2] = DFT4 over a of w16^(a k1) Y_a[k1]
        dft4(v[0], v[4], v[8], v[12]);
        dft4(v[1], v[5], v[9], v[13]);
        dft4(v[2], v[6], v[10], v[14]);
        dft4(v[3], v[7], v[11], v[15]);
        // Y_a[k1] now sits in v[a + 4*k1]
        v[5] = mul_w16<1>(v[5]);   v[6] = mul_w16<2>(v[6]);    v[7] = mul_w16<3>(v[7]);
        v[9] = mul_w16<2>(v[9]);   v[10] = mul_w16<4>(v[10]);  v[11] = mul_w16<6>(v[11]);
        v[13] = mul_w16<3>(v[13]); v[14] = mul_w16<6>(v[14]);  v[15] = mul_w16<9>(v[15]);
        dft4(v[0], v[1], v[2], v[3]);      // k1 = 0 -> X[0], X[4], X[8], X[12]
        dft4(v[4], v[5], v[6], v[7]);      // k1 = 1 -> X[1], X[5], X[9], X[13]
        dft4(v[8], v[9], v[10], v[11]);    // k1 = 2
        dft4(v[12], v[13], v[14], v[15]);  // k1 = 3
        // v[4*k1 + k2] = X[k1 + 4*k2]  -> transpose the 4x4 to natural order
        float2 t;
        t = v[1];  v[1] = v[4];   v[4] = t;
        t = v[2];  v[2] = v[8];   v[8] = t;
        t = v[3];  v[3] = v[12];  v[12] = t;
        t = v[6];  v[6] = v[9];   v[9] = t;
        t = v[7];  v[7] = v[13];  v[13] = t;
        t = v[11]; v[11] = v[14]; v[14] = t;
    }
};

// ---------------------------------------------------------------------------------------------
// Executors.  each(f): run f(tid, state) for every thread of the CTA.  sync(): CTA barrier.
// ---------------------------------------------------------------------------------------------
static constexpr int kValsPerThread = 16;  // complex values a thread carries between barriers

// Twiddle preload (WSO_TW_PRELOAD, default on): the one table value w_{NS*R}^k a thread needs per radix-16 stage depends only on
// its thread index, so it is requested at the top of the kernel - together with the first global loads - and waits in
// two or three registers, instead of being requested between a stage's shared-memory loads and its first multiply
// (where its L1 / L2 round trip showed up as 4-6 % of the warp time of K1 / K2, profiles/r3_ab_persistent.md).
#ifndef WSO_TW_PRELOAD
#define WSO_TW_PRELOAD 1
#endif
static constexpr bool kTwPreload = WSO_TW_PRELOAD != 0;
static constexpr int kMaxStages = 4;

struct ThreadState {
    float2 v[kValsPerThread];
    float2 tw[kMaxStages];  // preloaded twiddle base of stage SI (radix-16 stages behind the first one)
    float pre[6];           // K1's fused front end: wave numbers requested together with the records (kz of its row pairs, kx of its column pair)
};

#if defined(__CUDACC__)
struct DeviceExec {
    ThreadState st;
    template <class F>
    __device__ __forceinline__ void each(F&& f) {
        f((int)threadIdx.x, st);
    }
    __device__ __forceinline__ void sync() { __syncthreads(); }

    // Programmatic dependent launch (the launches carry cudaLaunchAttributeProgrammaticStreamSerialization).
    // pdl_wait(): block until the preceding kernel of the stream has completed and its writes are visible.
    // pdl_release(): let the NEXT kernel of the stream start being scheduled.  Every kernel releases only after its
    // own wait, so when a kernel starts, everything up to its predecessor's predecessor is complete.
    __device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
    __device__ __forceinline__ void pdl_release() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

    // 16-byte asynchronous copy global -> shared (cp.async / LDGSTS): no destination registers, completion awaited by
    // the issuing thread with async_wait() before it - or, behind a barrier, anyone - reads the shared-memory copy.
    __device__ __forceinline__ void async_copy16(void* smem_dst, const void* gsrc) {
        const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
    }
    __device__ __forceinline__ void async_wait() { asm volatile("cp.async.wait_all;" ::: "memory"); }

    // Barrier over the G consecutive threads [g*G, (g+1)*G) that share one FFT line (or line pair), instead of
    // the whole CTA: lines are independent between the evolve / split / pack phases, so a CTA-wide barrier per
    // stage would only make 16 warps wait for the slowest one.  G <= 32: the group lives inside one warp;
    // otherwise a named barrier (ids 1..15; id 0 is __syncthreads).
    template <int G, int T>
    __device__ __forceinline__ void sync_group(int id_base) {
        if constexpr (G >= T) {
            __syncthreads();
        } else if constexpr (G <= 32) {
            __syncwarp();
        } else {
            static_assert(G % 32 == 0, "group must be whole warps");
            const int id = id_base + (int)threadIdx.x / G;
            asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(G) : "memory");
        }
    }

    // Producer / consumer barrier per column pair, behind K1's fused front end.  There the H2 threads [cp*H2, (cp+1)*H2) write
    // the first-stage output of the NF lines of column pair cp, and the next stage reads line l with the G threads [l*G, (l+1)*G)
    // (lines l = fl*CP + cp): every thread announces its writes on its producer column pair (bar.arrive) and waits on the
    // column pair of the line it reads next (bar.sync); a column pair whose four warps are done moves on while the others
    // still evolve, instead of all warps of the CTA meeting at __syncthreads().
    template <int CP, int NF, int H2, int G>
    __device__ __forceinline__ void sync_colpair(int id_base) {
        static_assert(H2 % 32 == 0 && G % 32 == 0, "whole warps on both sides");
        constexpr int COUNT = H2 + NF * G;  // arrivals + waiters per column pair
        const int idp = id_base + (int)threadIdx.x / H2;
        const int idc = id_base + ((int)threadIdx.x / G) % CP;
        asm volatile("bar.arrive %0, %1;" ::"r"(idp), "n"(COUNT) : "memory");
        asm volatile("bar.sync %0, %1;" ::"r"(idc), "n"(COUNT) : "memory");
    }

    // Fold the (min,max) every thread left in st.v[0] into out[0] (min) / out[1] (max): warp-shuffle butterfly,
    // one partial per warp through shared memory, then ONE pair of atomics per CTA (all CTAs of a tile-frame hit the
    // same two words, and same-address atomics serialise in one L2 slice).  Float ordering through the sign-aware
    // int/uint trick, valid for any mix of signs.
    __device__ __forceinline__ void commit_minmax(float* out) {
        __shared__ float2 partial[32];
        float mn = st.v[0].x, mx = st.v[0].y;
        const unsigned nthreads = blockDim.x;
        const bool full_warps = (nthreads & 31u) == 0u;
        if (full_warps) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
                mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
            }
            const unsigned nwarps = nthreads >> 5;
            if (nwarps > 1) {
                if ((threadIdx.x & 31u) == 0u) partial[threadIdx.x >> 5] = make_float2(mn, mx);
                __syncthreads();
                if (threadIdx.x >= 32u) return;
                const float2 p = partial[threadIdx.x < nwarps ? threadIdx.x : 0];
                mn = p.x;
                mx = p.y;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
                    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                }
            }
        }
        if (!full_warps || threadIdx.x == 0u) {
            if (mn >= 0.0f) atomicMin(reinterpret_cast<int*>(out), __float_as_int(mn));
            else atomicMax(reinterpret_cast<unsigned int*>(out), __float_as_uint(mn));
            if (mx >= 0.0f) atomicMax(reinterpret_cast<int*>(out + 1), __float_as_int(mx));
            else atomicMin(reinterpret_cast<unsigned int*>(out + 1), __float_as_uint(mx));
        }
    }
};
#endif

struct HostExec {
    int nthreads;
    ThreadState* states;  // [nthreads]
    template <class F>
    void each(F&& f) {
        for (int t = 0; t < nthreads; ++t) f(t, states[t]);
    }
    void sync() {}
    void pdl_wait() {}
    void pdl_release() {}
    void async_copy16(void* smem_dst, const void* gsrc) { memcpy(smem_dst, gsrc, 16); }
    void async_wait() {}
    template <int G, int T>
    void sync_group(int) {}
    template <int CP, int NF, int H2, int G>
    void sync_colpair(int) {}
    void commit_minmax(float* out) {
        for (int t = 0; t < nthreads; ++t) {
            if (states[t].v[0].x < out[0]) out[0] = states[t].v[0].x;
            if (states[t].v[0].y > out[1]) out[1] = states[t].v[0].y;
        }
    }
};

// ---------------------------------------------------------------------------------------------
// One Stockham stage over B lines of length N held in shared memory (in place: all loads, barrier,
// butterflies + stores, barrier).  CTA size T = B*N/16; every thread carries 16 values; the N/16 threads
// [line*G, (line+1)*G) own one line, so the barriers are per line (sync_group).
//   radix R, NS = product of the radices of the earlier stages.
//   load : v[r] = x[j + r*N/R]                         (unit stride across threads)
//   twid : v[r] *= w_{NS*R}^{(j % NS) * r}
//   store: y[(j/NS)*NS*R + (j%NS) + r*NS] = DFT_R(v)[r]
// ---------------------------------------------------------------------------------------------
template <int N, int B, int R, int NS>
struct Stage {
    static constexpr int T = B * N / kValsPerThread;
    static constexpr int G = N / kValsPerThread;   // threads that share one line: tid/G = line, tid%G = lane in line
    static constexpr int NB = kValsPerThread / R;  // butterflies per thread: j = tid%G + G*i
    static constexpr int LS = LineStride<N>::value;
    static constexpr int JN = N / R;               // butterflies per line

    // All shared-memory offsets below are (per-thread base) + (compile-time constant): with JN and NS*R
    // multiples of 16 (or NS < 16 dividing 16) the padding term of element base + r*stride is
    // pad(base) + r*stride + ((r*stride) >> 4).
    static constexpr int kLoadStep = JN + (JN >> 4);   // pad_idx(j + r*JN) - pad_idx(j + (r-1)*JN), JN % 16 == 0
    static constexpr bool kLoadConst = (JN % 16) == 0;

    static WSO_HD void load(const float2* smem, int tid, ThreadState& st) {
#pragma unroll
        for (int i = 0; i < NB; ++i) {
            const int line = tid / G;
            const int j = tid % G + G * i;
            const float2* x = smem + line * LS;
            if (kLoadConst) {
                const float2* xb = x + pad_idx(j);
#pragma unroll
                for (int r = 0; r < R; ++r) st.v[i * R + r] = xb[r * kLoadStep];
            } else {
#pragma unroll
                for (int r = 0; r < R; ++r) st.v[i * R + r] = x[pad_idx(j + r * JN)];
            }
        }
    }

    // Twiddles w^r, r = 1..R-1, from ONE table load (w = w_{NS*R}^k) and a product tree of depth <= 4
    // (w^r = w^floor(r/2) * w^ceil(r/2)); fifteen scattered 8-byte loads per radix-16 butterfly would
    // otherwise dominate the load/store pipe.
    template <int RR>
    static WSO_HD void apply_powers(float2* v, float2 w1) {
        float2 w[RR > 1 ? RR : 2];
        w[1] = w1;
        v[1] = cmul(v[1], w1);
#pragma unroll
        for (int r = 2; r < RR; ++r) {
            w[r] = cmul(w[r >> 1], w[(r + 1) >> 1]);
            v[r] = cmul(v[r], w[r]);
        }
    }

    static WSO_HD void twiddle_dft(const float2* __restrict__ tw, int tid, ThreadState& st) {
#pragma unroll
        for (int i = 0; i < NB; ++i) {
            if (NS > 1) {
                const int j = tid % G + G * i;
                const int k = j % NS;
                constexpr int tstep = N / (NS * R);
                apply_powers<R>(&st.v[i * R], tw[tstep * k]);
            }
            Dft<R>::run(&st.v[i * R]);
        }
    }
    // one butterfly per thread (R == 16) and a preloaded table value
    static constexpr bool kCanPreload = (NB == 1) && (NS > 1);
    static WSO_HD float2 twiddle_of(const float2* __restrict__ tw, int tid) {
        constexpr int tstep = N / (NS * R);
        return tw[tstep * ((tid % G) % NS)];
    }
    static WSO_HD void twiddle_dft_pre(float2 w1, ThreadState& st) {
        apply_powers<R>(&st.v[0], w1);
        Dft<R>::run(&st.v[0]);
    }

    // store offsets: element base + r*NS with base = (j/NS)*NS*R + k, k < NS.
    //   NS % 16 == 0 : pad(base + r*NS) = pad(base) + r*(NS + NS/16)
    //   NS < 16      : base % 16 == k when NS*R % 16 == 0 (or base % R == 0 with R | 16 when NS == 1), so
    //                  pad(base + r*NS) = pad(base) + r*NS + ((r*NS) >> 4)
    static constexpr bool kStoreConst =
        (NS % 16 == 0) || ((NS * R) % 16 == 0 && 16 % NS == 0) || (NS == 1 && 16 % R == 0);
    static WSO_HD constexpr int store_off(int r) {
        return (NS % 16 == 0) ? r * (NS + (NS >> 4)) : r * NS + ((r * NS) >> 4);
    }

    static WSO_HD void store(float2* smem, int tid, const ThreadState& st) {
#pragma unroll
        for (int i = 0; i < NB; ++i) {
            const int line = tid / G;
            const int j = tid % G + G * i;
            const int k = j % NS;
            const int base = (j / NS) * NS * R + k;
            float2* y = smem + line * LS;
            if (kStoreConst) {
                float2* yb = y + pad_idx(base);
#pragma unroll
                for (int r = 0; r < R; ++r) yb[store_off(r)] = st.v[i * R + r];
            } else {
#pragma unroll
                for (int r = 0; r < R; ++r) y[pad_idx(base + r * NS)] = st.v[i * R + r];
            }
        }
    }
};

// Runs stages FIRST..S-1 of Plan<LOGN> on data already in smem (natural order in, natural order out).
// KEEP_LAST: the outputs of the last stage stay in the registers of the thread that computed them (st.v[i*R + r] =
// X[(tid%G + G*i) + r*N/R] of line tid/G) instead of going back to shared memory - for consumers that only reduce them.
template <int LOGN, int B, int SI, int NS, class Exec, bool KEEP_LAST = false>
struct RunStages {
    static WSO_HD void run(Exec& ex, float2* smem, const float2* __restrict__ tw) {
        constexpr int N = 1 << LOGN;
        constexpr int R = Plan<LOGN>::R[SI];
        constexpr bool kKeep = KEEP_LAST && (SI + 1 == Plan<LOGN>::S);
        using St = Stage<N, B, R, NS>;
        // only the threads of one line have to agree on that line's loads and stores
        ex.each([&](int tid, ThreadState& st) { St::load(smem, tid, st); });
        ex.template sync_group<St::G, St::T>(1);
        ex.each([&](int tid, ThreadState& st) {
            if constexpr (kTwPreload && St::kCanPreload) St::twiddle_dft_pre(st.tw[SI], st);
            else St::twiddle_dft(tw, tid, st);
            if (!kKeep) St::store(smem, tid, st);
        });
        if (!kKeep) ex.template sync_group<St::G, St::T>(1);
        if constexpr (SI + 1 < Plan<LOGN>::S) RunStages<LOGN, B, SI + 1, NS * R, Exec, KEEP_LAST>::run(ex, smem, tw);
    }
    // Requests the table values run() will use (stages SI..S-1); call it early, next to the kernel's first global loads.
    static WSO_HD void preload(Exec& ex, const float2* __restrict__ tw) {
        if constexpr (kTwPreload) {
            constexpr int N = 1 << LOGN;
            constexpr int R = Plan<LOGN>::R[SI];
            using St = Stage<N, B, R, NS>;
            if constexpr (St::kCanPreload) ex.each([&](int tid, ThreadState& st) { st.tw[SI] = St::twiddle_of(tw, tid); });
            if constexpr (SI + 1 < Plan<LOGN>::S) RunStages<LOGN, B, SI + 1, NS * R, Exec, KEEP_LAST>::preload(ex, tw);
        }
    }
};

}  // namespace wso
