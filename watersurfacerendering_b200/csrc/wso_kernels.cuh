// wso_kernels.cuh — CTA bodies of the three hot-path kernels (see DESIGN.md §3 for the derivation).
//
//   K1  Pass1  : spectrum evolve h0 -> h~(k,t) -> 4 real packed spectra Z_f, fused with the first 1-D
//                transform (along m, two real columns per complex FFT) -> Hermitian half W[m'][f][slot]
//   K2  Pass2  : second 1-D transform (along n) fused with sign fix, lambda and packing into the
//                RGBA32F (or, opt-in, RGBA16F) displacement / normal maps + height min/max
//   K3  Normalize : disp.y *= 1/A,  A = max(|min|,|max|)       (reference: WSTessendorf.cpp:443-455)
//
// Replaces reference WSTessendorf::ComputeWaves (src/scene/WSTessendorf.cpp:284-441) including the
// seven fftwf_execute calls (cpp:338-378).
#pragma once

#include <cstring>
#include <type_traits>

#include "wso_device.cuh"

namespace wso {

static constexpr int kMaxChunk = 64;   // batch items (tile-frames) per kernel launch
static constexpr int kMaxTable = 1024;  // entries of the per-frame sincos table kept in shared memory

// Per-tile constants, device pointers (written once per Prepare()).
struct TileDev {
    // [jl][half][m] one 16-byte record per wave vector (m,n), grouped by column PAIR: local pair jl = j - j0,
    // half 0 = column n = j, half 1 = its mirror column n = N-j (n = N/2 for j = 0); m runs contiguously:
    //   x,y = heightAmp re,im (reference h0 record)          z = 1/|k| (0 where |k| <= 1e-5: WSTessendorf.h:135)
    //   w   = quantised dispersion omega (WSTessendorf.h:284-287), or - when table_len > 0 - its integer
    //         multiple j of the base frequency (omega == fl(float(j)*omega0) exactly, checked at Prepare)
    const float4* h0;
    // [jl][half][i] (hs_index) for column pair j = j0 + jl = (j, N-j) and row pair i = (i, N-i), i in [0, N/2): the same
    // record with the amplitude replaced by the sum over the mirror pair, h0(k) + h0(-k):
    //   half 0: k = (m=i, n=j)     half 1: k = (m=i, n=N-j)
    // Only Re FFT is kept, so away from the index-0 / N/2 lines every field depends on h~ only through
    // h~(k) + h~(-k) (same omega for k and -k): one record and one (cos,sin) lookup serve two wave vectors.
    const float4* hs;
    const float* kv;     // [N]: kv[i] = (float)(M_PI*(2.0f*i-N)/L)  (reference: WSTessendorf.cpp:75-80)
    float lambda;        // displacement scale (reference: WSTessendorf.h:181)
    float omega0;        // base frequency (float)(2*pi/T)
    int table_len;       // j_max+1 when the per-frame sincos table is usable, else 0
    int use_pairs;       // 1 when omega(k) == omega(-k) everywhere (always true for Prepare()-built h0): hs is valid
    int j0;              // first column pair held by this device (0 unless the grid is slab-decomposed, DESIGN.md §7)
};

// Position of wave vector (m, n) in TileDev::h0 for a device whose first column pair is j0.
WSO_HD size_t h0_index(int n, int m, int N, int j0) {
    const int H = N >> 1;
    const int j = (n < H) ? n : ((n == H) ? 0 : N - n);
    const int half = (n < H) ? 0 : 1;
    return ((size_t)(j - j0) * 2 + half) * N + m;
}

// Position of the pair-summed record (row pair i, column pair jl, half) in TileDev::hs.  The two halves of a column pair
// are separate planes [jl][half][i]: the threads of a warp walk i, so each 16-byte load of a warp is one contiguous
// 512-byte run (4 cache lines).  Interleaved as [jl][i][2] every load touched 8 lines for the same bytes - 8 of K1's 18
// global load instructions, a sixth of its L1 wavefronts (profiles/r3_hs_layout.md); -DWSO_EXP_HS_AOS restores that.
WSO_HD size_t hs_index(int jl, int i, int half, int H) {
#ifdef WSO_EXP_HS_AOS
    return ((size_t)jl * H + i) * 2 + half;
#else
    return ((size_t)jl * 2 + half) * H + i;
#endif
}

struct BatchItem {
    uint32_t tile;  // which h0 / parameter set (host bookkeeping; the kernels read td[] below)
    uint32_t slot;  // which output map slot
    float t;        // time
};

// CAP: item capacity of the parameter block.  Batched launches use kMaxChunk; a launch of a few tile-frames uses
// a small block (kernel parameters are copied into the command stream at every launch).
template <int CAP>
struct LaunchArgsT {
    static constexpr int kCap = CAP;
    const float2* tw;      // [N] exp(+2*pi*i*k/N)
    float2* W;             // chunk scratch: [item][N/2][4][N]
    float4* disp;          // [slot][N*N]  (RGBA16F maps: the K2 instantiations with TEX = Half4 read it as Half4*)
    float4* norm;          // [slot][N*N]
    float* minmax;         // [slot][2]
    float* amp_out;        // [slot] amplitude A
    // Slab decomposition of ONE grid over P = 2^slab_shift devices (DESIGN.md §7): this device runs K1 on the column
    // pairs [rank*Hl, (rank+1)*Hl), Hl = N/2/P, and K2h/K2 on the row items m' of the same range.  K1 writes the block
    // [ml][f][half][jl] destined for the owner d of row item m' = d*Hl + ml through Wdst[d] (the owner's receive
    // buffer over NVLink peer memory, or the local send buffer of an all-to-all); K2h/K2 read W = [src][ml][f][half][jl].
    int slab_shift;
    int slab_rank;
    float2* Wdst[8];
    // Slab K1, staged store (NULL: store through Wdst in the exchange layout right away).  K1 writes what it separates
    // where consecutive threads hold consecutive m': stage[f][half][jl][m'], m' over the WHOLE half spectrum - contiguous
    // 8-byte stores - and the transposing exchange kernel (wso_slab_kernels.cu) carries the Hl x Hl blocks to their
    // owners in 256-byte rows.  (The direct layout costs one 32-byte sector per 8 useful bytes when a line is so long
    // that a CTA holds a single column pair, DESIGN.md 7.)
    float2* slab_stage;
    int slab_field0;  // slab K1 launched field group by field group (exchange pipelined behind it): first field group
    BatchItem items[CAP];
    // the tile constants of every item travel by value in the kernel parameters (constant bank): no dependent
    // global load sits between CTA start and the first h0 request
    TileDev td[CAP];
};
using LaunchArgs = LaunchArgsT<kMaxChunk>;
static constexpr int kSmallChunk = 4;
using LaunchArgsSmall = LaunchArgsT<kSmallChunk>;

// Layout of the intermediate W of one tile-frame (not slab-decomposed), complex [m'][f][N]:
//   paired  : element 2*j + half  - the two columns (n = j, n = N-j) that K1 separates out of one complex transform
//             sit next to each other: K1 stores them as ONE 16-byte word, and K2/K2h fetch both inputs of a
//             first-stage butterfly pair (u, JN0-u) with one 16-byte load
//   legacy  : element half*N/2 + j (two 8-byte stores N/2 apart; sizes whose first radix is 16 keep it, their K2
//             threads own a single first-stage butterfly)
// half 0: column n = j; half 1: n = N-j (n = N/2 for j = 0).
template <int LOGN>
struct WLayout {
#ifdef WSO_EXP_LEGACY_W
    static constexpr bool paired = false;
#else
    static constexpr bool paired = Plan<LOGN>::S > 1 && Plan<LOGN>::R[0] <= 8;
#endif
};

// reference: WSTessendorf.cpp:289-290 — max starts at FLT_MIN (smallest positive), min at FLT_MAX
static constexpr float kInitMax = 1.17549435e-38f;
static constexpr float kInitMin = 3.402823466e+38f;

struct Point {
    float H, kx, kz, ux, uz;
};

// compile-time loop: f(std::integral_constant<int, I>) for I = 0..N-1 (register arrays need constant indices)
template <int I>
struct IntC {
    static constexpr int value = I;
};
template <int I, int N, class F>
WSO_HD void static_for(F&& f) {
    if constexpr (I < N) {
        f(IntC<I>{});
        static_for<I + 1, N>(f);
    }
}

// h~(k,t) for the wave vector whose 16-byte record is q.
// reference: WaveHeightFT, WSTessendorf.h:265-275 with heightAmp_conj == conj(heightAmp) (validated at
// import): h~ = 2*(a*cos(wt) - b*sin(wt)), imaginary part exactly 0.
// The phase w*t is the same single fp32 product as the reference's; with TABLE the (cos,sin) pair comes
// from the per-frame table over j (bit-identical: the table entry is sincosf(fl(fl(j*omega0)*t))).
template <bool TABLE>
WSO_HD float eval_height(const float4 q, const float2* table, float t) {
    float s, c;
    if (TABLE) {
#if defined(__CUDA_ARCH__)
        const float2 cs = table[__float_as_int(q.w)];
#else
        int j;
        std::memcpy(&j, &q.w, 4);
        const float2 cs = table[j];
#endif
        c = cs.x;
        s = cs.y;
    } else {
        sincos_acc(rmul(q.w, t), &s, &c);
    }
    const float x = rsub(rmul(q.x, c), rmul(q.y, s));
    return radd(x, x);
}

// Even-type (real spectrum) and odd-type (imaginary spectrum i*V) member of packed field F.
//   F=0: (height, Dx)   F=1: (none, Dz)   F=2: (dxDx, slopeX)   F=3: (dzDz, slopeZ)
// reference: WSTessendorf.cpp:303-336 (same products in the same order).  ux,uz: WSTessendorf.h:133-136.
// JAC (SURVEY row f-4, reference COMPUTE_JACOBIAN: WSTessendorf.cpp:330-335): the otherwise empty real slot of packed
// field 1 carries dzDx = i*kz * Dx = kz*ux*h~ (a real spectrum; dxDz = i*kx * Dz = kx*uz*h~ is the same field).
template <int F, bool JAC = false>
WSO_HD void field_values(const Point& p, float* R, float* V) {
    if (F == 0) { *R = p.H;                              *V = rmul(-p.ux, p.H); }
    if (F == 1) { *R = JAC ? rmul(p.kz, rmul(p.ux, p.H)) : 0.0f;  *V = rmul(-p.uz, p.H); }
    if (F == 2) { *R = rmul(p.kx, rmul(p.ux, p.H));      *V = rmul(p.kx, p.H); }
    if (F == 3) { *R = rmul(p.kz, rmul(p.uz, p.H));      *V = rmul(p.kz, p.H); }
}

// GENERAL packing (any mirror pattern): Z = even(R) - odd(V) under DFT-index reflection, for the 4 points
// q = 2*a + b, a = row (mA,mB), b = column (nA,nB).  MASK bit1: the rows mirror into each other (i >= 1);
// bit0: the columns do (j >= 1).  Used on the index-0 (Nyquist) and N/2 (DC) lines, where the mirror of
// a point keeps one of its wave numbers; everywhere else pack_interior applies.
template <int F, bool JAC = false>
WSO_HD void pack_general(const Point (&pt)[4], int mask, float2* outA, float2* outB) {
    float R[4], V[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) field_values<F, JAC>(pt[q], &R[q], &V[q]);
    float z[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        // mirror partner q ^ mask, selected without dynamic register indexing
        const float Rm = (mask == 3) ? R[q ^ 3] : (mask == 2) ? R[q ^ 2] : (mask == 1) ? R[q ^ 1] : R[q];
        const float Vm = (mask == 3) ? V[q ^ 3] : (mask == 2) ? V[q ^ 2] : (mask == 1) ? V[q ^ 1] : V[q];
        z[q] = 0.5f * (R[q] + Rm) - 0.5f * (V[q] - Vm);
    }
    *outA = make_float2(z[0], z[1]);  // complex sample of row mA: Z(mA,nA) + i Z(mA,nB)
    *outB = make_float2(z[2], z[3]);
}

// INTERIOR packing (i >= 1 and j >= 1): the mirror of (m,n) is (N-m,N-n) with BOTH wave numbers negated, so
// every packed field depends on h~ only through S = h~(k) + h~(-k):
//   F0: Z(k) = S/2 * (1 + ux)      F1: Z(k) = S/2 * uz      F2: Z(k) = S/2 * kx*(ux - 1)     F3: same with z
// and Z(-k) follows by ux -> -ux, kx -> -kx.  s0 = S(mA,nA)/2, s1 = S(mA,nB)/2; (kx,kz,inv) of those two points.
template <int F, bool JAC = false>
WSO_HD void pack_interior(float s0, float kx0, float kz0, float inv0, float s1, float kx1, float kz1, float inv1,
                          float2* outA, float2* outB) {
    float z0, z1, z2, z3;
    if (F == 0) {
        const float a = kx0 * inv0 * s0, b = kx1 * inv1 * s1;
        z0 = s0 + a; z3 = s0 - a; z1 = s1 + b; z2 = s1 - b;
    } else if (F == 1 && JAC) {
        // Z(k) = S/2 * (kz*ux + uz); the even part kz*ux keeps its sign under k -> -k, uz flips
        const float a0 = kz0 * inv0 * s0, a1 = kz1 * inv1 * s1;
        const float r0 = kz0 * (kx0 * inv0) * s0, r1 = kz1 * (kx1 * inv1) * s1;
        z0 = r0 + a0; z3 = r0 - a0; z1 = r1 + a1; z2 = r1 - a1;
    } else if (F == 1) {
        z0 = kz0 * inv0 * s0; z3 = -z0; z1 = kz1 * inv1 * s1; z2 = -z1;
    } else if (F == 2) {
        const float g0 = kx0 * s0, g1 = kx1 * s1;
        const float a = kx0 * inv0 * g0, b = kx1 * inv1 * g1;
        z0 = a - g0; z3 = a + g0; z1 = b - g1; z2 = b + g1;
    } else {
        const float g0 = kz0 * s0, g1 = kz1 * s1;
        const float a = kz0 * inv0 * g0, b = kz1 * inv1 * g1;
        z0 = a - g0; z3 = a + g0; z1 = b - g1; z2 = b + g1;
    }
    *outA = make_float2(z0, z1);
    *outB = make_float2(z2, z3);
}

// -------------------------------------------------------------------------------------------------
// K1
// -------------------------------------------------------------------------------------------------
// FAST: the launch guarantees table_len > 0 and use_pairs for every item (any h0 built by Prepare()): the direct
// sincosf and per-point-record variants of the evolve loop are not instantiated - the kernel's code shrinks from
// ~170 KB to what the hot path needs (instruction-cache misses showed up as 7 % of K1's stall cycles).
template <int LOGN, int CP, int NF, bool SLAB = false, bool FAST = false, bool JAC = false>
struct Pass1 {
    static constexpr int N = 1 << LOGN;
    static constexpr int H = N / 2;
    static constexpr int B = CP * NF;                 // FFT lines per CTA
    static constexpr int T = B * N / kValsPerThread;  // threads per CTA
    static constexpr int LS = LineStride<N>::value;
    // + per column pair the four per-point records of the row pair (0, N/2) (fused front end, see special_request)
    static constexpr int SMEM_BYTES = (B * LS + kMaxTable) * (int)sizeof(float2) + CP * 4 * (int)sizeof(float4);
    static_assert(T >= 1 && T <= 1024, "bad CTA size");
    static_assert(H % CP == 0 && 4 % NF == 0, "bad tiling");
    // evolve work split: IT threads walk the row pairs i, CG thread groups walk the column pairs
    static constexpr int IT = (T < H) ? T : H;
    static constexpr int CG = T / IT;
    static_assert(T % IT == 0 && (CG <= CP), "bad evolve split");

    template <int F>
    static WSO_HD void put(float2* smem, int fl, int cp, int eA, int eB, float2 a, float2 b) {
        (void)F;
        smem[(fl * CP + cp) * LS + eA] = a;
        smem[(fl * CP + cp) * LS + eB] = b;
    }

    // Writes the NF packed fields of one interior work item given s = (h~(k) + h~(-k)) / 2 at its two wave vectors.
    static WSO_HD void pack_interior_item(float2* smem, int fg, int cp, int eA, int eB, float s0, float s1,
                                          float kxA, float kxB, float kzA, float inv0, float inv1) {
        float2 a, b;
        if (NF == 4 || (NF == 2 && fg == 0) || (NF == 1 && fg == 0)) {
            pack_interior<0, JAC>(s0, kxA, kzA, inv0, s1, kxB, kzA, inv1, &a, &b);
            put<0>(smem, 0, cp, eA, eB, a, b);
        }
        if (NF == 4 || (NF == 2 && fg == 0) || (NF == 1 && fg == 1)) {
            pack_interior<1, JAC>(s0, kxA, kzA, inv0, s1, kxB, kzA, inv1, &a, &b);
            put<1>(smem, NF == 1 ? 0 : 1, cp, eA, eB, a, b);
        }
        if (NF == 4 || (NF == 2 && fg == 1) || (NF == 1 && fg == 2)) {
            pack_interior<2, JAC>(s0, kxA, kzA, inv0, s1, kxB, kzA, inv1, &a, &b);
            put<2>(smem, NF == 4 ? 2 : 0, cp, eA, eB, a, b);
        }
        if (NF == 4 || (NF == 2 && fg == 1) || (NF == 1 && fg == 3)) {
            pack_interior<3, JAC>(s0, kxA, kzA, inv0, s1, kxB, kzA, inv1, &a, &b);
            put<3>(smem, NF == 4 ? 3 : (NF == 2 ? 1 : 0), cp, eA, eB, a, b);
        }
    }

    // one work item on the index-0 / N/2 lines (or any item when the pair records are unusable):
    // rows (mA,mB) x columns (nA,nB) = 4 wave vectors from the per-point records, general mirror pattern
    // jl: column pair index local to this device (storage), j = td.j0 + jl: global (wave numbers, special cases)
    template <bool TABLE>
    static WSO_HD void evolve_item_general(const TileDev& td, const float2* table, float t, int fg, float2* smem,
                                           int cp, int i, int jl) {
        const int j = td.j0 + jl;
        const int mA = i, mB = (i == 0) ? H : N - i;
        const int nA = j, nB = (j == 0) ? H : N - j;
        const float kxA = td.kv[nA], kxB = td.kv[nB], kzA = td.kv[mA], kzB = td.kv[mB];
        const int eA = pad_idx(mA), eB = pad_idx(mB);
        const float4* colA = td.h0 + (size_t)jl * 2 * N;
        const float4* colB = colA + N;
        const float4 q0 = colA[mA], q1 = colB[mA];
        const float4 q2 = colA[mB], q3 = colB[mB];
        const float h0 = eval_height<TABLE>(q0, table, t), h1 = eval_height<TABLE>(q1, table, t);
        const float h2 = eval_height<TABLE>(q2, table, t), h3 = eval_height<TABLE>(q3, table, t);
        const int mask = ((i != 0) ? 2 : 0) | ((j != 0) ? 1 : 0);
        Point pt[4];
        pt[0] = Point{h0, kxA, kzA, rmul(kxA, q0.z), rmul(kzA, q0.z)};
        pt[1] = Point{h1, kxB, kzA, rmul(kxB, q1.z), rmul(kzA, q1.z)};
        pt[2] = Point{h2, kxA, kzB, rmul(kxA, q2.z), rmul(kzB, q2.z)};
        pt[3] = Point{h3, kxB, kzB, rmul(kxB, q3.z), rmul(kzB, q3.z)};
        float2 a, b;
        if (NF == 4 || (NF == 2 && fg == 0) || (NF == 1 && fg == 0)) {
            pack_general<0, JAC>(pt, mask, &a, &b);
            put<0>(smem, 0, cp, eA, eB, a, b);
        }
        if (NF == 4 || (NF == 2 && fg == 0) || (NF == 1 && fg == 1)) {
            pack_general<1, JAC>(pt, mask, &a, &b);
            put<1>(smem, NF == 1 ? 0 : 1, cp, eA, eB, a, b);
        }
        if (NF == 4 || (NF == 2 && fg == 1) || (NF == 1 && fg == 2)) {
            pack_general<2, JAC>(pt, mask, &a, &b);
            put<2>(smem, NF == 4 ? 2 : 0, cp, eA, eB, a, b);
        }
        if (NF == 4 || (NF == 2 && fg == 1) || (NF == 1 && fg == 3)) {
            pack_general<3, JAC>(pt, mask, &a, &b);
            put<3>(smem, NF == 4 ? 3 : (NF == 2 ? 1 : 0), cp, eA, eB, a, b);
        }
    }

    // evolve phase of one thread: its row pairs i = i0, i0+IT, ... and column pairs cp = cg, cg+CG, ...
    // Interior items read the pair-summed records; all records of a row pair are requested before any is
    // used, so the L2 latency is paid once per row pair instead of once per item.
    static constexpr int CPT = CP / CG;  // column pairs per thread
    // The records of a thread's FIRST row pair are requested at the very top of the kernel (prefetch_thread) and
    // parked in the 16 complex registers that the transform stages use later: the L2 round trip overlaps the
    // sincos-table build, its barrier and the special row pair below.
    // Measured on B200 (profiles/r1h_ab_variants.txt): neutral at 1024^2 (one row pair per thread), but at 2048^2,
    // where a thread walks two row pairs, parking the first pair's records costs more than it hides (K1 68.3 ->
    // 56.3 us per tile-frame without it): only grids whose threads own a single row pair prefetch.
#ifndef WSO_TUNE_PREFETCH_MAX_LOGN
#define WSO_TUNE_PREFETCH_MAX_LOGN 10
#endif
#ifdef WSO_EXP_NO_PREFETCH
    static constexpr bool kPrefetch = false;
#else
    static constexpr bool kPrefetch = (LOGN <= WSO_TUNE_PREFETCH_MAX_LOGN) &&
                                      (2 * CPT * (int)sizeof(float4) <= kValsPerThread * (int)sizeof(float2));
#endif

    static WSO_HD const float4* pair_record(const TileDev& td, int bx, int cg, int k, int i, int half) {
        const int jl = bx * CP + cg + k * CG;
        return td.hs + hs_index(jl, i, half, H);
    }

    // the parking space holds the records of ONE row pair: threads that walk a single row pair can always prefetch
    // (the persistent form does, whatever the size: there the request is a whole store phase ahead of its use)
    static constexpr bool kPrefetchShape = (IT == H) && (2 * CPT * (int)sizeof(float4) <= kValsPerThread * (int)sizeof(float2));
    template <bool PF = kPrefetch>
    static WSO_HD void prefetch_thread(const TileDev& td, int bx, int tid, ThreadState& st) {
        if (!PF || (!FAST && !td.use_pairs)) return;
        const int i0 = tid % IT, cg = tid / IT;
        if (i0 == 0) return;
#pragma unroll
        for (int k = 0; k < CPT; ++k) {
            const float4 a = *pair_record(td, bx, cg, k, i0, 0), b = *pair_record(td, bx, cg, k, i0, 1);
            st.v[4 * k + 0] = make_float2(a.x, a.y);
            st.v[4 * k + 1] = make_float2(a.z, a.w);
            st.v[4 * k + 2] = make_float2(b.x, b.y);
            st.v[4 * k + 3] = make_float2(b.z, b.w);
        }
    }

    template <bool TABLE, bool PF = kPrefetch>
    static WSO_HD void evolve_thread(const TileDev& td, const float2* table, float t, int fg, float2* smem, int bx,
                                     int tid, const ThreadState& st) {
        const int i0 = tid % IT, cg = tid / IT;
        if (!FAST && !td.use_pairs) {  // foreign h0 (omega(k) != omega(-k)): every item through the per-point records
            for (int i = i0; i < H; i += IT)
                for (int cp = cg; cp < CP; cp += CG) evolve_item_general<TABLE>(td, table, t, fg, smem, cp, i, bx * CP + cp);
            return;
        }
        // The row pair i = 0 (rows 0 and N/2, their own mirrors) needs the general path: four dependent record
        // requests per item.  Its CP items are dealt to the last lanes of CP different warps so that they overlap
        // instead of serialising in the one thread that owns i0 == 0.
        if (T >= 32 * CP) {
            if ((tid & 31) == 31 && (tid >> 5) < CP) evolve_item_general<TABLE>(td, table, t, fg, smem, tid >> 5, 0, bx * CP + (tid >> 5));
        } else if (tid < CP) {
            evolve_item_general<TABLE>(td, table, t, fg, smem, tid, 0, bx * CP + tid);
        }
        for (int i = i0; i < H; i += IT) {
            if (i == 0) continue;
            float4 q0[CPT], q1[CPT];
            if (PF && i == i0) {
#pragma unroll
                for (int k = 0; k < CPT; ++k) {
                    q0[k] = make_float4(st.v[4 * k + 0].x, st.v[4 * k + 0].y, st.v[4 * k + 1].x, st.v[4 * k + 1].y);
                    q1[k] = make_float4(st.v[4 * k + 2].x, st.v[4 * k + 2].y, st.v[4 * k + 3].x, st.v[4 * k + 3].y);
                }
            } else {
#pragma unroll
                for (int k = 0; k < CPT; ++k) {
                    q0[k] = *pair_record(td, bx, cg, k, i, 0);
                    q1[k] = *pair_record(td, bx, cg, k, i, 1);
                }
            }
            const float kzA = td.kv[i];
            const int eA = pad_idx(i), eB = pad_idx(N - i);
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                const int cp = cg + k * CG;
                const int j = td.j0 + bx * CP + cp;
                if (j != 0) {
                    const float s0 = 0.5f * eval_height<TABLE>(q0[k], table, t);
                    const float s1 = 0.5f * eval_height<TABLE>(q1[k], table, t);
                    pack_interior_item(smem, fg, cp, eA, eB, s0, s1, td.kv[j], td.kv[N - j], kzA, q0[k].z, q1[k].z);
                } else {
                    evolve_item_general<TABLE>(td, table, t, fg, smem, cp, i, bx * CP + cp);
                }
            }
        }
    }

    // ---------------------------------------------------------------------------------------------------------
    // Fused front end (FAST launches whose tiling has NF * R0 == 8): evolve + FIRST Stockham stage in registers.
    // The first stage's butterfly j of a line reads rows j + r*JN0 (r < R0); the Hermitian mirror of those rows is
    // butterfly JN0 - j read backwards.  A thread that owns the butterfly pair (u, JN0-u) of the NF lines of one
    // column pair therefore needs exactly R0 row pairs (a, N-a) - the unit the pair-summed records are stored in -
    // and ends up with 2 * R0 * NF = 16 complex values: it runs the radix-R0 butterflies on them and writes the
    // stage-0 OUTPUT.  Against "evolve -> shared memory -> stage-0 load" this saves 16 STS.64 + 16 LDS.64 per thread
    // and one barrier (K1's transform phase runs at ~2/3 of the shared-memory wavefront bound, DESIGN.md §6).
    //   thread u >= 1: butterflies X = u, Y = JN0 - u.   thread u == 0: the two self-mirrored butterflies X = 0
    //   (rows r*JN0, holds the special rows 0 and N/2) and Y = JN0/2.
    // v[(fl*2 + bf)*R0 + idx]: line slot fl, bf 0 = X / 1 = Y, idx = input index r of that butterfly.
    static constexpr int R0 = Plan<LOGN>::R[0];
    static constexpr int JN0 = N / R0;
    static constexpr int H2 = JN0 / 2;  // threads per column pair
#ifdef WSO_EXP_NO_FUSE0
    static constexpr bool kFuse0 = false;
#else
    static constexpr bool kFuse0 = FAST && Plan<LOGN>::S > 1 && NF * R0 == 8 && H2 >= 2 && T == CP * H2;
#endif
    static constexpr bool kPrefetchF = kFuse0 && 4 * R0 <= kValsPerThread;  // all 2*R0 records fit the parking space
    // barrier behind the fused front end per column pair instead of CTA-wide (DeviceExec::sync_colpair); the named barriers
    // 1..B belong to the lines when a line is more than one warp
    static constexpr int kColPairIdBase = (N / kValsPerThread > 32) ? 1 + B : 1;
    // split + store dealt to the field groups, with a barrier per field group in front of it (split_store)
    static constexpr int kFieldIdBase = kColPairIdBase + CP;
#ifdef WSO_EXP_NO_FIELD_SPLIT
    static constexpr bool kFieldSplit = false;
#else
    // (measured per size, profiles/r3_memory_instructions.md section 9: 2048^2 K1 -3 %, 512^2 batches -2 %, but the 1024^2 path
    // 0.45 % slower in four pairs of runs although K1 alone is equal - that size keeps the CTA-wide barrier)
#ifndef WSO_TUNE_FIELD_SPLIT_SKIP_LOGN
#define WSO_TUNE_FIELD_SPLIT_SKIP_LOGN 10
#endif
    static constexpr bool kFieldSplit = !SLAB && NF > 1 && (T / NF) % 32 == 0 && (T / NF) % CP == 0 && H % (T / NF / CP) == 0 &&
                                        kFieldIdBase + NF - 1 <= 15 && LOGN != WSO_TUNE_FIELD_SPLIT_SKIP_LOGN;
#endif
#ifdef WSO_EXP_NO_COLPAIR_SYNC
    static constexpr bool kColPairSync = false;
#else
    static constexpr bool kColPairSync = kFuse0 && CP > 1 && H2 % 32 == 0 && (N / kValsPerThread) % 32 == 0 &&
                                         kColPairIdBase + CP - 1 <= 15;
#endif

    // packed field in line slot FL of field group fg: F = fg*NF + FL (fg is CTA-uniform)
    template <int FL>
    static WSO_HD void interior_fl(int fg, float s0, float kx0, float kz0, float inv0, float s1, float kx1, float kz1,
                                   float inv1, float2* a, float2* b) {
        if constexpr (NF == 4) {
            pack_interior<FL, JAC>(s0, kx0, kz0, inv0, s1, kx1, kz1, inv1, a, b);
        } else if constexpr (NF == 2) {
            if (fg == 0) pack_interior<FL, JAC>(s0, kx0, kz0, inv0, s1, kx1, kz1, inv1, a, b);
            else pack_interior<FL + 2, JAC>(s0, kx0, kz0, inv0, s1, kx1, kz1, inv1, a, b);
        } else {
            if (fg == 0) pack_interior<0, JAC>(s0, kx0, kz0, inv0, s1, kx1, kz1, inv1, a, b);
            else if (fg == 1) pack_interior<1, JAC>(s0, kx0, kz0, inv0, s1, kx1, kz1, inv1, a, b);
            else if (fg == 2) pack_interior<2, JAC>(s0, kx0, kz0, inv0, s1, kx1, kz1, inv1, a, b);
            else pack_interior<3, JAC>(s0, kx0, kz0, inv0, s1, kx1, kz1, inv1, a, b);
        }
    }
    template <int FL>
    static WSO_HD void general_fl(int fg, const Point (&pt)[4], int mask, float2* a, float2* b) {
        if constexpr (NF == 4) {
            pack_general<FL, JAC>(pt, mask, a, b);
        } else if constexpr (NF == 2) {
            if (fg == 0) pack_general<FL, JAC>(pt, mask, a, b);
            else pack_general<FL + 2, JAC>(pt, mask, a, b);
        } else {
            if (fg == 0) pack_general<0, JAC>(pt, mask, a, b);
            else if (fg == 1) pack_general<1, JAC>(pt, mask, a, b);
            else if (fg == 2) pack_general<2, JAC>(pt, mask, a, b);
            else pack_general<3, JAC>(pt, mask, a, b);
        }
    }

    // the four wave vectors of work item (row pair i, column pair jl) from the per-point records (same loads and
    // products as evolve_item_general)
    template <bool TABLE>
    static WSO_HD int general_points(const TileDev& td, const float2* table, float t, int i, int jl, Point (&pt)[4]) {
        const int mA = i, mB = (i == 0) ? H : N - i;
        const float4* colA = td.h0 + (size_t)jl * 2 * N;
        const float4* colB = colA + N;
        const float4 q[4] = {colA[mA], colB[mA], colA[mB], colB[mB]};
        return general_points_of<TABLE>(td, table, t, i, jl, q, pt);
    }
    // ... from records already at hand (q: the four per-point records in the order general_points reads them)
    template <bool TABLE>
    static WSO_HD int general_points_of(const TileDev& td, const float2* table, float t, int i, int jl, const float4* q,
                                        Point (&pt)[4]) {
        const int j = td.j0 + jl;
        const int mA = i, mB = (i == 0) ? H : N - i;
        const int nA = j, nB = (j == 0) ? H : N - j;
        const float kxA = td.kv[nA], kxB = td.kv[nB], kzA = td.kv[mA], kzB = td.kv[mB];
        const float4 q0 = q[0], q1 = q[1], q2 = q[2], q3 = q[3];
        const float h0 = eval_height<TABLE>(q0, table, t), h1 = eval_height<TABLE>(q1, table, t);
        const float h2 = eval_height<TABLE>(q2, table, t), h3 = eval_height<TABLE>(q3, table, t);
        pt[0] = Point{h0, kxA, kzA, rmul(kxA, q0.z), rmul(kzA, q0.z)};
        pt[1] = Point{h1, kxB, kzA, rmul(kxB, q1.z), rmul(kzA, q1.z)};
        pt[2] = Point{h2, kxA, kzB, rmul(kxA, q2.z), rmul(kzB, q2.z)};
        pt[3] = Point{h3, kxB, kzB, rmul(kxB, q3.z), rmul(kzB, q3.z)};
        return ((i != 0) ? 2 : 0) | ((j != 0) ? 1 : 0);
    }

    // register slot of the row-A / row-B output of work item K in the GENERIC arrangement (u >= 1):
    //   K <  R0/2 : a = u + K*JN0          A -> X[K]         B -> Y[R0-1-K]
    //   K >= R0/2 : a = JN0-u + (K-R0/2)*JN0  A -> Y[K-R0/2]   B -> X[R0-1-(K-R0/2)]
    template <int FL, int K>
    static constexpr int slot_a() { return K < R0 / 2 ? (FL * 2 + 0) * R0 + K : (FL * 2 + 1) * R0 + (K - R0 / 2); }
    template <int FL, int K>
    static constexpr int slot_b() {
        return K < R0 / 2 ? (FL * 2 + 1) * R0 + (R0 - 1 - K) : (FL * 2 + 0) * R0 + (R0 - 1 - (K - R0 / 2));
    }

    // The row pair (0, N/2) of a column pair goes through the per-point records (four 16-byte loads by the one thread
    // u == 0) - a dependent L2 round trip in front of the CTA-wide barrier behind the evolve, which held up the other 15
    // warps of the CTA for 7 % of K1's warp time (profiles/r3_ab_persistent.md).  The thread requests them at the top of
    // the kernel as asynchronous copies into a 64-byte scratch per column pair (no registers to park them in) and reads
    // them from there.
#ifdef WSO_EXP_NO_SPECIAL_ASYNC
    static constexpr bool kSpecialAsync = false;
#else
    static constexpr bool kSpecialAsync = kFuse0;
#endif
    static WSO_HD float4* special_scratch(float2* smem) { return reinterpret_cast<float4*>(smem + B * LS + kMaxTable); }
    template <class Exec>
    static WSO_HD void special_request(Exec& ex, const TileDev& td, float2* smem, int bx, int tid) {
        if constexpr (kSpecialAsync) {
            const int cp = tid / H2, u = tid - cp * H2;
            if (u != 0) return;
            const int jl = bx * CP + cp;
            const float4* colA = td.h0 + (size_t)jl * 2 * N;
            const float4* colB = colA + N;
            float4* dst = special_scratch(smem) + cp * 4;
            ex.async_copy16(dst + 0, colA);      // (m = 0, n = j)
            ex.async_copy16(dst + 1, colB);      // (0, N-j)
            ex.async_copy16(dst + 2, colA + H);  // (N/2, j)
            ex.async_copy16(dst + 3, colB + H);  // (N/2, N-j)
        }
    }

    static WSO_HD void prefetch_fused(const TileDev& td, int bx, int tid, ThreadState& st) {
        if (!kPrefetchF) return;
        const int cp = tid / H2, u = tid - cp * H2;
        const int jl = bx * CP + cp;
        const int base2 = u ? JN0 - u : JN0 / 2;
        static_for<0, R0>([&](auto kc) {
            constexpr int K = decltype(kc)::value;
            const int a = K < R0 / 2 ? u + K * JN0 : base2 + (K - R0 / 2) * JN0;
            const float4 q0 = ld_ro(td.hs + hs_index(jl, a, 0, H)), q1 = ld_ro(td.hs + hs_index(jl, a, 1, H));
            st.v[4 * K + 0] = make_float2(q0.x, q0.y);
            st.v[4 * K + 1] = make_float2(q0.z, q0.w);
            st.v[4 * K + 2] = make_float2(q1.x, q1.y);
            st.v[4 * K + 3] = make_float2(q1.z, q1.w);
        });
        // ... and the wave numbers the packing multiplies them with (td.kv is a table in global memory: requested here
        // they arrive with the records instead of after the table barrier)
        if constexpr (kPrefetchKv) {
            const int j = td.j0 + jl;
            static_for<0, R0>([&](auto kc) {
                constexpr int K = decltype(kc)::value;
                const int a = K < R0 / 2 ? u + K * JN0 : base2 + (K - R0 / 2) * JN0;
                st.pre[K] = td.kv[a];
            });
            st.pre[4] = td.kv[j];
            st.pre[5] = td.kv[j ? N - j : 0];
        }
    }
#ifdef WSO_EXP_NO_KV_PREFETCH
    static constexpr bool kPrefetchKv = false;
#else
    static constexpr bool kPrefetchKv = kPrefetchF && R0 <= 4;
#endif

    static WSO_HD void fused_thread(const TileDev& td, const float2* table, float t, int fg, float2* smem, int bx,
                                    int tid, ThreadState& st) {
        const int cp = tid / H2, u = tid - cp * H2;
        const int jl = bx * CP + cp, j = td.j0 + jl;
        const int base2 = u ? JN0 - u : JN0 / 2;
        float2 out[kValsPerThread];
        if (j != 0) {
            float4 q0[R0], q1[R0];
            static_for<0, R0>([&](auto kc) {
                constexpr int K = decltype(kc)::value;
                if (kPrefetchF) {
                    q0[K] = make_float4(st.v[4 * K + 0].x, st.v[4 * K + 0].y, st.v[4 * K + 1].x, st.v[4 * K + 1].y);
                    q1[K] = make_float4(st.v[4 * K + 2].x, st.v[4 * K + 2].y, st.v[4 * K + 3].x, st.v[4 * K + 3].y);
                } else {
                    const int a = K < R0 / 2 ? u + K * JN0 : base2 + (K - R0 / 2) * JN0;
                    q0[K] = ld_ro(td.hs + hs_index(jl, a, 0, H));
                    q1[K] = ld_ro(td.hs + hs_index(jl, a, 1, H));
                }
            });
            const float kxA = kPrefetchKv ? st.pre[4] : td.kv[j], kxB = kPrefetchKv ? st.pre[5] : td.kv[N - j];
            static_for<0, R0>([&](auto kc) {
                constexpr int K = decltype(kc)::value;
                const int a = K < R0 / 2 ? u + K * JN0 : base2 + (K - R0 / 2) * JN0;
                const float kz = kPrefetchKv ? st.pre[K] : td.kv[a];
                const float s0 = 0.5f * eval_height<true>(q0[K], table, t);
                const float s1 = 0.5f * eval_height<true>(q1[K], table, t);
                static_for<0, NF>([&](auto fc) {
                    constexpr int FL = decltype(fc)::value;
                    interior_fl<FL>(fg, s0, kxA, kz, q0[K].z, s1, kxB, kz, q1[K].z, &out[slot_a<FL, K>()],
                                    &out[slot_b<FL, K>()]);
                });
            });
        } else {  // column pair (0, N/2): every item through the per-point records
            static_for<0, R0>([&](auto kc) {
                constexpr int K = decltype(kc)::value;
                const int a = K < R0 / 2 ? u + K * JN0 : base2 + (K - R0 / 2) * JN0;
                Point pt[4];
                const int mask = general_points<true>(td, table, t, a, jl, pt);
                static_for<0, NF>([&](auto fc) {
                    constexpr int FL = decltype(fc)::value;
                    general_fl<FL>(fg, pt, mask, &out[slot_a<FL, K>()], &out[slot_b<FL, K>()]);
                });
            });
        }
        if (u == 0) {
            // item 0 of this thread is the row pair (0, N/2): its interior evaluation above read the (zero) record of
            // i = 0 and is replaced by the general one
            if (j != 0) {
                Point pt[4];
                const int mask = kSpecialAsync ? general_points_of<true>(td, table, t, 0, jl, special_scratch(smem) + cp * 4, pt)
                                               : general_points<true>(td, table, t, 0, jl, pt);
                static_for<0, NF>([&](auto fc) {
                    constexpr int FL = decltype(fc)::value;
                    general_fl<FL>(fg, pt, mask, &out[slot_a<FL, 0>()], &out[slot_b<FL, 0>()]);
                });
            }
            // self-mirrored butterflies: row B of item K < R0/2 belongs to X (index R0-K, or R0/2 for the row pair
            // (0, N/2)), row B of item R0/2 + r to Y (index R0-1-r): swap the upper halves accordingly
            static_for<0, NF>([&](auto fc) {
                constexpr int FL = decltype(fc)::value;
                float2 x_hi[R0 / 2], y_hi[R0 / 2];
                static_for<0, R0 / 2>([&](auto rc) {
                    constexpr int r = decltype(rc)::value;
                    x_hi[r] = out[(FL * 2 + 0) * R0 + R0 / 2 + r];
                    y_hi[r] = out[(FL * 2 + 1) * R0 + R0 / 2 + r];
                });
                static_for<0, R0 / 2>([&](auto rc) {
                    constexpr int r = decltype(rc)::value;  // r-th upper slot, index R0/2 + r
                    // new X[R0/2] = old Y[R0-1] (item 0);  new X[R0-K] = old Y[R0-1-K], K = 1..R0/2-1
                    if constexpr (r == 0) out[(FL * 2 + 0) * R0 + R0 / 2] = y_hi[R0 / 2 - 1];
                    else out[(FL * 2 + 0) * R0 + R0 / 2 + r] = y_hi[r - 1];
                    // new Y[R0-1-r'] = old X[R0-1-r']
                    out[(FL * 2 + 1) * R0 + R0 / 2 + r] = x_hi[r];
                });
            });
        }
        // first Stockham stage (NS = 1: no twiddles) and its store: y[j*R0 + r] = DFT_R0(x[j + r*JN0])[r]
        static_for<0, NF>([&](auto fc) {
            constexpr int FL = decltype(fc)::value;
            static_for<0, 2>([&](auto bc) {
                constexpr int BF = decltype(bc)::value;
                float2* x = &out[(FL * 2 + BF) * R0];
                Dft<R0>::run(x);
                const int jb = BF == 0 ? u : base2;
                float2* y = smem + (FL * CP + cp) * LS + pad_idx(jb * R0);
#pragma unroll
                for (int r = 0; r < R0; ++r) y[r] = x[r];
            });
        });
    }

    // bx: column-pair group, by: field group, bz: item within the chunk
    template <class Exec, class Args>
    static WSO_HD void run(Exec& ex, float2* smem, int bx, int by, int bz, const Args& args) {
        const BatchItem item = args.items[bz];
        const TileDev& td = args.td[bz];
        const float t = item.t;

        // ---- request the first row pair's records before anything else ---------------------------------
        ex.each([&](int tid, ThreadState& st) {
            if constexpr (kFuse0) prefetch_fused(td, bx, tid, st);
            else prefetch_thread(td, bx, tid, st);
        });
        if constexpr (kFuse0) RunStages<LOGN, B, 1, R0, Exec>::preload(ex, args.tw);
        else RunStages<LOGN, B, 0, 1, Exec>::preload(ex, args.tw);
        if constexpr (kFuse0) ex.each([&](int tid, ThreadState&) { special_request(ex, td, smem, bx, tid); });

        // ---- per-frame (cos,sin)(omega_j * t) table: omega takes few distinct values j*omega0 ------
        float2* table = smem + B * LS;
        const bool use_table = FAST || td.table_len > 0;
        if (use_table) {
            ex.each([&](int tid, ThreadState&) {
                for (int j = tid; j < td.table_len; j += T) {
                    float s, c;
                    sincos_acc(rmul(rmul((float)j, td.omega0), t), &s, &c);
                    table[j] = make_float2(c, s);
                }
            });
            if constexpr (kFuse0 && kSpecialAsync) ex.each([&](int, ThreadState&) { ex.async_wait(); });
            ex.sync();
        }

        // ---- evolve: 4 wave vectors per work item, all NF fields ------------------------------------
#ifndef WSO_EXP_SKIP_EVOLVE
        ex.each([&](int tid, ThreadState& st) {
            if constexpr (kFuse0) fused_thread(td, table, t, by, smem, bx, tid, st);
            else if (FAST || use_table) evolve_thread<true>(td, table, t, by, smem, bx, tid, st);
            else if constexpr (!FAST) evolve_thread<false>(td, table, t, by, smem, bx, tid, st);
        });
#endif
        if constexpr (kColPairSync) ex.template sync_colpair<CP, NF, H2, N / kValsPerThread>(kColPairIdBase);
        else ex.sync();

        // ---- B complex FFTs of length N along m ---------------------------------------------------
#ifndef WSO_EXP_SKIP_FFT1
        if constexpr (kFuse0) RunStages<LOGN, B, 1, R0, Exec>::run(ex, smem, args.tw);  // stage 0 ran in registers
        else RunStages<LOGN, B, 0, 1, Exec>::run(ex, smem, args.tw);
#endif
        // the split below reads the CP lines of a packed field per work item: with the split dealt to the field groups
        // (kFieldSplit) only the T/NF threads that own those lines have to meet, otherwise the whole CTA
        if constexpr (kFieldSplit) ex.template sync_group<T / NF, T>(kFieldIdBase);
        else ex.sync();
#ifdef WSO_EXP_SKIP_STORE1
        if (args.W != nullptr) return;
#endif
        // Everything above touched only per-tile constants and shared memory, so it may overlap the tail of the
        // previous kernel in the stream (the previous tile-frame's K2, which still reads W and the slot's min/max).
        ex.pdl_wait();
        ex.pdl_release();
        // the height min/max accumulators of this item's slot are reset here, ahead of K2h
        if (bx == 0 && by == 0) {
            ex.each([&](int tid, ThreadState&) {
                if (tid == 0) {
                    args.minmax[2 * item.slot + 0] = kInitMin;
                    args.minmax[2 * item.slot + 1] = kInitMax;
                }
            });
        }

        split_store(ex, smem, bx, by, bz, args);
    }

    template <class Exec, class Args>
    static WSO_HD void split_store(Exec& ex, const float2* smem, int bx, int by, int bz, const Args& args) {
        // ---- split the two real columns, keep m' in [0, N/2), store W[m'][f][slot] ---------------
        // thread -> fixed column pair cp = tid % CP (CP adjacent slots = one 8*CP-byte segment per m'),
        // and (field, m') pairs rest = tid/CP + k*(T/CP)
        // The sweep structure is compile-time: SWEEPS = 8 fully unrolled iterations (all shared-memory loads of a thread
        // are in flight together; a rolled loop paid one LDS round trip and ~20 index instructions per iteration -
        // 22 % of K1's executed instructions in profiles/r1h_ncu_c2.txt).
        // kFieldSplit: the T/NF threads that transformed the lines of packed field fl (threads [fl*T/NF, (fl+1)*T/NF)) also
        // split and store that field, so the barrier in front of the split is theirs alone (run()); otherwise every thread
        // walks all NF fields.  Same number of sweeps per thread, same store segments either way.
        float2* Wit = args.W + (size_t)bz * ((size_t)H * 4 * N);
        constexpr int TG = kFieldSplit ? T / NF : T;   // threads that share the split of one field (or of all)
        constexpr int STEP = TG / CP;                  // m' values covered per sweep
        constexpr int PER_LINE = H / STEP;             // sweeps per packed field
        constexpr int SWEEPS = (kFieldSplit ? 1 : NF) * PER_LINE;  // = 8
        static_assert(STEP >= 1 && H % STEP == 0 && SWEEPS * STEP * (kFieldSplit ? NF : 1) == NF * H, "bad split tiling");
        ex.each([&](int tid, ThreadState&) {
            const int tl = tid % TG;
            const int cp = tl % CP;
            const int jl = bx * CP + cp;
            const int b = tl / CP;               // m' of the first sweep, < STEP
#pragma unroll
            for (int k = 0; k < SWEEPS; ++k) {
                const int fl = kFieldSplit ? tid / TG : k / PER_LINE;
                const int mp = b + (k % PER_LINE) * STEP;
                const float2* line = smem + (fl * CP + cp) * LS;
                const float2 c1 = line[pad_idx(mp)];
                const float2 c2 = line[pad_idx((N - mp) & (N - 1))];
                // column n=j: (c1 + conj(c2))/2, column n=N-j: -i*(c1 - conj(c2))/2
                float2 wa = cscale(0.5f, cadd_conj(c1, c2));
                const float2 d = csub_conj(c1, c2);
                float2 wb = cscale(0.5f, make_float2(d.y, -d.x));
                if (k % PER_LINE == 0) {
                    if (mp == 0) {  // pack the (real) Nyquist bin m'=N/2 into the imaginary part of m'=0
                        const float2 ch = line[pad_idx(H)];
                        wa.y = ch.x;
                        wb.y = ch.y;
                    }
                }
                const int f = by * NF + fl;
                if constexpr (SLAB) {
                    const int hl_log = LOGN - 1 - args.slab_shift;
                    const int Hl = 1 << hl_log;
                    if (args.slab_stage != nullptr) {
                        float2* dst = args.slab_stage + ((size_t)(f * 2) * Hl + jl) * H + mp;
                        dst[0] = wa;
                        dst[(size_t)Hl * H] = wb;
                    } else {
                        // the store IS the transpose: block of the device that owns row item m'
                        float2* dst = args.Wdst[mp >> hl_log] + ((size_t)((mp & (Hl - 1)) * 4 + f) * 2) * Hl + jl;
                        dst[0] = wa;
                        dst[Hl] = wb;
                    }
                } else if constexpr (WLayout<LOGN>::paired) {
                    float4* dst = reinterpret_cast<float4*>(Wit + ((size_t)mp * 4 + f) * N) + jl;
                    st_keep(dst, make_float4(wa.x, wa.y, wb.x, wb.y));
                } else {
                    float2* dst = Wit + ((size_t)mp * 4 + f) * N + jl;
                    dst[0] = wa;
                    dst[H] = wb;
                }
            }
        });
    }

    // ---------------------------------------------------------------------------------------------------------
    // Persistent form (batched launches of the fused tilings): a fixed grid of CTAs walks the work items
    // w = cta, cta + ncta, ... (w -> column-pair group bx fastest, then field group by, then tile-frame bz).
    // What a CTA pays once per work item when every item is its own CTA - instruction fetch and parameter loads at
    // start, the L2 round trip of the records with nothing else to do, the drain of its W stores before the
    // next CTA can take its place (together a quarter of K1's warp time in the ncu source view of the one-CTA-per-item
    // kernel, profiles/r2_ncu_c2.txt) - is paid once per CTA here: the records of item w + ncta are requested right
    // before the split / store phase of item w, into the 16 complex registers that phase does not use, and have
    // arrived when the next evolve starts.
    static constexpr bool kPersistOk = FAST && !SLAB && !JAC && ((kFuse0 && kPrefetchF) || (!kFuse0 && kPrefetchShape));
    template <class Exec, class Args>
    static WSO_HD void run_persistent(Exec& ex, float2* smem, int cta, int ncta, int n_items, const Args& args) {
        static_assert(kPersistOk, "persistent K1: a tiling whose threads can park the records of their next item");
        constexpr int GX = H / CP, GY = 4 / NF;
        const int total = GX * GY * n_items;
        float2* table = smem + B * LS;
        int w = cta;
        if (w >= total) {  // (the launch sizes the grid <= total)
            ex.pdl_wait();
            ex.pdl_release();
            return;
        }
        int bx = w % GX, by = (w / GX) % GY, bz = w / (GX * GY);
        auto request = [&](int bzr, int bxr) {
            ex.each([&](int tid, ThreadState& st) {
                if constexpr (kFuse0) prefetch_fused(args.td[bzr], bxr, tid, st);
                else prefetch_thread<true>(args.td[bzr], bxr, tid, st);
            });
        };
        // (the scratch of the special row pair is read during the evolve only: it is rewritten at the loop top, behind
        // the barriers that follow the previous item's evolve)
        auto request_special = [&](int bzr, int bxr) {
            if constexpr (kFuse0) ex.each([&](int tid, ThreadState&) { special_request(ex, args.td[bzr], smem, bxr, tid); });
        };
        request(bz, bx);
        if constexpr (kFuse0) RunStages<LOGN, B, 1, R0, Exec>::preload(ex, args.tw);
        else RunStages<LOGN, B, 0, 1, Exec>::preload(ex, args.tw);
        int table_bz = -1;
        bool first = true;
        for (;;) {
            const TileDev& td = args.td[bz];
            const float t = args.items[bz].t;
            // (cos,sin)(omega_j t) of this tile-frame; every thread is past the previous item's evolve (barriers below)
            request_special(bz, bx);
            if (bz != table_bz) {
                ex.each([&](int tid, ThreadState&) {
                    for (int j = tid; j < td.table_len; j += T) {
                        float sn, cs;
                        sincos_acc(rmul(rmul((float)j, td.omega0), t), &sn, &cs);
                        table[j] = make_float2(cs, sn);
                    }
                });
                table_bz = bz;
            }
            if constexpr (kFuse0 && kSpecialAsync) ex.each([&](int, ThreadState&) { ex.async_wait(); });
            ex.sync();  // table visible; the previous item's split has finished reading the lines
            ex.each([&](int tid, ThreadState& st) {
                if constexpr (kFuse0) fused_thread(td, table, t, by, smem, bx, tid, st);
                else evolve_thread<true, true>(td, table, t, by, smem, bx, tid, st);
            });
            ex.sync();
            if constexpr (kFuse0) RunStages<LOGN, B, 1, R0, Exec>::run(ex, smem, args.tw);
            else RunStages<LOGN, B, 0, 1, Exec>::run(ex, smem, args.tw);
            ex.sync();
            const int wn = w + ncta;
            if (first) {  // W of the previous chunk in this lane is still being read until its K2 has completed
                ex.pdl_wait();
                first = false;
            }
            if (wn >= total) ex.pdl_release();
            if (bx == 0 && by == 0) {
                const BatchItem item = args.items[bz];
                ex.each([&](int tid, ThreadState&) {
                    if (tid == 0) {
                        args.minmax[2 * item.slot + 0] = kInitMin;
                        args.minmax[2 * item.slot + 1] = kInitMax;
                    }
                });
            }
            int bxn = 0, byn = 0, bzn = 0;
            if (wn < total) { bxn = wn % GX; byn = (wn / GX) % GY; bzn = wn / (GX * GY); }
#ifndef WSO_EXP_P_NOAHEAD
            if (wn < total) request(bzn, bxn);
#endif
            split_store(ex, smem, bx, by, bz, args);
#ifdef WSO_EXP_P_NOAHEAD
            if (wn < total) request(bzn, bxn);
#endif
            if (wn >= total) break;
            w = wn; bx = bxn; by = byn; bz = bzn;
        }
    }
};

// -------------------------------------------------------------------------------------------------
// K2 (maps) and K2h (height extrema only)
// -------------------------------------------------------------------------------------------------
WSO_HD int slot_of_column(int n, int N) {
    const int H = N >> 1;
    return (n < H) ? n : ((n == H) ? H : H + (N - n));
}

// reference: NormalizeHeights, WSTessendorf.cpp:443-455
WSO_HD float amplitude_of(float mn, float mx) {
    const float a = mn < 0.0f ? -mn : mn;
    const float b = mx < 0.0f ? -mx : mx;
    return a > b ? a : b;
}

// HEIGHT_ONLY = true : K2h - transforms only packed field 0 of every row item and reduces min/max of the height
//                      (A = max(|min|,|max|) must be known before any disp.y can be written normalised).
// HEIGHT_ONLY = false: K2  - all four fields; by = 0 writes the displacement map (fields 0,1; disp.y already
//                      multiplied by 1/A), by = 1 the normal map (fields 2,3).
// SLAB : the grid is slab-decomposed over several devices (LaunchArgsT::slab_*): W is read in the received block
//        layout and the two output rows of local row item ml go to local rows ml and Hl + ml.
// PAIR : the two lines of a row item live in the two CTAs of a thread-block cluster (a 16384-point line pair does not
//        fit one SM's shared memory): each CTA transforms one line, then packs ONE of the two output rows, reading
//        its partner's line through distributed shared memory.
// JAC  : SURVEY row f-4 (reference COMPUTE_JACOBIAN, WSTessendorf.cpp:421-428): one CTA transforms all FOUR packed
//        fields of a row item (by = 0 only) and writes both maps, disp.w = the Jacobian of the horizontal displacement.
// TEX  : output texel, float4 (RGBA32F) or Half4 (RGBA16F, wso_device.cuh): LaunchArgsT::disp / norm are read as arrays
//        of TEX.  The arithmetic is the same; only the final store converts.  Single-device kernels only.
template <int LOGN, int RI, bool HEIGHT_ONLY, bool SLAB = false, bool PAIR = false, bool JAC = false, class TEX = float4>
struct Pass2 {
    static constexpr int N = 1 << LOGN;
    static constexpr int H = N / 2;
    static constexpr int LPI = HEIGHT_ONLY ? 1 : (JAC ? 4 : 2);  // lines per row item
    static constexpr int LPC = PAIR ? 1 : LPI;       // ... of which this CTA holds
    static constexpr int B = RI * LPC;
    static constexpr int T = B * N / kValsPerThread;
    static constexpr int G = N / kValsPerThread;     // threads per line
    static constexpr int GI = LPC * G;               // threads per row item
    static constexpr int LS = LineStride<N>::value;
    static constexpr int SMEM_BYTES = B * LS * (int)sizeof(float2);
    static_assert(T >= 1 && T <= 1024, "bad CTA size");
    static_assert(H % RI == 0, "bad tiling");
    static_assert(!PAIR || (!HEIGHT_ONLY && RI == 1), "cluster pairs: one row item per CTA pair");
    static_assert(!JAC || (!HEIGHT_ONLY && !SLAB && !PAIR), "Jacobian variant: single-device maps kernel only");
    static_assert(std::is_same<TEX, float4>::value || (std::is_same<TEX, Half4>::value && !SLAB && !PAIR),
                  "RGBA16F maps: single-device kernels only");

    template <class Args>
    static WSO_HD int hl_log(const Args& args) { return SLAB ? LOGN - 1 - args.slab_shift : LOGN - 1; }

    // K2h only reduces the transformed heights: the outputs of the last stage are folded into min/max straight from
    // the registers (no final store, barrier and re-load: a third of K2h's shared-memory traffic); only the line
    // that carries rows 0 and N/2 as one complex transform goes through shared memory (it needs mirrored columns).
#ifdef WSO_EXP_NO_REG_REDUCE
    static constexpr bool kReduceFromRegs = false;
#else
    static constexpr bool kReduceFromRegs = HEIGHT_ONLY && Plan<LOGN>::S > 1 && (G % 2 == 0);
#endif

    // K2 packs from the registers of the last stage.  After the last stage (radix 16: thread j of a line holds X[j + r*N/16],
    // r < 16) the thread of packed-field line 0 keeps its columns r < 8 and the thread j of line 1 its columns r >= 8; each
    // hands the OTHER half to its partner through its own shared-memory line (8 stores, one barrier of the row item's
    // threads, 8 loads) and packs both output rows of its 8 columns - lanes = consecutive columns, 512-byte store
    // segments as before.  Against "store the whole last stage, barrier, re-load both lines" this is 16 instead of 32
    // shared-memory accesses per thread (a sixth of K2's; the LSU data pipe is what K2 runs closest to, DESIGN.md 6).
    // Same arithmetic on the same values: bit-identical maps.  Row item 0 (rows 0 and N/2 in one complex line: needs
    // mirrored columns) keeps the old route.
    static constexpr int RLast = Plan<LOGN>::R[Plan<LOGN>::S - 1];
#ifdef WSO_EXP_NO_PACK_REGS
    static constexpr bool kPackFromRegs = false;
#else
    static constexpr bool kPackFromRegs = !HEIGHT_ONLY && !SLAB && !PAIR && !JAC && Plan<LOGN>::S > 1 &&
                                          RLast == kValsPerThread && G >= 32 && ((N / RLast) % 16 == 0);
#endif

    // K2h, two row items per transform.  The height of row item m' is Re FFT(w), w = its packed-field-0 line; the real
    // part of a transform is the transform of the conjugate-even part e[n] = (w[n] + conj(w[N-n])) / 2, and the paired W
    // layout hands a thread w[n] and w[N-n] in ONE 16-byte word.  So one complex transform of e_a + i e_b yields the
    // heights of row items a (real part) and b (imaginary part): K2h runs half as many lines for one more load per
    // point.  Line 0 keeps row item 0 alone (rows 0 and N/2 travel as one complex line and need both parts); line
    // l >= 1 carries the row items 2l-1 and 2l (the last line its single item twice).  The factor 1/2 is applied to the
    // heights (exact).  Sizes >= 512^2.
    // Build option, OFF: measured on B200 (profiles/r3_ab_persistent.md) K2h alone gets 14 % faster (1024^2: 3.28 -> 2.81 us,
    // 2048^2: 13.3 -> 11.5 us per tile-frame) - it is bound by the latency of its loads, not by the transform - and the
    // whole path does not move (K2h runs underneath K1 / K2 of the other compute lane), while the extrema stop being
    // bit-identical to the heights K2 writes and to the slab path's.
#ifdef WSO_EXP_K2H_PAIRS
    static constexpr bool kTwoForOne = HEIGHT_ONLY && !SLAB && !PAIR && !JAC && WLayout<LOGN>::paired && LOGN >= 9 && kReduceFromRegs;
#else
    static constexpr bool kTwoForOne = false;
#endif
    static constexpr int kLines = kTwoForOne ? 1 + H / 2 : H;            // K2h / K2 lines groups per tile-frame
    static WSO_HD constexpr int grid_x() { return (kLines + RI - 1) / RI; }
    // row items (a, b) of global line gl of the two-for-one K2h (gl >= 1)
    static WSO_HD void items_of_line(int gl, int& a, int& b) {
        if (gl > H / 2) gl = H / 2;  // lines past the end of a partially filled CTA repeat the last one
        a = 2 * gl - 1;
        b = (2 * gl < H) ? 2 * gl : a;
    }

    // ---- first stage in the paired W layout --------------------------------------------------------------
    // A thread owns first-stage butterfly PAIRS (p, JN-p) - the mirror column N-n of every column n of butterfly p
    // belongs to butterfly JN-p - so each 16-byte word (column n, column N-n) feeds one input of each.  Pair 0 is the
    // two self-mirrored butterflies (0, JN/2); its upper halves are re-slotted exactly as in K1's fused front end.
    // first_load only requests the words (into the registers the butterflies run in); first_compute runs the
    // butterflies and stores the stage output: the persistent K2 issues the loads of its NEXT row items ahead of the
    // pack phase of the current ones.
    static constexpr int R1st = Plan<LOGN>::R[0];
    static constexpr int JN1st = N / R1st;
    static constexpr int NP1st = (2 * R1st <= kValsPerThread) ? kValsPerThread / (2 * R1st) : 1;  // butterfly pairs per thread
    static WSO_HD void first_load(int tid, ThreadState& st, const float2* Wit, int bx, int by, int crank) {
        constexpr int R = R1st, JN = JN1st, NP = NP1st;
        static_assert(!WLayout<LOGN>::paired || (G * NP == JN / 2), "paired first stage: bad shape");
        const int line = tid / G, lt = tid % G;
        if constexpr (kTwoForOne) {
            const int gl = bx * RI + line;
            if (gl != 0) {
                int ia, ib;
                items_of_line(gl, ia, ib);
                const float4* srcA = reinterpret_cast<const float4*>(Wit + ((size_t)ia * 4) * N);
                const float4* srcB = reinterpret_cast<const float4*>(Wit + ((size_t)ib * 4) * N);
                static_for<0, NP>([&](auto ic) {
                    constexpr int I = decltype(ic)::value;
                    const int p = lt + G * I;
                    const int base2 = p ? JN - p : JN / 2;
                    float2* v = &st.v[I * 2 * R];
                    static_for<0, R>([&](auto kc) {
                        constexpr int K = decltype(kc)::value;
                        const int n = K < R / 2 ? p + K * JN : base2 + (K - R / 2) * JN;
                        const float4 qa = srcA[n], qb = srcB[n];
                        constexpr int sa = K < R / 2 ? K : R + (K - R / 2);
                        constexpr int sb = K < R / 2 ? R + (R - 1 - K) : (R - 1 - (K - R / 2));
                        // 2 e[n] = w[n] + conj(w[N-n]) of both items; x[n] = 2 e_a[n] + i 2 e_b[n], x[N-n] = conj(2 e_a[n]) + i conj(2 e_b[n])
                        const float ax = qa.x + qa.z, ay = qa.y - qa.w, bx2 = qb.x + qb.z, by2 = qb.y - qb.w;
                        float2 xn = make_float2(ax - by2, ay + bx2), xm = make_float2(ax + by2, bx2 - ay);
                        if (K == 0 && n == 0) {  // the word (w[0], w[N/2]): both bins are their own mirrors, e = Re w
                            xn = make_float2(qa.x + qa.x, qb.x + qb.x);
                            xm = make_float2(qa.z + qa.z, qb.z + qb.z);
                        }
                        v[sa] = xn;
                        v[sb] = xm;
                    });
                });
                return;
            }
        }
        const int ml = kTwoForOne ? 0 : bx * RI + line / LPC;
        const int f = HEIGHT_ONLY ? 0 : (JAC ? line % LPC : by * 2 + (PAIR ? crank : line % LPC));
        const float4* src = reinterpret_cast<const float4*>(Wit + ((size_t)ml * 4 + f) * N);
        static_for<0, NP>([&](auto ic) {
            constexpr int I = decltype(ic)::value;
            const int p = lt + G * I;
            const int base2 = p ? JN - p : JN / 2;
            float2* v = &st.v[I * 2 * R];  // v[bf*R + idx]
            static_for<0, R>([&](auto kc) {
                constexpr int K = decltype(kc)::value;
                const int n = K < R / 2 ? p + K * JN : base2 + (K - R / 2) * JN;
                const float4 q = HEIGHT_ONLY ? src[n] : ld_last(src + n);  // K2 is W's last reader
                constexpr int sa = K < R / 2 ? K : R + (K - R / 2);
                constexpr int sb = K < R / 2 ? R + (R - 1 - K) : (R - 1 - (K - R / 2));
                v[sa] = make_float2(q.x, q.y);
                v[sb] = make_float2(q.z, q.w);
            });
        });
    }
    static WSO_HD void first_compute(int tid, ThreadState& st, float2* smem) {
        constexpr int R = R1st, JN = JN1st, NP = NP1st;
        const int line = tid / G, lt = tid % G;
        float2* y = smem + line * LS;
        static_for<0, NP>([&](auto ic) {
            constexpr int I = decltype(ic)::value;
            const int p = lt + G * I;
            const int base2 = p ? JN - p : JN / 2;
            float2* v = &st.v[I * 2 * R];
            if (p == 0) {
                float2 x_hi[R / 2], y_hi[R / 2];
                static_for<0, R / 2>([&](auto rc) {
                    constexpr int r = decltype(rc)::value;
                    x_hi[r] = v[R / 2 + r];
                    y_hi[r] = v[R + R / 2 + r];
                });
                static_for<0, R / 2>([&](auto rc) {
                    constexpr int r = decltype(rc)::value;
                    if constexpr (r == 0) v[R / 2] = y_hi[R / 2 - 1];
                    else v[R / 2 + r] = y_hi[r - 1];
                    v[R + R / 2 + r] = x_hi[r];
                });
            }
            static_for<0, 2>([&](auto bc) {
                constexpr int BF = decltype(bc)::value;
                Dft<R>::run(&v[BF * R]);
                float2* yb = y + pad_idx((BF == 0 ? p : base2) * R);
#pragma unroll
                for (int r = 0; r < R; ++r) yb[r] = v[BF * R + r];
            });
        });
    }

    // ---- transform phase: first stage straight from global memory (W rows are contiguous), rest in shared memory
    // crank: rank of this CTA in its cluster pair (PAIR only)
    template <class Exec, class Args>
    static WSO_HD void transform(Exec& ex, float2* smem, int bx, int by, int bz, int crank, const Args& args) {
        const float2* Wit = args.W + (SLAB ? (size_t)0 : (size_t)bz * ((size_t)H * 4 * N));
        // K2h consumes what K1 (its predecessor in the stream) wrote: wait first.  K2 is released by K2h only after
        // K2h's own wait, i.e. K1 is complete when K2 starts: K2 transforms W right away and waits (for K2h's
        // min/max) only before the pack phase.
        if constexpr (HEIGHT_ONLY) {
            ex.pdl_wait();
            ex.pdl_release();
        }
        constexpr int R = Plan<LOGN>::R[0];
        using St = Stage<N, B, R, 1>;
        const int hlog = hl_log(args);
        if constexpr (Plan<LOGN>::S > 1) RunStages<LOGN, B, 1, R, Exec, kReduceFromRegs || kPackFromRegs>::preload(ex, args.tw);
        if constexpr (!SLAB && WLayout<LOGN>::paired) {
            ex.each([&](int tid, ThreadState& st) { first_load(tid, st, Wit, bx, by, crank); });
            ex.each([&](int tid, ThreadState& st) { first_compute(tid, st, smem); });
            ex.template sync_group<G, T>(1);
            if constexpr (Plan<LOGN>::S > 1) RunStages<LOGN, B, 1, R, Exec, kReduceFromRegs || kPackFromRegs>::run(ex, smem, args.tw);
            return;
        }
        ex.each([&](int tid, ThreadState& st) {
            const int line = tid / G;
            const int ml = bx * RI + line / LPC;
            const int f = HEIGHT_ONLY ? 0 : (JAC ? line % LPC : by * 2 + (PAIR ? crank : line % LPC));
            const float2* src = Wit + ((size_t)ml * 4 + f) * 2 * ((size_t)1 << hlog);  // [ml][f][half][jl] of source 0
#pragma unroll
            for (int i = 0; i < St::NB; ++i) {
                const int j = tid % G + G * i;
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int slot = slot_of_column(j + r * St::JN, N);
                    if constexpr (SLAB) {
                        const int half = slot >> (LOGN - 1), jj = slot & (H - 1);
                        const size_t blk = (size_t)8 << (2 * hlog);  // elements per source block: Hl*4*2*Hl
                        st.v[i * R + r] = src[(size_t)(jj >> hlog) * blk + ((size_t)half << hlog) + (jj & ((1 << hlog) - 1))];
                    } else {
                        st.v[i * R + r] = src[slot];
                    }
                }
            }
            St::twiddle_dft(args.tw, tid, st);
            St::store(smem, tid, st);
        });
        ex.template sync_group<G, T>(1);
        if constexpr (Plan<LOGN>::S > 1) RunStages<LOGN, B, 1, R, Exec, kReduceFromRegs || kPackFromRegs>::run(ex, smem, args.tw);
    }

    // ---- K2h: min/max of the height = Re of packed field 0
    template <class Exec, class Args>
    static WSO_HD void reduce_heights(Exec& ex, float2* smem, int bx, int bz, const Args& args) {
        const BatchItem item = args.items[bz];
        const int hlog = hl_log(args);
        if constexpr (kReduceFromRegs) {
            constexpr int RL = Plan<LOGN>::R[Plan<LOGN>::S - 1];  // radix of the last stage
            constexpr int NSL = N / RL;                            // its output stride: st.v[i*RL + r] = X[j_i + r*NSL]
            using StL = Stage<N, B, RL, NSL>;
            const int mp0 = (SLAB ? (args.slab_rank << hlog) : 0) + bx * RI;  // row item of this CTA's first line
            const bool has_special = (mp0 == 0);                              // CTA-uniform
            ex.each([&](int tid, ThreadState& st) {
                const int ri = tid / GI, lt = tid % GI;
                const int mp = mp0 + ri;   // two-for-one: the global line index (0 = row item 0 alone)
                if (kTwoForOne && mp != 0) {
                    int ia, ib;
                    items_of_line(mp, ia, ib);
                    // column parity is one value per thread (G and NSL are even); the transform ran on 2 e
                    const float sa = ((ia + lt) & 1) ? -0.5f : 0.5f, sb = ((ib + lt) & 1) ? -0.5f : 0.5f;
                    float mn = kInitMin, mx = kInitMax;
#pragma unroll
                    for (int k = 0; k < kValsPerThread; ++k) {
                        const float ha = rmul(st.v[k].x, sa), hb = rmul(st.v[k].y, sb);
                        mn = ha < mn ? ha : mn;
                        mx = ha > mx ? ha : mx;
                        mn = hb < mn ? hb : mn;
                        mx = hb > mx ? hb : mx;
                    }
                    st.v[0] = make_float2(mn, mx);
                } else if (mp != 0) {
                    // column c = lt + G*i + r*NSL: G and NSL are even, so (-1)^(row+col) is one sign per thread
                    const float s = ((mp + lt) & 1) ? -1.0f : 1.0f;
                    float mn = kInitMin, mx = kInitMax;
#pragma unroll
                    for (int k = 0; k < kValsPerThread; ++k) {
                        const float h = rmul(st.v[k].x, s);
                        mn = h < mn ? h : mn;
                        mx = h > mx ? h : mx;
                    }
                    st.v[0] = make_float2(mn, mx);
                } else {
                    StL::store(smem, tid, st);
                }
            });
            if (has_special) {
                ex.template sync_group<G, T>(1);
                ex.each([&](int tid, ThreadState& st) {
                    const int ri = tid / GI, lt = tid % GI;
                    if (mp0 + ri != 0) return;
                    const float2* l0 = smem + ri * LS;
                    float mn = kInitMin, mx = kInitMax;
                    const float s = (lt & 1) ? -1.0f : 1.0f;
                    for (int c = lt; c < N; c += GI) {
                        const float2 a = l0[pad_idx(c)], m = l0[pad_idx((N - c) & (N - 1))];
                        const float hA = rmul(0.5f * (a.x + m.x), s), hB = rmul(0.5f * (a.y + m.y), s);
                        mn = hA < mn ? hA : mn; mx = hA > mx ? hA : mx;
                        mn = hB < mn ? hB : mn; mx = hB > mx ? hB : mx;
                    }
                    st.v[0] = make_float2(mn, mx);
                });
            }
            ex.commit_minmax(args.minmax + 2 * item.slot);
            return;
        }
        ex.each([&](int tid, ThreadState& st) {
            float mn = kInitMin, mx = kInitMax;
            const int ri = tid / GI, lt = tid % GI;
            const int mp = (SLAB ? (args.slab_rank << hlog) : 0) + bx * RI + ri;
            const float2* l0 = smem + ri * LS;
            // (-1)^(row+col): loop invariant when the column stride GI is even (N >= 32)
            float s = ((mp + lt) & 1) ? -1.0f : 1.0f;
            if (mp != 0) {
#pragma unroll
                for (int k = 0; k < N / GI; ++k) {  // compile-time trip count: the loads of a thread overlap
                    const int c = lt + k * GI;
                    if (GI & 1) s = ((mp + c) & 1) ? -1.0f : 1.0f;
                    const float h = rmul(l0[pad_idx(c)].x, s);
                    mn = h < mn ? h : mn;
                    mx = h > mx ? h : mx;
                }
            } else {  // rows 0 and N/2 were transformed as one complex line
                for (int c = lt; c < N; c += GI) {
                    if (GI & 1) s = (c & 1) ? -1.0f : 1.0f;
                    const float2 a = l0[pad_idx(c)], m = l0[pad_idx((N - c) & (N - 1))];
                    const float hA = rmul(0.5f * (a.x + m.x), s), hB = rmul(0.5f * (a.y + m.y), s);
                    mn = hA < mn ? hA : mn; mx = hA > mx ? hA : mx;
                    mn = hB < mn ? hB : mn; mx = hB > mx ? hB : mx;
                }
            }
            st.v[0] = make_float2(mn, mx);
        });
        ex.commit_minmax(args.minmax + 2 * item.slot);
    }

    // ---- K2 pack: each transformed line pair (l0, l1) yields output rows A = m' and B = N-m' (rows 0 and N/2 for
    // m' = 0).  rows: bit 0 = write row A, bit 1 = write row B.
    // reference: WSTessendorf.cpp:385-437 (sign, lambda, packing) and :443-455 (normalisation)
    // STRIDE: threads per row item.  The column loop stays rolled: fully unrolled (all 16 shared-memory loads of a
    // thread in flight) it measured 6-8 % SLOWER on B200 (K2 9.35 -> 10.1 us per 1024^2 tile-frame, profiles/
    // r1i_sweep.txt) - the map stores of K2 are what bounds it, and they issue best interleaved with the loads.
#ifndef WSO_TUNE_PACK_UNROLL
#define WSO_TUNE_PACK_UNROLL 1
#endif
    static constexpr int kPackUnroll = WSO_TUNE_PACK_UNROLL;
    template <int STRIDE>
    static WSO_HD void pack_item(const float2* l0, const float2* l1, int mp, TEX* outA, TEX* outB, int by,
                                 float lambda, float inv_amp, int lt, int rows) {
        static_assert(N % STRIDE == 0, "bad pack stride");
        constexpr int VISITS = N / STRIDE;
        // (-1)^(row+col) is the same for both output rows and every column this thread visits (stride is even)
        const float s = ((mp + lt) & 1) ? -1.0f : 1.0f;
        const float sl = rmul(s, lambda);
        if (mp != 0) {
            if (by == 0) {
#pragma unroll kPackUnroll
                for (int k = 0; k < VISITS; ++k) {
                    const int c = lt + k * STRIDE;
                    const int e = pad_idx(c);
                    const float2 a0 = l0[e], a1 = l1[e];
                    const int cm = (N - c) & (N - 1);   // row N-m' is the conjugate mirror of row m'
                    const float y = rmul(rmul(a0.x, s), inv_amp);
                    const float x = rmul(sl, a0.y), z = rmul(sl, a1.y);
                    if (rows & 1) st_texel(&outA[c], x, y, z, 1.0f);
                    if (rows & 2) st_texel(&outB[cm], -x, y, -z, 1.0f);
                }
            } else {
#pragma unroll kPackUnroll
                for (int k = 0; k < VISITS; ++k) {
                    const int c = lt + k * STRIDE;
                    const int e = pad_idx(c);
                    const float2 a0 = l0[e], a1 = l1[e];
                    const int cm = (N - c) & (N - 1);
                    const float4 ta = make_float4(s * a0.y, s * a1.y, s * a0.x, s * a1.x);
                    if (rows & 1) st_texel(&outA[c], ta.x, ta.y, ta.z, ta.w);
                    if (rows & 2) st_texel(&outB[cm], -ta.x, -ta.y, ta.z, ta.w);
                }
            }
        } else {
            // rows 0 and N/2 were transformed as one complex line: separate them
            for (int c = lt; c < N; c += STRIDE) {
                const int e = pad_idx(c), em = pad_idx((N - c) & (N - 1));
                const float2 p0 = l0[e], p1 = l1[e], m0 = l0[em], m1 = l1[em];
                const float2 a0 = make_float2(0.5f * (p0.x + m0.x), 0.5f * (p0.y - m0.y));
                const float2 a1 = make_float2(0.5f * (p1.x + m1.x), 0.5f * (p1.y - m1.y));
                const float2 b0 = make_float2(0.5f * (p0.y + m0.y), -0.5f * (p0.x - m0.x));
                const float2 b1 = make_float2(0.5f * (p1.y + m1.y), -0.5f * (p1.x - m1.x));
                if (by == 0) {
                    if (rows & 1) st_texel(&outA[c], rmul(sl, a0.y), rmul(rmul(a0.x, s), inv_amp), rmul(sl, a1.y), 1.0f);
                    if (rows & 2) st_texel(&outB[c], rmul(sl, b0.y), rmul(rmul(b0.x, s), inv_amp), rmul(sl, b1.y), 1.0f);
                } else {
                    if (rows & 1) st_texel(&outA[c], s * a0.y, s * a1.y, s * a0.x, s * a1.x);
                    if (rows & 2) st_texel(&outB[c], s * b0.y, s * b1.y, s * b0.x, s * b1.x);
                }
            }
        }
    }

    // Jacobian variant: lines l0..l3 = packed fields 0..3 of the row item; writes rows A = m' and B = N-m' of BOTH maps.
    // reference: WSTessendorf.cpp:421-428  J = (1 + l*s*dxDx)(1 + l*s*dzDz) - (l*s*dxDz)(l*s*dzDx), dxDz == dzDx
    static WSO_HD float jacobian_of(float lambda, float dxdx, float dzdz, float dzdx) {
        const float c = rmul(lambda, dzdx);
        return rsub(rmul(radd(1.0f, rmul(lambda, dxdx)), radd(1.0f, rmul(lambda, dzdz))), rmul(c, c));
    }
    template <int STRIDE>
    static WSO_HD void pack_item_jac(const float2* l0, const float2* l1, const float2* l2, const float2* l3, int mp,
                                     TEX* dA, TEX* dB, TEX* nA, TEX* nB, float lambda, float inv_amp,
                                     int lt) {
        const float s = ((mp + lt) & 1) ? -1.0f : 1.0f;
        const float sl = rmul(s, lambda);
        if (mp != 0) {
            for (int c = lt; c < N; c += STRIDE) {
                const int e = pad_idx(c);
                const float2 a0 = l0[e], a1 = l1[e], a2 = l2[e], a3 = l3[e];
                const int cm = (N - c) & (N - 1);
                const float y = rmul(rmul(a0.x, s), inv_amp);
                const float x = rmul(sl, a0.y), z = rmul(sl, a1.y);
                const float j = jacobian_of(lambda, s * a2.x, s * a3.x, s * a1.x);
                st_texel(&dA[c], x, y, z, j);
                st_texel(&dB[cm], -x, y, -z, j);
                const float4 ta = make_float4(s * a2.y, s * a3.y, s * a2.x, s * a3.x);
                st_texel(&nA[c], ta.x, ta.y, ta.z, ta.w);
                st_texel(&nB[cm], -ta.x, -ta.y, ta.z, ta.w);
            }
        } else {
            // rows 0 and N/2 were transformed as one complex line per field: separate them
            for (int c = lt; c < N; c += STRIDE) {
                const int e = pad_idx(c), em = pad_idx((N - c) & (N - 1));
                float2 a[4], b[4];
                const float2* ls[4] = {l0, l1, l2, l3};
#pragma unroll
                for (int f = 0; f < 4; ++f) {
                    const float2 p = ls[f][e], m = ls[f][em];
                    a[f] = make_float2(0.5f * (p.x + m.x), 0.5f * (p.y - m.y));
                    b[f] = make_float2(0.5f * (p.y + m.y), -0.5f * (p.x - m.x));
                }
                st_texel(&dA[c], rmul(sl, a[0].y), rmul(rmul(a[0].x, s), inv_amp), rmul(sl, a[1].y),
                         jacobian_of(lambda, s * a[2].x, s * a[3].x, s * a[1].x));
                st_texel(&dB[c], rmul(sl, b[0].y), rmul(rmul(b[0].x, s), inv_amp), rmul(sl, b[1].y),
                         jacobian_of(lambda, s * b[2].x, s * b[3].x, s * b[1].x));
                st_texel(&nA[c], s * a[2].y, s * a[3].y, s * a[2].x, s * a[3].x);
                st_texel(&nB[c], s * b[2].y, s * b[3].y, s * b[2].x, s * b[3].x);
            }
        }
    }

    // smem_peer: the partner CTA's line (PAIR only; distributed shared memory on the device)
    template <class Exec, class Args>
    static WSO_HD void pack(Exec& ex, const float2* smem, const float2* smem_peer, int bx, int by, int bz, int crank,
                            const Args& args) {
        // Only the displacement map needs K2h's result (disp.y is written already divided by A): the CTAs of the normal
        // map pack right away and fill the device while K2h drains.
        const bool needs_amp = JAC || by == 0;
        if (needs_amp) ex.pdl_wait();
        ex.pdl_release();
        pack_body(ex, smem, smem_peer, bx, by, bz, crank, args);
    }
    // (the caller has waited for K2h where by == 0)
    template <class Exec, class Args>
    static WSO_HD void pack_body(Exec& ex, const float2* smem, const float2* smem_peer, int bx, int by, int bz, int crank,
                                 const Args& args) {
        const BatchItem item = args.items[bz];
        const bool needs_amp = JAC || by == 0;
        const float lambda = args.td[bz].lambda;
        const float amp = needs_amp ? amplitude_of(args.minmax[2 * item.slot], args.minmax[2 * item.slot + 1]) : 1.0f;
        const float inv_amp = rdiv(1.0f, amp);
        if (bx == 0 && by == 0 && crank == 0) {
            ex.each([&](int tid, ThreadState&) {
                if (tid == 0) args.amp_out[item.slot] = amp;
            });
        }
        const int hlog = hl_log(args);
        const size_t rows_per_slot = SLAB ? ((size_t)2 << hlog) : (size_t)N;
        if constexpr (JAC) {
            TEX* outd = reinterpret_cast<TEX*>(args.disp) + (size_t)item.slot * ((size_t)N * N);
            TEX* outn = reinterpret_cast<TEX*>(args.norm) + (size_t)item.slot * ((size_t)N * N);
            ex.each([&](int tid, ThreadState&) {
                const int ri = tid / GI, lt = tid % GI;
                const int mp = bx * RI + ri;
                const float2* l0 = smem + (ri * 4) * LS;
                const size_t ra = (size_t)mp * N, rb = (size_t)(mp == 0 ? H : N - mp) * N;
                pack_item_jac<GI>(l0, l0 + LS, l0 + 2 * LS, l0 + 3 * LS, mp, outd + ra, outd + rb, outn + ra, outn + rb,
                                  lambda, inv_amp, lt);
            });
            return;
        }
        TEX* out = reinterpret_cast<TEX*>(by == 0 ? args.disp : args.norm) + (size_t)item.slot * (rows_per_slot * N);
        ex.each([&](int tid, ThreadState&) {
            const int ri = tid / GI, lt = tid % GI;
            const int ml = bx * RI + ri;
            const int mp = (SLAB ? (args.slab_rank << hlog) : 0) + ml;
            const float2 *l0, *l1;
            int rows = 3;
            if constexpr (PAIR) {
                l0 = crank == 0 ? smem : smem_peer;
                l1 = crank == 0 ? smem_peer : smem;
                rows = crank == 0 ? 1 : 2;
            } else {
                l0 = smem + (ri * 2 + 0) * LS;
                l1 = l0 + LS;
            }
            TEX* outA = out + (size_t)(SLAB ? ml : mp) * N;
            TEX* outB = out + (size_t)(SLAB ? (1 << hlog) + ml : (mp == 0 ? H : N - mp)) * N;
            pack_item<GI>(l0, l1, mp, outA, outB, by, lambda, inv_amp, lt, rows);
        });
    }

    // one CTA holds whole row items (every size whose line pair fits shared memory)
    template <class Exec, class Args>
    static WSO_HD void run(Exec& ex, float2* smem, int bx, int by, int bz, const Args& args) {
        static_assert(!PAIR, "cluster pairs are driven phase by phase (transform / cluster barrier / pack)");
        transform(ex, smem, bx, by, bz, 0, args);
        if constexpr (HEIGHT_ONLY) {
            reduce_heights(ex, smem, bx, bz, args);
        } else {
            if constexpr (kPackFromRegs) {
                pack_from_regs(ex, smem, bx, by, bz, args);
            } else {
                // the pack phase of a row item reads both of its lines: barrier over that pair of line groups
                ex.template sync_group<GI, T>(1 + (G > 32 ? B : 0));
                pack(ex, smem, nullptr, bx, by, bz, 0, args);
            }
        }
    }

    template <class Exec, class Args>
    static WSO_HD void pack_from_regs(Exec& ex, float2* smem, int bx, int by, int bz, const Args& args) {
        constexpr int NSL = N / RLast, HALF = RLast / 2;
        constexpr int STEP = NSL + (NSL >> 4);  // pad(j + r*NSL) = pad(j) + r*STEP  (NSL % 16 == 0, j < NSL)
        using StL = Stage<N, B, RLast, NSL>;
        ex.each([&](int tid, ThreadState& st) {
            const int line = tid / G, j = tid % G;
            if (bx * RI + line / 2 == 0) {  // row item 0: whole lines, old route
                StL::store(smem, tid, st);
                return;
            }
            float2* y = smem + line * LS + pad_idx(j);
            if ((line & 1) == 0) {
#pragma unroll
                for (int r = HALF; r < RLast; ++r) y[r * STEP] = st.v[r];
            } else {
#pragma unroll
                for (int r = 0; r < HALF; ++r) y[r * STEP] = st.v[r];
            }
        });
        ex.template sync_group<GI, T>(1 + (G > 32 ? B : 0));
        const BatchItem item = args.items[bz];
        const bool needs_amp = by == 0;
        if (needs_amp) ex.pdl_wait();
        ex.pdl_release();
        const float lambda = args.td[bz].lambda;
        const float amp = needs_amp ? amplitude_of(args.minmax[2 * item.slot], args.minmax[2 * item.slot + 1]) : 1.0f;
        const float inv_amp = rdiv(1.0f, amp);
        if (bx == 0 && by == 0) {
            ex.each([&](int tid, ThreadState&) {
                if (tid == 0) args.amp_out[item.slot] = amp;
            });
        }
        TEX* out = reinterpret_cast<TEX*>(by == 0 ? args.disp : args.norm) + (size_t)item.slot * ((size_t)N * N);
        ex.each([&](int tid, ThreadState& st) {
            const int line = tid / G, j = tid % G;
            const int mp = bx * RI + line / 2;
            TEX* outA = out + (size_t)mp * N;
            TEX* outB = out + (size_t)(mp == 0 ? H : N - mp) * N;
            if (mp == 0) {
                const float2* l0 = smem + (line & ~1) * LS;
                pack_item<GI>(l0, l0 + LS, mp, outA, outB, by, lambda, inv_amp, tid % GI, 3);
                return;
            }
            const float2* yp = smem + (line ^ 1) * LS + pad_idx(j);
            // (-1)^(row+col): the columns j + r*NSL of a thread share the parity of j
            const float s = ((mp + j) & 1) ? -1.0f : 1.0f;
            const float sl = rmul(s, lambda);
            auto emit = [&](int c, float2 a0, float2 a1) {
                const int cm = (N - c) & (N - 1);  // row N-m' is the conjugate mirror of row m'
                if (by == 0) {
                    const float y = rmul(rmul(a0.x, s), inv_amp);
                    const float x = rmul(sl, a0.y), z = rmul(sl, a1.y);
                    st_texel(&outA[c], x, y, z, 1.0f);
                    st_texel(&outB[cm], -x, y, -z, 1.0f);
                } else {
                    const float4 ta = make_float4(s * a0.y, s * a1.y, s * a0.x, s * a1.x);
                    st_texel(&outA[c], ta.x, ta.y, ta.z, ta.w);
                    st_texel(&outB[cm], -ta.x, -ta.y, ta.z, ta.w);
                }
            };
            if ((line & 1) == 0) {  // this thread holds packed field 0 (or 2): columns r < HALF
#pragma unroll
                for (int r = 0; r < HALF; ++r) emit(j + r * NSL, st.v[r], yp[r * STEP]);
            } else {                // packed field 1 (or 3): columns r >= HALF
#pragma unroll
                for (int r = HALF; r < RLast; ++r) emit(j + r * NSL, yp[r * STEP], st.v[r]);
            }
        });
    }

    // Persistent form of K2 (batched launches, paired W layout): a fixed grid of CTAs walks the work items
    // w = cta, cta + ncta, ...; the first half of the item range is the normal map of every tile-frame (needs nothing
    // from K2h), the second half the displacement map - a CTA reaches its first displacement item, and only there waits
    // for K2h, after one or two normal-map items.  The W words of item w + ncta are requested before the pack phase of
    // item w (the 16 complex registers are free there): the L2 round trip that tops the stall list of the one-CTA-per-item
    // kernel (a third of its warp time, profiles/r2_ncu_c2.txt) overlaps the map stores.
    template <class Exec, class Args>
    static WSO_HD void run_persistent(Exec& ex, float2* smem, int cta, int ncta, int n_items, const Args& args) {
        static_assert(!HEIGHT_ONLY && !SLAB && !PAIR && !JAC && WLayout<LOGN>::paired, "persistent K2: paired layout, maps only");
        constexpr int GX = H / RI;
        const int half = GX * n_items, total = 2 * half;
        int w = cta;
        if (w >= total) {  // (the launch sizes the grid <= total)
            ex.pdl_wait();
            ex.pdl_release();
            return;
        }
        auto decode = [&](int wi, int& bx, int& by, int& bz) {
            by = wi < half ? 1 : 0;
            const int rem = wi < half ? wi : wi - half;
            bz = rem / GX;
            bx = rem - bz * GX;
        };
        int bx, by, bz;
        decode(w, bx, by, bz);
        if constexpr (Plan<LOGN>::S > 1) RunStages<LOGN, B, 1, R1st, Exec, false>::preload(ex, args.tw);
        ex.each([&](int tid, ThreadState& st) {
            first_load(tid, st, args.W + (size_t)bz * ((size_t)H * 4 * N), bx, by, 0);
        });
        bool waited = false;
        for (;;) {
            ex.each([&](int tid, ThreadState& st) { first_compute(tid, st, smem); });
            ex.template sync_group<G, T>(1);
            if constexpr (Plan<LOGN>::S > 1) RunStages<LOGN, B, 1, R1st, Exec, false>::run(ex, smem, args.tw);
            ex.template sync_group<GI, T>(1 + (G > 32 ? B : 0));
            const int wn = w + ncta;
            if (by == 0 && !waited) {
                ex.pdl_wait();
                waited = true;
            }
            if (wn >= total) ex.pdl_release();
            int bxn = 0, byn = 0, bzn = 0;
            if (wn < total) decode(wn, bxn, byn, bzn);
#ifndef WSO_EXP_P_NOAHEAD
            if (wn < total)
                ex.each([&](int tid, ThreadState& st) {
                    first_load(tid, st, args.W + (size_t)bzn * ((size_t)H * 4 * N), bxn, byn, 0);
                });
#endif
            pack_body(ex, smem, nullptr, bx, by, bz, 0, args);
#ifdef WSO_EXP_P_NOAHEAD
            if (wn < total)
                ex.each([&](int tid, ThreadState& st) {
                    first_load(tid, st, args.W + (size_t)bzn * ((size_t)H * 4 * N), bxn, byn, 0);
                });
#endif
            if (wn >= total) break;
            // the lines of a row item are rewritten by the threads of that item only
            ex.template sync_group<GI, T>(1 + (G > 32 ? B : 0));
            w = wn; bx = bxn; by = byn; bz = bzn;
        }
    }
};

}  // namespace wso
