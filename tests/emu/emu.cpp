// TEST INFRASTRUCTURE — CPU emulation of the CUDA kernel bodies.
//
// Compiles watersurfacerendering_b200/csrc/wso_kernels.cuh with g++ and steps every CTA thread by thread
// (HostExec) so that the index / Hermitian-layout logic of the sm_100a kernels can be checked against the
// oracle in the GPU-less build container.  Never linked into the product library; tests only.
#include <cstdio>
#include <cstring>
#include <vector>

#include "wso_kernels.cuh"
#include "wso_tilings.h"

using namespace wso;

// JAC: the Jacobian-channel kernels (SURVEY row f-4): K1's general body with field 1's real slot filled, K2 with four
// lines per CTA (by = 0 only).
// PERSIST: bit 0 = K1, bit 2 = K2 through their persistent forms (run_persistent: a few emulated CTAs walk the work items,
// each with its own shared memory and thread states that live across items - the prefetched inputs of the next item
// sit in them while the current item is stored)
template <int LOGN, int CP, int NF, int RI, bool JAC = false, int PERSIST = 0>
static int run_cfg(const float* amp_t, const float* omega_t, const float* kv, float omega0, float lambda,
                   float t, float* disp, float* norm, float* minmax, float* amp_out, float* w_out) {
    constexpr int N = 1 << LOGN, H = N / 2;
    using P1 = Pass1<LOGN, CP, NF, false, false, JAC>;
    using P2 = Pass2<LOGN, JAC ? 1 : RI, false, false, false, JAC>;
    using PH = Pass2<LOGN, RI, true>;
    constexpr int RI2 = JAC ? 1 : RI;
    std::vector<float2> tw(N);
    for (int k = 0; k < N; ++k) {
        const double a = 2.0 * 3.14159265358979323846 * k / N;
        tw[k] = make_float2((float)cos(a), (float)sin(a));
    }
    // same record / table decision as upload_h0() in wso_api.cu (omega0 <= 0: force the direct sincos path)
    std::vector<float4> rec((size_t)N * N);
    int jmax = 0;
    bool table_ok = omega0 > 0.0f;
    for (size_t i = 0; i < (size_t)N * N && table_ok; ++i) {
        const float jf = std::nearbyint(omega_t[i] / omega0);
        if (!(jf >= 0.0f && jf < (float)kMaxTable) || jf * omega0 != omega_t[i]) table_ok = false;
        else if ((int)jf > jmax) jmax = (int)jf;
    }
    for (int n = 0; n < N; ++n)
        for (int m = 0; m < N; ++m) {
            const size_t i = (size_t)n * N + m;
            const float d = kv[n] * kv[n] + kv[m] * kv[m];
            const float inv = std::sqrt(d) > 0.00001f ? 1.0f / std::sqrt(d) : 0.0f;
            float wf = omega_t[i];
            if (table_ok) {
                const int j = (int)std::nearbyint(omega_t[i] / omega0);
                std::memcpy(&wf, &j, 4);
            }
            rec[h0_index(n, m, N, 0)] = make_float4(amp_t[2 * i], amp_t[2 * i + 1], inv, wf);
        }
    const int hN = N / 2;
    std::vector<float4> recs((size_t)hN * hN * 2, make_float4(0.f, 0.f, 0.f, 0.f));
    bool pairs_ok = true;
    for (int j = 1; j < hN; ++j)
        for (int i = 1; i < hN; ++i) {
            const float4 a0 = rec[h0_index(j, i, N, 0)], a3 = rec[h0_index(N - j, N - i, N, 0)];
            const float4 a1 = rec[h0_index(N - j, i, N, 0)], a2 = rec[h0_index(j, N - i, N, 0)];
            if (std::memcmp(&a0.w, &a3.w, 4) != 0 || std::memcmp(&a1.w, &a2.w, 4) != 0) pairs_ok = false;
            recs[hs_index((int)j, (int)i, 0, (int)hN)] = make_float4(a0.x + a3.x, a0.y + a3.y, a0.z, a0.w);
            recs[hs_index((int)j, (int)i, 1, (int)hN)] = make_float4(a1.x + a2.x, a1.y + a2.y, a1.z, a1.w);
        }
    TileDev td;
    td.h0 = rec.data();
    td.hs = recs.data();
    td.kv = kv;
    td.lambda = lambda;
    td.omega0 = omega0;
    td.table_len = table_ok ? jmax + 1 : 0;
    td.use_pairs = pairs_ok ? 1 : 0;
    td.j0 = 0;
    std::vector<float2> W((size_t)H * 4 * N);
    LaunchArgs args;
    std::memset(&args, 0, sizeof(args));
    args.td[0] = td;
    args.tw = tw.data();
    args.W = W.data();
    args.disp = reinterpret_cast<float4*>(disp);
    args.norm = reinterpret_cast<float4*>(norm);
    args.minmax = minmax;
    args.amp_out = amp_out;
    args.items[0].tile = 0;
    args.items[0].slot = 0;
    args.items[0].t = t;
    {
        // same choice as launch_tiled() in wso_kernels.cu: the lean instantiation when every item qualifies
        using P1F = Pass1<LOGN, CP, NF, false, true>;
        const bool fast = !JAC && td.table_len > 0 && td.use_pairs != 0;
        std::vector<float2> smem(P1::SMEM_BYTES / sizeof(float2));
        std::vector<ThreadState> st(P1::T);
        if constexpr ((PERSIST & 1) != 0) {
            if (!fast) return -2;
            const int ncta = 5;
            for (int cta = 0; cta < ncta; ++cta) {
                for (auto& v : smem) v = make_float2(NAN, NAN);
                for (auto& x : st) for (auto& v : x.v) v = make_float2(NAN, NAN);
                HostExec ex{P1::T, st.data()};
                P1F::run_persistent(ex, smem.data(), cta, ncta, 1, args);
            }
        } else {
        for (int by = 0; by < 4 / NF; ++by)
            for (int bx = 0; bx < H / CP; ++bx) {
                for (auto& v : smem) v = make_float2(NAN, NAN);
                HostExec ex{P1::T, st.data()};
                if (fast) P1F::run(ex, smem.data(), bx, by, 0, args);
                else P1::run(ex, smem.data(), bx, by, 0, args);
            }
        }
    }
    if (w_out) std::memcpy(w_out, W.data(), W.size() * sizeof(float2));
    {   // K2h: height extrema
        std::vector<float2> smem(PH::SMEM_BYTES / sizeof(float2));
        std::vector<ThreadState> st(PH::T);
        for (int bx = 0; bx < PH::grid_x(); ++bx) {
            for (auto& v : smem) v = make_float2(NAN, NAN);
            HostExec ex{PH::T, st.data()};
            PH::run(ex, smem.data(), bx, 0, 0, args);
        }
    }
    {
        std::vector<float2> smem(P2::SMEM_BYTES / sizeof(float2));
        std::vector<ThreadState> st(P2::T);
        if constexpr ((PERSIST & 4) != 0) {
            const int ncta = 7;
            for (int cta = 0; cta < ncta; ++cta) {
                for (auto& v : smem) v = make_float2(NAN, NAN);
                for (auto& x : st) for (auto& v : x.v) v = make_float2(NAN, NAN);
                HostExec ex{P2::T, st.data()};
                P2::run_persistent(ex, smem.data(), cta, ncta, 1, args);
            }
        } else {
        for (int by = 0; by < (JAC ? 1 : 2); ++by)
            for (int bx = 0; bx < H / RI2; ++bx) {
                for (auto& v : smem) v = make_float2(NAN, NAN);
                HostExec ex{P2::T, st.data()};
                P2::run(ex, smem.data(), bx, by, 0, args);
            }
        }
    }
    return 0;
}

// Slab decomposition over P = 2^shift emulated devices (all in this process): every rank runs K1 on its column pairs
// and writes the blocks of the row owners directly (the fused peer-store mode), then K2h, a min/max reduction over
// ranks, and K2 on its rows; the local rows are scattered back to full maps for comparison.  PAIR = the cluster-pair
// variant of K2 (two CTAs, one line each, partner line through "distributed shared memory").
template <int LOGN, int CP, int NF, int RI, bool PAIR>
static int run_slab_cfg(int shift, const float* amp_t, const float* omega_t, const float* kv, float omega0, float lambda,
                        float t, float* disp, float* norm, float* minmax, float* amp_out) {
    constexpr int N = 1 << LOGN, H = N / 2;
    const int P = 1 << shift, Hl = H >> shift;
    using P1 = Pass1<LOGN, CP, NF, true>;
    using P2 = Pass2<LOGN, RI, false, true, PAIR>;
    using PH = Pass2<LOGN, RI, true, true, false>;
    if (Hl % CP != 0 || Hl % RI != 0) return -2;
    std::vector<float2> tw(N);
    for (int k = 0; k < N; ++k) {
        const double a = 2.0 * 3.14159265358979323846 * k / N;
        tw[k] = make_float2((float)cos(a), (float)sin(a));
    }
    int jmax = 0;
    bool table_ok = omega0 > 0.0f;
    for (size_t i = 0; i < (size_t)N * N && table_ok; ++i) {
        const float jf = std::nearbyint(omega_t[i] / omega0);
        if (!(jf >= 0.0f && jf < (float)kMaxTable) || jf * omega0 != omega_t[i]) table_ok = false;
        else if ((int)jf > jmax) jmax = (int)jf;
    }
    auto record = [&](int n, int m) {
        const size_t i = (size_t)n * N + m;
        const float d = kv[n] * kv[n] + kv[m] * kv[m];
        const float inv = std::sqrt(d) > 0.00001f ? 1.0f / std::sqrt(d) : 0.0f;
        float wf = omega_t[i];
        if (table_ok) {
            const int j = (int)std::nearbyint(omega_t[i] / omega0);
            std::memcpy(&wf, &j, 4);
        }
        return make_float4(amp_t[2 * i], amp_t[2 * i + 1], inv, wf);
    };
    const size_t blk = (size_t)Hl * 4 * 2 * Hl;
    std::vector<std::vector<float2>> recv(P, std::vector<float2>(blk * P, make_float2(NAN, NAN)));
    std::vector<std::vector<float4>> rec(P), recs(P);
    std::vector<TileDev> tds(P);
    for (int r = 0; r < P; ++r) {
        const int j0 = r * Hl;
        rec[r].assign((size_t)2 * Hl * N, make_float4(0.f, 0.f, 0.f, 0.f));
        recs[r].assign((size_t)Hl * H * 2, make_float4(0.f, 0.f, 0.f, 0.f));
        for (int jl = 0; jl < Hl; ++jl) {
            const int j = j0 + jl;
            const int nA = j, nB = (j == 0) ? H : N - j;
            for (int m = 0; m < N; ++m) {
                rec[r][h0_index(nA, m, N, j0)] = record(nA, m);
                rec[r][h0_index(nB, m, N, j0)] = record(nB, m);
            }
            if (j == 0) continue;
            for (int i = 1; i < H; ++i) {
                const float4 a0 = record(j, i), a3 = record(N - j, N - i), a1 = record(N - j, i), a2 = record(j, N - i);
                recs[r][hs_index((int)jl, (int)i, 0, (int)H)] = make_float4(a0.x + a3.x, a0.y + a3.y, a0.z, a0.w);
                recs[r][hs_index((int)jl, (int)i, 1, (int)H)] = make_float4(a1.x + a2.x, a1.y + a2.y, a1.z, a1.w);
            }
        }
        TileDev& td = tds[r];
        td.h0 = rec[r].data();
        td.hs = recs[r].data();
        td.kv = kv;
        td.lambda = lambda;
        td.omega0 = omega0;
        td.table_len = table_ok ? jmax + 1 : 0;
        td.use_pairs = 1;
        td.j0 = j0;
    }
    std::vector<std::vector<float4>> ldisp(P, std::vector<float4>((size_t)2 * Hl * N)), lnorm(P, std::vector<float4>((size_t)2 * Hl * N));
    std::vector<float> lmm((size_t)2 * P), lamp(P);
    auto make_args = [&](int r) {
        LaunchArgs a;
        std::memset(&a, 0, sizeof(a));
        a.tw = tw.data();
        a.W = recv[r].data();
        a.disp = ldisp[r].data();
        a.norm = lnorm[r].data();
        a.minmax = &lmm[2 * r];
        a.amp_out = &lamp[r];
        a.slab_shift = shift;
        a.slab_rank = r;
        for (int d = 0; d < P; ++d) a.Wdst[d] = recv[d].data() + (size_t)r * blk;
        a.items[0].tile = 0;
        a.items[0].slot = 0;
        a.items[0].t = t;
        a.td[0] = tds[r];
        return a;
    };
    for (int r = 0; r < P; ++r) {  // K1 everywhere (stores land in the owners' receive buffers)
        LaunchArgs args = make_args(r);
        std::vector<float2> smem(P1::SMEM_BYTES / sizeof(float2));
        std::vector<ThreadState> st(P1::T);
        for (int by = 0; by < 4 / NF; ++by)
            for (int bx = 0; bx < Hl / CP; ++bx) {
                for (auto& v : smem) v = make_float2(NAN, NAN);
                HostExec ex{P1::T, st.data()};
                P1::run(ex, smem.data(), bx, by, 0, args);
            }
    }
    float gmin = kInitMin, gmax = kInitMax;
    for (int r = 0; r < P; ++r) {  // K2h + reduction over ranks
        LaunchArgs args = make_args(r);
        std::vector<float2> smem(PH::SMEM_BYTES / sizeof(float2));
        std::vector<ThreadState> st(PH::T);
        for (int bx = 0; bx < Hl / RI; ++bx) {
            for (auto& v : smem) v = make_float2(NAN, NAN);
            HostExec ex{PH::T, st.data()};
            PH::run(ex, smem.data(), bx, 0, 0, args);
        }
        if (lmm[2 * r] < gmin) gmin = lmm[2 * r];
        if (lmm[2 * r + 1] > gmax) gmax = lmm[2 * r + 1];
    }
    for (int r = 0; r < P; ++r) {
        lmm[2 * r] = gmin;
        lmm[2 * r + 1] = gmax;
    }
    for (int r = 0; r < P; ++r) {  // K2
        LaunchArgs args = make_args(r);
        std::vector<ThreadState> st(P2::T);
        for (int by = 0; by < 2; ++by)
            for (int bx = 0; bx < Hl / RI; ++bx) {
                if constexpr (PAIR) {
                    std::vector<float2> sm0(P2::SMEM_BYTES / sizeof(float2), make_float2(NAN, NAN)), sm1(sm0);
                    HostExec ex{P2::T, st.data()};
                    P2::transform(ex, sm0.data(), bx, by, 0, 0, args);
                    P2::transform(ex, sm1.data(), bx, by, 0, 1, args);
                    P2::pack(ex, sm0.data(), sm1.data(), bx, by, 0, 0, args);
                    P2::pack(ex, sm1.data(), sm0.data(), bx, by, 0, 1, args);
                } else {
                    std::vector<float2> smem(P2::SMEM_BYTES / sizeof(float2), make_float2(NAN, NAN));
                    HostExec ex{P2::T, st.data()};
                    P2::run(ex, smem.data(), bx, by, 0, args);
                }
            }
        // local rows -> global rows
        for (int ml = 0; ml < Hl; ++ml) {
            const int mp = r * Hl + ml;
            const int rowA = mp, rowB = (mp == 0) ? H : N - mp;
            std::memcpy(disp + (size_t)rowA * N * 4, &ldisp[r][(size_t)ml * N], sizeof(float4) * N);
            std::memcpy(disp + (size_t)rowB * N * 4, &ldisp[r][(size_t)(Hl + ml) * N], sizeof(float4) * N);
            std::memcpy(norm + (size_t)rowA * N * 4, &lnorm[r][(size_t)ml * N], sizeof(float4) * N);
            std::memcpy(norm + (size_t)rowB * N * 4, &lnorm[r][(size_t)(Hl + ml) * N], sizeof(float4) * N);
        }
    }
    minmax[0] = gmin;
    minmax[1] = gmax;
    amp_out[0] = lamp[0];
    return 0;
}

// One phase of ONE rank of the slab path in its unfused form (K1 fills the send blocks; the caller transposes them
// with an all-to-all) - lets the CPU tests drive the real multi-process orchestration over gloo.
//   phase 0: K1 -> send[world][blk]     1: K2h(recv) -> minmax[2]     2: K2(recv, minmax) -> ldisp/lnorm [2*Hl][N]
template <int LOGN, int CP, int NF, int RI, bool PAIR>
static int slab_rank_phase(int shift, int rank, int phase, const float* amp_t, const float* omega_t, const float* kv,
                           float omega0, float lambda, float t, float* send, float* recv, float* minmax, float* ldisp,
                           float* lnorm, float* amp_out) {
    constexpr int N = 1 << LOGN, H = N / 2;
    const int P = 1 << shift, Hl = H >> shift, j0 = rank * Hl;
    using P1 = Pass1<LOGN, CP, NF, true>;
    using P2 = Pass2<LOGN, RI, false, true, PAIR>;
    using PH = Pass2<LOGN, RI, true, true, false>;
    if (Hl % CP != 0 || Hl % RI != 0) return -2;
    std::vector<float2> tw(N);
    for (int k = 0; k < N; ++k) {
        const double a = 2.0 * 3.14159265358979323846 * k / N;
        tw[k] = make_float2((float)cos(a), (float)sin(a));
    }
    int jmax = 0;
    for (size_t i = 0; i < (size_t)N * N; ++i) {
        const int j = (int)std::nearbyint(omega_t[i] / omega0);
        if (j > jmax) jmax = j;
    }
    auto record = [&](int n, int m) {
        const size_t i = (size_t)n * N + m;
        const float d = kv[n] * kv[n] + kv[m] * kv[m];
        const float inv = std::sqrt(d) > 0.00001f ? 1.0f / std::sqrt(d) : 0.0f;
        const int j = (int)std::nearbyint(omega_t[i] / omega0);
        float wf;
        std::memcpy(&wf, &j, 4);
        return make_float4(amp_t[2 * i], amp_t[2 * i + 1], inv, wf);
    };
    std::vector<float4> rec((size_t)2 * Hl * N), recs((size_t)Hl * H * 2, make_float4(0.f, 0.f, 0.f, 0.f));
    if (phase == 0)
        for (int jl = 0; jl < Hl; ++jl) {
            const int j = j0 + jl;
            const int nA = j, nB = (j == 0) ? H : N - j;
            for (int m = 0; m < N; ++m) {
                rec[h0_index(nA, m, N, j0)] = record(nA, m);
                rec[h0_index(nB, m, N, j0)] = record(nB, m);
            }
            if (j == 0) continue;
            for (int i = 1; i < H; ++i) {
                const float4 a0 = record(j, i), a3 = record(N - j, N - i), a1 = record(N - j, i), a2 = record(j, N - i);
                recs[hs_index((int)jl, (int)i, 0, (int)H)] = make_float4(a0.x + a3.x, a0.y + a3.y, a0.z, a0.w);
                recs[hs_index((int)jl, (int)i, 1, (int)H)] = make_float4(a1.x + a2.x, a1.y + a2.y, a1.z, a1.w);
            }
        }
    TileDev td;
    td.h0 = rec.data();
    td.hs = recs.data();
    td.kv = kv;
    td.lambda = lambda;
    td.omega0 = omega0;
    td.table_len = jmax + 1;
    td.use_pairs = 1;
    td.j0 = j0;
    const size_t blk = (size_t)Hl * 4 * 2 * Hl;
    LaunchArgs args;
    std::memset(&args, 0, sizeof(args));
    args.tw = tw.data();
    args.W = reinterpret_cast<float2*>(recv);
    args.disp = reinterpret_cast<float4*>(ldisp);
    args.norm = reinterpret_cast<float4*>(lnorm);
    args.minmax = minmax;
    args.amp_out = amp_out;
    args.slab_shift = shift;
    args.slab_rank = rank;
    for (int d = 0; d < P; ++d) args.Wdst[d] = reinterpret_cast<float2*>(send) + (size_t)d * blk;
    args.items[0].t = t;
    args.td[0] = td;
    if (phase == 0) {
        std::vector<float2> smem(P1::SMEM_BYTES / sizeof(float2));
        std::vector<ThreadState> st(P1::T);
        for (int by = 0; by < 4 / NF; ++by)
            for (int bx = 0; bx < Hl / CP; ++bx) {
                for (auto& v : smem) v = make_float2(NAN, NAN);
                HostExec ex{P1::T, st.data()};
                P1::run(ex, smem.data(), bx, by, 0, args);
            }
    } else if (phase == 1) {
        std::vector<float2> smem(PH::SMEM_BYTES / sizeof(float2));
        std::vector<ThreadState> st(PH::T);
        for (int bx = 0; bx < Hl / RI; ++bx) {
            for (auto& v : smem) v = make_float2(NAN, NAN);
            HostExec ex{PH::T, st.data()};
            PH::run(ex, smem.data(), bx, 0, 0, args);
        }
    } else {
        std::vector<ThreadState> st(P2::T);
        for (int by = 0; by < 2; ++by)
            for (int bx = 0; bx < Hl / RI; ++bx) {
                if constexpr (PAIR) {
                    std::vector<float2> sm0(P2::SMEM_BYTES / sizeof(float2), make_float2(NAN, NAN)), sm1(sm0);
                    HostExec ex{P2::T, st.data()};
                    P2::transform(ex, sm0.data(), bx, by, 0, 0, args);
                    P2::transform(ex, sm1.data(), bx, by, 0, 1, args);
                    P2::pack(ex, sm0.data(), sm1.data(), bx, by, 0, 0, args);
                    P2::pack(ex, sm1.data(), sm0.data(), bx, by, 0, 1, args);
                } else {
                    std::vector<float2> smem(P2::SMEM_BYTES / sizeof(float2), make_float2(NAN, NAN));
                    HostExec ex{P2::T, st.data()};
                    P2::run(ex, smem.data(), bx, by, 0, args);
                }
            }
    }
    return 0;
}

extern "C" int wso_emu_slab_rank_phase(int logn, int variant, int shift, int rank, int phase, const float* amp_t,
                                       const float* omega_t, const float* kv, float omega0, float lambda, float t,
                                       float* send, float* recv, float* minmax, float* ldisp, float* lnorm,
                                       float* amp_out) {
#define RCFG(L, V, CP, NF, RI, PAIR) \
    if (logn == L && variant == V) return slab_rank_phase<L, CP, NF, RI, PAIR>(shift, rank, phase, amp_t, omega_t, kv, omega0, lambda, t, send, recv, minmax, ldisp, lnorm, amp_out);
    RCFG(6, 0, 2, 2, 2, false)
    RCFG(6, 1, 1, 1, 1, true)
#undef RCFG
    return -1;
}

extern "C" int wso_emu_compute_slab(int logn, int variant, int shift, const float* amp_t, const float* omega_t,
                                    const float* kv, float omega0, float lambda, float t, float* disp, float* norm,
                                    float* minmax, float* amp_out) {
#define SCFG(L, V, CP, NF, RI, PAIR) \
    if (logn == L && variant == V) return run_slab_cfg<L, CP, NF, RI, PAIR>(shift, amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out);
    SCFG(6, 0, 2, 2, 2, false)
    SCFG(6, 1, 1, 1, 1, true)
    SCFG(8, 0, 4, 2, 2, false)
    SCFG(8, 1, 1, 1, 1, true)
#undef SCFG
    return -1;
}

extern "C" int wso_emu_compute(int logn, int variant, const float* amp_t, const float* omega_t,
                               const float* kv, float omega0, float lambda, float t, float* disp, float* norm,
                               float* minmax, float* amp_out, float* w_out) {
#define CFG(L, V, CP, NF, RI) \
    if (logn == L && variant == V) return run_cfg<L, CP, NF, RI>(amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out, w_out);
    CFG(4, 0, 8, 4, 8)
    CFG(4, 1, 2, 1, 1)
    CFG(5, 0, 8, 4, 8)
    CFG(6, 0, 8, 4, 8)
    CFG(6, 1, 4, 2, 2)
    CFG(6, 2, 1, 1, 1)
    CFG(7, 0, 4, 4, 8)
    CFG(8, 0, 4, 4, 4)
    CFG(8, 1, 4, 2, 2)
    CFG(9, 0, 4, 4, 4)
    CFG(9, 1, 4, 2, 2)
    CFG(10, 0, 4, 2, 4)
    CFG(11, 0, 4, 1, 2)
#undef CFG
    // variants 200+: the persistent forms of K1 / K2 (the tilings batched launches run)
#define PCFG(L, V, CP, NF, RI, PM) \
    if (logn == L && variant == 200 + V) return run_cfg<L, CP, NF, RI, false, PM>(amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out, w_out);
    PCFG(9, 0, 4, 4, 1, 5)
    PCFG(9, 1, 4, 4, 1, 1)
    PCFG(10, 0, 4, 2, 2, 5)
    PCFG(10, 1, 4, 2, 2, 4)
    PCFG(11, 0, 4, 2, 1, 5)
#undef PCFG
    // variants 100+: the Jacobian-channel kernels with the same K1 / K2h tilings
#define JCFG(L, V, CP, NF, RI) \
    if (logn == L && variant == 100 + V) return run_cfg<L, CP, NF, RI, true>(amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out, w_out);
    JCFG(4, 0, 8, 4, 8)
    JCFG(6, 1, 4, 2, 2)
    JCFG(8, 0, 4, 4, 4)
    JCFG(9, 0, 4, 4, 4)
    JCFG(10, 0, 4, 2, 4)
#undef JCFG
    return -1;
}

// ---------------------------------------------------------------------------------------------------------------------
// The tilings the library ships (wso_tilings.h), run as launch_tiled() / launch_tiled_jacobian() in wso_kernels.cu run
// them: one launch of n_items tile-frames, item i with its own spectrum, wave numbers, lambda and time, written to slot i.
// ---------------------------------------------------------------------------------------------------------------------

// Same records, table and pair decision as upload_h0() in wso_api.cu; returns the tile constants.
static TileDev make_tile(int N, const float* amp_t, const float* omega_t, const float* kv, float omega0, float lambda,
                         std::vector<float4>& rec, std::vector<float4>& recs) {
    const size_t n2 = (size_t)N * N;
    int jmax = 0;
    bool table_ok = omega0 > 0.0f;
    for (size_t i = 0; i < n2 && table_ok; ++i) {
        const float jf = std::nearbyint(omega_t[i] / omega0);
        if (!(jf >= 0.0f && jf < (float)kMaxTable) || jf * omega0 != omega_t[i]) table_ok = false;
        else if ((int)jf > jmax) jmax = (int)jf;
    }
    rec.assign(n2, make_float4(0.f, 0.f, 0.f, 0.f));
    for (int n = 0; n < N; ++n)
        for (int m = 0; m < N; ++m) {
            const size_t i = (size_t)n * N + m;
            const float d = kv[n] * kv[n] + kv[m] * kv[m];
            const float inv = std::sqrt(d) > 0.00001f ? 1.0f / std::sqrt(d) : 0.0f;
            float wf = omega_t[i];
            if (table_ok) {
                const int j = (int)std::nearbyint(omega_t[i] / omega0);
                std::memcpy(&wf, &j, 4);
            }
            rec[h0_index(n, m, N, 0)] = make_float4(amp_t[2 * i], amp_t[2 * i + 1], inv, wf);
        }
    const int hN = N / 2;
    recs.assign((size_t)hN * hN * 2, make_float4(0.f, 0.f, 0.f, 0.f));
    bool pairs_ok = true;
    for (int j = 1; j < hN; ++j)
        for (int i = 1; i < hN; ++i) {
            const float4 a0 = rec[h0_index(j, i, N, 0)], a3 = rec[h0_index(N - j, N - i, N, 0)];
            const float4 a1 = rec[h0_index(N - j, i, N, 0)], a2 = rec[h0_index(j, N - i, N, 0)];
            if (std::memcmp(&a0.w, &a3.w, 4) != 0 || std::memcmp(&a1.w, &a2.w, 4) != 0) pairs_ok = false;
            recs[hs_index(j, i, 0, hN)] = make_float4(a0.x + a3.x, a0.y + a3.y, a0.z, a0.w);
            recs[hs_index(j, i, 1, hN)] = make_float4(a1.x + a2.x, a1.y + a2.y, a1.z, a1.w);
        }
    TileDev td;
    std::memset(&td, 0, sizeof(td));
    td.h0 = rec.data();
    td.hs = recs.data();
    td.kv = kv;
    td.lambda = lambda;
    td.omega0 = omega0;
    td.table_len = table_ok ? jmax + 1 : 0;
    td.use_pairs = pairs_ok ? 1 : 0;
    td.j0 = 0;
    return td;
}

// PERSIST: bit 0 = K1, bit 2 = K2 in their persistent forms, taken - as in launch_tiled() - only where PersistOk allows
// them and every item has the table and the pair records.  JAC: launch_tiled_jacobian() (general K1, one row item per K2
// CTA).  amp_t / omega_t / kv: [n_items] consecutive arrays of the layout wso_emu_compute takes.
template <int LOGN, class TL, bool JAC, int PERSIST, class TEX>
static int run_launch(int n_items, const float* amp_t, const float* omega_t, const float* kv, const float* omega0,
                      const float* lambda, const float* t, void* disp, void* norm, float* minmax, float* amp_out,
                      float* w_out) {
    constexpr int N = 1 << LOGN, H = N / 2;
    const size_t n2 = (size_t)N * N;
    if (n_items < 1 || n_items > LaunchArgs::kCap) return -3;
    using P1 = Pass1<LOGN, TL::CP, TL::NF, false, false, JAC>;
    using P1F = Pass1<LOGN, TL::CP, TL::NF, false, true>;
    using P2 = Pass2<LOGN, JAC ? 1 : TL::RI, false, false, false, JAC, TEX>;
    using PH = Pass2<LOGN, TL::RH, true>;
    constexpr int RI2 = JAC ? 1 : TL::RI;
    std::vector<float2> tw(N);
    for (int k = 0; k < N; ++k) {
        const double a = 2.0 * 3.14159265358979323846 * k / N;
        tw[k] = make_float2((float)cos(a), (float)sin(a));
    }
    std::vector<std::vector<float4>> rec(n_items), recs(n_items);
    std::vector<float2> W((size_t)n_items * H * 4 * N);
    LaunchArgs args;
    std::memset(&args, 0, sizeof(args));
    bool fast = !JAC;
    for (int i = 0; i < n_items; ++i) {
        args.td[i] = make_tile(N, amp_t + 2 * n2 * i, omega_t + n2 * i, kv + (size_t)N * i, omega0[i], lambda[i], rec[i], recs[i]);
        fast = fast && args.td[i].table_len > 0 && args.td[i].use_pairs != 0;
        args.items[i].tile = (uint32_t)i;
        args.items[i].slot = (uint32_t)i;
        args.items[i].t = t[i];
    }
    args.tw = tw.data();
    args.W = W.data();
    args.disp = reinterpret_cast<float4*>(disp);
    args.norm = reinterpret_cast<float4*>(norm);
    args.minmax = minmax;
    args.amp_out = amp_out;
    constexpr bool p1 = (PERSIST & 1) && PersistOk<LOGN, TL>::k1, p2 = (PERSIST & 4) && PersistOk<LOGN, TL>::k2;
    {   // K1
        std::vector<float2> smem(P1::SMEM_BYTES / sizeof(float2));
        std::vector<ThreadState> st(P1::T);
        if (p1 && fast) {
            if constexpr (p1) {
                const int ncta = 5;
                for (int cta = 0; cta < ncta; ++cta) {
                    for (auto& v : smem) v = make_float2(NAN, NAN);
                    for (auto& x : st) for (auto& v : x.v) v = make_float2(NAN, NAN);
                    HostExec ex{P1::T, st.data()};
                    P1F::run_persistent(ex, smem.data(), cta, ncta, n_items, args);
                }
            }
        } else {
            for (int bz = 0; bz < n_items; ++bz)
                for (int by = 0; by < 4 / TL::NF; ++by)
                    for (int bx = 0; bx < H / TL::CP; ++bx) {
                        for (auto& v : smem) v = make_float2(NAN, NAN);
                        HostExec ex{P1::T, st.data()};
                        if (fast) P1F::run(ex, smem.data(), bx, by, bz, args);
                        else P1::run(ex, smem.data(), bx, by, bz, args);
                    }
        }
    }
    if (w_out) std::memcpy(w_out, W.data(), W.size() * sizeof(float2));
    {   // K2h: height extrema
        std::vector<float2> smem(PH::SMEM_BYTES / sizeof(float2));
        std::vector<ThreadState> st(PH::T);
        for (int bz = 0; bz < n_items; ++bz)
            for (int bx = 0; bx < PH::grid_x(); ++bx) {
                for (auto& v : smem) v = make_float2(NAN, NAN);
                HostExec ex{PH::T, st.data()};
                PH::run(ex, smem.data(), bx, 0, bz, args);
            }
    }
    {   // K2
        std::vector<float2> smem(P2::SMEM_BYTES / sizeof(float2));
        std::vector<ThreadState> st(P2::T);
        if (p2 && fast) {
            if constexpr (p2) {
                const int ncta = 7;
                for (int cta = 0; cta < ncta; ++cta) {
                    for (auto& v : smem) v = make_float2(NAN, NAN);
                    for (auto& x : st) for (auto& v : x.v) v = make_float2(NAN, NAN);
                    HostExec ex{P2::T, st.data()};
                    P2::run_persistent(ex, smem.data(), cta, ncta, n_items, args);
                }
            }
        } else {
            for (int bz = 0; bz < n_items; ++bz)
                for (int by = 0; by < (JAC ? 1 : 2); ++by)
                    for (int bx = 0; bx < H / RI2; ++bx) {
                        for (auto& v : smem) v = make_float2(NAN, NAN);
                        HostExec ex{P2::T, st.data()};
                        P2::run(ex, smem.data(), bx, by, bz, args);
                    }
        }
    }
    return 0;
}

// kind: 0 = Cfg<L>::Lat, 1 = Cfg<L>::Bulk, 2 = Bulk with the persistent K1 and K2 where PersistOk allows them,
// 3 = the Jacobian launch (Bulk tiling).  Sizes 16^2 ... 2048^2.
enum { kEmuLat = 0, kEmuBulk = 1, kEmuPersist = 2, kEmuJacobian = 3, kEmuKinds = 4 };
constexpr int kEmuMinLogN = 4, kEmuMaxLogN = 11;

template <int LOGN, class TEX>
static int shipped(int kind, int n_items, const float* amp_t, const float* omega_t, const float* kv, const float* omega0,
                   const float* lambda, const float* t, void* disp, void* norm, float* minmax, float* amp_out, float* w_out) {
    using B = typename Cfg<LOGN>::Bulk;
    using L = typename Cfg<LOGN>::Lat;
    switch (kind) {
        case kEmuLat: return run_launch<LOGN, L, false, 0, TEX>(n_items, amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out, w_out);
        case kEmuBulk: return run_launch<LOGN, B, false, 0, TEX>(n_items, amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out, w_out);
        case kEmuPersist:
            if (!(PersistOk<LOGN, B>::k1 || PersistOk<LOGN, B>::k2)) return -1;
            return run_launch<LOGN, B, false, 5, TEX>(n_items, amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out, w_out);
        case kEmuJacobian: return run_launch<LOGN, B, true, 0, TEX>(n_items, amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out, w_out);
        default: return -1;
    }
}

// half = 0: disp / norm receive [n_items][N*N] RGBA32F texels, half = 1: RGBA16F texels (4 x binary16).
extern "C" int wso_emu_compute_shipped(int logn, int kind, int half, int n_items, const float* amp_t, const float* omega_t,
                                       const float* kv, const float* omega0, const float* lambda, const float* t,
                                       void* disp, void* norm, float* minmax, float* amp_out, float* w_out) {
#define SHIP(L)                                                                                                              \
    if (logn == L)                                                                                                       \
        return half ? shipped<L, Half4>(kind, n_items, amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out, w_out) \
                    : shipped<L, float4>(kind, n_items, amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out, w_out);
    SHIP(4) SHIP(5) SHIP(6) SHIP(7) SHIP(8) SHIP(9) SHIP(10) SHIP(11)
#undef SHIP
    return -1;
}

// The tilings launch_all() can pick, from the same header as the library.  Row r = 7 ints: logn, kind (0 = Lat,
// 1 = Bulk), CP, NF, RI, RH, persistent forms of Bulk (bit 0 = K1, bit 2 = K2).  Returns the row count (two per size,
// logn 4 ... 13; wso_emu_compute_shipped runs logn 4 ... 11 of them).
template <int LOGN>
static int tiling_rows(int* out) {
    using B = typename Cfg<LOGN>::Bulk;
    using L = typename Cfg<LOGN>::Lat;
    const int pm = (PersistOk<LOGN, B>::k1 ? 1 : 0) | (PersistOk<LOGN, B>::k2 ? 4 : 0);
    const int rows[2][7] = {{LOGN, 0, L::CP, L::NF, L::RI, L::RH, 0}, {LOGN, 1, B::CP, B::NF, B::RI, B::RH, pm}};
    std::memcpy(out, rows, sizeof(rows));
    return 2;
}
extern "C" int wso_emu_tilings(int* out) {
    int n = 0;
#define ROWS(L) n += tiling_rows<L>(out + 7 * n);
    ROWS(4) ROWS(5) ROWS(6) ROWS(7) ROWS(8) ROWS(9) ROWS(10) ROWS(11) ROWS(12) ROWS(13)
#undef ROWS
    return n;
}
