// TEST INFRASTRUCTURE — CPU emulation of the RGBA16F map kernels (wso_set_map_format).
//
// The same thread-by-thread stepping of the wso_kernels.cuh bodies as emu.cpp, with K2 instantiated for both output
// texel types (float4 = RGBA32F, Half4 = RGBA16F), plus the host build's float -> binary16 conversion of
// wso_device.cuh.  Built and loaded by tests/test_map_format.py; never linked into the product library.
#include <cstdio>
#include <cstring>
#include <vector>

#include "wso_kernels.cuh"

using namespace wso;

// JAC: the Jacobian-channel kernels (SURVEY row f-4): K1's general body with field 1's real slot filled, K2 with four
// lines per CTA (by = 0 only).
// PERSIST: bit 0 = K1, bit 2 = K2 through their persistent forms (run_persistent: a few emulated CTAs walk the work items,
// each with its own shared memory and thread states that live across items - the prefetched inputs of the next item
// sit in them while the current item is stored)
// TEX: texel type of the maps K2 writes (float4 = RGBA32F, Half4 = RGBA16F); disp / norm hold N*N texels of it
template <int LOGN, int CP, int NF, int RI, bool JAC = false, int PERSIST = 0, class TEX = float4>
static int run_cfg(const float* amp_t, const float* omega_t, const float* kv, float omega0, float lambda,
                   float t, void* disp, void* norm, float* minmax, float* amp_out, float* w_out) {
    constexpr int N = 1 << LOGN, H = N / 2;
    using P1 = Pass1<LOGN, CP, NF, false, false, JAC>;
    using P2 = Pass2<LOGN, JAC ? 1 : RI, false, false, false, JAC, TEX>;
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

template <class TEX>
static int compute_variant(int logn, int variant, const float* amp_t, const float* omega_t, const float* kv, float omega0,
                           float lambda, float t, void* disp, void* norm, float* minmax, float* amp_out) {
    float* w_out = nullptr;
#define CFG(L, V, CP, NF, RI) \
    if (logn == L && variant == V) return run_cfg<L, CP, NF, RI, false, 0, TEX>(amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out, w_out);
    // the tilings of emu.cpp's wso_emu_compute (same variant numbers)
    CFG(4, 0, 8, 4, 8)
    CFG(4, 1, 2, 1, 1)
    CFG(6, 0, 8, 4, 8)
    CFG(6, 1, 4, 2, 2)
    CFG(6, 2, 1, 1, 1)
    CFG(8, 0, 4, 4, 4)
    CFG(8, 1, 4, 2, 2)
    CFG(9, 0, 4, 4, 4)
    CFG(9, 1, 4, 2, 2)
    CFG(10, 0, 4, 2, 4)
#undef CFG
    // variants 200+: the persistent forms of K1 / K2 (bit 0 / bit 2 of the last argument)
#define PCFG(L, V, CP, NF, RI, PM) \
    if (logn == L && variant == 200 + V) return run_cfg<L, CP, NF, RI, false, PM, TEX>(amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out, w_out);
    PCFG(9, 0, 4, 4, 1, 5)
    PCFG(9, 1, 4, 4, 1, 1)
    PCFG(10, 0, 4, 2, 2, 5)
    PCFG(10, 1, 4, 2, 2, 4)
#undef PCFG
    // variants 100+: the Jacobian-channel K2 (pack_item_jac)
#define JCFG(L, V, CP, NF, RI) \
    if (logn == L && variant == 100 + V) return run_cfg<L, CP, NF, RI, true, 0, TEX>(amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out, w_out);
    JCFG(4, 0, 8, 4, 8)
    JCFG(6, 1, 4, 2, 2)
    JCFG(8, 0, 4, 4, 4)
    JCFG(10, 0, 4, 2, 4)
#undef JCFG
    return -1;
}

// One tile-frame; half = 0: disp / norm receive N*N RGBA32F texels, half = 1: N*N texels of 4 binary16 values.
extern "C" int wso_emu16_compute(int logn, int variant, int half, const float* amp_t, const float* omega_t, const float* kv,
                                 float omega0, float lambda, float t, void* disp, void* norm, float* minmax, float* amp_out) {
    return half ? compute_variant<Half4>(logn, variant, amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out)
                : compute_variant<float4>(logn, variant, amp_t, omega_t, kv, omega0, lambda, t, disp, norm, minmax, amp_out);
}

// The host build's float -> binary16 conversion (wso_device.cuh) over an array.
extern "C" void wso_emu16_f32_to_f16(const float* x, uint16_t* out, size_t n) {
    for (size_t i = 0; i < n; ++i) out[i] = f32_to_f16_rn(x[i]);
}
