// wso_kernels.cu — __global__ entry points and launch dispatch for sm_100a.
#include "wso_launch.h"

#include <atomic>
#include <cstdlib>
#include <type_traits>

#include "wso_kernels.cuh"

namespace wso {

#ifndef WSO_K2_SPLIT_DEFAULT
#define WSO_K2_SPLIT_DEFAULT 0
#endif

// CTA tiling.  CP: column pairs per K1 CTA, NF: packed fields per K1 CTA, RI: row items (each = output rows m'
// and N-m') per K2 CTA, RH: row items per K2h CTA (one line each).  CTA threads = lines * N / 16.
template <int CP_, int NF_, int RI_, int RH_>
struct Tiling {
    static constexpr int CP = CP_, NF = NF_, RI = RI_, RH = RH_;
};
// Two tilings per tile size:
//   Bulk - batched launches (many tile-frames per launch): larger CTAs, 32-byte W store segments; tuned with
//          tools/sweep_build.py + tools/sweep_run.sh on B200 (profiles/r1b_sweep.md)
//   Lat  - a launch with few tile-frames (the reference's one ComputeWaves(t) per frame): small CTAs so that a single
//          512^2 or 1024^2 tile still spreads over all 148 SMs
template <int LOGN> struct Cfg;
template <> struct Cfg<4>  { using Bulk = Tiling<8, 4, 8, 8>;   using Lat = Tiling<2, 4, 2, 4>; };
template <> struct Cfg<5>  { using Bulk = Tiling<8, 4, 8, 16>;  using Lat = Tiling<2, 4, 2, 4>; };
template <> struct Cfg<6>  { using Bulk = Tiling<8, 4, 8, 16>;  using Lat = Tiling<2, 4, 2, 4>; };
template <> struct Cfg<7>  { using Bulk = Tiling<4, 4, 8, 16>;  using Lat = Tiling<2, 4, 2, 4>; };
template <> struct Cfg<8>  { using Bulk = Tiling<4, 4, 4, 8>;   using Lat = Tiling<2, 2, 1, 2>; };
// (the WSO_TUNE_* macros exist for tuning sweeps: tools/tune_build.sh builds variant libraries)
#ifndef WSO_TUNE_CP9
#define WSO_TUNE_CP9 4
#define WSO_TUNE_NF9 4
#define WSO_TUNE_RI9 1
#define WSO_TUNE_RH9 4
#endif
#ifndef WSO_TUNE_CP10
#define WSO_TUNE_CP10 4
#define WSO_TUNE_NF10 2
#define WSO_TUNE_RI10 2
#define WSO_TUNE_RH10 4
#endif
#ifndef WSO_TUNE_CP11
#define WSO_TUNE_CP11 4
#define WSO_TUNE_NF11 2
#define WSO_TUNE_RI11 1
#define WSO_TUNE_RH11 2
#endif
#ifndef WSO_TUNE_LCP9
#define WSO_TUNE_LCP9 2
#define WSO_TUNE_LNF9 2
#define WSO_TUNE_LRI9 1
#define WSO_TUNE_LRH9 2
#endif
#ifndef WSO_TUNE_LCP10
#define WSO_TUNE_LCP10 2
#define WSO_TUNE_LNF10 2
#define WSO_TUNE_LRI10 1
#define WSO_TUNE_LRH10 2
#endif
template <> struct Cfg<9> {
    using Bulk = Tiling<WSO_TUNE_CP9, WSO_TUNE_NF9, WSO_TUNE_RI9, WSO_TUNE_RH9>;
    using Lat = Tiling<WSO_TUNE_LCP9, WSO_TUNE_LNF9, WSO_TUNE_LRI9, WSO_TUNE_LRH9>;
};
template <> struct Cfg<10> {
    using Bulk = Tiling<WSO_TUNE_CP10, WSO_TUNE_NF10, WSO_TUNE_RI10, WSO_TUNE_RH10>;
    using Lat = Tiling<WSO_TUNE_LCP10, WSO_TUNE_LNF10, WSO_TUNE_LRI10, WSO_TUNE_LRH10>;
};
template <> struct Cfg<11> {
    using Bulk = Tiling<WSO_TUNE_CP11, WSO_TUNE_NF11, WSO_TUNE_RI11, WSO_TUNE_RH11>;
    using Lat = Bulk;
};
template <> struct Cfg<12> { using Bulk = Tiling<4, 1, 2, 4>; using Lat = Bulk; };
template <> struct Cfg<13> { using Bulk = Tiling<2, 1, 1, 2>; using Lat = Bulk; };

// 1024 resident threads per SM at <= 64 registers: every thread carries 16 complex values between barriers
constexpr int min_blocks(int threads) { return threads >= 1024 ? 1 : (1024 / threads > 8 ? 8 : 1024 / threads); }

// FAST = every item of the launch has the sincos table and the pair-summed records (any Prepare()-built h0): the
// lean instantiation of K1.  FAST = false serves imported spectra that lack either property.
// JAC: packed field 1 also carries dzDx (the Jacobian channel, SURVEY row f-4); served by the general (FAST = false) body.
template <int LOGN, class TL, class Args, bool FAST, bool JAC = false>
__global__ void __launch_bounds__(Pass1<LOGN, TL::CP, TL::NF>::T, min_blocks(Pass1<LOGN, TL::CP, TL::NF>::T))
wso_pass1_kernel(const __grid_constant__ Args args) {
    extern __shared__ __align__(16) float2 smem[];
    DeviceExec ex;
#ifdef WSO_EXP_STAGGER_K1_NS
    // experiment: the CTAs that fill the second resident slot of every SM in the first wave start late, so that the two
    // co-resident CTAs are in different phases (evolve = L2 latency, transform = shared memory, split = stores)
    {
        const unsigned lin = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
        if (lin >= 148u && lin < 296u) __nanosleep(WSO_EXP_STAGGER_K1_NS);
    }
#endif
    Pass1<LOGN, TL::CP, TL::NF, false, FAST, JAC>::run(ex, smem, blockIdx.x, blockIdx.y, blockIdx.z, args);
}

// TEX: output texel of the maps kernels (float4 = RGBA32F, Half4 = RGBA16F; wso_set_map_format)
template <int LOGN, class TL, class Args, class TEX = float4>
__global__ void __launch_bounds__(Pass2<LOGN, TL::RI, false>::T, min_blocks(Pass2<LOGN, TL::RI, false>::T))
wso_pass2_kernel(const __grid_constant__ Args args) {
    extern __shared__ __align__(16) float2 smem[];
    DeviceExec ex;
    Pass2<LOGN, TL::RI, false, false, false, false, TEX>::run(ex, smem, blockIdx.x, blockIdx.y, blockIdx.z, args);
}

// Persistent forms (Pass1::run_persistent / Pass2::run_persistent): a fixed 1-D grid of CTAs - as many as the device
// holds at once - walks the work items of the launch and requests the inputs of its next item ahead of the store phase
// of the current one.  Batched launches of the fused K1 tilings (512^2, 1024^2) and of the paired-W K2 (512^2 ... 2048^2).
// experiment hook: co-resident persistent CTAs (slot = blockIdx.x / SMs) start `ns` apart so that they stay in different phases
__device__ __forceinline__ void exp_stagger(unsigned ns) {
    if (ns == 0) return;
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    do {
        __nanosleep(200);
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    } while (t1 - t0 < ns);
}
template <int LOGN, class TL>
struct PersistOk {
    static constexpr bool k1 = Pass1<LOGN, TL::CP, TL::NF, false, true>::kPersistOk && LOGN >= 9 && LOGN <= 11;
    static constexpr bool k2 = WLayout<LOGN>::paired && LOGN >= 9 && LOGN <= 11;
};
template <int LOGN, class TL, class Args>
__global__ void __launch_bounds__(Pass1<LOGN, TL::CP, TL::NF>::T, min_blocks(Pass1<LOGN, TL::CP, TL::NF>::T))
wso_pass1p_kernel(const __grid_constant__ Args args, const int n_items) {
    extern __shared__ __align__(16) float2 smem[];
    DeviceExec ex;
#ifdef WSO_EXP_P_STAGGER1_NS
    exp_stagger((blockIdx.x / 148u) * (unsigned)(WSO_EXP_P_STAGGER1_NS));
#endif
    if constexpr (PersistOk<LOGN, TL>::k1)
        Pass1<LOGN, TL::CP, TL::NF, false, true>::run_persistent(ex, smem, blockIdx.x, gridDim.x, n_items, args);
}
template <int LOGN, class TL, class Args, class TEX = float4>
__global__ void __launch_bounds__(Pass2<LOGN, TL::RI, false>::T, min_blocks(Pass2<LOGN, TL::RI, false>::T))
wso_pass2p_kernel(const __grid_constant__ Args args, const int n_items) {
    extern __shared__ __align__(16) float2 smem[];
    DeviceExec ex;
#ifdef WSO_EXP_P_STAGGER2_NS
    exp_stagger((blockIdx.x / 148u) * (unsigned)(WSO_EXP_P_STAGGER2_NS));
#endif
    if constexpr (PersistOk<LOGN, TL>::k2)
        Pass2<LOGN, TL::RI, false, false, false, false, TEX>::run_persistent(ex, smem, blockIdx.x, gridDim.x, n_items, args);
}

// "K2nh": the height pre-pass and the NORMAL map in one launch (blockIdx.y = 0: normal-map CTAs, 1: height CTAs), followed
// by wso_pass2_kernel for the displacement map only.  The normal map does not need the amplitude A, so K2h - a partial
// wave of latency-bound CTAs when launched alone - runs underneath the store-bound normal-map CTAs instead of in front of
// both maps.  Needs equal CTA sizes of the two bodies.
template <int LOGN, class TL>
struct K2Split {
    using P2 = Pass2<LOGN, TL::RI, false>;
    static constexpr int RHS = 2 * TL::RI;  // a height CTA holds as many lines as a map CTA: equal CTA sizes
    static constexpr bool possible = (RHS <= P2::H) && (RHS * P2::N / kValsPerThread <= 1024);
    using PH = Pass2<LOGN, possible ? RHS : 1, true>;
    static constexpr int SMEM = P2::SMEM_BYTES > PH::SMEM_BYTES ? P2::SMEM_BYTES : PH::SMEM_BYTES;
    static constexpr int GX = P2::H / TL::RI;  // >= the number of height CTAs, H / (2 RI)
};
template <int LOGN, class TL, class Args, class TEX = float4>
__global__ void __launch_bounds__(Pass2<LOGN, TL::RI, false>::T, min_blocks(Pass2<LOGN, TL::RI, false>::T))
wso_pass2nh_kernel(const __grid_constant__ Args args) {
    extern __shared__ __align__(16) float2 smem[];
    DeviceExec ex;
    if (blockIdx.y == 0) {
        if (blockIdx.x >= Pass2<LOGN, TL::RI, false>::H / TL::RI) return;
        // K1 (the predecessor in the stream) must have completed before W is read
        ex.pdl_wait();
        ex.pdl_release();
        Pass2<LOGN, TL::RI, false, false, false, false, TEX>::run(ex, smem, blockIdx.x, 1, blockIdx.z, args);
    } else {
        using PH = typename K2Split<LOGN, TL>::PH;
        if (blockIdx.x >= PH::grid_x()) return;
        PH::run(ex, smem, blockIdx.x, 0, blockIdx.z, args);
    }
}

// K2 with the Jacobian channel: one row item (all four packed fields) per CTA, both maps from one CTA.
// Sizes up to 4096^2 (four lines of shared memory and 4*N/16 <= 1024 threads).
constexpr bool jacobian_size_ok(int logn) { return logn <= 12; }
template <int LOGN, class Args, class TEX = float4>
__global__ void __launch_bounds__(Pass2<LOGN, 1, false, false, false, true>::T)
wso_pass2j_kernel(const __grid_constant__ Args args) {
    extern __shared__ __align__(16) float2 smem[];
    DeviceExec ex;
    Pass2<LOGN, 1, false, false, false, true, TEX>::run(ex, smem, blockIdx.x, 0, blockIdx.z, args);
}

// K2h: height extrema (min/max -> amplitude A) ahead of K2, so that K2 writes disp.y already normalised and no
// second pass over the displacement map is needed (reference: the serial NormalizeHeights sweep, WSTessendorf.cpp:443-455)
template <int LOGN, class TL, class Args>
__global__ void __launch_bounds__(Pass2<LOGN, TL::RH, true>::T, min_blocks(Pass2<LOGN, TL::RH, true>::T))
wso_heights_kernel(const __grid_constant__ Args args) {
    extern __shared__ __align__(16) float2 smem[];
    DeviceExec ex;
    Pass2<LOGN, TL::RH, true>::run(ex, smem, blockIdx.x, 0, blockIdx.z, args);
}

// Every launch carries the programmatic-stream-serialization attribute: the next kernel of the stream is
// scheduled while this one drains and blocks in griddepcontrol.wait (pdl_wait() at the top of each kernel body)
// until its predecessor has completed and flushed - stream order is preserved, launch latency is hidden.
// (frame graphs, see launch_frame_graph below: while a thread rewrites the parameters of an instantiated graph, the
// launch code runs as usual and every launch_pdl lands on the graph node of its kernel instead of in the stream)
struct GraphUpdate {
    FrameGraph* g;
    unsigned used;   // nodes rewritten so far (bit per node)
    bool mismatch;   // a launch for which the graph has no (unused) node: the sequence changed, capture again
};
static thread_local GraphUpdate* tl_graph_update = nullptr;

template <class Args, class Kern, class... Extra>
static cudaError_t launch_pdl(Kern kern, dim3 grid, int threads, int smem, cudaStream_t stream, const Args& args,
                              Extra... extra) {
    if (GraphUpdate* u = tl_graph_update) {
        int k = -1;
        for (int i = 0; i < u->g->n_nodes; ++i)
            if (u->g->func[i] == reinterpret_cast<void*>(kern)) k = i;
        if (k < 0 || (u->used >> k & 1u)) {
            u->mismatch = true;
            return cudaSuccess;
        }
        u->used |= 1u << k;
        void* params[] = {const_cast<Args*>(&args), static_cast<void*>(&extra)...};
        cudaKernelNodeParams p = {};
        p.func = reinterpret_cast<void*>(kern);
        p.gridDim = grid;
        p.blockDim = dim3((unsigned)threads, 1, 1);
        p.sharedMemBytes = (unsigned)smem;
        p.kernelParams = params;
        p.extra = nullptr;
        return cudaGraphExecKernelNodeSetParams(u->g->exec, u->g->node[k], &p);
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3((unsigned)threads, 1, 1);
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, args, extra...);
}

// Which of K1 / K2h / K2 (bits 0 / 1 / 2) of a qualifying batched launch run on the warp-per-line kernels of
// wso_kernels2.cu.  Default = what measured faster on B200 (profiles/r2_ab_kernel_sets.md): the height pre-pass K2h at
// 1024^2; everything else stays on the CTA-per-line kernels of this file.  WSO_WARP_CORE overrides the mask for every
// supported size (0 = none, 7 = all three) - used by the A/B measurements and the parity tests of both kernel sets.
// Bits 4 / 6 of the same mask: K1 / K2 of the CTA-per-line set in their PERSISTENT form (where a kernel is on the
// warp-per-line set, that wins).
static std::atomic<int> g_warp_core_override{-1};  // wso_select_kernels(): -1 = no override
void set_warp_core_override(int mask) { g_warp_core_override.store(mask < 0 ? -1 : (mask & 0x57), std::memory_order_relaxed); }

#ifndef WSO_PERSIST_DEFAULT
#define WSO_PERSIST_DEFAULT 0
#endif
static int kernel_choice_mask(int logn) {
    static const int env_mask = [] {
        const char* env = std::getenv("WSO_WARP_CORE");
        return env ? (std::atoi(env) & 0x57) : -1;
    }();
    const int forced = g_warp_core_override.load(std::memory_order_relaxed);
    if (forced >= 0) return forced & 0x57;
    if (env_mask >= 0) return env_mask;
    (void)logn;  // (round 2, second session: K2h at 1024^2 ran on the warp-per-line set; with the twiddle preload the CTA-per-line K2h is faster again)
    return WSO_PERSIST_DEFAULT;
}
static int warp_core_mask(int logn) { return kernel_choice_mask(logn) & 7; }

// CTAs of a persistent kernel = what the device holds at once (queried once per kernel and device)
template <class Kern>
static int resident_ctas(Kern kern, int threads, int smem, int dev) {
    int per_sm = 0, sms = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, (size_t)smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms < 1) sms = 148;
    return per_sm * sms;
}

// Jacobian mode: K1 (general body, field 1 with its real slot filled), K2h, K2 with four lines per CTA
template <int LOGN, class TL, class Args, class TEX>
static cudaError_t launch_tiled_jacobian(const Args& args, int n_items, cudaStream_t stream, cudaEvent_t* ev) {
    if constexpr (!jacobian_size_ok(LOGN)) {
        return cudaErrorNotSupported;
    } else {
        using P1 = Pass1<LOGN, TL::CP, TL::NF>;
        using PJ = Pass2<LOGN, 1, false, false, false, true>;
        using PH = Pass2<LOGN, TL::RH, true>;
        static std::atomic<bool> configured[16];  // per device: opt in to > 48 KB of dynamic shared memory once
        int dev = 0;
        cudaGetDevice(&dev);
        cudaError_t e;
        if (dev < 0 || dev >= 16 || !configured[dev].load(std::memory_order_acquire)) {
            e = cudaFuncSetAttribute(wso_pass1_kernel<LOGN, TL, Args, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, P1::SMEM_BYTES);
            if (e != cudaSuccess) return e;
            e = cudaFuncSetAttribute(wso_pass2j_kernel<LOGN, Args, TEX>, cudaFuncAttributeMaxDynamicSharedMemorySize, PJ::SMEM_BYTES);
            if (e != cudaSuccess) return e;
            e = cudaFuncSetAttribute(wso_heights_kernel<LOGN, TL, Args>, cudaFuncAttributeMaxDynamicSharedMemorySize, PH::SMEM_BYTES);
            if (e != cudaSuccess) return e;
            // (the attribute calls are idempotent: two threads racing here both complete them before either publishes)
            if (dev >= 0 && dev < 16) configured[dev].store(true, std::memory_order_release);
        }
        if (ev) cudaEventRecord(ev[0], stream);
        e = launch_pdl(wso_pass1_kernel<LOGN, TL, Args, false, true>, dim3(P1::H / TL::CP, 4 / TL::NF, n_items), P1::T,
                       P1::SMEM_BYTES, stream, args);
        if (e != cudaSuccess) return e;
        if (ev) cudaEventRecord(ev[1], stream);
        e = launch_pdl(wso_heights_kernel<LOGN, TL, Args>, dim3(PH::grid_x(), 1, n_items), PH::T, PH::SMEM_BYTES, stream, args);
        if (e != cudaSuccess) return e;
        if (ev) cudaEventRecord(ev[2], stream);
        e = launch_pdl(wso_pass2j_kernel<LOGN, Args, TEX>, dim3(PJ::H, 1, n_items), PJ::T, PJ::SMEM_BYTES, stream, args);
        if (e != cudaSuccess) return e;
        if (ev) cudaEventRecord(ev[3], stream);
        return cudaGetLastError();
    }
}

// K2h together with the normal map (wso_pass2nh_kernel) instead of in front of both maps: WSO_K2_SPLIT=0/1 overrides.
static std::atomic<int> g_k2_split_override{-1};
void set_k2_split_override(int on) { g_k2_split_override.store(on < 0 ? -1 : (on ? 1 : 0), std::memory_order_relaxed); }
static bool k2_split_enabled() {
    static const int env = [] {
        const char* e = std::getenv("WSO_K2_SPLIT");
        return e ? (std::atoi(e) != 0 ? 1 : 0) : -1;
    }();
    const int forced = g_k2_split_override.load(std::memory_order_relaxed);
    if (forced >= 0) return forced != 0;
    if (env >= 0) return env != 0;
    return WSO_K2_SPLIT_DEFAULT != 0;
}
bool k2_split_active() { return k2_split_enabled(); }

// Experiment hook: request at least this much dynamic shared memory for K1 / K2 (bytes; 0 = what the kernel needs).  A
// larger request lowers the number of CTAs of that kernel an SM can hold and leaves threads / registers / shared memory
// for the CTAs of the OTHER compute lane's kernel, i.e. it forces K1 and K2 of different chunks to share SMs.
static int exp_min_smem(const char* name) {
    const char* env = std::getenv(name);
    const int v = env ? std::atoi(env) : 0;
    return v > 0 && v <= 227 * 1024 ? v : 0;
}

template <int LOGN, class TL, class Args, class TEX>
static cudaError_t launch_tiled(const Args& args, int n_items, cudaStream_t stream, cudaEvent_t* ev) {
    using P1 = Pass1<LOGN, TL::CP, TL::NF>;
    using P2 = Pass2<LOGN, TL::RI, false>;
    using PH = Pass2<LOGN, TL::RH, true>;
    static const int k1_min = exp_min_smem("WSO_EXP_K1_SMEM"), k2_min = exp_min_smem("WSO_EXP_K2_SMEM");
    const int smem1 = P1::SMEM_BYTES > k1_min ? P1::SMEM_BYTES : k1_min;
    const int smem2 = P2::SMEM_BYTES > k2_min ? P2::SMEM_BYTES : k2_min;
    static std::atomic<bool> configured[16];  // per device: opt in to > 48 KB of dynamic shared memory once
    // persistent forms: batched launches (the big parameter block) only
    constexpr bool kPersist = std::is_same<Args, LaunchArgs>::value && (PersistOk<LOGN, TL>::k1 || PersistOk<LOGN, TL>::k2);
    static int ctas1[16], ctas2[16];  // resident CTAs of the persistent K1 / K2 per device (written before `configured`)
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 16 || !configured[dev].load(std::memory_order_acquire)) {
        cudaError_t e;
        e = cudaFuncSetAttribute(wso_pass1_kernel<LOGN, TL, Args, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem1);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(wso_pass1_kernel<LOGN, TL, Args, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem1);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(wso_pass2_kernel<LOGN, TL, Args, TEX>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(wso_heights_kernel<LOGN, TL, Args>, cudaFuncAttributeMaxDynamicSharedMemorySize, PH::SMEM_BYTES);
        if (e != cudaSuccess) return e;
        if constexpr (kPersist) {
            if constexpr (PersistOk<LOGN, TL>::k1) {
                e = cudaFuncSetAttribute(wso_pass1p_kernel<LOGN, TL, Args>, cudaFuncAttributeMaxDynamicSharedMemorySize, P1::SMEM_BYTES);
                if (e != cudaSuccess) return e;
                if (dev >= 0 && dev < 16) ctas1[dev] = resident_ctas(wso_pass1p_kernel<LOGN, TL, Args>, P1::T, P1::SMEM_BYTES, dev);
            }
            if constexpr (PersistOk<LOGN, TL>::k2) {
                e = cudaFuncSetAttribute(wso_pass2p_kernel<LOGN, TL, Args, TEX>, cudaFuncAttributeMaxDynamicSharedMemorySize, P2::SMEM_BYTES);
                if (e != cudaSuccess) return e;
                if (dev >= 0 && dev < 16) ctas2[dev] = resident_ctas(wso_pass2p_kernel<LOGN, TL, Args, TEX>, P2::T, P2::SMEM_BYTES, dev);
            }
        }
        if constexpr (K2Split<LOGN, TL>::possible) {
            const int smemnh = K2Split<LOGN, TL>::SMEM > k2_min ? K2Split<LOGN, TL>::SMEM : k2_min;
            e = cudaFuncSetAttribute(wso_pass2nh_kernel<LOGN, TL, Args, TEX>, cudaFuncAttributeMaxDynamicSharedMemorySize, smemnh);
            if (e != cudaSuccess) return e;
        }
        if (dev >= 0 && dev < 16) configured[dev].store(true, std::memory_order_release);
    }
    cudaError_t e;
    if (ev) cudaEventRecord(ev[0], stream);
    const dim3 g1(P1::H / TL::CP, 4 / TL::NF, n_items);
#ifdef WSO_EXP_NO_FAST
    bool fast = false;
#else
    bool fast = true;
#endif
    for (int i = 0; i < n_items; ++i) fast = fast && args.td[i].table_len > 0 && args.td[i].use_pairs != 0;
    // batched launches of 512^2 / 1024^2 / 2048^2 run on the warp-per-line kernels (wso_kernels2.cu); mask bit k = kernel k
    int warp_mask = 0;
    if constexpr (std::is_same<Args, LaunchArgs>::value) {
        if (fast && warp_core_supported(LOGN)) warp_mask = warp_core_mask(LOGN);
    }
    // the warp-per-line K2 writes RGBA32F only: RGBA16F maps always come from the CTA-per-line K2 (bit 2 ignored)
    if constexpr (!std::is_same<TEX, float4>::value) warp_mask &= ~4;
    if constexpr (std::is_same<Args, LaunchArgs>::value) {
        if (warp_mask & 1) e = launch_warp_core(LOGN, 0, args, n_items, stream);
    }
    int persist = 0;  // bit 0: K1, bit 2: K2 in the persistent form
    if constexpr (kPersist) {
        if (fast && dev >= 0 && dev < 16 && k1_min == 0 && k2_min == 0) persist = (kernel_choice_mask(LOGN) >> 4) & 5;
    }
    bool k1_done = (warp_mask & 1) != 0;
    if constexpr (kPersist && PersistOk<LOGN, TL>::k1) {
        if (!k1_done && (persist & 1)) {
            const int total = (int)(g1.x * g1.y * g1.z);
            const int grid = total < ctas1[dev] ? total : ctas1[dev];
            e = launch_pdl(wso_pass1p_kernel<LOGN, TL, Args>, dim3(grid, 1, 1), P1::T, P1::SMEM_BYTES, stream, args, n_items);
            k1_done = true;
        }
    }
    if (!k1_done)
        e = fast ? launch_pdl(wso_pass1_kernel<LOGN, TL, Args, true>, g1, P1::T, smem1, stream, args)
                 : launch_pdl(wso_pass1_kernel<LOGN, TL, Args, false>, g1, P1::T, smem1, stream, args);
    if (e != cudaSuccess) return e;
    if (ev) cudaEventRecord(ev[1], stream);
    if constexpr (K2Split<LOGN, TL>::possible) {
        if (!(warp_mask & 6) && k2_split_enabled()) {
            using KS = K2Split<LOGN, TL>;
            const int smemnh = KS::SMEM > k2_min ? KS::SMEM : k2_min;
            e = launch_pdl(wso_pass2nh_kernel<LOGN, TL, Args, TEX>, dim3(KS::GX, 2, n_items), P2::T, smemnh, stream, args);
            if (e != cudaSuccess) return e;
            if (ev) cudaEventRecord(ev[2], stream);
            e = launch_pdl(wso_pass2_kernel<LOGN, TL, Args, TEX>, dim3(P2::H / TL::RI, 1, n_items), P2::T, smem2, stream, args);
            if (e != cudaSuccess) return e;
            if (ev) cudaEventRecord(ev[3], stream);
            return cudaGetLastError();
        }
    }
    const dim3 gh(PH::grid_x(), 1, n_items);
    if constexpr (std::is_same<Args, LaunchArgs>::value) {
        if (warp_mask & 2) e = launch_warp_core(LOGN, 1, args, n_items, stream);
    }
    if (!(warp_mask & 2)) e = launch_pdl(wso_heights_kernel<LOGN, TL, Args>, gh, PH::T, PH::SMEM_BYTES, stream, args);
    if (e != cudaSuccess) return e;
    if (ev) cudaEventRecord(ev[2], stream);
    const dim3 g2(P2::H / TL::RI, 2, n_items);
    if constexpr (std::is_same<Args, LaunchArgs>::value) {
        if (warp_mask & 4) e = launch_warp_core(LOGN, 2, args, n_items, stream);
    }
    bool k2_done = (warp_mask & 4) != 0;
    if constexpr (kPersist && PersistOk<LOGN, TL>::k2) {
        if (!k2_done && (persist & 4)) {
            const int total = (int)(g2.x * g2.y * g2.z);
            const int grid = total < ctas2[dev] ? total : ctas2[dev];
            e = launch_pdl(wso_pass2p_kernel<LOGN, TL, Args, TEX>, dim3(grid, 1, 1), P2::T, P2::SMEM_BYTES, stream, args, n_items);
            k2_done = true;
        }
    }
    if (!k2_done) e = launch_pdl(wso_pass2_kernel<LOGN, TL, Args, TEX>, g2, P2::T, smem2, stream, args);
    if (e != cudaSuccess) return e;
    if (ev) cudaEventRecord(ev[3], stream);
    return cudaGetLastError();
}

template <int LOGN, class TEX>
static cudaError_t launch_all(const LaunchArgs& args, int n_items, cudaStream_t stream, bool jacobian, cudaEvent_t* ev) {
    using B = typename Cfg<LOGN>::Bulk;
    using L = typename Cfg<LOGN>::Lat;
    if (jacobian) return launch_tiled_jacobian<LOGN, B, LaunchArgs, TEX>(args, n_items, stream, ev);
    // few tile-frames in this launch: the Bulk grid of K1 would leave SMs idle -> fine-grained tiling and the
    // small parameter block
    constexpr int bulk_ctas_per_item = ((1 << LOGN) / 2 / B::CP) * (4 / B::NF);
    if (n_items <= kSmallChunk && n_items * bulk_ctas_per_item < 2 * 148) {
        LaunchArgsSmall sm = {};
        sm.tw = args.tw; sm.W = args.W; sm.disp = args.disp; sm.norm = args.norm;
        sm.minmax = args.minmax; sm.amp_out = args.amp_out;
        for (int i = 0; i < kSmallChunk; ++i) { sm.items[i] = args.items[i]; sm.td[i] = args.td[i]; }
        return launch_tiled<LOGN, L, LaunchArgsSmall, TEX>(sm, n_items, stream, ev);
    }
    return launch_tiled<LOGN, B, LaunchArgs, TEX>(args, n_items, stream, ev);
}
template <int LOGN>
static cudaError_t launch_all(const LaunchArgs& args, int n_items, cudaStream_t stream, bool jacobian, bool half,
                              cudaEvent_t* ev) {
    return half ? launch_all<LOGN, Half4>(args, n_items, stream, jacobian, ev)
                : launch_all<LOGN, float4>(args, n_items, stream, jacobian, ev);
}

cudaError_t launch_compute_waves(int logn, const LaunchArgs& args, int n_items, cudaStream_t stream,
                                 bool jacobian, bool half, cudaEvent_t* ev) {
    switch (logn) {
// WSO_ONLY_LOGN: tuning builds instantiate a single size (tools/tune_build.sh) to keep compile times short
#ifdef WSO_ONLY_LOGN
        case WSO_ONLY_LOGN: return launch_all<WSO_ONLY_LOGN>(args, n_items, stream, jacobian, half, ev);
#else
        case 4: return launch_all<4>(args, n_items, stream, jacobian, half, ev);
        case 5: return launch_all<5>(args, n_items, stream, jacobian, half, ev);
        case 6: return launch_all<6>(args, n_items, stream, jacobian, half, ev);
        case 7: return launch_all<7>(args, n_items, stream, jacobian, half, ev);
        case 8: return launch_all<8>(args, n_items, stream, jacobian, half, ev);
        case 9: return launch_all<9>(args, n_items, stream, jacobian, half, ev);
        case 10: return launch_all<10>(args, n_items, stream, jacobian, half, ev);
        case 11: return launch_all<11>(args, n_items, stream, jacobian, half, ev);
        case 12: return launch_all<12>(args, n_items, stream, jacobian, half, ev);
        case 13: return launch_all<13>(args, n_items, stream, jacobian, half, ev);
#endif
        default: return cudaErrorInvalidValue;
    }
}

int kernels_per_launch() { return 3; }

void destroy_frame_graph(FrameGraph& g) {
    if (g.exec) cudaGraphExecDestroy(g.exec);
    if (g.graph) cudaGraphDestroy(g.graph);
    g.exec = nullptr;
    g.graph = nullptr;
    g.n_nodes = 0;
    g.logn = g.jacobian = g.half = -1;
}

// Capture the launch sequence of one tile-frame into g (stream must not be capturing already).  false: not capturable here.
static bool capture_frame_graph(FrameGraph& g, int logn, const LaunchArgs& args, cudaStream_t stream, bool jacobian,
                                bool half) {
    destroy_frame_graph(g);
    if (cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    const cudaError_t le = launch_compute_waves(logn, args, 1, stream, jacobian, half, nullptr);
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(stream, &graph);
    bool ok = le == cudaSuccess && ce == cudaSuccess && graph != nullptr;
    size_t n = 0;
    ok = ok && cudaGraphGetNodes(graph, nullptr, &n) == cudaSuccess && n >= 1 && n <= (size_t)FrameGraph::kMaxNodes;
    ok = ok && cudaGraphGetNodes(graph, g.node, &n) == cudaSuccess;
    for (size_t i = 0; ok && i < n; ++i) {
        cudaGraphNodeType type;
        cudaKernelNodeParams p = {};
        ok = cudaGraphNodeGetType(g.node[i], &type) == cudaSuccess && type == cudaGraphNodeTypeKernel &&
             cudaGraphKernelNodeGetParams(g.node[i], &p) == cudaSuccess;
        g.func[i] = p.func;
        for (size_t k = 0; ok && k < i; ++k) ok = g.func[k] != g.func[i];  // nodes are told apart by their kernel
    }
    ok = ok && cudaGraphInstantiate(&g.exec, graph, 0) == cudaSuccess;
    if (!ok) {
        if (graph) cudaGraphDestroy(graph);
        g.exec = nullptr;
        cudaGetLastError();
        return false;
    }
    g.graph = graph;
    g.n_nodes = (int)n;
    g.logn = logn;
    g.jacobian = jacobian ? 1 : 0;
    g.half = half ? 1 : 0;
    g.captures += 1;
    return true;
}

cudaError_t launch_frame_graph(FrameGraph& g, int logn, const LaunchArgs& args, cudaStream_t stream, bool jacobian,
                               bool half) {
    // kernels of wso_kernels2.cu (an explicit kernel-set choice) launch through their own helper: plain launches
    if (g.disabled || (kernel_choice_mask(logn) & 7) != 0) return launch_compute_waves(logn, args, 1, stream, jacobian, half, nullptr);
    // a caller that is capturing this stream into a graph of its own gets the three kernels recorded as they are
    cudaStreamCaptureStatus capturing = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(stream, &capturing) != cudaSuccess || capturing != cudaStreamCaptureStatusNone) {
        cudaGetLastError();
        return launch_compute_waves(logn, args, 1, stream, jacobian, half, nullptr);
    }
    if (g.warm_logn != logn || g.warm_jacobian != (jacobian ? 1 : 0) || g.warm_half != (half ? 1 : 0)) {
        // first frame of this shape: the plain launch also does the one-time kernel configuration (cudaFuncSetAttribute)
        const cudaError_t e = launch_compute_waves(logn, args, 1, stream, jacobian, half, nullptr);
        if (e == cudaSuccess) {
            g.warm_logn = logn;
            g.warm_jacobian = jacobian ? 1 : 0;
            g.warm_half = half ? 1 : 0;
        }
        return e;
    }
    for (int attempt = 0; attempt < 2; ++attempt) {
        if (!g.exec || g.logn != logn || g.jacobian != (jacobian ? 1 : 0) || g.half != (half ? 1 : 0)) {
            if (!capture_frame_graph(g, logn, args, stream, jacobian, half)) break;
            g.graph_launches += 1;
            return cudaGraphLaunch(g.exec, stream);  // captured with this call's parameters
        }
        GraphUpdate u{&g, 0u, false};
        tl_graph_update = &u;
        const cudaError_t e = launch_compute_waves(logn, args, 1, stream, jacobian, half, nullptr);
        tl_graph_update = nullptr;
        if (e == cudaSuccess && !u.mismatch && u.used == (1u << g.n_nodes) - 1u) {
            g.graph_launches += 1;
            return cudaGraphLaunch(g.exec, stream);
        }
        cudaGetLastError();
        destroy_frame_graph(g);  // another kernel variant serves this frame (e.g. an imported spectrum without the table)
    }
    g.disabled = true;
    destroy_frame_graph(g);
    return launch_compute_waves(logn, args, 1, stream, jacobian, half, nullptr);
}

}  // namespace wso
