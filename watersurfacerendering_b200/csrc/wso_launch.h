// wso_launch.h — host-side launch interface of the kernels in wso_kernels.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace wso {

template <int CAP>
struct LaunchArgsT;
using LaunchArgs = LaunchArgsT<64>;  // kMaxChunk (wso_kernels.cuh)

static constexpr int kMinLogN = 4;   // 16
static constexpr int kMaxLogN = 13;  // 8192 (single-CTA line transforms; larger grids: slab path, DESIGN.md §7)

// Enqueue K1 (evolve + first transform), K2h (height extrema) and K2 (second transform + pack) for
// n_items tile-frames described by args.items[0..n_items).
// ev: NULL, or 4 events recorded before K1, between the kernels and after K2 (opt-in profiling).
// jacobian: write disp.w = Jacobian of the horizontal displacement (SURVEY row f-4; sizes up to 4096^2, else
// cudaErrorNotSupported) instead of the reference default 1.0f.
// half: K2 writes RGBA16F texels (8 bytes, wso_device.cuh Half4) into args.disp / args.norm, slot stride 8*N*N bytes,
// instead of RGBA32F (always through the CTA-per-line K2, whatever the kernel-set mask says for K2).
cudaError_t launch_compute_waves(int logn, const LaunchArgs& args, int n_items, cudaStream_t stream,
                                 bool jacobian, bool half, cudaEvent_t* ev);
static constexpr int kMaxJacobianLogN = 12;
int kernels_per_launch();

// One tile-frame as a CUDA graph (the reference's calling pattern: one ComputeWaves(t) per rendered frame).  The three
// launches of a frame cost ~13 us of host enqueue through the runtime - more than the kernels take on the device at 512^2 -
// so a context keeps the launch sequence of its current (size, jacobian, map format) as an instantiated graph (captured from the very
// same launch code, programmatic-dependent-launch edges included), rewrites the kernel parameters of its nodes per call
// (cudaGraphExecKernelNodeSetParams) and pays one cudaGraphLaunch.
struct FrameGraph {
    static constexpr int kMaxNodes = 4;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    cudaGraphNode_t node[kMaxNodes] = {};
    void* func[kMaxNodes] = {};
    int n_nodes = 0;
    int logn = -1, jacobian = -1, half = -1;                  // what the instantiated graph was captured for
    int warm_logn = -1, warm_jacobian = -1, warm_half = -1;  // a plain launch of this shape has run (one-time kernel configuration done)
    bool disabled = false;                   // capture or instantiation failed once: plain launches from then on
    uint64_t graph_launches = 0, captures = 0;
};
// args.items[0] = the tile-frame.  Falls back to launch_compute_waves whenever the graph cannot be used.
cudaError_t launch_frame_graph(FrameGraph& g, int logn, const LaunchArgs& args, cudaStream_t stream, bool jacobian,
                               bool half);
void destroy_frame_graph(FrameGraph& g);

// Warp-per-line kernels (wso_kernels2.cu): 512^2, 1024^2 and 2048^2, every item with the sincos table and the pair-summed
// records, no Jacobian channel.  which: 0 = K1, 1 = K2h, 2 = K2 (same W layout and stream protocol as the kernels of
// wso_kernels.cu, so the two sets can be mixed kernel by kernel).
bool warp_core_supported(int logn);
// process-wide override of the kernel-set choice (bit k = kernel k on the warp-per-line set; -1 = built-in default)
void set_warp_core_override(int mask);
// K2h launched together with the normal map, the displacement map behind them (-1 = built-in default); what is active now
void set_k2_split_override(int on);
bool k2_split_active();
cudaError_t launch_warp_core(int logn, int which, const LaunchArgs& args, int n_items, cudaStream_t stream);

// Slab-decomposed path (one grid over several devices, DESIGN.md §7).  phase 0: K1 on this device's column pairs,
// 1: K2h on its row items, 2: K2 (pair = force the two-CTA cluster variant; always used when a line pair exceeds
// one SM's shared memory).
// nfields (phase 0 only): 0 = all four packed fields, else that many from field args.slab_field0 * NF on
cudaError_t launch_slab_phase(int logn, int phase, const LaunchArgsT<1>& args, bool pair, int nfields, cudaStream_t stream);
int slab_fields_per_group(int logn);
bool slab_size_supported(int logn);
// The slab exchange as one transposing kernel (wso_slab_kernels.cu): stage = K1's staged output on this device, dst.p[d]
// = where device d's row items go (block `src = this device` of d's receive buffer, or of a local send buffer).
struct XposeDst {
    float2* p[8];
};
cudaError_t launch_slab_exchange(const float2* stage, const XposeDst& dst, int world, int rank, int hl_log, int h_log,
                                 int field0, int nfields, cudaStream_t stream);

// Prepare() on the device (wso_prepare_kernels.cu, SURVEY row f-3).  One launch builds the per-point records
// h0[jl][half][m] and the pair-summed records hs[jl][i][2] of the column pairs j0 .. j0+n_pairs-1.
struct PrepareArgs {
    float4* h0;
    float4* hs;
    const float* kv;      // [n] wave numbers (device)
    const float2* xi;     // [n][n] Gaussian array in the reference's order (device), or NULL: counter-based
    uint64_t seed_mixed;  // counter_seed_mix(seed)
    int n, j0;
    float wind_x, wind_y, omega0, phillips_const, damping, inv_sqrt2, Lw2;
};
cudaError_t launch_prepare(const PrepareArgs& a, int n_pairs, cudaStream_t stream);
// device records of a whole (non-slab) tile -> reference 20-byte records [m][n] in out20 (device, 5 floats each)
cudaError_t launch_export_records(const float4* h0, float* out20, int n, float omega0, bool table, cudaStream_t stream);
uint64_t counter_seed_mix(uint64_t seed);

// Surface queries (wso_query_kernels.cu, body in wso_query.cuh): one launch, one thread per query over args.c[0..n_slots)
// (1..4 cascades); half: the maps hold RGBA16F texels.  args.n > 0.
struct QueryArgs;
cudaError_t launch_query_surface(const QueryArgs& args, int n_slots, bool half, cudaStream_t stream);
// Ray casts (same files): one launch, one thread per ray over args.q.c[0..n_slots).  args.n > 0.
struct RayArgs;
cudaError_t launch_raycast_surface(const RayArgs& args, int n_slots, bool half, cudaStream_t stream);
// Hydrostatics (wso_hydro.cu, body in wso_hydro.cuh): one launch, one 256-thread CTA per body over args.q.c[0..n_slots).
// 1 <= args.n < 2^31.
struct HydroArgs;
cudaError_t launch_hydrostatics(const HydroArgs& args, int n_slots, bool half, cudaStream_t stream);

}  // namespace wso
