// wso_api.cu — the C ABI (include/wsocean.h): context, buffers, Prepare(), batching, host copies.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include <cuda.h>  // types of the virtual-memory API only; entry points come from cudaGetDriverEntryPoint

#include "wso_host_prepare.h"
#include "wso_kernels.cuh"
#include "wso_launch.h"
#include "wso_query.cuh"
#include "wsocean.h"

static_assert(sizeof(wso_surface_sample) == 2 * sizeof(float4), "one query record = two float4 stores");
static_assert(sizeof(wso_ray_hit) == 48, "one ray record = three float4 stores");
static_assert(WSO_RAY_INVALID == wso::kRayInvalid && WSO_RAY_UNRESOLVED == wso::kRayUnresolved && WSO_RAY_HIT == wso::kRayHit,
              "ray status codes of the C ABI and the kernel body");

using wso::BatchItem;
using wso::LaunchArgs;
using wso::TileDev;

namespace {

std::mutex g_err_mutex;
std::string g_create_error;

struct Tile {
    wso_params params;          // as set (pending until the next prepare, except lambda)
    wso_params prepared;        // parameters the resident h0 was built with
    bool is_prepared = false;
    std::vector<wso_h0_record> h0;  // host copy in the reference layout (export / checkpoint)
};

// What a map slot holds, for the surface queries: whether a compute has written it since its maps were last reset, the
// tile_length of the tile that compute used (as prepared) and the lambda in effect.  Host-side bookkeeping only.
struct SlotFrame {
    bool valid = false;
    float length = 0.0f;
    float lambda = 0.0f;
};

enum BackingKind { kBackCudaMalloc = 0, kBackExportable = 1, kBackExternal = 2 };
struct MapBacking {
    int kind = kBackCudaMalloc;
    CUmemGenericAllocationHandle handle = 0;  // kBackExportable
    size_t mapped_bytes = 0;                  // kBackExportable: granularity-rounded size of the mapping
    cudaExternalMemory_t ext = nullptr;       // kBackExternal
};

}  // namespace

struct wso_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t copy_stream = nullptr;
    cudaStream_t aux_stream = nullptr;  // second compute lane: odd chunks of a batch (fills the tails of the even ones)
    cudaStream_t more_lanes[2] = {nullptr, nullptr};  // third / fourth compute lane of wso_compute_batch (WSO_LANES)
    cudaEvent_t ev_lane_join[2] = {nullptr, nullptr};
    int lanes = 2;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaEvent_t ev_async = nullptr;  // wso_compute_async
    cudaStream_t stream = nullptr;  // the one kernels run on (own_stream unless wso_set_stream)
    cudaEvent_t ev_chunk[2] = {nullptr, nullptr};
    cudaEvent_t ev_copied[2] = {nullptr, nullptr};
    uint32_t n = 0;
    int logn = 0;
    uint32_t max_tiles = 1, max_slots = 1;
    uint32_t chunk = 1;
    bool first_use = true;
    bool jacobian = false;  // disp.w = Jacobian instead of 1.0f (wso_set_compute_jacobian, SURVEY row f-4)
    int map_format = WSO_MAP_RGBA32F;  // texel format of both maps (wso_set_map_format); sizes: map_texel_bytes()
    uint64_t launches = 0;
    std::vector<Tile> tiles;
    // device
    float4* d_h0 = nullptr;      // [tile][n][m] (amp.re, amp.im, 1/|k|, omega or j)
    float4* d_hs = nullptr;      // [tile][j][i][2] pair-summed records (see TileDev::hs)
    float* d_kv = nullptr;       // [tile][N]
    float2* d_tw = nullptr;      // [N]
    float2* d_W = nullptr;       // [2][chunk][N/2][4][N]  (double buffered across chunks)
    wso::FrameGraph frame_graph;  // launch sequence of one tile-frame as an instantiated CUDA graph (wso_launch.h)
    int frame_graph_mode = 1;     // 0: plain launches, 1: graph for sizes up to 512^2, 2: graph for every size (WSO_FRAME_GRAPH)
    bool l2_policy_done = false; // WSO_EXP_L2_PERSIST_MB examined (experiment hook in wso_compute_batch)
    float4* d_disp = nullptr;    // [slot][N*N] texels of map_texel_bytes() each (RGBA16F: Half4, see map_slot)
    float4* d_norm = nullptr;
    float* d_minmax = nullptr;   // [slot][2]
    float* d_ampl = nullptr;     // [slot]
    std::vector<SlotFrame> slot_frames;  // [slot] (wso_query_surface)
    void* d_stage_in = nullptr;          // staging of the blocking surface queries and ray casts, grown on demand
    void* d_stage_out = nullptr;
    size_t stage_in_bytes = 0, stage_out_bytes = 0;
    // how each map array (0 = displacement, 1 = normal) is backed: cudaMalloc, an exportable virtual-memory
    // allocation, or memory imported from another API (wso_set_exportable / wso_import_external_fd)
    MapBacking map_mem[2];
    bool exportable = false;
    cudaExternalSemaphore_t ext_sem[2] = {nullptr, nullptr};
    // pinned host
    void* h_disp = nullptr;      // slot 0 mirror for wso_compute / wso_map_host_bytes (N*N texels in the map format)
    void* h_norm = nullptr;
    float* h_small = nullptr;    // [small_cap][3] amplitude,min,max staging
    size_t small_cap = 0;
    std::vector<TileDev> h_tiles;
    // opt-in per-kernel timing (wso_set_profiling): one event quad per chunk launch, resolved lazily
    bool profiling = false;
    std::vector<cudaEvent_t> prof_events;  // 4 per launch
    size_t prof_used = 0;                  // events handed out since the last resolve
    double prof_ms[3] = {0.0, 0.0, 0.0};
    uint64_t prof_launches = 0;
    uint64_t prof_items = 0;
    std::string err;
};

namespace {

int fail(wso_ctx* c, int code, const std::string& msg) {
    if (c) c->err = msg;
    else {
        std::lock_guard<std::mutex> lk(g_err_mutex);
        g_create_error = msg;
    }
    return code;
}
int fail_cuda(wso_ctx* c, cudaError_t e, const char* what) {
    const int code = (e == cudaErrorMemoryAllocation) ? WSO_ERR_OUT_OF_MEMORY : WSO_ERR_CUDA;
    return fail(c, code, std::string(what) + ": " + cudaGetErrorString(e));
}
#define WSO_CUDA(c, call)                                   \
    do {                                                    \
        cudaError_t e_ = (call);                            \
        if (e_ != cudaSuccess) return fail_cuda(c, e_, #call); \
    } while (0)

bool valid_tile_size(uint32_t n, int* logn) {
    if (n == 0 || (n & (n - 1)) != 0) return false;
    int l = 0;
    while ((1u << l) < n) ++l;
    if (l < wso::kMinLogN || l > wso::kMaxLogN) return false;
    if (logn) *logn = l;
    return true;
}

bool valid_params(const wso_params& p) {
    if (!(p.tile_length > 0.0f)) return false;
    if (!(p.wind_dir_x != 0.0f || p.wind_dir_y != 0.0f)) return false;
    if (!std::isfinite(p.wind_dir_x) || !std::isfinite(p.wind_dir_y)) return false;
    if (!(p.anim_period > 0.0f)) return false;
    if (!std::isfinite(p.wind_speed) || !std::isfinite(p.phillips_const) || !std::isfinite(p.damping) ||
        !std::isfinite(p.lambda))
        return false;
    return true;
}

// ---- CUDA virtual-memory API through the runtime's driver-entry-point lookup (libwsocean.so does not link libcuda)
struct VmmApi {
    CUresult (*GetGranularity)(size_t*, const CUmemAllocationProp*, CUmemAllocationGranularity_flags) = nullptr;
    CUresult (*Create)(CUmemGenericAllocationHandle*, size_t, const CUmemAllocationProp*, unsigned long long) = nullptr;
    CUresult (*AddressReserve)(CUdeviceptr*, size_t, size_t, CUdeviceptr, unsigned long long) = nullptr;
    CUresult (*Map)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long) = nullptr;
    CUresult (*SetAccess)(CUdeviceptr, size_t, const CUmemAccessDesc*, size_t) = nullptr;
    CUresult (*Unmap)(CUdeviceptr, size_t) = nullptr;
    CUresult (*Release)(CUmemGenericAllocationHandle) = nullptr;
    CUresult (*AddressFree)(CUdeviceptr, size_t) = nullptr;
    CUresult (*ExportHandle)(void*, CUmemGenericAllocationHandle, CUmemAllocationHandleType, unsigned long long) = nullptr;
    bool ok = false;
};

const VmmApi& vmm_api() {
    static const VmmApi api = [] {
        VmmApi a;
        bool ok = true;
        auto get = [&](const char* name, void** fn) {
            cudaDriverEntryPointQueryResult q;
            if (cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess ||
                *fn == nullptr)
                ok = false;
        };
        get("cuMemGetAllocationGranularity", (void**)&a.GetGranularity);
        get("cuMemCreate", (void**)&a.Create);
        get("cuMemAddressReserve", (void**)&a.AddressReserve);
        get("cuMemMap", (void**)&a.Map);
        get("cuMemSetAccess", (void**)&a.SetAccess);
        get("cuMemUnmap", (void**)&a.Unmap);
        get("cuMemRelease", (void**)&a.Release);
        get("cuMemAddressFree", (void**)&a.AddressFree);
        get("cuMemExportToShareableHandle", (void**)&a.ExportHandle);
        a.ok = ok;
        return a;
    }();
    return api;
}

float4*& map_ptr(wso_ctx* c, int which) { return which == 0 ? c->d_disp : c->d_norm; }

// Bytes of one map texel in the context's format: the one source for every size, offset and pitch of the map arrays,
// their pinned mirrors and the host copies.  Slot s of a map starts at byte s * map_texel_bytes * N*N.
size_t map_texel_bytes(const wso_ctx* c) { return c->map_format == WSO_MAP_RGBA16F ? sizeof(wso::Half4) : sizeof(float4); }
size_t map_slot_bytes(const wso_ctx* c) { return map_texel_bytes(c) * (size_t)c->n * c->n; }
char* map_slot(wso_ctx* c, int which, uint32_t slot) {
    return reinterpret_cast<char*>(map_ptr(c, which)) + map_slot_bytes(c) * slot;
}

// Every slot's maps are gone or reset: no slot holds a queryable frame until the next compute writes it.
void forget_frames(wso_ctx* c) {
    for (SlotFrame& f : c->slot_frames) f = SlotFrame{};
}

void free_map(wso_ctx* c, int which) {
    forget_frames(c);
    MapBacking& b = c->map_mem[which];
    float4*& p = map_ptr(c, which);
    if (p != nullptr) {
        if (b.kind == kBackExportable) {
            const VmmApi& v = vmm_api();
            v.Unmap((CUdeviceptr)p, b.mapped_bytes);
            v.Release(b.handle);
            v.AddressFree((CUdeviceptr)p, b.mapped_bytes);
        } else if (b.kind == kBackExternal) {
            cudaFree(p);  // releases the mapping of the imported object
            cudaDestroyExternalMemory(b.ext);
        } else {
            cudaFree(p);
        }
    }
    p = nullptr;
    b = MapBacking{};
}

// Allocate the [slot][N*N] array of one map: cudaMalloc, or - when the context is exportable - a physical allocation
// that can be exported as a POSIX file descriptor, mapped into a reserved address range.
int alloc_map(wso_ctx* c, int which, size_t bytes) {
    free_map(c, which);
    float4*& p = map_ptr(c, which);
    if (!c->exportable) {
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return fail_cuda(c, e, "cudaMalloc(map)");
        return WSO_OK;
    }
    const VmmApi& v = vmm_api();
    if (!v.ok) return fail(c, WSO_ERR_CUDA, "the CUDA driver does not provide the virtual-memory API");
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = c->device;
    prop.requestedHandleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
    size_t gran = 0;
    if (v.GetGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_MINIMUM) != CUDA_SUCCESS || gran == 0)
        return fail(c, WSO_ERR_CUDA, "cuMemGetAllocationGranularity failed");
    const size_t size = (bytes + gran - 1) / gran * gran;
    MapBacking b;
    b.kind = kBackExportable;
    b.mapped_bytes = size;
    CUresult r = v.Create(&b.handle, size, &prop, 0);
    if (r != CUDA_SUCCESS)
        return fail(c, r == CUDA_ERROR_OUT_OF_MEMORY ? WSO_ERR_OUT_OF_MEMORY : WSO_ERR_CUDA, "cuMemCreate(exportable map) failed");
    CUdeviceptr va = 0;
    if (v.AddressReserve(&va, size, 0, 0, 0) != CUDA_SUCCESS) {
        v.Release(b.handle);
        return fail(c, WSO_ERR_CUDA, "cuMemAddressReserve failed");
    }
    CUmemAccessDesc acc = {};
    acc.location = prop.location;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    if (v.Map(va, size, 0, b.handle, 0) != CUDA_SUCCESS || v.SetAccess(va, size, &acc, 1) != CUDA_SUCCESS) {
        v.Unmap(va, size);
        v.Release(b.handle);
        v.AddressFree(va, size);
        return fail(c, WSO_ERR_CUDA, "cuMemMap / cuMemSetAccess failed");
    }
    p = reinterpret_cast<float4*>(va);
    c->map_mem[which] = b;
    return WSO_OK;
}

void free_device_buffers(wso_ctx* c) {
    cudaFree(c->d_h0); c->d_h0 = nullptr;
    cudaFree(c->d_hs); c->d_hs = nullptr;
    cudaFree(c->d_kv); c->d_kv = nullptr;
    cudaFree(c->d_tw); c->d_tw = nullptr;
    cudaFree(c->d_W); c->d_W = nullptr;
    c->l2_policy_done = false;
    free_map(c, 0);
    free_map(c, 1);
    cudaFree(c->d_minmax); c->d_minmax = nullptr;
    cudaFree(c->d_ampl); c->d_ampl = nullptr;
    cudaFreeHost(c->h_disp); c->h_disp = nullptr;
    cudaFreeHost(c->h_norm); c->h_norm = nullptr;
    cudaFreeHost(c->h_small); c->h_small = nullptr;
}

// Map contents before the first ComputeWaves(): the reference's resize() defaults (WSTessendorf.cpp:48-54) -
// displacement (0,0,0,0), normal (0,1,0,0) - in every device slot and in the pinned host mirrors of slot 0.
// RGBA16F: the same values in binary16, normal (0, 1, 0, 0) = halves (0x0000, 0x3c00, 0x0000, 0x0000).
int reset_map_contents(wso_ctx* c, size_t n2, int which_mask = 3) {
    forget_frames(c);
    const size_t tb = map_texel_bytes(c);
    if (which_mask & 1) {
        WSO_CUDA(c, cudaMemsetAsync(c->d_disp, 0, tb * n2 * c->max_slots, c->stream));
        if (c->h_disp) std::memset(c->h_disp, 0, tb * n2);
    }
    if ((which_mask & 2) && c->h_norm) {
        if (c->map_format == WSO_MAP_RGBA16F) {
            const wso::Half4 up = {0x3c00u << 16, 0u};
            wso::Half4* h = static_cast<wso::Half4*>(c->h_norm);
            for (size_t i = 0; i < n2; ++i) h[i] = up;
        } else {
            const float4 up = make_float4(0.0f, 1.0f, 0.0f, 0.0f);
            float4* h = static_cast<float4*>(c->h_norm);
            for (size_t i = 0; i < n2; ++i) h[i] = up;
        }
        // (slot offsets from n2: while the buffers of a new size are allocated, c->n is still 0)
        for (uint32_t sl = 0; sl < c->max_slots; ++sl)
            WSO_CUDA(c, cudaMemcpyAsync(reinterpret_cast<char*>(c->d_norm) + tb * n2 * sl, c->h_norm, tb * n2,
                                        cudaMemcpyHostToDevice, c->stream));
    }
    return WSO_OK;
}

int allocate_buffers(wso_ctx* c, uint32_t n, int logn);

// (Re)allocate everything that depends on the tile size.
int allocate_for_size(wso_ctx* c, uint32_t n) {
    int logn = 0;
    if (!valid_tile_size(n, &logn)) return fail(c, WSO_ERR_BAD_TILE_SIZE, "tile size must be a power of two in [16, 8192]");
    WSO_CUDA(c, cudaSetDevice(c->device));
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    free_device_buffers(c);
    // Nothing is resident from here on: should any allocation below fail, the context stays in the "no tile prepared,
    // no size" state (compute calls answer WSO_ERR_NOT_PREPARED, the map accessors report zero texels) instead of
    // pointing kernels at freed buffers.
    c->n = 0;
    c->logn = 0;
    c->first_use = true;
    for (uint32_t t = 0; t < c->max_tiles; ++t) {
        c->tiles[t].is_prepared = false;
        c->tiles[t].h0.clear();
    }
    c->h_tiles.assign(c->max_tiles, TileDev{});
    const int rc_alloc = allocate_buffers(c, n, logn);
    if (rc_alloc != WSO_OK) {
        free_device_buffers(c);
        return rc_alloc;
    }
    c->n = n;
    c->logn = logn;
    return WSO_OK;
}

int allocate_buffers(wso_ctx* c, uint32_t n, int logn) {
    (void)logn;
    const size_t n2 = (size_t)n * n;
    // chunk: tile-frames per launch.  Keep the W scratch of one chunk around 64 MB so it stays in the
    // 126 MB L2 between K1 and K2 (DESIGN.md §4; 16/32/48/64/96 MB measured on B200, profiles/r1j_sweep.txt:
    // 1024^2 42.5k / 52.8k / 52.6k / 54.9k / 54.8k tile-frames/s).
    const size_t w_item = n2 * 16;
    size_t budget_mb = 64;
    if (const char* env = std::getenv("WSO_W_BUDGET_MB")) {
        const long v = std::atol(env);
        if (v > 0 && v <= 65536) budget_mb = (size_t)v;
    }
    size_t chunk = (budget_mb << 20) / w_item;
    if (chunk < 1) chunk = 1;
    if (chunk > (size_t)wso::kMaxChunk) chunk = wso::kMaxChunk;
    if (chunk > c->max_slots) chunk = c->max_slots;
    c->chunk = (uint32_t)chunk;
    WSO_CUDA(c, cudaMalloc(&c->d_h0, sizeof(float4) * n2 * c->max_tiles));
    WSO_CUDA(c, cudaMalloc(&c->d_hs, sizeof(float4) * (n2 / 2) * c->max_tiles));
    WSO_CUDA(c, cudaMalloc(&c->d_kv, sizeof(float) * n * c->max_tiles));
    WSO_CUDA(c, cudaMalloc(&c->d_tw, sizeof(float2) * n));
    WSO_CUDA(c, cudaMalloc(&c->d_W, w_item * chunk * (size_t)(c->lanes > 2 ? c->lanes : 2)));
    for (int which = 0; which < 2; ++which) {
        const int rc = alloc_map(c, which, map_texel_bytes(c) * n2 * c->max_slots);
        if (rc != WSO_OK) return rc;
    }
    WSO_CUDA(c, cudaMalloc(&c->d_minmax, sizeof(float) * 2 * c->max_slots));
    WSO_CUDA(c, cudaMalloc(&c->d_ampl, sizeof(float) * c->max_slots));
    WSO_CUDA(c, cudaMallocHost(&c->h_disp, map_texel_bytes(c) * n2));
    WSO_CUDA(c, cudaMallocHost(&c->h_norm, map_texel_bytes(c) * n2));
    c->small_cap = c->max_slots;
    WSO_CUDA(c, cudaMallocHost(&c->h_small, sizeof(float) * 3 * c->small_cap));
    {
        const int rc = reset_map_contents(c, n2);
        if (rc != WSO_OK) return rc;
    }
    // twiddles exp(+2 pi i k / N), computed in float64
    std::vector<float2> tw(n);
    for (uint32_t k = 0; k < n; ++k) {
        const double a = 2.0 * 3.14159265358979323846 * (double)k / (double)n;
        tw[k] = make_float2((float)std::cos(a), (float)std::sin(a));
    }
    WSO_CUDA(c, cudaMemcpyAsync(c->d_tw, tw.data(), sizeof(float2) * n, cudaMemcpyHostToDevice, c->stream));
    for (uint32_t t = 0; t < c->max_tiles; ++t) {
        c->h_tiles[t].h0 = c->d_h0 + n2 * t;
        c->h_tiles[t].hs = c->d_hs + (n2 / 2) * t;
        c->h_tiles[t].kv = c->d_kv + (size_t)n * t;
        c->h_tiles[t].lambda = c->tiles[t].params.lambda;
        c->h_tiles[t].omega0 = 0.0f;
        c->h_tiles[t].table_len = 0;
        c->h_tiles[t].use_pairs = 0;
        c->tiles[t].is_prepared = false;
        c->tiles[t].h0.clear();
    }
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    return WSO_OK;
}

// Upload one tile's h0 (reference layout, row-major [m][n]) as the transposed compact arrays the kernels read.
int upload_h0(wso_ctx* c, uint32_t tile, const wso_h0_record* h0) {
    const uint32_t n = c->n;
    const size_t n2 = (size_t)n * n;
    for (size_t i = 0; i < n2; ++i) {
        // every reference-built h0 has heightAmp_conj == conj(heightAmp) (WSTessendorf.cpp:132-135)
        if (!(h0[i].amp_conj_re == h0[i].amp_re && h0[i].amp_conj_im == -h0[i].amp_im))
            return fail(c, WSO_ERR_H0_NOT_CONJUGATE, "h0: heightAmp_conj != conj(heightAmp)");
    }
    std::vector<float> kv;
    wso::host_wave_numbers(n, c->tiles[tile].params.tile_length, kv);
    // The quantised dispersion takes few distinct values j*omega0 (reference: QDispersion, WSTessendorf.h:284-287).
    // When every omega is EXACTLY fl(float(j)*omega0) with a small j, the kernels use a per-frame (cos,sin) table
    // over j instead of one sincosf per wave vector - bit-identical, since the table entry evaluates the same
    // fp32 phase fl(omega*t).  Otherwise (e.g. an imported h0 with foreign dispersion) omega itself is stored.
    const float omega0 = wso::derive_params(c->tiles[tile].params).base_freq;
    int jmax = 0;
    bool table_ok = omega0 > 0.0f;
    for (size_t i = 0; i < n2 && table_ok; ++i) {
        const float w = h0[i].dispersion;
        const float jf = std::nearbyint(w / omega0);
        if (!(jf >= 0.0f && jf < (float)wso::kMaxTable) || jf * omega0 != w) table_ok = false;
        else if ((int)jf > jmax) jmax = (int)jf;
    }
    std::vector<float4> rec(n2);
    for (uint32_t m = 0; m < n; ++m)
        for (uint32_t k = 0; k < n; ++k) {
            const wso_h0_record& r = h0[(size_t)m * n + k];
            // 1/|k| exactly as glm::normalize computes it (reference: WSTessendorf.h:133-136)
            const float d = kv[k] * kv[k] + kv[m] * kv[m];
            const float inv = std::sqrt(d) > 0.00001f ? 1.0f / std::sqrt(d) : 0.0f;
            float wfield = r.dispersion;
            if (table_ok) {
                const int j = (int)std::nearbyint(r.dispersion / omega0);
                std::memcpy(&wfield, &j, sizeof(float));
            }
            rec[wso::h0_index((int)k, (int)m, (int)n, 0)] = make_float4(r.amp_re, r.amp_im, inv, wfield);
        }
    // pair-summed records for the interior (i,j >= 1): amplitude h0(k) + h0(-k); 1/|k| and omega are even in k
    const uint32_t hN = n / 2;
    std::vector<float4> recs((size_t)hN * hN * 2, make_float4(0.f, 0.f, 0.f, 0.f));
    bool pairs_ok = true;  // needs omega(k) == omega(-k): true for any dispersion that depends on |k| only
    for (uint32_t j = 1; j < hN; ++j)
        for (uint32_t i = 1; i < hN; ++i) {
            const int N_ = (int)n;
            const float4 a0 = rec[wso::h0_index((int)j, (int)i, N_, 0)], a3 = rec[wso::h0_index(N_ - (int)j, N_ - (int)i, N_, 0)];
            const float4 a1 = rec[wso::h0_index(N_ - (int)j, (int)i, N_, 0)], a2 = rec[wso::h0_index((int)j, N_ - (int)i, N_, 0)];
            if (std::memcmp(&a0.w, &a3.w, 4) != 0 || std::memcmp(&a1.w, &a2.w, 4) != 0) pairs_ok = false;
            recs[wso::hs_index((int)j, (int)i, 0, (int)hN)] = make_float4(a0.x + a3.x, a0.y + a3.y, a0.z, a0.w);
            recs[wso::hs_index((int)j, (int)i, 1, (int)hN)] = make_float4(a1.x + a2.x, a1.y + a2.y, a1.z, a1.w);
        }
    WSO_CUDA(c, cudaSetDevice(c->device));
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    WSO_CUDA(c, cudaMemcpy(c->d_h0 + n2 * tile, rec.data(), sizeof(float4) * n2, cudaMemcpyHostToDevice));
    WSO_CUDA(c, cudaMemcpy(c->d_hs + (n2 / 2) * tile, recs.data(), sizeof(float4) * (n2 / 2), cudaMemcpyHostToDevice));
    WSO_CUDA(c, cudaMemcpy(c->d_kv + (size_t)n * tile, kv.data(), sizeof(float) * n, cudaMemcpyHostToDevice));
    c->h_tiles[tile].omega0 = omega0;
    c->h_tiles[tile].table_len = table_ok ? jmax + 1 : 0;
    c->h_tiles[tile].use_pairs = pairs_ok ? 1 : 0;
    Tile& tl = c->tiles[tile];
    if (tl.h0.data() != h0) tl.h0.assign(h0, h0 + n2);
    tl.prepared = tl.params;
    tl.is_prepared = true;
    return WSO_OK;
}

// lambda takes effect at the next compute without a Prepare (reference: SetLambda, WSTessendorf.h:181); the tile
// constants travel by value with every launch, so refreshing the host copy is all there is to do
int push_lambdas(wso_ctx* c) {
    for (uint32_t t = 0; t < c->max_tiles; ++t) c->h_tiles[t].lambda = c->tiles[t].params.lambda;
    return WSO_OK;
}

// Prepare step shared by wso_prepare / wso_prepare_gauss: apply pending params (possibly a new size).
int begin_prepare(wso_ctx* c, uint32_t tile) {
    if (!c) return WSO_ERR_INVALID_ARG;
    if (tile >= c->max_tiles) return fail(c, WSO_ERR_INVALID_ARG, "tile index out of range");
    const wso_params& p = c->tiles[tile].params;
    if (p.tile_size != c->n) {
        const int rc = allocate_for_size(c, p.tile_size);
        if (rc != WSO_OK) return rc;
    }
    return WSO_OK;
}

static constexpr int kFrameGraphMaxLogN = 9;

int enqueue_chunk(wso_ctx* c, uint32_t n_items, const uint32_t* tiles, const float* t, uint32_t first_slot,
                  int wbuf, cudaStream_t stream) {
    LaunchArgs args;
    args.tw = c->d_tw;
    args.W = c->d_W + (size_t)wbuf * c->chunk * ((size_t)c->n * c->n * 2);
    args.disp = c->d_disp;
    args.norm = c->d_norm;
    args.minmax = c->d_minmax;
    args.amp_out = c->d_ampl;
    for (uint32_t i = 0; i < n_items; ++i) {
        args.items[i].tile = tiles ? tiles[i] : 0u;
        args.items[i].slot = first_slot + i;
        args.items[i].t = t[i];
        args.td[i] = c->h_tiles[args.items[i].tile];
    }
    for (uint32_t i = n_items; i < (uint32_t)wso::kMaxChunk; ++i) {
        args.items[i] = BatchItem{0u, 0u, 0.0f};
        args.td[i] = TileDev{};
    }
    cudaEvent_t* ev = nullptr;
    if (c->profiling) {
        if (c->prof_used + 4 > c->prof_events.size()) {
            for (int i = 0; i < 4; ++i) {
                cudaEvent_t x;
                cudaError_t ee = cudaEventCreate(&x);
                if (ee != cudaSuccess) return fail_cuda(c, ee, "cudaEventCreate");
                c->prof_events.push_back(x);
            }
        }
        ev = c->prof_events.data() + c->prof_used;
        c->prof_used += 4;
        c->prof_launches += 1;
        c->prof_items += n_items;
    }
    if (c->jacobian && c->logn > wso::kMaxJacobianLogN)
        return fail(c, WSO_ERR_INVALID_ARG, "the Jacobian channel is available for tile sizes up to 4096");
    // a single tile-frame (the reference's one ComputeWaves(t) per rendered frame) goes out as one graph launch
    // (up to 512^2, where the three launches cost more host time than the kernels take; from 1024^2 on plain launches are
    // faster back to back - K1 of the next frame overlaps K2 of this one through programmatic dependent launch, which does not
    // reach across graph launches: profiles/r3_frame_graph.md.  Mode 2 = every size.)
    const bool as_graph = n_items == 1 && ev == nullptr &&
                          (c->frame_graph_mode == 2 || (c->frame_graph_mode == 1 && c->logn <= kFrameGraphMaxLogN));
    const bool half = c->map_format == WSO_MAP_RGBA16F;
    cudaError_t e = as_graph ? wso::launch_frame_graph(c->frame_graph, c->logn, args, stream, c->jacobian, half)
                             : wso::launch_compute_waves(c->logn, args, (int)n_items, stream, c->jacobian, half, ev);
    if (e != cudaSuccess) return fail_cuda(c, e, "kernel launch");
    c->first_use = false;
    c->launches += (uint64_t)wso::kernels_per_launch();
    for (uint32_t i = 0; i < n_items; ++i) {
        const uint32_t tl = args.items[i].tile;
        c->slot_frames[args.items[i].slot] = SlotFrame{true, c->tiles[tl].prepared.tile_length, args.td[i].lambda};
    }
    return WSO_OK;
}

// Prepare() on the device (SURVEY row f-3): one kernel builds both record arrays of the tile from a Gaussian array
// already in device memory (d_xi) or from the counter-based generator (d_xi == NULL).
int prepare_on_device(wso_ctx* c, uint32_t tile, const float2* d_xi, uint64_t seed) {
    const uint32_t n = c->n;
    Tile& tl = c->tiles[tile];
    const wso::DerivedParams d = wso::derive_params(tl.params);
    std::vector<float> kv;
    wso::host_wave_numbers(n, tl.params.tile_length, kv);
    // largest multiple j of the base frequency: the wave vector of index (0,0) has the largest |k|, and
    // floor(sqrt(g k)/omega0) is monotone in |k| (same fp32 operations as the kernel)
    const float kmax = std::sqrt(kv[0] * kv[0] + kv[0] * kv[0]);
    const float jf = std::floor(std::sqrt(9.81f * kmax) / d.base_freq);
    if (!(d.base_freq > 0.0f) || !(jf >= 0.0f && jf < (float)wso::kMaxTable))
        return fail(c, WSO_ERR_INVALID_ARG, "device Prepare: dispersion table would exceed 1024 entries (use wso_prepare)");
    wso::PrepareArgs a;
    a.h0 = c->d_h0 + (size_t)n * n * tile;
    a.hs = c->d_hs + ((size_t)n * n / 2) * tile;
    a.kv = c->d_kv + (size_t)n * tile;
    a.xi = d_xi;
    a.seed_mixed = wso::counter_seed_mix(seed);
    a.n = (int)n;
    a.j0 = 0;
    a.wind_x = d.wind_x;
    a.wind_y = d.wind_y;
    a.omega0 = d.base_freq;
    a.phillips_const = tl.params.phillips_const;
    a.damping = tl.params.damping;
    a.inv_sqrt2 = 1.0f / std::sqrt(2.0f);
    const float Lw = d.wind_speed * d.wind_speed / 9.81f;
    a.Lw2 = Lw * Lw;
    WSO_CUDA(c, cudaSetDevice(c->device));
    WSO_CUDA(c, cudaMemcpyAsync(c->d_kv + (size_t)n * tile, kv.data(), sizeof(float) * n, cudaMemcpyHostToDevice, c->stream));
    WSO_CUDA(c, wso::launch_prepare(a, (int)(n / 2), c->stream));
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    c->launches += 1;
    c->h_tiles[tile].omega0 = d.base_freq;
    c->h_tiles[tile].table_len = (int)jf + 1;
    c->h_tiles[tile].use_pairs = 1;
    tl.h0.clear();  // the records live on the device only; wso_export_h0 reads them back
    tl.prepared = tl.params;
    tl.is_prepared = true;
    return WSO_OK;
}

int check_batch(wso_ctx* c, uint32_t n, const uint32_t* tiles, const float* t, uint32_t first_slot) {
    if (!c) return WSO_ERR_INVALID_ARG;
    if (!t) return fail(c, WSO_ERR_INVALID_ARG, "t is NULL");
    if ((uint64_t)first_slot + n > c->max_slots) return fail(c, WSO_ERR_INVALID_ARG, "slots out of range");
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t tl = tiles ? tiles[i] : 0u;
        if (tl >= c->max_tiles) return fail(c, WSO_ERR_INVALID_ARG, "tile index out of range");
        if (!c->tiles[tl].is_prepared) return fail(c, WSO_ERR_NOT_PREPARED, "Prepare() has not been called for this tile");
    }
    return WSO_OK;
}

}  // namespace

extern "C" {

int wso_default_params(wso_params* p) {
    if (!p) return WSO_ERR_INVALID_ARG;
    p->tile_size = 512;       // reference: WSTessendorf.h:36-43
    p->tile_length = 1000.0f;
    p->wind_dir_x = 1.0f;
    p->wind_dir_y = 1.0f;
    p->wind_speed = 30.0f;
    p->anim_period = 200.0f;
    p->phillips_const = 3e-7f;
    p->damping = 0.1f;
    p->lambda = -1.0f;        // reference: WSTessendorf.h:181
    return WSO_OK;
}

int wso_create(const wso_params* p, int device, uint32_t max_tiles, uint32_t max_slots, wso_ctx** out) {
    if (!p || !out || max_tiles == 0 || max_slots == 0) return fail(nullptr, WSO_ERR_INVALID_ARG, "bad argument");
    *out = nullptr;
    if (!valid_tile_size(p->tile_size, nullptr))
        return fail(nullptr, WSO_ERR_BAD_TILE_SIZE, "tile size must be a power of two in [16, 8192]");
    if (!valid_params(*p)) return fail(nullptr, WSO_ERR_INVALID_ARG, "invalid parameters");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, WSO_ERR_CUDA, std::string("no usable CUDA device (no CPU fallback exists): ") +
                                               (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    if (device < 0 || device >= ndev) return fail(nullptr, WSO_ERR_INVALID_ARG, "device ordinal out of range");
    wso_ctx* c = new (std::nothrow) wso_ctx();
    if (!c) return fail(nullptr, WSO_ERR_OUT_OF_MEMORY, "host allocation failed");
    c->device = device;
    c->max_tiles = max_tiles;
    c->max_slots = max_slots;
    c->tiles.resize(max_tiles);
    c->slot_frames.resize(max_slots);
    wso_params p0 = *p;
    wso::normalise_like_setters(p0, nullptr);
    for (auto& tl : c->tiles) tl.params = p0;
    int rc = WSO_OK;
    do {
        if ((e = cudaSetDevice(device)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaSetDevice"); break; }
        if ((e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaStreamCreate"); break; }
        if ((e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaStreamCreate"); break; }
        if ((e = cudaStreamCreateWithFlags(&c->aux_stream, cudaStreamNonBlocking)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaStreamCreate"); break; }
        if (const char* env = std::getenv("WSO_FRAME_GRAPH")) {
            const int v = std::atoi(env);
            c->frame_graph_mode = v < 0 ? 0 : (v > 2 ? 2 : v);
        }
        if (const char* env = std::getenv("WSO_LANES")) {  // compute lanes of a batched call (default 2)
            const int v = std::atoi(env);
            if (v >= 1 && v <= 4) c->lanes = v;
        }
        for (int i = 0; i < 2 && rc == WSO_OK; ++i) {
            if ((e = cudaStreamCreateWithFlags(&c->more_lanes[i], cudaStreamNonBlocking)) != cudaSuccess) rc = fail_cuda(nullptr, e, "cudaStreamCreate");
            else if ((e = cudaEventCreateWithFlags(&c->ev_lane_join[i], cudaEventDisableTiming)) != cudaSuccess) rc = fail_cuda(nullptr, e, "cudaEventCreate");
        }
        if (rc != WSO_OK) break;
        if ((e = cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaEventCreate"); break; }
        if ((e = cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming)) != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaEventCreate"); break; }
        for (int i = 0; i < 2; ++i) {
            if ((e = cudaEventCreateWithFlags(&c->ev_chunk[i], cudaEventDisableTiming)) != cudaSuccess) break;
            if ((e = cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming)) != cudaSuccess) break;
        }
        if (e != cudaSuccess) { rc = fail_cuda(nullptr, e, "cudaEventCreate"); break; }
        c->stream = c->own_stream;
        rc = allocate_for_size(c, p->tile_size);
        if (rc != WSO_OK) fail(nullptr, rc, c->err);
    } while (0);
    if (rc != WSO_OK) {
        wso_destroy(c);
        return rc;
    }
    *out = c;
    return WSO_OK;
}

int wso_destroy(wso_ctx* c) {
    if (!c) return WSO_OK;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    if (c->aux_stream) cudaStreamSynchronize(c->aux_stream);
    wso::destroy_frame_graph(c->frame_graph);
    free_device_buffers(c);
    cudaFree(c->d_stage_in);
    cudaFree(c->d_stage_out);
    for (int i = 0; i < 2; ++i)
        if (c->ext_sem[i]) cudaDestroyExternalSemaphore(c->ext_sem[i]);
    if (c->ev_async) cudaEventDestroy(c->ev_async);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    if (c->aux_stream) cudaStreamDestroy(c->aux_stream);
    for (int i = 0; i < 2; ++i) {
        if (c->more_lanes[i]) {
            cudaStreamSynchronize(c->more_lanes[i]);
            cudaStreamDestroy(c->more_lanes[i]);
        }
        if (c->ev_lane_join[i]) cudaEventDestroy(c->ev_lane_join[i]);
    }
    for (int i = 0; i < 2; ++i) {
        if (c->ev_chunk[i]) cudaEventDestroy(c->ev_chunk[i]);
        if (c->ev_copied[i]) cudaEventDestroy(c->ev_copied[i]);
    }
    for (cudaEvent_t x : c->prof_events) cudaEventDestroy(x);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    delete c;
    return WSO_OK;
}

int wso_set_params(wso_ctx* c, uint32_t tile, const wso_params* p) {
    if (!c || !p) return WSO_ERR_INVALID_ARG;
    if (tile >= c->max_tiles) return fail(c, WSO_ERR_INVALID_ARG, "tile index out of range");
    if (!valid_tile_size(p->tile_size, nullptr))
        return fail(c, WSO_ERR_BAD_TILE_SIZE, "tile size must be a power of two in [16, 8192]; unchanged");
    if (p->tile_size != c->n && c->max_tiles != 1)
        return fail(c, WSO_ERR_INVALID_ARG, "tile size can only change on a single-tile context");
    if (!valid_params(*p)) return fail(c, WSO_ERR_INVALID_ARG, "invalid parameters");
    wso_params np = *p;
    wso::normalise_like_setters(np, &c->tiles[tile].params);
    c->tiles[tile].params = np;
    return WSO_OK;
}

int wso_get_params(const wso_ctx* c, uint32_t tile, wso_params* p) {
    if (!c || !p || tile >= c->max_tiles) return WSO_ERR_INVALID_ARG;
    *p = c->tiles[tile].params;  // wind direction normalised / speed clamped at set time, like the reference
    return WSO_OK;
}

int wso_set_lambda(wso_ctx* c, uint32_t tile, float lambda) {
    if (!c || tile >= c->max_tiles || !std::isfinite(lambda)) return WSO_ERR_INVALID_ARG;
    c->tiles[tile].params.lambda = lambda;
    return WSO_OK;
}

int wso_set_compute_jacobian(wso_ctx* c, int on) {
    if (!c) return WSO_ERR_INVALID_ARG;
    if (on && c->logn > wso::kMaxJacobianLogN)
        return fail(c, WSO_ERR_INVALID_ARG, "the Jacobian channel is available for tile sizes up to 4096");
    c->jacobian = on != 0;
    return WSO_OK;
}

int wso_get_compute_jacobian(const wso_ctx* c, int* on) {
    if (!c || !on) return WSO_ERR_INVALID_ARG;
    *on = c->jacobian ? 1 : 0;
    return WSO_OK;
}

int wso_prepare(wso_ctx* c, uint32_t tile, int reseed, unsigned seed) {
    int rc = begin_prepare(c, tile);
    if (rc != WSO_OK) return rc;
    if (reseed) std::srand(seed);
    std::vector<float> xi;
    wso::host_gauss_array_from_rand(c->n, xi);
    return wso_prepare_gauss(c, tile, xi.data());
}

int wso_prepare_gauss(wso_ctx* c, uint32_t tile, const float* xi) {
    int rc = begin_prepare(c, tile);
    if (rc != WSO_OK) return rc;
    if (!xi) return fail(c, WSO_ERR_INVALID_ARG, "xi is NULL");
    Tile& tl = c->tiles[tile];
    wso::host_base_wave_heights(tl.params, xi, tl.h0);
    return upload_h0(c, tile, tl.h0.data());
}

int wso_prepare_gauss_device(wso_ctx* c, uint32_t tile, const float* xi) {
    int rc = begin_prepare(c, tile);
    if (rc != WSO_OK) return rc;
    if (!xi) return fail(c, WSO_ERR_INVALID_ARG, "xi is NULL");
    const size_t bytes = sizeof(float2) * (size_t)c->n * c->n;
    float2* d_xi = nullptr;
    WSO_CUDA(c, cudaSetDevice(c->device));
    WSO_CUDA(c, cudaMalloc(&d_xi, bytes));
    cudaError_t e = cudaMemcpyAsync(d_xi, xi, bytes, cudaMemcpyHostToDevice, c->stream);
    if (e != cudaSuccess) {
        cudaFree(d_xi);
        return fail_cuda(c, e, "cudaMemcpyAsync(xi)");
    }
    rc = prepare_on_device(c, tile, d_xi, 0);
    cudaFree(d_xi);
    return rc;
}

int wso_prepare_counter(wso_ctx* c, uint32_t tile, uint64_t seed) {
    int rc = begin_prepare(c, tile);
    if (rc != WSO_OK) return rc;
    return prepare_on_device(c, tile, nullptr, seed);
}

int wso_import_h0(wso_ctx* c, uint32_t tile, const wso_h0_record* h0) {
    int rc = begin_prepare(c, tile);
    if (rc != WSO_OK) return rc;
    if (!h0) return fail(c, WSO_ERR_INVALID_ARG, "h0 is NULL");
    return upload_h0(c, tile, h0);
}

int wso_export_h0(const wso_ctx* c, uint32_t tile, wso_h0_record* h0) {
    if (!c || !h0 || tile >= c->max_tiles) return WSO_ERR_INVALID_ARG;
    const Tile& tl = c->tiles[tile];
    if (!tl.is_prepared) return WSO_ERR_NOT_PREPARED;
    if (!tl.h0.empty()) {
        std::memcpy(h0, tl.h0.data(), sizeof(wso_h0_record) * tl.h0.size());
        return WSO_OK;
    }
    // prepared on the device: rebuild the reference records from the device arrays
    static_assert(sizeof(wso_h0_record) == 20, "reference BaseWaveHeight is 5 floats");
    const size_t n2 = (size_t)c->n * c->n;
    float* d_out = nullptr;
    if (cudaSetDevice(c->device) != cudaSuccess || cudaMalloc(&d_out, n2 * 20) != cudaSuccess) return WSO_ERR_CUDA;
    const TileDev& td = c->h_tiles[tile];
    cudaError_t e = wso::launch_export_records(td.h0, d_out, (int)c->n, td.omega0, td.table_len > 0, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h0, d_out, n2 * 20, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d_out);
    return e == cudaSuccess ? WSO_OK : WSO_ERR_CUDA;
}

// Compact form of the spectrum (SURVEY 8b): heightAmp_conj == conj(heightAmp) in every reference-built h0
// (WSTessendorf.cpp:132-135), so 12 bytes per wave vector - (amp.re, amp.im, dispersion) - carry all of it.
int wso_import_h0_compact(wso_ctx* c, uint32_t tile, const float* h0_3f) {
    int rc = begin_prepare(c, tile);
    if (rc != WSO_OK) return rc;
    if (!h0_3f) return fail(c, WSO_ERR_INVALID_ARG, "h0 is NULL");
    const size_t n2 = (size_t)c->n * c->n;
    std::vector<wso_h0_record> full(n2);
    for (size_t i = 0; i < n2; ++i) {
        full[i].amp_re = h0_3f[3 * i + 0];
        full[i].amp_im = h0_3f[3 * i + 1];
        full[i].amp_conj_re = h0_3f[3 * i + 0];
        full[i].amp_conj_im = -h0_3f[3 * i + 1];
        full[i].dispersion = h0_3f[3 * i + 2];
    }
    return upload_h0(c, tile, full.data());
}

int wso_export_h0_compact(const wso_ctx* c, uint32_t tile, float* h0_3f) {
    if (!c || !h0_3f || tile >= c->max_tiles) return WSO_ERR_INVALID_ARG;
    if (!c->tiles[tile].is_prepared) return WSO_ERR_NOT_PREPARED;
    const size_t n2 = (size_t)c->n * c->n;
    std::vector<wso_h0_record> full(n2);
    const int rc = wso_export_h0(c, tile, full.data());
    if (rc != WSO_OK) return rc;
    for (size_t i = 0; i < n2; ++i) {
        h0_3f[3 * i + 0] = full[i].amp_re;
        h0_3f[3 * i + 1] = full[i].amp_im;
        h0_3f[3 * i + 2] = full[i].dispersion;
    }
    return WSO_OK;
}

// Asynchronous ComputeWaves(t): tile 0 -> device slot 0 on the context's stream, no host copy, no synchronisation.
// *event_out (a cudaEvent_t owned by the context, valid until the next call) completes when both maps and A are final;
// a CUDA caller orders its own stream behind it (cudaStreamWaitEvent), any caller can block with wso_wait_event.
int wso_compute_async(wso_ctx* c, float t, void** event_out) {
    int rc = check_batch(c, 1, nullptr, &t, 0);
    if (rc != WSO_OK) return rc;
    WSO_CUDA(c, cudaSetDevice(c->device));
    if (!c->ev_async) WSO_CUDA(c, cudaEventCreateWithFlags(&c->ev_async, cudaEventDisableTiming));
    if ((rc = push_lambdas(c)) != WSO_OK) return rc;
    if ((rc = enqueue_chunk(c, 1, nullptr, &t, 0, 0, c->stream)) != WSO_OK) return rc;
    WSO_CUDA(c, cudaEventRecord(c->ev_async, c->stream));
    if (event_out) *event_out = c->ev_async;
    return WSO_OK;
}

int wso_wait_event(wso_ctx* c, void* event) {
    if (!c || !event) return WSO_ERR_INVALID_ARG;
    WSO_CUDA(c, cudaSetDevice(c->device));
    WSO_CUDA(c, cudaEventSynchronize(static_cast<cudaEvent_t>(event)));
    return WSO_OK;
}

int wso_compute_batch(wso_ctx* c, uint32_t n, const uint32_t* tiles, const float* t, uint32_t first_slot) {
    int rc = check_batch(c, n, tiles, t, first_slot);
    if (rc != WSO_OK) return rc;
    WSO_CUDA(c, cudaSetDevice(c->device));
    if ((rc = push_lambdas(c)) != WSO_OK) return rc;
    // Two compute lanes: even chunks on the caller-visible stream, odd chunks on an internal one, each lane with
    // its own W scratch.  Chunks are independent, so the second lane's kernels fill the partial last wave and the
    // launch gaps of the first.  Fork/join events keep everything ordered with respect to c->stream.
    const uint32_t n_chunks = (n + c->chunk - 1) / c->chunk;
    // per-kernel event timing wants the kernels serialised
    const int lanes = c->profiling ? 1 : (int)(n_chunks < (uint32_t)c->lanes ? n_chunks : (uint32_t)c->lanes);
    auto lane_stream = [&](int l) { return l == 0 ? c->stream : (l == 1 ? c->aux_stream : c->more_lanes[l - 2]); };
    // Experiment hook (WSO_EXP_L2_PERSIST_MB=<carve-out>): the W scratch of every lane as a persisting-L2 access-policy window of
    // that lane's stream, so that the map stores streaming through L2 do not push W out between K1 and K2.  Measured result in
    // profiles/r3_memory_instructions.md; off by default.
    if (!c->l2_policy_done) {
        c->l2_policy_done = true;
        if (const char* env = std::getenv("WSO_EXP_L2_PERSIST_MB")) {
            const long mb = std::atol(env);
            cudaDeviceProp prop;
            if (mb > 0 && cudaGetDeviceProperties(&prop, c->device) == cudaSuccess && prop.persistingL2CacheMaxSize > 0) {
                size_t carve = (size_t)mb << 20;
                if (carve > (size_t)prop.persistingL2CacheMaxSize) carve = (size_t)prop.persistingL2CacheMaxSize;
                cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve);
                const size_t lane_bytes = (size_t)c->chunk * c->n * c->n * 16;
                float ratio = 1.0f;
                if (const char* r = std::getenv("WSO_EXP_L2_PERSIST_RATIO")) ratio = (float)std::atof(r);
                for (int l = 0; l < (c->lanes > 2 ? c->lanes : 2); ++l) {
                    cudaStreamAttrValue v = {};
                    v.accessPolicyWindow.base_ptr = reinterpret_cast<char*>(c->d_W) + (size_t)l * lane_bytes;
                    size_t win = lane_bytes;
                    if (win > (size_t)prop.accessPolicyMaxWindowSize) win = (size_t)prop.accessPolicyMaxWindowSize;
                    v.accessPolicyWindow.num_bytes = win;
                    v.accessPolicyWindow.hitRatio = ratio;
                    v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
                    v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
                    cudaStreamSetAttribute(lane_stream(l), cudaStreamAttributeAccessPolicyWindow, &v);
                }
                std::fprintf(stderr, "wsocean: persisting L2 carve-out %zu MB (max %d MB), window %zu MB per lane (max %d MB), ratio %.2f\n",
                             carve >> 20, prop.persistingL2CacheMaxSize >> 20, lane_bytes >> 20, prop.accessPolicyMaxWindowSize >> 20, ratio);
                cudaGetLastError();
            }
        }
    }
    if (lanes > 1) {
        WSO_CUDA(c, cudaEventRecord(c->ev_fork, c->stream));
        for (int l = 1; l < lanes; ++l) WSO_CUDA(c, cudaStreamWaitEvent(lane_stream(l), c->ev_fork, 0));
    }
    int lane = 0;
    for (uint32_t done = 0; done < n; done += c->chunk) {
        const uint32_t m = (n - done < c->chunk) ? (n - done) : c->chunk;
        rc = enqueue_chunk(c, m, tiles ? tiles + done : nullptr, t + done, first_slot + done, lane, lane_stream(lane));
        if (rc != WSO_OK) return rc;
        lane = (lane + 1 == lanes) ? 0 : lane + 1;
    }
    for (int l = 1; l < lanes; ++l) {
        cudaEvent_t ev = l == 1 ? c->ev_join : c->ev_lane_join[l - 2];
        WSO_CUDA(c, cudaEventRecord(ev, lane_stream(l)));
        WSO_CUDA(c, cudaStreamWaitEvent(c->stream, ev, 0));
    }
    return WSO_OK;
}

int wso_sync(wso_ctx* c) {
    if (!c) return WSO_ERR_INVALID_ARG;
    WSO_CUDA(c, cudaSetDevice(c->device));
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    WSO_CUDA(c, cudaStreamSynchronize(c->aux_stream));
    WSO_CUDA(c, cudaStreamSynchronize(c->copy_stream));
    return WSO_OK;
}

int wso_read_heights(wso_ctx* c, uint32_t first_slot, uint32_t n, float* amplitude, float* min_height,
                     float* max_height) {
    if (!c) return WSO_ERR_INVALID_ARG;
    if ((uint64_t)first_slot + n > c->max_slots) return fail(c, WSO_ERR_INVALID_ARG, "slots out of range");
    WSO_CUDA(c, cudaSetDevice(c->device));
    float* ha = c->h_small;
    float* hm = c->h_small + c->small_cap;
    WSO_CUDA(c, cudaMemcpyAsync(ha, c->d_ampl + first_slot, sizeof(float) * n, cudaMemcpyDeviceToHost, c->stream));
    WSO_CUDA(c, cudaMemcpyAsync(hm, c->d_minmax + 2 * first_slot, sizeof(float) * 2 * n, cudaMemcpyDeviceToHost, c->stream));
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    for (uint32_t i = 0; i < n; ++i) {
        if (amplitude) amplitude[i] = ha[i];
        if (min_height) min_height[i] = hm[2 * i];
        if (max_height) max_height[i] = hm[2 * i + 1];
    }
    return WSO_OK;
}

int wso_compute(wso_ctx* c, float t, float* amplitude) {
    int rc = check_batch(c, 1, nullptr, &t, 0);
    if (rc != WSO_OK) return rc;
    WSO_CUDA(c, cudaSetDevice(c->device));
    if ((rc = push_lambdas(c)) != WSO_OK) return rc;
    if ((rc = enqueue_chunk(c, 1, nullptr, &t, 0, 0, c->stream)) != WSO_OK) return rc;
    const size_t bytes = map_slot_bytes(c);
    WSO_CUDA(c, cudaMemcpyAsync(c->h_disp, c->d_disp, bytes, cudaMemcpyDeviceToHost, c->stream));
    WSO_CUDA(c, cudaMemcpyAsync(c->h_norm, c->d_norm, bytes, cudaMemcpyDeviceToHost, c->stream));
    WSO_CUDA(c, cudaMemcpyAsync(c->h_small, c->d_ampl, sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    if (amplitude) *amplitude = c->h_small[0];
    return WSO_OK;
}

int wso_compute_to_host(wso_ctx* c, uint32_t n, const uint32_t* tiles, const float* t, float* disp_host,
                        float* norm_host, float* amplitude, float* min_height, float* max_height) {
    if (!c) return WSO_ERR_INVALID_ARG;
    if (c->map_format != WSO_MAP_RGBA32F)
        return fail(c, WSO_ERR_INVALID_ARG, "wso_compute_to_host takes RGBA32F maps: use wso_compute_to_host_bytes");
    return wso_compute_to_host_bytes(c, n, tiles, t, disp_host, norm_host, (size_t)n * map_slot_bytes(c), amplitude,
                                     min_height, max_height);
}

int wso_compute_to_host_bytes(wso_ctx* c, uint32_t n, const uint32_t* tiles, const float* t, void* disp_host,
                              void* norm_host, size_t bytes_each, float* amplitude, float* min_height,
                              float* max_height) {
    if (!c) return WSO_ERR_INVALID_ARG;
    if (!disp_host || !norm_host) return fail(c, WSO_ERR_INVALID_ARG, "host buffers are NULL");
    if (bytes_each < (size_t)n * map_slot_bytes(c))
        return fail(c, WSO_ERR_INVALID_ARG, "host buffers too small: n * N*N texels of the map format each");
    // Slots are recycled: chunk k uses slots [ (k&1)*chunk , (k&1)*chunk + m ).
    const uint32_t need = (n <= c->chunk) ? n : 2 * c->chunk;
    if (need > c->max_slots) return fail(c, WSO_ERR_INVALID_ARG, "wso_compute_to_host needs max_slots >= 2*chunk");
    int rc = check_batch(c, 0, nullptr, t, 0);
    if (rc != WSO_OK) return rc;
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t tl = tiles ? tiles[i] : 0u;
        if (tl >= c->max_tiles) return fail(c, WSO_ERR_INVALID_ARG, "tile index out of range");
        if (!c->tiles[tl].is_prepared) return fail(c, WSO_ERR_NOT_PREPARED, "Prepare() has not been called for this tile");
    }
    WSO_CUDA(c, cudaSetDevice(c->device));
    if ((rc = push_lambdas(c)) != WSO_OK) return rc;
    const size_t map_bytes = map_slot_bytes(c);
    if (n > c->small_cap) {  // pinned staging for amplitude/min/max of every tile-frame
        WSO_CUDA(c, cudaStreamSynchronize(c->stream));
        cudaFreeHost(c->h_small);
        c->h_small = nullptr;
        c->small_cap = 0;
        WSO_CUDA(c, cudaMallocHost(&c->h_small, sizeof(float) * 3 * n));
        c->small_cap = n;
    }
    float* small = c->h_small;
    int k = 0;
    for (uint32_t done = 0; done < n; done += c->chunk, ++k) {
        const uint32_t m = (n - done < c->chunk) ? (n - done) : c->chunk;
        const int b = k & 1;
        const uint32_t slot0 = (uint32_t)b * c->chunk;
        // the slots (and W buffer) of parity b are free once the copy issued two chunks ago is done
        cudaStream_t lane = b ? c->aux_stream : c->stream;
        if (k == 1) {  // first use of the second lane: order it after whatever preceded this call on c->stream
            WSO_CUDA(c, cudaEventRecord(c->ev_fork, c->stream));
            WSO_CUDA(c, cudaStreamWaitEvent(c->aux_stream, c->ev_fork, 0));
        }
        if (k >= 2) WSO_CUDA(c, cudaStreamWaitEvent(lane, c->ev_copied[b], 0));
        rc = enqueue_chunk(c, m, tiles ? tiles + done : nullptr, t + done, slot0, b, lane);
        if (rc != WSO_OK) return rc;
        WSO_CUDA(c, cudaEventRecord(c->ev_chunk[b], lane));
        WSO_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->ev_chunk[b], 0));
        WSO_CUDA(c, cudaMemcpyAsync(static_cast<char*>(disp_host) + (size_t)done * map_bytes, map_slot(c, 0, slot0),
                                    map_bytes * m, cudaMemcpyDeviceToHost, c->copy_stream));
        WSO_CUDA(c, cudaMemcpyAsync(static_cast<char*>(norm_host) + (size_t)done * map_bytes, map_slot(c, 1, slot0),
                                    map_bytes * m, cudaMemcpyDeviceToHost, c->copy_stream));
        WSO_CUDA(c, cudaMemcpyAsync(small + done, c->d_ampl + slot0, sizeof(float) * m,
                                    cudaMemcpyDeviceToHost, c->copy_stream));
        WSO_CUDA(c, cudaMemcpyAsync(small + n + 2 * (size_t)done, c->d_minmax + 2 * slot0,
                                    sizeof(float) * 2 * m, cudaMemcpyDeviceToHost, c->copy_stream));
        WSO_CUDA(c, cudaEventRecord(c->ev_copied[b], c->copy_stream));
    }
    WSO_CUDA(c, cudaStreamSynchronize(c->copy_stream));
    WSO_CUDA(c, cudaStreamSynchronize(c->aux_stream));
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    for (uint32_t i = 0; i < n; ++i) {
        if (amplitude) amplitude[i] = small[i];
        if (min_height) min_height[i] = small[n + 2 * (size_t)i];
        if (max_height) max_height[i] = small[n + 2 * (size_t)i + 1];
    }
    return WSO_OK;
}

int wso_map_host(wso_ctx* c, int which, const float** ptr, size_t* texels) {
    if (!c || !ptr) return WSO_ERR_INVALID_ARG;
    if (c->map_format != WSO_MAP_RGBA32F)
        return fail(c, WSO_ERR_INVALID_ARG, "wso_map_host returns RGBA32F maps: use wso_map_host_bytes");
    const void* p = nullptr;
    const int rc = wso_map_host_bytes(c, which, &p, nullptr);
    if (rc != WSO_OK) return rc;
    *ptr = static_cast<const float*>(p);
    if (texels) *texels = (size_t)c->n * c->n;
    return WSO_OK;
}

int wso_map_host_bytes(wso_ctx* c, int which, const void** ptr, size_t* bytes) {
    if (!c || !ptr) return WSO_ERR_INVALID_ARG;
    if (which != WSO_MAP_DISPLACEMENT && which != WSO_MAP_NORMAL) return fail(c, WSO_ERR_INVALID_ARG, "bad map id");
    *ptr = which == WSO_MAP_DISPLACEMENT ? c->h_disp : c->h_norm;
    if (bytes) *bytes = map_slot_bytes(c);
    return WSO_OK;
}

int wso_map_device(wso_ctx* c, int which, uint32_t slot, void** dptr, size_t* texels) {
    if (!c || !dptr) return WSO_ERR_INVALID_ARG;
    if (which != WSO_MAP_DISPLACEMENT && which != WSO_MAP_NORMAL) return fail(c, WSO_ERR_INVALID_ARG, "bad map id");
    if (slot >= c->max_slots) return fail(c, WSO_ERR_INVALID_ARG, "slot out of range");
    *dptr = map_slot(c, which, slot);
    if (texels) *texels = (size_t)c->n * c->n;
    return WSO_OK;
}

int wso_copy_map(wso_ctx* c, int which, uint32_t slot, float* dst) {
    if (c && c->map_format != WSO_MAP_RGBA32F)
        return fail(c, WSO_ERR_INVALID_ARG, "wso_copy_map copies RGBA32F maps: use wso_copy_map_bytes");
    return wso_copy_map_bytes(c, which, slot, dst, c ? map_slot_bytes(c) : 0);
}

int wso_copy_map_bytes(wso_ctx* c, int which, uint32_t slot, void* dst, size_t dst_bytes) {
    void* src = nullptr;
    int rc = wso_map_device(c, which, slot, &src, nullptr);
    if (rc != WSO_OK) return rc;
    if (!dst) return fail(c, WSO_ERR_INVALID_ARG, "dst is NULL");
    const size_t bytes = map_slot_bytes(c);
    if (dst_bytes < bytes) return fail(c, WSO_ERR_INVALID_ARG, "dst too small: N*N texels of the map format");
    WSO_CUDA(c, cudaSetDevice(c->device));
    WSO_CUDA(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    return WSO_OK;
}

int wso_set_exportable(wso_ctx* c, int on) {
    if (!c) return WSO_ERR_INVALID_ARG;
    const bool want = on != 0;
    if (want == c->exportable && c->map_mem[0].kind != kBackExternal && c->map_mem[1].kind != kBackExternal) return WSO_OK;
    WSO_CUDA(c, cudaSetDevice(c->device));
    int rc = wso_sync(c);
    if (rc != WSO_OK) return rc;
    const bool before = c->exportable;
    c->exportable = want;
    const size_t bytes = map_slot_bytes(c) * c->max_slots;
    for (int which = 0; which < 2; ++which) {
        rc = alloc_map(c, which, bytes);
        if (rc != WSO_OK) {  // fall back to what worked before; the maps must stay usable
            c->exportable = before;
            const std::string msg = c->err;
            for (int w = 0; w < 2; ++w)
                if (map_ptr(c, w) == nullptr) alloc_map(c, w, bytes);
            return fail(c, rc, msg);
        }
    }
    rc = reset_map_contents(c, (size_t)c->n * c->n);
    if (rc != WSO_OK) return rc;
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    return WSO_OK;
}

// Switch both maps between RGBA32F and RGBA16F: like wso_set_exportable, the map arrays (own or exportable memory; an
// imported array returns to own memory) and the pinned mirrors are reallocated at the new size and reset to the
// resize() defaults.  Prepare() state, the tile size and the exportable switch are kept.
int wso_set_map_format(wso_ctx* c, int format) {
    if (!c) return WSO_ERR_INVALID_ARG;
    if (format != WSO_MAP_RGBA32F && format != WSO_MAP_RGBA16F)
        return fail(c, WSO_ERR_INVALID_ARG, "map format must be WSO_MAP_RGBA32F or WSO_MAP_RGBA16F; unchanged");
    if (format == c->map_format) return WSO_OK;
    WSO_CUDA(c, cudaSetDevice(c->device));
    int rc = wso_sync(c);
    if (rc != WSO_OK) return rc;
    const int before = c->map_format;
    c->map_format = format;
    if (c->n == 0) return WSO_OK;  // no size allocated (a failed size change): the next allocation uses the format
    const size_t n2 = (size_t)c->n * c->n;
    auto reallocate = [&]() -> int {
        cudaFreeHost(c->h_disp); c->h_disp = nullptr;
        cudaFreeHost(c->h_norm); c->h_norm = nullptr;
        for (int which = 0; which < 2; ++which) free_map(c, which);
        WSO_CUDA(c, cudaMallocHost(&c->h_disp, map_texel_bytes(c) * n2));
        WSO_CUDA(c, cudaMallocHost(&c->h_norm, map_texel_bytes(c) * n2));
        for (int which = 0; which < 2; ++which) {
            const int r = alloc_map(c, which, map_slot_bytes(c) * c->max_slots);
            if (r != WSO_OK) return r;
        }
        const int r = reset_map_contents(c, n2);
        if (r != WSO_OK) return r;
        WSO_CUDA(c, cudaStreamSynchronize(c->stream));
        return WSO_OK;
    };
    rc = reallocate();
    if (rc != WSO_OK) {  // fall back to the previous format; the maps must stay usable
        const std::string msg = c->err;
        c->map_format = before;
        if (reallocate() != WSO_OK) {
            // not even the previous size fits any more: no size is resident (compute calls answer WSO_ERR_NOT_PREPARED)
            free_device_buffers(c);
            c->n = 0;
            c->logn = 0;
            for (uint32_t t = 0; t < c->max_tiles; ++t) c->tiles[t].is_prepared = false;
        }
        return fail(c, rc, msg);
    }
    return WSO_OK;
}

int wso_get_map_format(const wso_ctx* c, int* format) {
    if (!c || !format) return WSO_ERR_INVALID_ARG;
    *format = c->map_format;
    return WSO_OK;
}

}  // extern "C"

namespace {

// Everything wso_query_surface checks before it touches the device; fills the cascade constants of a launch.
int check_query(wso_ctx* c, uint32_t n_slots, const uint32_t* slots, uint32_t iterations, wso::QueryArgs* a) {
    if (!c) return WSO_ERR_INVALID_ARG;
    if (!slots) return fail(c, WSO_ERR_INVALID_ARG, "slots is NULL");
    if (n_slots < 1 || n_slots > (uint32_t)wso::kMaxQueryCascades)
        return fail(c, WSO_ERR_INVALID_ARG, "n_slots must be 1..4");
    if (iterations > (uint32_t)wso::kMaxQueryIterations) return fail(c, WSO_ERR_INVALID_ARG, "iterations must be <= 16");
    *a = wso::QueryArgs{};
    for (uint32_t i = 0; i < n_slots; ++i) {
        const uint32_t s = slots[i];
        if (s >= c->max_slots) return fail(c, WSO_ERR_INVALID_ARG, "slot out of range");
        const SlotFrame& f = c->slot_frames[s];
        if (!f.valid || c->n == 0)
            return fail(c, WSO_ERR_INVALID_ARG, "slot " + std::to_string(s) + " holds no computed frame");
        a->c[i] = wso::make_query_cascade(map_slot(c, 0, s), map_slot(c, 1, s), c->d_ampl + s, c->n, f.length, f.lambda);
    }
    a->mask = c->n - 1;
    a->logn = c->logn;
    a->iterations = (int)iterations;
    return WSO_OK;
}

// wso_raycast_surface's checks: those of the queries plus the march parameters.
int check_raycast(wso_ctx* c, uint32_t n_slots, const uint32_t* slots, const wso_ray_params* p, wso::RayArgs* a) {
    if (!c) return WSO_ERR_INVALID_ARG;
    if (!p) return fail(c, WSO_ERR_INVALID_ARG, "ray params are NULL");
    const int rc = check_query(c, n_slots, slots, p->iterations, &a->q);
    if (rc != WSO_OK) return rc;
    if (!(p->step > 0.0f && p->step <= FLT_MAX)) return fail(c, WSO_ERR_INVALID_ARG, "step must be finite and > 0");
    if (p->max_steps < 1 || p->max_steps > wso::kMaxRaySteps)
        return fail(c, WSO_ERR_INVALID_ARG, "max_steps must be 1..4096");
    if (p->refine > wso::kMaxRayRefine) return fail(c, WSO_ERR_INVALID_ARG, "refine must be <= 24");
    a->step = p->step;
    a->max_steps = p->max_steps;
    a->refine = p->refine;
    return WSO_OK;
}

// The device staging of the blocking query / ray-cast forms: at least in_bytes and out_bytes, grown on demand.
int grow_staging(wso_ctx* c, size_t in_bytes, size_t out_bytes) {
    if (in_bytes <= c->stage_in_bytes && out_bytes <= c->stage_out_bytes) return WSO_OK;
    in_bytes = std::max(in_bytes, c->stage_in_bytes);
    out_bytes = std::max(out_bytes, c->stage_out_bytes);
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    cudaFree(c->d_stage_in);
    cudaFree(c->d_stage_out);
    c->d_stage_in = nullptr;
    c->d_stage_out = nullptr;
    c->stage_in_bytes = c->stage_out_bytes = 0;
    WSO_CUDA(c, cudaMalloc(&c->d_stage_in, in_bytes));
    WSO_CUDA(c, cudaMalloc(&c->d_stage_out, out_bytes));
    c->stage_in_bytes = in_bytes;
    c->stage_out_bytes = out_bytes;
    return WSO_OK;
}

}  // namespace

extern "C" {

int wso_query_surface(wso_ctx* c, uint32_t n_slots, const uint32_t* slots, uint32_t iterations, uint32_t n,
                      const float* xz_dev, wso_surface_sample* out_dev) {
    wso::QueryArgs a;
    int rc = check_query(c, n_slots, slots, iterations, &a);
    if (rc != WSO_OK) return rc;
    if (n == 0) return WSO_OK;
    if (!xz_dev || !out_dev) return fail(c, WSO_ERR_INVALID_ARG, "xz or out is NULL");
    if (reinterpret_cast<uintptr_t>(out_dev) % 16 != 0) return fail(c, WSO_ERR_INVALID_ARG, "out is not 16-byte aligned");
    a.xz = xz_dev;
    a.out = reinterpret_cast<float4*>(out_dev);
    a.n = n;
    WSO_CUDA(c, cudaSetDevice(c->device));
    WSO_CUDA(c, wso::launch_query_surface(a, (int)n_slots, c->map_format == WSO_MAP_RGBA16F, c->stream));
    c->launches += 1;
    return WSO_OK;
}

int wso_query_surface_host(wso_ctx* c, uint32_t n_slots, const uint32_t* slots, uint32_t iterations, uint32_t n,
                           const float* xz_host, wso_surface_sample* out_host) {
    wso::QueryArgs a;
    int rc = check_query(c, n_slots, slots, iterations, &a);
    if (rc != WSO_OK) return rc;
    if (n == 0) return WSO_OK;
    if (!xz_host || !out_host) return fail(c, WSO_ERR_INVALID_ARG, "xz or out is NULL");
    WSO_CUDA(c, cudaSetDevice(c->device));
    rc = grow_staging(c, sizeof(float) * 2 * (size_t)n, sizeof(wso_surface_sample) * (size_t)n);
    if (rc != WSO_OK) return rc;
    WSO_CUDA(c, cudaMemcpyAsync(c->d_stage_in, xz_host, sizeof(float) * 2 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    a.xz = static_cast<const float*>(c->d_stage_in);
    a.out = static_cast<float4*>(c->d_stage_out);
    a.n = n;
    WSO_CUDA(c, wso::launch_query_surface(a, (int)n_slots, c->map_format == WSO_MAP_RGBA16F, c->stream));
    c->launches += 1;
    WSO_CUDA(c, cudaMemcpyAsync(out_host, c->d_stage_out, sizeof(wso_surface_sample) * (size_t)n, cudaMemcpyDeviceToHost,
                                c->stream));
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    return WSO_OK;
}

int wso_raycast_surface(wso_ctx* c, uint32_t n_slots, const uint32_t* slots, const wso_ray_params* p, uint32_t n,
                        const float* rays_dev, wso_ray_hit* out_dev) {
    wso::RayArgs a;
    int rc = check_raycast(c, n_slots, slots, p, &a);
    if (rc != WSO_OK) return rc;
    if (n == 0) return WSO_OK;
    if (!rays_dev || !out_dev) return fail(c, WSO_ERR_INVALID_ARG, "rays or out is NULL");
    if (reinterpret_cast<uintptr_t>(rays_dev) % 16 != 0 || reinterpret_cast<uintptr_t>(out_dev) % 16 != 0)
        return fail(c, WSO_ERR_INVALID_ARG, "rays or out is not 16-byte aligned");
    a.rays = reinterpret_cast<const float4*>(rays_dev);
    a.out = reinterpret_cast<float4*>(out_dev);
    a.n = n;
    WSO_CUDA(c, cudaSetDevice(c->device));
    WSO_CUDA(c, wso::launch_raycast_surface(a, (int)n_slots, c->map_format == WSO_MAP_RGBA16F, c->stream));
    c->launches += 1;
    return WSO_OK;
}

int wso_raycast_surface_host(wso_ctx* c, uint32_t n_slots, const uint32_t* slots, const wso_ray_params* p, uint32_t n,
                             const float* rays_host, wso_ray_hit* out_host) {
    wso::RayArgs a;
    int rc = check_raycast(c, n_slots, slots, p, &a);
    if (rc != WSO_OK) return rc;
    if (n == 0) return WSO_OK;
    if (!rays_host || !out_host) return fail(c, WSO_ERR_INVALID_ARG, "rays or out is NULL");
    WSO_CUDA(c, cudaSetDevice(c->device));
    rc = grow_staging(c, sizeof(float) * 8 * (size_t)n, sizeof(wso_ray_hit) * (size_t)n);
    if (rc != WSO_OK) return rc;
    WSO_CUDA(c, cudaMemcpyAsync(c->d_stage_in, rays_host, sizeof(float) * 8 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    a.rays = static_cast<const float4*>(c->d_stage_in);
    a.out = static_cast<float4*>(c->d_stage_out);
    a.n = n;
    WSO_CUDA(c, wso::launch_raycast_surface(a, (int)n_slots, c->map_format == WSO_MAP_RGBA16F, c->stream));
    c->launches += 1;
    WSO_CUDA(c, cudaMemcpyAsync(out_host, c->d_stage_out, sizeof(wso_ray_hit) * (size_t)n, cudaMemcpyDeviceToHost,
                                c->stream));
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    return WSO_OK;
}

int wso_export_fd(wso_ctx* c, int which, int* fd, size_t* bytes) {
    if (!c || !fd) return WSO_ERR_INVALID_ARG;
    if (which != WSO_MAP_DISPLACEMENT && which != WSO_MAP_NORMAL) return fail(c, WSO_ERR_INVALID_ARG, "bad map id");
    const MapBacking& b = c->map_mem[which];
    if (b.kind != kBackExportable)
        return fail(c, WSO_ERR_INVALID_ARG, "map memory is not exportable: call wso_set_exportable(ctx, 1) first");
    WSO_CUDA(c, cudaSetDevice(c->device));
    int out = -1;
    if (vmm_api().ExportHandle(&out, b.handle, CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR, 0) != CUDA_SUCCESS || out < 0)
        return fail(c, WSO_ERR_CUDA, "cuMemExportToShareableHandle failed");
    *fd = out;
    if (bytes) *bytes = b.mapped_bytes;
    return WSO_OK;
}

int wso_import_external_fd(wso_ctx* c, int which, int fd, size_t bytes, size_t offset) {
    if (!c || fd < 0) return WSO_ERR_INVALID_ARG;
    if (which != WSO_MAP_DISPLACEMENT && which != WSO_MAP_NORMAL) return fail(c, WSO_ERR_INVALID_ARG, "bad map id");
    const size_t need = map_slot_bytes(c) * c->max_slots;
    if (offset % 16 != 0 || offset > bytes || bytes - offset < need)
        return fail(c, WSO_ERR_INVALID_ARG, "external memory too small for max_slots maps at this offset (or offset not 16-byte aligned)");
    WSO_CUDA(c, cudaSetDevice(c->device));
    int rc = wso_sync(c);
    if (rc != WSO_OK) return rc;
    cudaExternalMemoryHandleDesc hd = {};
    hd.type = cudaExternalMemoryHandleTypeOpaqueFd;
    hd.handle.fd = fd;
    hd.size = bytes;
    cudaExternalMemory_t ext = nullptr;
    cudaError_t e = cudaImportExternalMemory(&ext, &hd);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail_cuda(c, e, "cudaImportExternalMemory");
    }
    cudaExternalMemoryBufferDesc bd = {};
    bd.offset = offset;
    bd.size = need;
    void* ptr = nullptr;
    e = cudaExternalMemoryGetMappedBuffer(&ptr, ext, &bd);
    if (e != cudaSuccess) {
        cudaGetLastError();
        cudaDestroyExternalMemory(ext);
        return fail_cuda(c, e, "cudaExternalMemoryGetMappedBuffer");
    }
    free_map(c, which);
    map_ptr(c, which) = static_cast<float4*>(ptr);
    c->map_mem[which].kind = kBackExternal;
    c->map_mem[which].ext = ext;
    {
        const int rc = reset_map_contents(c, (size_t)c->n * c->n, which == WSO_MAP_DISPLACEMENT ? 1 : 2);
        if (rc != WSO_OK) return rc;
    }
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    return WSO_OK;
}

int wso_import_semaphore_fd(wso_ctx* c, int index, int fd, int is_timeline) {
    if (!c || fd < 0 || index < 0 || index > 1) return WSO_ERR_INVALID_ARG;
    WSO_CUDA(c, cudaSetDevice(c->device));
    cudaExternalSemaphoreHandleDesc sd = {};
    sd.type = is_timeline ? cudaExternalSemaphoreHandleTypeTimelineSemaphoreFd : cudaExternalSemaphoreHandleTypeOpaqueFd;
    sd.handle.fd = fd;
    cudaExternalSemaphore_t sem = nullptr;
    cudaError_t e = cudaImportExternalSemaphore(&sem, &sd);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail_cuda(c, e, "cudaImportExternalSemaphore");
    }
    if (c->ext_sem[index]) {
        cudaStreamSynchronize(c->stream);
        cudaDestroyExternalSemaphore(c->ext_sem[index]);
    }
    c->ext_sem[index] = sem;
    return WSO_OK;
}

int wso_signal_semaphore(wso_ctx* c, int index, uint64_t value) {
    if (!c || index < 0 || index > 1) return WSO_ERR_INVALID_ARG;
    if (!c->ext_sem[index]) return fail(c, WSO_ERR_INVALID_ARG, "no semaphore imported at this index");
    WSO_CUDA(c, cudaSetDevice(c->device));
    cudaExternalSemaphoreSignalParams sp = {};
    sp.params.fence.value = value;
    WSO_CUDA(c, cudaSignalExternalSemaphoresAsync(&c->ext_sem[index], &sp, 1, c->stream));
    return WSO_OK;
}

int wso_wait_semaphore(wso_ctx* c, int index, uint64_t value) {
    if (!c || index < 0 || index > 1) return WSO_ERR_INVALID_ARG;
    if (!c->ext_sem[index]) return fail(c, WSO_ERR_INVALID_ARG, "no semaphore imported at this index");
    WSO_CUDA(c, cudaSetDevice(c->device));
    cudaExternalSemaphoreWaitParams wp = {};
    wp.params.fence.value = value;
    WSO_CUDA(c, cudaWaitExternalSemaphoresAsync(&c->ext_sem[index], &wp, 1, c->stream));
    return WSO_OK;
}

int wso_set_stream(wso_ctx* c, void* cuda_stream) {
    if (!c) return WSO_ERR_INVALID_ARG;
    WSO_CUDA(c, cudaSetDevice(c->device));
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    c->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : c->own_stream;
    return WSO_OK;
}

int wso_alloc_host(size_t bytes, void** ptr) {
    if (!ptr) return WSO_ERR_INVALID_ARG;
    cudaError_t e = cudaMallocHost(ptr, bytes);
    if (e != cudaSuccess) return fail_cuda(nullptr, e, "cudaMallocHost");
    return WSO_OK;
}

int wso_select_kernels(int mask) {
    if (mask < -1 || (mask & ~0x57) != 0) return WSO_ERR_INVALID_ARG;
    wso::set_warp_core_override(mask);
    return WSO_OK;
}

int wso_register_host(void* ptr, size_t bytes) {
    if (!ptr || bytes == 0) return WSO_ERR_INVALID_ARG;
    const cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return e == cudaErrorMemoryAllocation ? WSO_ERR_OUT_OF_MEMORY : WSO_ERR_CUDA;
    }
    return WSO_OK;
}

int wso_unregister_host(void* ptr) {
    if (!ptr) return WSO_ERR_INVALID_ARG;
    const cudaError_t e = cudaHostUnregister(ptr);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return WSO_ERR_CUDA;
    }
    return WSO_OK;
}

int wso_free_host(void* ptr) {
    cudaError_t e = cudaFreeHost(ptr);
    return e == cudaSuccess ? WSO_OK : WSO_ERR_CUDA;
}

int wso_set_profiling(wso_ctx* c, int on) {
    if (!c) return WSO_ERR_INVALID_ARG;
    WSO_CUDA(c, cudaSetDevice(c->device));
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    c->profiling = on != 0;
    c->prof_used = 0;
    c->prof_ms[0] = c->prof_ms[1] = c->prof_ms[2] = 0.0;
    c->prof_launches = 0;
    c->prof_items = 0;
    return WSO_OK;
}

int wso_get_profile(wso_ctx* c, double* kernel_ms, uint64_t* launches, uint64_t* tile_frames) {
    if (!c) return WSO_ERR_INVALID_ARG;
    WSO_CUDA(c, cudaSetDevice(c->device));
    WSO_CUDA(c, cudaStreamSynchronize(c->stream));
    for (size_t i = 0; i + 3 < c->prof_used; i += 4)
        for (int k = 0; k < 3; ++k) {
            float ms = 0.0f;
            WSO_CUDA(c, cudaEventElapsedTime(&ms, c->prof_events[i + k], c->prof_events[i + k + 1]));
            c->prof_ms[k] += (double)ms;
        }
    c->prof_used = 0;
    if (kernel_ms) for (int k = 0; k < 3; ++k) kernel_ms[k] = c->prof_ms[k];
    if (launches) *launches = c->prof_launches;
    if (tile_frames) *tile_frames = c->prof_items;
    return WSO_OK;
}

int wso_set_frame_graph(wso_ctx* c, int on) {
    if (!c) return WSO_ERR_INVALID_ARG;
    c->frame_graph_mode = on < 0 ? 0 : (on > 2 ? 2 : on);
    return WSO_OK;
}

int wso_get_frame_graph_stats(const wso_ctx* c, uint64_t* graph_launches, uint64_t* captures) {
    if (!c) return WSO_ERR_INVALID_ARG;
    if (graph_launches) *graph_launches = c->frame_graph.graph_launches;
    if (captures) *captures = c->frame_graph.captures;
    return WSO_OK;
}

int wso_get_stats(const wso_ctx* c, uint64_t* kernel_launches, uint32_t* chunk) {
    if (!c) return WSO_ERR_INVALID_ARG;
    if (kernel_launches) *kernel_launches = c->launches;
    if (chunk) *chunk = c->chunk;
    return WSO_OK;
}

const char* wso_last_error(const wso_ctx* c) {
    if (c) return c->err.c_str();
    std::lock_guard<std::mutex> lk(g_err_mutex);
    static thread_local std::string copy;
    copy = g_create_error;
    return copy.c_str();
}

const char* wso_version(void) { return "wsocean 0.1 (sm_100a)"; }

}  // extern "C"
