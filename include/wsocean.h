/* wsocean.h — C ABI of the B200-native Tessendorf wave-synthesis library (libwsocean.so).
 *
 * Drop-in boundary for ONE hot path of kentril0/WaterSurfaceRendering: the CPU surface model
 * `class WSTessendorf` (reference: src/scene/WSTessendorf.h:33-321, src/scene/WSTessendorf.cpp).
 * Each entry point below names the reference interface it replaces.  Plain pointers and sizes only;
 * no C++ / CUDA / torch types cross this boundary.  Every function returns a wso_status (0 = ok) and
 * never throws or aborts; wso_last_error() gives the text of the last failure.
 *
 * Threading (reference: single frame-loop thread, model not re-entrant): one context = one CUDA
 * device + one stream; calls on a context must be serialised by the caller; contexts are independent.
 *
 * All kernels are hand-written sm_100a CUDA (no cuFFT).  There is no CPU fallback: on a machine
 * without a usable GPU wso_create() fails with WSO_ERR_CUDA.
 */
#ifndef WSOCEAN_H_
#define WSOCEAN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WSO_API __attribute__((visibility("default")))

typedef struct wso_ctx wso_ctx;

typedef enum wso_status {
    WSO_OK = 0,
    WSO_ERR_INVALID_ARG = -1,
    WSO_ERR_BAD_TILE_SIZE = -2,   /* not a power of two in [16, 8192]; state unchanged
                                     (reference SetTileSize silently ignores non-pow2: WSTessendorf.cpp:459-468) */
    WSO_ERR_NOT_PREPARED = -3,    /* ComputeWaves before Prepare */
    WSO_ERR_CUDA = -4,
    WSO_ERR_OUT_OF_MEMORY = -5,
    WSO_ERR_H0_NOT_CONJUGATE = -6 /* imported h0 violates heightAmp_conj == conj(heightAmp), which every
                                     reference-built h0 satisfies (WSTessendorf.cpp:132-135) and the kernels rely on */
} wso_status;

/* The reference's tunables (setters: WSTessendorf.cpp:459-505; defaults: WSTessendorf.h:36-43,181). */
typedef struct wso_params {
    uint32_t tile_size;    /* N: points == waves per side, power of two      (SetTileSize)        */
    float tile_length;     /* L: world-space tile length                      (SetTileLength)      */
    float wind_dir_x;      /* any non-zero vector; normalised on use          (SetWindDirection)   */
    float wind_dir_y;
    float wind_speed;      /* clamped to >= 1e-4                              (SetWindSpeed)       */
    float anim_period;     /* T; base frequency w0 = 2*pi/T                   (SetAnimationPeriod) */
    float phillips_const;  /* A of the Phillips spectrum                      (SetPhillipsConst)   */
    float damping;         /* suppresses wave lengths below it                (SetDamping)         */
    float lambda;          /* choppy-displacement scale; no Prepare() needed  (SetLambda)          */
} wso_params;

/* The reference's 20-byte h0 record (struct BaseWaveHeight, WSTessendorf.h:142-147). */
typedef struct wso_h0_record {
    float amp_re, amp_im;            /* heightAmp       */
    float amp_conj_re, amp_conj_im;  /* heightAmp_conj  */
    float dispersion;                /* quantised omega */
} wso_h0_record;

enum { WSO_MAP_DISPLACEMENT = 0, WSO_MAP_NORMAL = 1 };

/* Fill *p with the reference defaults (WSTessendorf.h:36-43, lambda = -1: WSTessendorf.h:181). */
WSO_API int wso_default_params(wso_params* p);

/* Replaces: WSTessendorf::WSTessendorf(tileSize, tileLength) (WSTessendorf.cpp:13-26).
 * device: CUDA ordinal.  max_tiles: independent parameter sets / h0 fields sharing tile_size (>= 1).
 * max_slots: output map pairs kept resident on the device (>= 1; a batch writes one slot per tile-frame). */
WSO_API int wso_create(const wso_params* p, int device, uint32_t max_tiles, uint32_t max_slots,
                       wso_ctx** out);
/* Replaces: WSTessendorf::~WSTessendorf (WSTessendorf.cpp:28-34). */
WSO_API int wso_destroy(wso_ctx* ctx);

/* Replaces: the Set* family (WSTessendorf.cpp:459-505).  tile_size / length / wind / period / A / damping
 * take effect at the next wso_prepare* of that tile (as in the reference); lambda takes effect at the
 * next compute.  A tile_size different from the context's is accepted only while max_tiles == 1. */
WSO_API int wso_set_params(wso_ctx* ctx, uint32_t tile, const wso_params* p);
/* Replaces: the Get* family (WSTessendorf.h:82-89); wind direction is returned normalised. */
WSO_API int wso_get_params(const wso_ctx* ctx, uint32_t tile, wso_params* p);
WSO_API int wso_set_lambda(wso_ctx* ctx, uint32_t tile, float lambda);
/* Replaces: the compile-time switch COMPUTE_JACOBIAN (WSTessendorf.cpp:158-175, 330-335, 368-377, 421-428; dead code in
 * the reference - it does not compile there - so this is an extension with no reference output to pin it to, SURVEY
 * row f-4).  on != 0: every following compute writes displacement.w = J = (1 + l*dxDx)(1 + l*dzDz) - (l*dxDz)(l*dzDx)
 * (l = lambda, all four derivatives already carrying the (-1)^(m+n) sign) instead of 1.0f; J < 0 marks folded
 * (foam) texels.  No extra transform: dxDz == dzDx rides in the empty real slot of the packed field that carries Dz.
 * Tile sizes up to 4096; not available on the slab path.  Default off = the reference's behaviour. */
WSO_API int wso_set_compute_jacobian(wso_ctx* ctx, int on);
WSO_API int wso_get_compute_jacobian(const wso_ctx* ctx, int* on);

/* Replaces: WSTessendorf::Prepare() (WSTessendorf.cpp:36-58) — wave vectors, Gaussian array drawn from
 * the C library rand() exactly like glm::gaussRand does (libs/glm/glm/gtc/random.inl:218-232), Phillips
 * h0(k) and dispersion; buffers (re)sized.  reseed != 0 calls srand(seed) first (the reference app seeds
 * once with the wall clock: core/Application.cpp:21). */
WSO_API int wso_prepare(wso_ctx* ctx, uint32_t tile, int reseed, unsigned seed);
/* Same, with a caller-supplied Gaussian array xi: N*N complex<float> (re,im), row-major [m][n]
 * (the array ComputeGaussRandomArray returns, WSTessendorf.cpp:87-103). */
WSO_API int wso_prepare_gauss(wso_ctx* ctx, uint32_t tile, const float* xi);
/* Prepare() ON THE DEVICE (replaces the CPU passes ComputeWaveVectors + ComputeBaseWaveHeightField,
 * WSTessendorf.cpp:60-85, 105-148, with PhillipsSpectrum / BaseWaveHeightFT / QDispersion, WSTessendorf.h:237-297):
 * one kernel builds the spectrum records straight in device memory from the uploaded Gaussian array xi (same
 * layout as above).  Dispersion, 1/|k| and layout are bit-identical to wso_prepare_gauss; amplitudes agree to
 * 1 ulp (the two exp() are evaluated in float64 on the device).  No host copy of h0 is kept: wso_export_h0 reads
 * the records back. */
WSO_API int wso_prepare_gauss_device(wso_ctx* ctx, uint32_t tile, const float* xi);
/* Same, the Gaussian array drawn in the kernel from the counter-based generator (seed, m*N+n) - a reproducible
 * stand-in for the reference's serial rand() stream (ComputeGaussRandomArray, WSTessendorf.cpp:87-103); the host
 * build of the same generator is wso_counter_h0. */
WSO_API int wso_prepare_counter(wso_ctx* ctx, uint32_t tile, uint64_t seed);
/* Import / export h0 in the reference's own layout: N*N records, row-major [m][n]
 * (m_BaseWaveHeights, WSTessendorf.h:197).  Import replaces the spectrum of a tile whose parameters
 * (tile_length in particular) were set beforehand; this is also the checkpoint/restore mechanism. */
WSO_API int wso_import_h0(wso_ctx* ctx, uint32_t tile, const wso_h0_record* h0);
WSO_API int wso_export_h0(const wso_ctx* ctx, uint32_t tile, wso_h0_record* h0);
/* Compact form, 12 bytes per wave vector (amp.re, amp.im, dispersion), row-major [m][n]: heightAmp_conj == conj(heightAmp)
 * in every reference-built h0 (WSTessendorf.cpp:132-135), so nothing is lost against the 20-byte BaseWaveHeight record. */
WSO_API int wso_import_h0_compact(wso_ctx* ctx, uint32_t tile, const float* h0_3f);
WSO_API int wso_export_h0_compact(const wso_ctx* ctx, uint32_t tile, float* h0_3f);

/* Replaces: float WSTessendorf::ComputeWaves(float t) (WSTessendorf.cpp:284-441) for tile 0 -> slot 0.
 * Blocking.  On return both maps are in pinned host memory (wso_map_host) and on the device
 * (wso_map_device); *amplitude receives the return value A. */
WSO_API int wso_compute(wso_ctx* ctx, float t, float* amplitude);
/* The same frame without the host copy and without blocking: tile 0 -> device slot 0 on the context's stream.  *event_out
 * is a cudaEvent_t (as void*) owned by the context and valid until the next call; it completes when both maps, A and
 * min/max of the frame are final on the device (wso_map_device, wso_read_heights).  A CUDA caller orders its own stream
 * behind it with cudaStreamWaitEvent; wso_wait_event blocks the host. */
WSO_API int wso_compute_async(wso_ctx* ctx, float t, void** event_out);
WSO_API int wso_wait_event(wso_ctx* ctx, void* event);

/* Batched form: n tile-frames.  Item i evolves tile tiles[i] (NULL = all tile 0) to time t[i] and writes
 * device map slot first_slot + i.  Asynchronous on the context's stream; results stay on the device. */
WSO_API int wso_compute_batch(wso_ctx* ctx, uint32_t n, const uint32_t* tiles, const float* t,
                              uint32_t first_slot);
/* Batched form with host output: like wso_compute_batch, then streams each tile-frame's maps into
 * disp_host / norm_host (n * N*N*4 floats each, ideally pinned: wso_alloc_host) overlapping copies with
 * the next chunk's kernels; amplitude/min/max may be NULL.  Blocking. */
WSO_API int wso_compute_to_host(wso_ctx* ctx, uint32_t n, const uint32_t* tiles, const float* t,
                                float* disp_host, float* norm_host, float* amplitude,
                                float* min_height, float* max_height);
WSO_API int wso_sync(wso_ctx* ctx);

/* Replaces: GetMinHeight()/GetMaxHeight() (WSTessendorf.h:90-91) and the ComputeWaves return value,
 * for n slots starting at first_slot.  Blocking (small device->host read).  Any pointer may be NULL. */
WSO_API int wso_read_heights(wso_ctx* ctx, uint32_t first_slot, uint32_t n, float* amplitude,
                             float* min_height, float* max_height);

/* Replaces: GetDisplacements()/GetNormals() + Get*Count() (WSTessendorf.h:95-101): tightly packed
 * RGBA32F texels, row-major [m][n], N*N of them.
 *   displacement = (lambda*Dx, height/A, lambda*Dz, 1)      normal = (dh/dx, dh/dz, dDx/dx, dDz/dz)
 * wso_map_host: pinned host copy of slot 0 written by wso_compute (valid until the next compute/prepare).
 *   Between Prepare() and the first compute every texel holds the reference's resize() defaults
 *   (WSTessendorf.cpp:48-54): displacement (0,0,0,0), normal (0,1,0,0) - on the host mirrors and in every device slot.
 * wso_map_device: device pointer of any slot (valid until destroy / tile-size change).
 * wso_copy_map: blocking copy of one slot's map into caller memory. */
WSO_API int wso_map_host(wso_ctx* ctx, int which, const float** ptr, size_t* texels);
WSO_API int wso_map_device(wso_ctx* ctx, int which, uint32_t slot, void** dptr, size_t* texels);
WSO_API int wso_copy_map(wso_ctx* ctx, int which, uint32_t slot, float* dst_host);

/* ------------------------------------------------------------------------------------------------------------
 * Map format (an extension; the reference writes RGBA32F only).  Both maps of a context are in one format:
 *   WSO_MAP_RGBA32F (default): 4 x fp32 per texel, 16 bytes, VK_FORMAT_R32G32B32A32_SFLOAT - everything above.
 *   WSO_MAP_RGBA16F: (x, y, z, w) as 4 x IEEE binary16, little-endian, tightly packed: 8 bytes per texel,
 *       VK_FORMAT_R16G16B16A16_SFLOAT (a mandatory sampled format with linear filtering).  Each channel is the value the
 *       RGBA32F path computes, rounded to nearest even; magnitudes >= 65520 become +-inf, NaN stays NaN (IEEE conversion).
 *       Half the device memory, half the device->host bytes and half of K2's stores.  disp.y is normalised to [-1, 1];
 *       at the 512^2 defaults |lambda*Dx| <= 23 (about 1 cm of binary16 spacing there) and the normals <= 1.1.
 * wso_set_map_format reallocates both map arrays and the pinned mirrors at the new size (in the current backing: own or
 * exportable memory; an array imported with wso_import_external_fd returns to own memory) and resets their contents
 * to the resize() defaults in the new format (displacement 0, normal (0, 1, 0, 0)).  Prepare() state, the tile size,
 * the Jacobian switch and wso_set_exportable are kept; the format survives Prepare(), tile-size changes and
 * wso_set_exportable.  Any other value: WSO_ERR_INVALID_ARG, state unchanged.
 * Layout in either format: [slot][N*N] texels, slot s at byte s*B*N*N, row pitch B*N (B = 16 or 8 bytes per texel); this
 * is the layout of wso_map_device, wso_export_fd (which then reports the smaller array) and of the memory
 * wso_import_external_fd needs (max_slots*B*N*N bytes).
 * The float-typed calls wso_map_host, wso_copy_map and wso_compute_to_host serve RGBA32F only and answer
 * WSO_ERR_INVALID_ARG in RGBA16F; their byte-typed counterparts below work in both formats:
 *   wso_map_host_bytes       : pinned host copy of slot 0 (as wso_map_host); *bytes = B*N*N
 *   wso_copy_map_bytes       : blocking copy of one slot into dst_host, which must hold dst_bytes >= B*N*N
 *   wso_compute_to_host_bytes: wso_compute_to_host into buffers of bytes_each >= n*B*N*N bytes each
 * Not on the slab path (RGBA32F only).  RGBA16F maps always come from the CTA-per-line K2 (wso_select_kernels bit 2
 * does not apply to them). */
enum { WSO_MAP_RGBA32F = 0, WSO_MAP_RGBA16F = 1 };
WSO_API int wso_set_map_format(wso_ctx* ctx, int format);
WSO_API int wso_get_map_format(const wso_ctx* ctx, int* format);
WSO_API int wso_map_host_bytes(wso_ctx* ctx, int which, const void** ptr, size_t* bytes);
WSO_API int wso_copy_map_bytes(wso_ctx* ctx, int which, uint32_t slot, void* dst_host, size_t dst_bytes);
WSO_API int wso_compute_to_host_bytes(wso_ctx* ctx, uint32_t n, const uint32_t* tiles, const float* t,
                                      void* disp_host, void* norm_host, size_t bytes_each, float* amplitude,
                                      float* min_height, float* max_height);

/* ------------------------------------------------------------------------------------------------------------
 * Surface queries (an extension): height, normal and undisplaced origin of the surface at arbitrary world points
 * (buoyancy, collision, spray, wake placement), sampled on the device from the maps of 1..4 slots (cascades: tiles of
 * different tile_length, e.g. the tiles of a max_tiles context, each computed into its own slot), in either map format.
 * Slot s was last written by a compute of tile t; N = tile size, L_s = tile_length t was PREPARED with, l_s = lambda in
 * effect for that compute, A_s = that frame's amplitude (wso_read_heights), D_s / G_s = its displacement / normal map
 * (RGBA16F decoded to fp32).
 *   Coordinates: texel [m][n] is the field at world (x, z) = (n*L/N, m*L/N) (rows = z, columns = x), L-periodic.
 *   Sampling S_s[F](x, z): u = x*N/L_s, v = z*N/L_s, n0 = floor(u), m0 = floor(v), fu = u - n0, fv = v - m0; bilinear
 *       blend of texels [m0|m0+1][n0|n0+1], indices wrapped mod N (any x, z, negative or many tiles away).  x and z are
 *       reduced mod L_s once per cascade in float64; the rest is fp32, so far-away queries are as accurate as near ones.
 *   Inversion: choppy displacement moves points sideways.  The surface point above q = (x, z) started at p with
 *       p + Dh(p) = q, Dh(p) = sum_s (S_s[D.x](p), S_s[D.z](p)) (D.x, D.z carry lambda).  `iterations` = I fixed-point
 *       steps held as offsets from q:  d_0 = 0, d_{k+1} = -Dh(q + d_k), p = q + d_I.  I = 0: the point that started at q.
 *   Record (32 bytes):
 *       height   = sum_s A_s * S_s[D.y](p)
 *       normal   = normalize(-sx/ex, 1, -sz/ez), sx = sum_s S_s[G.x](p), sz = sum_s S_s[G.y](p),
 *                  ex = 1 + sum_s l_s*S_s[G.z](p), ez = 1 + sum_s l_s*S_s[G.w](p)   (one slot: the reference's vertex
 *                  shader normal, WaterSurfaceMesh.vert:33-38)
 *       offset   = d_I = p - q
 *       residual = |d_I + Dh(p)|, world units: how far the answer is from q.  Where the surface folds (J < 0) the
 *                  iteration need not converge; a large residual says so, it is not an error.
 *       w        = S_{s0}[D.w](p) of the first slot: 1, or J if that frame had the Jacobian on.
 * wso_query_surface: xz_dev = n (x, z) float pairs, out_dev = n records (16-byte aligned), both device pointers;
 *   asynchronous on the context's stream, ONE kernel launch, so it follows a compute on that stream without a host sync.
 * wso_query_surface_host: host pointers; blocking; stages through library-owned device memory grown on demand.
 * 1 <= n_slots <= 4, iterations <= 16, n == 0 is a no-op.  WSO_ERR_INVALID_ARG (state unchanged): a slot >= max_slots, a
 * slot that holds no computed frame (every compute entry point records one; wso_set_map_format, wso_set_exportable,
 * wso_import_external_fd and a Prepare that changes the tile size clear them all), a NULL pointer, a misaligned out_dev,
 * a limit exceeded.  Non-finite coordinates give NaN records (device data is not inspected).  Not on the slab path. */
typedef struct wso_surface_sample {
    float height;
    float normal_x, normal_y, normal_z;
    float offset_x, offset_z;
    float residual;
    float w;
} wso_surface_sample;
WSO_API int wso_query_surface(wso_ctx* ctx, uint32_t n_slots, const uint32_t* slots, uint32_t iterations,
                              uint32_t n, const float* xz_dev, wso_surface_sample* out_dev);
WSO_API int wso_query_surface_host(wso_ctx* ctx, uint32_t n_slots, const uint32_t* slots, uint32_t iterations,
                                   uint32_t n, const float* xz_host, wso_surface_sample* out_host);

/* ------------------------------------------------------------------------------------------------------------
 * Ray casts (an extension): the first point of a segment at or under the displaced surface (projectiles, line of
 * sight, picking, camera under water), marched on the device over the same 1..4 slots as the surface queries.
 * H(q) below is the height of a surface query (same slots, same iterations I) evaluated at slot-local positions q_s.
 * All fp32 operations are round-to-nearest and happen in this order ("fl" = one rounding):
 *   Ray: o = (ox, oy, oz), range tmax, direction d.  m = max(|dx|, |dy|, |dz|); v = fl(d / m) per component;
 *       len = fl(sqrt(fl(fl(vx*vx + vy*vy) + vz*vz))); d^ = fl(v / len) per component.
 *   INVALID: o or d has a non-finite component, d = 0, or tmax is NaN or negative (+inf is allowed).  distance, x, z
 *       and the sample are NaN.  Rays are checked one by one on the device: bad data is never a call error.
 *   Slab: Hb = fl(fl(sum_s |A_s|) * (1 + 2^-10)) > |every height a query or the march can return| (proof in
 *       csrc/wso_query.cuh).  oy < -Hb: ORIGIN_BELOW.  Otherwise, d^y != 0: t1 = fl(fl(Hb - oy) / d^y),
 *       t2 = fl(fl(-Hb - oy) / d^y), entry = min, exit = max; d^y = 0: entry = -inf, exit = +inf if oy <= Hb else -inf.
 *       s0 = max(0, entry), s_end = min(tmax, exit).  s0 > s_end: MISS without any sample.
 *   March positions: per cascade p_s = (reduce_mod(ox, L_s), reduce_mod(oz, L_s)) (float64 mod L_s, rounded once, as
 *       the queries do); at parameter t: q_s = (fl(p_s.x + fl(t*d^x)), fl(p_s.z + fl(t*d^z))), y = fl(oy + fl(t*d^y)).
 *       The point is at or under the surface, f(t) <= 0, when y <= H(q).  Accuracy depends on the distance marched,
 *       not on |o|.
 *   March: t_k = fl(s0 + fl(k*step)) for k = 0, 1, ... while t_k < s_end, then t = s_end; at most max_steps samples.
 *       The first sample with f <= 0 ends the march: at k = 0 with s0 = 0 it is ORIGIN_BELOW; otherwise a HIT
 *       bracketed by [a, b] = [previous sample, this sample] (at k = 0 with s0 > 0: [s0, s0]).  The sample at s_end
 *       with f > 0: MISS.  max_steps samples taken before s_end: UNRESOLVED.
 *   Refine (HIT): `refine` times m = fl(a + fl(0.5 * fl(b - a))); f(m) > 0 ? a = m : b = m.  distance = b: a point
 *       at or under the surface at most step * 2^-refine past the first sign change the march saw.
 *   Record (48 bytes): HIT / ORIGIN_BELOW (distance b = 0): x = fl(ox + fl(b*d^x)), z = fl(oz + fl(b*d^z)) and
 *       `surface` = bit for bit the wso_surface_sample wso_query_surface returns at (x, z) with the same slots and
 *       iterations (surface.height is the hit's y).  MISS: distance +inf.  UNRESOLVED: distance = the parameter of the
 *       last sample; continue with origin o + distance*d^ and range tmax - distance.  Both: x, z, surface NaN.
 * A march step costs one H evaluation: 4 * n_slots * (I + 1) displacement texels; the normal maps are read only for
 * the record.  Choose step at most the finest texel spacing L_s/N: a ray can pass through a wave crest thinner than
 * step between two samples without seeing it (tunnelling).
 * wso_raycast_surface: rays_dev = n x 8 floats (ox, oy, oz, tmax, dx, dy, dz, unused), out_dev = n records, device
 *   pointers, both 16-byte aligned; asynchronous on the context's stream, ONE kernel launch.
 * wso_raycast_surface_host: host pointers; blocking; stages through library-owned device memory grown on demand.
 * WSO_ERR_INVALID_ARG (state unchanged): everything wso_query_surface rejects (slots, n_slots, iterations > 16), a NULL
 * p, step not finite and > 0, max_steps outside 1..4096, refine > 24, a NULL or misaligned pointer.  n == 0 is a no-op.
 * Not on the slab path. */
typedef struct wso_ray_params {
    float step;           /* march spacing along the ray, world units, finite and > 0 */
    uint32_t max_steps;   /* march samples per ray, 1..4096 */
    uint32_t refine;      /* bisection steps after a bracket, 0..24 */
    uint32_t iterations;  /* inversion steps of every H evaluation, 0..16 (as wso_query_surface) */
} wso_ray_params;
enum { WSO_RAY_MISS = 0, WSO_RAY_HIT = 1, WSO_RAY_ORIGIN_BELOW = 2, WSO_RAY_UNRESOLVED = 3, WSO_RAY_INVALID = 4 };
typedef struct wso_ray_hit {
    float distance;               /* along d^: b (hit), 0 (origin below), +inf (miss), last sample (unresolved), NaN */
    float x, z;                   /* world position of the hit */
    uint32_t status;              /* WSO_RAY_* */
    wso_surface_sample surface;   /* wso_query_surface at (x, z) */
} wso_ray_hit;
WSO_API int wso_raycast_surface(wso_ctx* ctx, uint32_t n_slots, const uint32_t* slots, const wso_ray_params* p,
                                uint32_t n, const float* rays_dev, wso_ray_hit* out_dev);
WSO_API int wso_raycast_surface_host(wso_ctx* ctx, uint32_t n_slots, const uint32_t* slots, const wso_ray_params* p,
                                     uint32_t n, const float* rays_host, wso_ray_hit* out_host);

/* ------------------------------------------------------------------------------------------------------------
 * External-memory interop (SURVEY row f-2): the maps land in memory a Vulkan device can bind, so the renderer's
 * vkCmdCopyBufferToImage reads them where K2 wrote them.  Replaces: the two 16*N*N-byte memcpy calls into the mapped
 * staging buffer and the PCIe upload behind them (WaterSurfaceMesh.cpp:701-755, vulkan/Texture2D.cpp:175-226).
 * Both directions of VK_KHR_external_memory_fd are offered:
 *   wso_set_exportable + wso_export_fd : the library allocates the map arrays with the CUDA virtual-memory API
 *       (POSIX-fd shareable) and hands out a file descriptor; Vulkan imports it with VkImportMemoryFdInfoKHR
 *       { handleType = VK_EXTERNAL_MEMORY_HANDLE_TYPE_OPAQUE_FD_BIT } and binds a VkBuffer of *bytes to it.
 *       The caller owns the returned fd (close() it, or let the Vulkan import consume it).
 *   wso_import_external_fd : Vulkan allocated and exported the memory (vkGetMemoryFdKHR); the library maps
 *       [offset, offset + max_slots*16*N*N) of it as the output array of map `which` (8*N*N per slot in RGBA16F).  On success the fd belongs
 *       to CUDA.  A tile-size change (Prepare after SetTileSize) drops the import and returns to own memory.
 * Layout either way: [slot][N*N] RGBA32F texels, slot s at byte offset s*16*N*N (+ offset), row pitch 16*N
 * (RGBA16F maps, wso_set_map_format: 8*N*N and 8*N).
 * Map contents are reset to zero by wso_set_exportable / wso_import_external_fd; Prepare() state is kept.
 * Ordering with the renderer: wso_import_semaphore_fd binds an exported VkSemaphore (binary: is_timeline = 0,
 * timeline: 1; `index` 0 or 1); wso_signal_semaphore / wso_wait_semaphore enqueue a signal / wait on the context's
 * stream after / before the work enqueued around them (value ignored for binary semaphores). */
WSO_API int wso_set_exportable(wso_ctx* ctx, int on);
WSO_API int wso_export_fd(wso_ctx* ctx, int which, int* fd, size_t* bytes);
WSO_API int wso_import_external_fd(wso_ctx* ctx, int which, int fd, size_t bytes, size_t offset);
WSO_API int wso_import_semaphore_fd(wso_ctx* ctx, int index, int fd, int is_timeline);
WSO_API int wso_signal_semaphore(wso_ctx* ctx, int index, uint64_t value);
WSO_API int wso_wait_semaphore(wso_ctx* ctx, int index, uint64_t value);

/* Plumbing: run on a caller-owned CUDA stream (cudaStream_t as void*; NULL = the context's own), and
 * pinned host allocations for wso_compute_to_host. */
WSO_API int wso_set_stream(wso_ctx* ctx, void* cuda_stream);
WSO_API int wso_alloc_host(size_t bytes, void** ptr);
WSO_API int wso_free_host(void* ptr);
/* Page-lock memory the CALLER owns (e.g. the storage of the std::vector<glm::vec4> the reference's accessors hand out,
 * WSTessendorf.h:95-101) so that wso_compute_to_host copies straight into it at full PCIe speed; unregister before
 * the memory is freed or reallocated.  Failing to register is not fatal: the copies then go through pageable memory. */
WSO_API int wso_register_host(void* ptr, size_t bytes);
WSO_API int wso_unregister_host(void* ptr);

/* Two implementations of the three hot-path kernels exist for 512^2, 1024^2 and 2048^2 batched launches: CTA-per-line
 * (Stockham stages through shared memory) and warp-per-line (radix-32 register stages, shuffle exchanges, bulk-copy line
 * pipeline).  They produce the same maps within the parity tolerance and share the intermediate layout.  mask bit 0 / 1 /
 * 2 puts K1 / K2h / K2 on the warp-per-line set; bits 4 / 6 (0x10 / 0x40) run K1 / K2 of the CTA-per-line set in their
 * persistent form (a fixed grid of CTAs walks the work items and requests the inputs of its next item ahead of the store
 * phase of the current one; bit-identical results); -1 restores the built-in choice (what measured faster per size).
 * Any other bit: WSO_ERR_INVALID_ARG.  Process-wide; meant for A/B measurements and for the parity tests, which run
 * every form.  A context with RGBA16F maps (wso_set_map_format) runs the CTA-per-line K2 whatever bit 2 says (the
 * warp-per-line K2 writes RGBA32F only); the K1 / K2h choice and bit 6 apply as usual. */
WSO_API int wso_select_kernels(int mask);

/* Introspection used by the benchmark: number of kernels launched so far by this context, the chunk
 * (tile-frames per launch) the batched calls use, and the CTA tiling of the two transform kernels. */
WSO_API int wso_get_stats(const wso_ctx* ctx, uint64_t* kernel_launches, uint32_t* chunk);

/* A call that computes ONE tile-frame (wso_compute, wso_compute_async, wso_compute_to_host or wso_compute_batch with
 * n == 1 - the reference's one ComputeWaves(t) per rendered frame, WaterSurfaceMesh.cpp:123-154) is enqueued as one
 * launch of an instantiated CUDA graph holding the frame's three kernels, whose parameters are rewritten per call,
 * instead of three kernel launches.  on = 1 (default): for tile sizes up to 512, where the launches cost more host time
 * than the kernels take on the device (12.3 instead of 15.6 us per 512^2 frame back to back on B200); larger tiles keep
 * plain launches, whose programmatic dependent launch overlaps consecutive frames.  on = 2: every size; on = 0: never
 * (also: environment WSO_FRAME_GRAPH=0|1|2).  The counters say how many frames went out as graph launches and how often
 * the graph was (re)captured. */
WSO_API int wso_set_frame_graph(wso_ctx* ctx, int on);
WSO_API int wso_get_frame_graph_stats(const wso_ctx* ctx, uint64_t* graph_launches, uint64_t* captures);

/* Opt-in per-kernel device timing (the analogue of the reference's VKP_PROFILE_SCOPE table,
 * core/Profile.h:16-32): with profiling on, every launch is bracketed by CUDA events on the compute
 * stream.  wso_get_profile synchronises and returns the accumulated milliseconds of
 * {K1 evolve+first transform, K2h height extrema, K2 second transform+pack}, the number of launches of each
 * and the tile-frames they covered since wso_set_profiling(ctx, 1). */
WSO_API int wso_set_profiling(wso_ctx* ctx, int on);
WSO_API int wso_get_profile(wso_ctx* ctx, double* kernel_ms3, uint64_t* launches, uint64_t* tile_frames);

/* ------------------------------------------------------------------------------------------------------------
 * Slab-decomposed path: ONE large grid (2048..16384 per side) spread over P = 1, 2, 4 or 8 devices, one process
 * and one wso_slab per device (BASELINE.json configs[4]; no reference counterpart - the reference caps the tile at
 * 1024^2, WaterSurfaceMesh.h:45-46 - the arithmetic is the same ComputeWaves, WSTessendorf.cpp:284-441).
 * Rank r evolves and transforms (along m) the column pairs (n, N-n) for n in [r*N/2P, (r+1)*N/2P) and, after the
 * exchange, transforms (along n) and packs the rows m' and N-m' for m' in the same range.  Per tile-frame:
 *     wso_slab_pass1(t)  ->  wso_slab_exchange  ->  wso_slab_heights  ->  all-reduce (min, max)  ->  wso_slab_pass2
 * pass1 stores what it separates where its threads hold it (coalesced); wso_slab_exchange is ONE transposing kernel
 * that carries the Hl x Hl blocks to the owners of the row items in 256-byte rows:
 *   fused   - straight into the owners' receive buffers over NVLink peer mappings (wso_slab_ipc_handle /
 *             wso_slab_open_peer / wso_slab_set_fused), followed by any stream-ordered inter-rank barrier of the caller's;
 *             the receive buffers alternate by frame parity, so frames may be enqueued back to back without host syncs;
 *   unfused - into the `world` equal blocks of the local send buffer, which the caller then moves with ONE all-to-all
 *             into the receive buffer (e.g. torch.distributed.all_to_all_single over NCCL) on the slab's stream.
 * The all-reduce (min over [0], max over [1] of the 2-float minmax buffer) is the caller's as well. */
typedef struct wso_slab wso_slab;
WSO_API int wso_slab_create(const wso_params* p, int device, uint32_t rank, uint32_t world, wso_slab** out);
WSO_API int wso_slab_destroy(wso_slab* s);
/* Spectrum of this rank's columns: from a full N*N array in the reference layout (small grids, tests), or generated
 * in place from a counter-based Gaussian source (seed, m*N+n) with the reference's Phillips/dispersion arithmetic
 * (WSTessendorf.cpp:105-148).  wso_counter_h0 evaluates the same records for rows [m0, m0+rows) - for checkers. */
WSO_API int wso_slab_import_h0(wso_slab* s, const wso_h0_record* h0_full);
WSO_API int wso_slab_prepare_counter(wso_slab* s, uint64_t seed);
/* the same spectrum built by the device Prepare kernel (this rank's column pairs only; no host pass) */
WSO_API int wso_slab_prepare_counter_device(wso_slab* s, uint64_t seed);
WSO_API int wso_counter_h0(const wso_params* p, uint64_t seed, uint32_t m0, uint32_t rows, wso_h0_record* out);
WSO_API int wso_slab_set_lambda(wso_slab* s, float lambda);
WSO_API int wso_slab_set_stream(wso_slab* s, void* cuda_stream);
/* Exchange buffers: send/recv = `world` blocks of block_bytes each (block d of send goes to rank d; block r of recv
 * came from rank r); minmax = 2 floats written by wso_slab_heights, to be all-reduced before wso_slab_pass2. */
WSO_API int wso_slab_buffers(wso_slab* s, void** send, void** recv, size_t* block_bytes, void** minmax);
/* Fused exchange: 64-byte CUDA IPC handle of this rank's receive buffer; map every peer's, then switch on. */
WSO_API int wso_slab_ipc_handle(wso_slab* s, void* handle64);
WSO_API int wso_slab_open_peer(wso_slab* s, uint32_t peer, const void* handle64);
WSO_API int wso_slab_set_fused(wso_slab* s, int on);
/* Use the two-CTA cluster variant of K2 (always used at 16384, where a line pair exceeds one SM's shared memory). */
WSO_API int wso_slab_force_pair(wso_slab* s, int on);
WSO_API int wso_slab_pass1(wso_slab* s, float t);
WSO_API int wso_slab_exchange(wso_slab* s);
/* Pipelined form of the two calls above: packed fields [field0, field0 + nfields) only (whole field groups,
 * wso_slab_fields_per_group), the exchange on `cuda_stream` (NULL = the slab's stream), so that the transfer of one field
 * overlaps the transform of the next.  wso_slab_pass1_fields with field0 == 0 starts a new tile-frame. */
WSO_API int wso_slab_pass1_fields(wso_slab* s, float t, int field0, int nfields);
WSO_API int wso_slab_exchange_fields(wso_slab* s, int field0, int nfields, void* cuda_stream);
WSO_API int wso_slab_fields_per_group(const wso_slab* s);
WSO_API int wso_slab_heights(wso_slab* s);
WSO_API int wso_slab_pass2(wso_slab* s);
WSO_API int wso_slab_sync(wso_slab* s);
WSO_API int wso_slab_read_heights(wso_slab* s, float* amplitude, float* min_height, float* max_height);
/* Output: this rank's 2*N/2P rows of each map, N RGBA32F texels per row; wso_slab_row_index gives the global row
 * of every local row (local row ml < N/2P is row m' = r*N/2P + ml, local row N/2P + ml its mirror N-m'; N/2 for m'=0). */
WSO_API int wso_slab_map_device(wso_slab* s, int which, void** dptr, uint32_t* rows);
WSO_API int wso_slab_copy_rows(wso_slab* s, int which, float* dst_host);
WSO_API int wso_slab_row_index(const wso_slab* s, uint32_t* rows);
WSO_API const char* wso_slab_last_error(const wso_slab* s);

WSO_API const char* wso_last_error(const wso_ctx* ctx); /* ctx may be NULL: last create failure */
WSO_API const char* wso_version(void);

#ifdef __cplusplus
}
#endif
#endif /* WSOCEAN_H_ */
