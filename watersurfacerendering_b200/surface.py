"""Python mirror of the reference surface-model interface, on top of the C ABI.

`WSTessendorf` keeps the reference's method names, argument meaning and error behaviour
(reference: src/scene/WSTessendorf.h:58-122, src/scene/WSTessendorf.cpp:459-505) so the parity tests read
like tests of the reference class; the batched / multi-tile calls are the B200 extensions
(BASELINE.json configs 2-4).  All arithmetic happens in libwsocean.so (hand-written sm_100a kernels).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _lib as L

# reference: WSTessendorf.h:142-147
H0_DTYPE = np.dtype(
    [("re", "<f4"), ("im", "<f4"), ("re_c", "<f4"), ("im_c", "<f4"), ("omega", "<f4")]
)
# wso_surface_sample: height, normal (x, y, z), offset (x, z) = undisplaced origin - query, residual, w
SURFACE_SAMPLE_DTYPE = np.dtype(L.SURFACE_SAMPLE_DTYPE)
# wso_ray_hit: distance, hit x / z, status (WSO_RAY_*), then the wso_surface_sample at (x, z)
RAY_HIT_DTYPE = np.dtype(L.RAY_HIT_DTYPE)
# wso_body: rotation (row-major, body -> world), position, center (reference point), vertex / triangle ranges
BODY_DTYPE = np.dtype(L.BODY_DTYPE)
# wso_hydro_result: force (world axes), wetted area, torque (about position + rotation @ center), status (WSO_HYDRO_*)
HYDRO_RESULT_DTYPE = np.dtype(L.HYDRO_RESULT_DTYPE)


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


SPECTRUM_KINDS = {"phillips": L.WSO_SPECTRUM_PHILLIPS, "pierson_moskowitz": L.WSO_SPECTRUM_PIERSON_MOSKOWITZ,
                  "jonswap": L.WSO_SPECTRUM_JONSWAP, "tma": L.WSO_SPECTRUM_TMA}


def make_spectrum(kind="phillips", *, fetch: float = 1e5, depth: float = np.inf, gamma: float = 3.3,
                  spread: float = 0.0, k_band=(0.0, np.inf), scale: float = 1.0) -> "L.WsoSpectrum":
    """A struct wso_spectrum; ``kind`` is a WSO_SPECTRUM_* value or one of SPECTRUM_KINDS' names.  The defaults are
    wso_default_spectrum's.  Validation happens in the library (wso_set_spectrum / wso_spectrum_h0)."""
    s = L.WsoSpectrum()
    s.kind = SPECTRUM_KINDS[kind.lower()] if isinstance(kind, str) else int(kind)
    s.fetch, s.depth, s.gamma, s.spread = float(fetch), float(depth), float(gamma), float(spread)
    s.k_min, s.k_max = float(k_band[0]), float(k_band[1])
    s.scale = float(scale)
    return s


def spectrum_dict(s: "L.WsoSpectrum") -> dict:
    return {"kind": int(s.kind), "fetch": s.fetch, "depth": s.depth, "gamma": s.gamma, "spread": s.spread,
            "k_band": (s.k_min, s.k_max), "scale": s.scale}


def spectrum_h0(params: "L.WsoParams", spectrum: "L.WsoSpectrum", xi: Optional[np.ndarray] = None, seed: int = 0,
                m0: int = 0, rows: Optional[int] = None) -> np.ndarray:
    """Host build of the spectrum records (wso_spectrum_h0), rows [m0, m0+rows) in the reference layout: from the
    N*N Gaussian array ``xi`` (as PrepareWithGauss), or from the counter generator of PrepareCounterOnDevice (``seed``)."""
    n = int(params.tile_size)
    rows = n - m0 if rows is None else int(rows)
    if xi is not None:
        xi = np.ascontiguousarray(xi, np.complex64).reshape(n, n)
    out = np.zeros((rows, n), H0_DTYPE)
    L.check(L.load().wso_spectrum_h0(C.byref(params), C.byref(spectrum), _ptr(xi), int(seed), int(m0), rows,
                                     out.ctypes.data_as(C.c_void_p)))
    return out


class PinnedBuffer:
    """Page-locked host memory (wso_alloc_host) exposed as a NumPy array."""

    def __init__(self, shape, dtype=np.float32):
        self._lib = L.load()
        self.shape = tuple(shape)
        self.nbytes = int(np.prod(self.shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        L.check(self._lib.wso_alloc_host(self.nbytes, C.byref(p)))
        self._p = p
        buf = (C.c_char * self.nbytes).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=dtype).reshape(self.shape)

    def close(self):
        if self._p is not None:
            self.array = None
            self._lib.wso_free_host(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class WSTessendorf:
    """Tessendorf ocean surface model, computed on a B200.

    Reference call sequence: construct, set parameters, ``Prepare()``, then ``ComputeWaves(t)`` per frame
    and read ``GetDisplacements()`` / ``GetNormals()``.
    """

    s_kDefaultTileSize = 512          # reference: WSTessendorf.h:36-43
    s_kDefaultTileLength = 1000.0
    s_kDefaultWindDir = (1.0, 1.0)
    s_kDefaultWindSpeed = 30.0
    s_kDefaultAnimPeriod = 200.0
    s_kDefaultPhillipsConst = 3e-7
    s_kDefaultPhillipsDamping = 0.1

    def __init__(self, tileSize: int = 512, tileLength: float = 1000.0, *, device: int = 0,
                 max_tiles: int = 1, max_slots: int = 1):
        self._lib = L.load()
        p = L.WsoParams()
        L.check(self._lib.wso_default_params(C.byref(p)))
        p.tile_size = int(tileSize)
        p.tile_length = float(tileLength)
        h = C.c_void_p()
        L.check(self._lib.wso_create(C.byref(p), int(device), int(max_tiles), int(max_slots), C.byref(h)))
        self._h = h
        self.device = int(device)
        self.max_tiles = int(max_tiles)
        self.max_slots = int(max_slots)
        self._min = np.float32(-1.0)   # reference: WSTessendorf.h:226-227
        self._max = np.float32(1.0)
        self._map_dtype = np.float32   # texel channel type of both maps (set_map_format)

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.wso_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ------------------------------------------------------------------ parameters
    def _get(self, tile=0) -> L.WsoParams:
        p = L.WsoParams()
        L.check(self._lib.wso_get_params(self._h, tile, C.byref(p)), self._h)
        return p

    def _raw(self, tile=0) -> L.WsoParams:
        return self._get(tile)

    def _set(self, tile, **kw) -> int:
        p = self._get(tile)
        for k, v in kw.items():
            setattr(p, k, v)
        return self._lib.wso_set_params(self._h, tile, C.byref(p))

    def GetTileSize(self, tile=0): return int(self._get(tile).tile_size)
    def GetTileLength(self, tile=0): return float(self._get(tile).tile_length)
    def GetWindDir(self, tile=0):
        p = self._get(tile)
        return np.array([p.wind_dir_x, p.wind_dir_y], np.float32)
    def GetWindSpeed(self, tile=0): return float(self._get(tile).wind_speed)
    def GetAnimationPeriod(self, tile=0): return float(self._get(tile).anim_period)
    def GetPhillipsConst(self, tile=0): return float(self._get(tile).phillips_const)
    def GetDamping(self, tile=0): return float(self._get(tile).damping)
    def GetDisplacementLambda(self, tile=0): return float(self._get(tile).lambda_)
    def GetMinHeight(self): return self._min
    def GetMaxHeight(self): return self._max

    def SetTileSize(self, size: int, tile=0):
        """Non power-of-two sizes are ignored, like the reference (WSTessendorf.cpp:459-468)."""
        rc = self._set(tile, tile_size=int(size)) if 0 < int(size) < 2 ** 32 else L.WSO_ERR_BAD_TILE_SIZE
        if rc not in (L.WSO_OK, L.WSO_ERR_BAD_TILE_SIZE):
            L.check(rc, self._h)
        return rc == L.WSO_OK

    def SetTileLength(self, length: float, tile=0): L.check(self._set(tile, tile_length=float(length)), self._h)
    def SetWindDirection(self, w: Sequence[float], tile=0):
        L.check(self._set(tile, wind_dir_x=float(w[0]), wind_dir_y=float(w[1])), self._h)
    def SetWindSpeed(self, v: float, tile=0): L.check(self._set(tile, wind_speed=float(v)), self._h)
    def SetAnimationPeriod(self, T: float, tile=0): L.check(self._set(tile, anim_period=float(T)), self._h)
    def SetPhillipsConst(self, A: float, tile=0): L.check(self._set(tile, phillips_const=float(A)), self._h)
    def SetDamping(self, d: float, tile=0): L.check(self._set(tile, damping=float(d)), self._h)
    def SetLambda(self, lam: float, tile=0): L.check(self._lib.wso_set_lambda(self._h, tile, float(lam)), self._h)

    def SetComputeJacobian(self, on: bool = True):
        """The reference's COMPUTE_JACOBIAN switch (WSTessendorf.cpp:421-428, dead code there) at run time:
        displacement.w = Jacobian of the horizontal displacement instead of 1."""
        L.check(self._lib.wso_set_compute_jacobian(self._h, 1 if on else 0), self._h)

    def GetComputeJacobian(self) -> bool:
        v = C.c_int()
        L.check(self._lib.wso_get_compute_jacobian(self._h, C.byref(v)), self._h)
        return bool(v.value)

    # ------------------------------------------------------------------ wave spectra
    def set_spectrum(self, kind="phillips", tile: int = 0, **kw):
        """Spectrum of ``tile`` from its next Prepare on (wso_set_spectrum): ``kind`` = "phillips" (default, the
        reference's), "pierson_moskowitz", "jonswap" or "tma"; keywords fetch, depth, gamma, spread, k_band = (k_min,
        k_max), scale as in make_spectrum."""
        s = make_spectrum(kind, **kw)
        L.check(self._lib.wso_set_spectrum(self._h, tile, C.byref(s)), self._h)

    def get_spectrum(self, tile: int = 0) -> dict:
        s = L.WsoSpectrum()
        L.check(self._lib.wso_get_spectrum(self._h, tile, C.byref(s)), self._h)
        return spectrum_dict(s)

    # ------------------------------------------------------------------ prepare
    def Prepare(self, seed: Optional[int] = None, tile: int = 0):
        """reference Prepare(); ``seed`` = srand(seed) first (the reference app seeds with the clock)."""
        L.check(self._lib.wso_prepare(self._h, tile, 0 if seed is None else 1, 0 if seed is None else int(seed)),
                self._h)

    def PrepareWithGauss(self, xi: np.ndarray, tile: int = 0):
        n = self.GetTileSize(tile)
        xi = np.ascontiguousarray(xi, np.complex64).reshape(n, n)
        L.check(self._lib.wso_prepare_gauss(self._h, tile, _ptr(xi)), self._h)

    def PrepareWithGaussOnDevice(self, xi: np.ndarray, tile: int = 0):
        """Prepare() with the spectrum built by the device kernel (wso_prepare_gauss_device) from the Gaussian array."""
        n = self.GetTileSize(tile)
        xi = np.ascontiguousarray(xi, np.complex64).reshape(n, n)
        L.check(self._lib.wso_prepare_gauss_device(self._h, tile, _ptr(xi)), self._h)

    def PrepareCounterOnDevice(self, seed: int, tile: int = 0):
        """Prepare() entirely on the device: counter-based Gaussian array + spectrum (wso_prepare_counter)."""
        L.check(self._lib.wso_prepare_counter(self._h, tile, int(seed)), self._h)

    def ImportH0(self, h0: np.ndarray, tile: int = 0):
        n = self.GetTileSize(tile)
        if h0.dtype != H0_DTYPE:
            h0 = np.ascontiguousarray(h0, np.float32).reshape(n, n, 5).view(H0_DTYPE)
        h0 = np.ascontiguousarray(h0).reshape(n, n)
        L.check(self._lib.wso_import_h0(self._h, tile, _ptr(h0)), self._h)

    def ExportH0(self, tile: int = 0) -> np.ndarray:
        n = self.GetTileSize(tile)
        h0 = np.zeros((n, n), H0_DTYPE)
        L.check(self._lib.wso_export_h0(self._h, tile, _ptr(h0)), self._h)
        return h0

    def ImportH0Compact(self, h0_3f: np.ndarray, tile: int = 0):
        """(N,N,3) fp32 (amp.re, amp.im, dispersion): 12 bytes per wave vector instead of the reference's 20."""
        n = self.GetTileSize(tile)
        a = np.ascontiguousarray(h0_3f, np.float32).reshape(n, n, 3)
        L.check(self._lib.wso_import_h0_compact(self._h, tile, _ptr(a)), self._h)

    def ExportH0Compact(self, tile: int = 0) -> np.ndarray:
        n = self.GetTileSize(tile)
        a = np.zeros((n, n, 3), np.float32)
        L.check(self._lib.wso_export_h0_compact(self._h, tile, _ptr(a)), self._h)
        return a

    def ComputeWavesAsync(self, t: float) -> int:
        """Enqueue one frame (tile 0 -> device slot 0), no host copy, no synchronisation. -> cudaEvent_t handle (int)."""
        ev = C.c_void_p()
        L.check(self._lib.wso_compute_async(self._h, float(t), C.byref(ev)), self._h)
        return ev.value

    def WaitEvent(self, event: int):
        L.check(self._lib.wso_wait_event(self._h, C.c_void_p(event)), self._h)

    # ------------------------------------------------------------------ per-frame (reference API)
    def ComputeWaves(self, t: float) -> np.float32:
        a = C.c_float()
        L.check(self._lib.wso_compute(self._h, float(t), C.byref(a)), self._h)
        mn, mx = np.zeros(1, np.float32), np.zeros(1, np.float32)
        L.check(self._lib.wso_read_heights(self._h, 0, 1, None, _ptr(mn), _ptr(mx)), self._h)
        self._min, self._max = mn[0], mx[0]
        return np.float32(a.value)

    def _host_map(self, which) -> np.ndarray:
        n = self.GetTileSize()
        if self._map_dtype is np.float16:
            p, nbytes = C.c_void_p(), C.c_size_t()
            L.check(self._lib.wso_map_host_bytes(self._h, which, C.byref(p), C.byref(nbytes)), self._h)
            buf = (C.c_char * nbytes.value).from_address(p.value)
            return np.frombuffer(buf, dtype=np.float16).reshape(n, n, 4)
        p, cnt = C.c_void_p(), C.c_size_t()
        L.check(self._lib.wso_map_host(self._h, which, C.byref(p), C.byref(cnt)), self._h)
        buf = (C.c_float * (cnt.value * 4)).from_address(p.value)
        return np.frombuffer(buf, dtype=np.float32).reshape(n, n, 4)

    # ---- map format (extension: RGBA16F maps, half the bytes of the reference's RGBA32F)
    def set_map_format(self, fmt: str):
        """"rgba32f" (default, the reference's format) or "rgba16f": 4 x binary16 per texel, each channel the fp32 value
        rounded to nearest even.  Reallocates the maps (contents reset to the resize() defaults); Prepare() state is kept.
        In "rgba16f" the map accessors return np.float16 arrays."""
        code = {"rgba32f": L.WSO_MAP_RGBA32F, "rgba16f": L.WSO_MAP_RGBA16F}.get(fmt)
        if code is None:
            raise ValueError(f"map format must be 'rgba32f' or 'rgba16f', not {fmt!r}")
        L.check(self._lib.wso_set_map_format(self._h, code), self._h)
        self._map_dtype = np.float16 if code == L.WSO_MAP_RGBA16F else np.float32

    def get_map_format(self) -> str:
        v = C.c_int()
        L.check(self._lib.wso_get_map_format(self._h, C.byref(v)), self._h)
        return "rgba16f" if v.value == L.WSO_MAP_RGBA16F else "rgba32f"

    def GetDisplacementCount(self): return self.GetTileSize() ** 2
    def GetNormalCount(self): return self.GetTileSize() ** 2
    def GetDisplacements(self) -> np.ndarray:
        """(N,N,4) view of the pinned host copy written by ComputeWaves (valid until the next call); np.float16 with
        RGBA16F maps."""
        return self._host_map(L.WSO_MAP_DISPLACEMENT)
    def GetNormals(self) -> np.ndarray:
        return self._host_map(L.WSO_MAP_NORMAL)

    # ------------------------------------------------------------------ batched / device-resident
    def compute_batch(self, times, tiles=None, first_slot: int = 0):
        t = np.ascontiguousarray(times, np.float32)
        tl = None if tiles is None else np.ascontiguousarray(tiles, np.uint32)
        L.check(self._lib.wso_compute_batch(self._h, t.size, _ptr(tl), _ptr(t), int(first_slot)), self._h)

    def compute_to_host(self, times, disp_out: np.ndarray, norm_out: np.ndarray, tiles=None):
        """Streams every tile-frame's maps into host arrays (ideally PinnedBuffer.array, np.float16 with RGBA16F maps).
        -> (A, min, max)"""
        t = np.ascontiguousarray(times, np.float32)
        tl = None if tiles is None else np.ascontiguousarray(tiles, np.uint32)
        a = np.zeros(t.size, np.float32)
        mn = np.zeros(t.size, np.float32)
        mx = np.zeros(t.size, np.float32)
        assert disp_out.dtype == self._map_dtype and norm_out.dtype == self._map_dtype
        assert disp_out.flags.c_contiguous and norm_out.flags.c_contiguous
        need = t.size * self.GetTileSize() ** 2 * 4
        assert disp_out.size >= need and norm_out.size >= need
        if self._map_dtype is np.float16:
            L.check(self._lib.wso_compute_to_host_bytes(self._h, t.size, _ptr(tl), _ptr(t), _ptr(disp_out),
                                                        _ptr(norm_out), min(disp_out.nbytes, norm_out.nbytes),
                                                        _ptr(a), _ptr(mn), _ptr(mx)), self._h)
            return a, mn, mx
        L.check(self._lib.wso_compute_to_host(self._h, t.size, _ptr(tl), _ptr(t), _ptr(disp_out),
                                              _ptr(norm_out), _ptr(a), _ptr(mn), _ptr(mx)), self._h)
        return a, mn, mx

    def sync(self):
        L.check(self._lib.wso_sync(self._h), self._h)

    def read_heights(self, first_slot: int, n: int):
        a = np.zeros(n, np.float32)
        mn = np.zeros(n, np.float32)
        mx = np.zeros(n, np.float32)
        L.check(self._lib.wso_read_heights(self._h, first_slot, n, _ptr(a), _ptr(mn), _ptr(mx)), self._h)
        return a, mn, mx

    def copy_map(self, which: int, slot: int = 0) -> np.ndarray:
        n = self.GetTileSize()
        if self._map_dtype is np.float16:
            out = np.empty((n, n, 4), np.float16)
            L.check(self._lib.wso_copy_map_bytes(self._h, which, slot, _ptr(out), out.nbytes), self._h)
            return out
        out = np.empty((n, n, 4), np.float32)
        L.check(self._lib.wso_copy_map(self._h, which, slot, _ptr(out)), self._h)
        return out

    def map_device(self, which: int, slot: int = 0) -> int:
        p, cnt = C.c_void_p(), C.c_size_t()
        L.check(self._lib.wso_map_device(self._h, which, slot, C.byref(p), C.byref(cnt)), self._h)
        return int(p.value)

    # ---- surface queries (extension: the surface at arbitrary world points, sampled on the device)
    @staticmethod
    def _slots(slots):
        sl = np.ascontiguousarray(np.atleast_1d(np.asarray(slots)), np.uint32)
        return sl, int(sl.size)

    def query_surface(self, xz, slots=(0,), iterations: int = 4) -> np.ndarray:
        """Height, normal and undisplaced origin of the surface above the world points xz ((n, 2) or (2,) array of
        (x, z)), summed over the cascades `slots` (1..4 slots holding computed frames), with `iterations` fixed-point steps
        of the choppy-displacement inversion.  Blocking (wso_query_surface_host).  -> structured array of n records
        (SURFACE_SAMPLE_DTYPE: height, normal_x/y/z, offset_x/z, residual, w)."""
        q = np.ascontiguousarray(xz, np.float32).reshape(-1, 2)
        out = np.zeros(q.shape[0], SURFACE_SAMPLE_DTYPE)
        sl, ns = self._slots(slots)
        L.check(self._lib.wso_query_surface_host(self._h, ns, _ptr(sl), int(iterations), q.shape[0], _ptr(q),
                                                 _ptr(out)), self._h)
        return out

    def query_surface_device(self, xz_ptr: int, out_ptr: int, n: int, slots=(0,), iterations: int = 4):
        """The same on device memory (e.g. tensor.data_ptr()): xz_ptr = n (x, z) float pairs, out_ptr = n 32-byte records
        (16-byte aligned).  Asynchronous on the context's stream (wso_query_surface)."""
        sl, ns = self._slots(slots)
        L.check(self._lib.wso_query_surface(self._h, ns, _ptr(sl), int(iterations), int(n), C.c_void_p(xz_ptr or 0),
                                            C.c_void_p(out_ptr or 0)), self._h)

    # ---- ray casts (extension: first hit of a segment with the displaced surface, marched on the device)
    @staticmethod
    def _ray_params(step, max_steps, refine, iterations):
        return L.WsoRayParams(float(step), int(max_steps), int(refine), int(iterations))

    def raycast_surface(self, origins, directions, tmax=np.inf, slots=(0,), *, step: float, max_steps: int = 1024,
                        refine: int = 16, iterations: int = 4) -> np.ndarray:
        """First point at or under the surface of each ray o + t*d/|d|, 0 <= t <= tmax: origins / directions = (n, 3)
        or (3,) arrays of (x, y, z) (broadcast against each other), tmax a scalar or n ranges.  Marched every `step` world
        units (at most the finest texel spacing L/N; at most `max_steps` samples), the bracket refined by `refine`
        bisection steps, every height with `iterations` inversion steps over the cascades `slots`.  Blocking
        (wso_raycast_surface_host).  -> structured array of n records (RAY_HIT_DTYPE: distance, x, z, status =
        WSO_RAY_*, then the surface query at (x, z))."""
        o, d = np.broadcast_arrays(np.atleast_2d(np.asarray(origins, np.float32)),
                                   np.atleast_2d(np.asarray(directions, np.float32)))
        rays = np.zeros((o.shape[0], 8), np.float32)
        rays[:, 0:3] = o
        rays[:, 3] = np.broadcast_to(np.asarray(tmax, np.float32), (o.shape[0],))
        rays[:, 4:7] = d
        out = np.zeros(rays.shape[0], RAY_HIT_DTYPE)
        sl, ns = self._slots(slots)
        p = self._ray_params(step, max_steps, refine, iterations)
        L.check(self._lib.wso_raycast_surface_host(self._h, ns, _ptr(sl), C.byref(p), rays.shape[0], _ptr(rays),
                                                   _ptr(out)), self._h)
        return out

    def raycast_surface_device(self, rays_ptr: int, out_ptr: int, n: int, slots=(0,), *, step: float,
                               max_steps: int = 1024, refine: int = 16, iterations: int = 4):
        """The same on device memory (e.g. tensor.data_ptr()): rays_ptr = n x 8 floats (ox, oy, oz, tmax, dx, dy, dz,
        unused), out_ptr = n 48-byte records, both 16-byte aligned.  Asynchronous on the context's stream
        (wso_raycast_surface)."""
        sl, ns = self._slots(slots)
        p = self._ray_params(step, max_steps, refine, iterations)
        L.check(self._lib.wso_raycast_surface(self._h, ns, _ptr(sl), C.byref(p), int(n), C.c_void_p(rays_ptr or 0),
                                              C.c_void_p(out_ptr or 0)), self._h)

    # ---- hydrostatics (extension: buoyancy force and torque on triangle hulls, integrated on the device)
    @staticmethod
    def _hydro_params(iterations, density, gravity):
        return L.WsoHydroParams(float(density), float(gravity), int(iterations), 0)

    def hydrostatics(self, bodies, vertices, triangles, slots=(0,), iterations: int = 4, density: float = 1025.0,
                     gravity: float = 9.81) -> np.ndarray:
        """Hydrostatic force and torque on each body of `bodies` (BODY_DTYPE array, or one record), a triangle hull in
        `vertices` ((n, 3) or (n, 4) body coordinates) and `triangles` ((m, 3) indices relative to each body's
        vertex_first, counter-clockwise seen from outside), floating in the surface summed over the cascades `slots`
        with `iterations` inversion steps per height.  Blocking (wso_hydrostatics_host).  -> structured array of records
        (HYDRO_RESULT_DTYPE: force, wetted_area, torque about the body's world reference point, status = WSO_HYDRO_*)."""
        b = np.ascontiguousarray(np.atleast_1d(np.asarray(bodies, BODY_DTYPE)))
        v = np.atleast_2d(np.asarray(vertices, np.float32))
        if v.ndim != 2 or v.shape[1] not in (3, 4):
            raise ValueError("vertices must be an (n, 3) or (n, 4) array")
        v4 = np.zeros((v.shape[0], 4), np.float32)
        v4[:, :v.shape[1]] = v
        t = np.ascontiguousarray(triangles, np.uint32).reshape(-1, 3)
        out = np.zeros(b.shape[0], HYDRO_RESULT_DTYPE)
        sl, ns = self._slots(slots)
        p = self._hydro_params(iterations, density, gravity)
        L.check(self._lib.wso_hydrostatics_host(self._h, ns, _ptr(sl), C.byref(p), b.shape[0], _ptr(b), v4.shape[0],
                                                _ptr(v4), t.shape[0], _ptr(t), _ptr(out)), self._h)
        return out

    def hydrostatics_device(self, bodies_ptr: int, n_bodies: int, vertices_ptr: int, n_vertices: int,
                            triangles_ptr: int, n_triangles: int, out_ptr: int, slots=(0,), iterations: int = 4,
                            density: float = 1025.0, gravity: float = 9.81):
        """The same on device memory (e.g. tensor.data_ptr()): n_bodies 80-byte wso_body records, n_vertices x 4 floats,
        n_triangles x 3 uint32, out_ptr = n_bodies 32-byte records; bodies, vertices and out 16-byte aligned.
        Asynchronous on the context's stream (wso_hydrostatics)."""
        sl, ns = self._slots(slots)
        p = self._hydro_params(iterations, density, gravity)
        L.check(self._lib.wso_hydrostatics(self._h, ns, _ptr(sl), C.byref(p), int(n_bodies), C.c_void_p(bodies_ptr or 0),
                                           int(n_vertices), C.c_void_p(vertices_ptr or 0), int(n_triangles),
                                           C.c_void_p(triangles_ptr or 0), C.c_void_p(out_ptr or 0)), self._h)

    # ---- external-memory interop (SURVEY row f-2; replaces the staging memcpy of WaterSurfaceMesh.cpp:701-755)
    def set_exportable(self, on: bool = True):
        """Back the map arrays with memory that can be exported as a POSIX fd (Vulkan: VK_KHR_external_memory_fd)."""
        L.check(self._lib.wso_set_exportable(self._h, 1 if on else 0), self._h)

    def export_fd(self, which: int):
        """-> (fd, bytes) of the whole [slot][N*N] array of one map (RGBA32F, or RGBA16F); the caller owns the fd."""
        fd, nbytes = C.c_int(-1), C.c_size_t()
        L.check(self._lib.wso_export_fd(self._h, which, C.byref(fd), C.byref(nbytes)), self._h)
        return int(fd.value), int(nbytes.value)

    def import_external_fd(self, which: int, fd: int, nbytes: int, offset: int = 0):
        """Write one map into memory exported by another API (e.g. vkGetMemoryFdKHR); CUDA takes the fd over."""
        L.check(self._lib.wso_import_external_fd(self._h, which, fd, nbytes, offset), self._h)

    def import_semaphore_fd(self, index: int, fd: int, timeline: bool = False):
        L.check(self._lib.wso_import_semaphore_fd(self._h, index, fd, 1 if timeline else 0), self._h)

    def signal_semaphore(self, index: int, value: int = 0):
        L.check(self._lib.wso_signal_semaphore(self._h, index, value), self._h)

    def wait_semaphore(self, index: int, value: int = 0):
        L.check(self._lib.wso_wait_semaphore(self._h, index, value), self._h)

    def set_stream(self, cuda_stream_ptr: Optional[int]):
        L.check(self._lib.wso_set_stream(self._h, C.c_void_p(cuda_stream_ptr or 0)), self._h)

    def set_profiling(self, on: bool):
        L.check(self._lib.wso_set_profiling(self._h, 1 if on else 0), self._h)

    def profile(self):
        """-> dict(ms=[K1,K2,K3] accumulated device ms, launches, tile_frames) since set_profiling(True)."""
        ms = np.zeros(3, np.float64)
        n, f = C.c_uint64(), C.c_uint64()
        L.check(self._lib.wso_get_profile(self._h, _ptr(ms), C.byref(n), C.byref(f)), self._h)
        return {"ms": ms.tolist(), "launches": int(n.value), "tile_frames": int(f.value)}

    def stats(self):
        k, c = C.c_uint64(), C.c_uint32()
        L.check(self._lib.wso_get_stats(self._h, C.byref(k), C.byref(c)), self._h)
        g, r = C.c_uint64(), C.c_uint64()
        L.check(self._lib.wso_get_frame_graph_stats(self._h, C.byref(g), C.byref(r)), self._h)
        return {"kernel_launches": int(k.value), "chunk": int(c.value), "frame_graph_launches": int(g.value),
                "frame_graph_captures": int(r.value)}

    def set_frame_graph(self, on, every_size: bool = False):
        """Single tile-frame calls as one CUDA-graph launch (default: tile sizes up to 512; every_size: all) or as three
        plain kernel launches (on = False)."""
        L.check(self._lib.wso_set_frame_graph(self._h, (2 if every_size else 1) if on else 0), self._h)
