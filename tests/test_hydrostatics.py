"""Hydrostatics (wso_hydrostatics): buoyancy force and torque on triangle hulls floating in the surface of 1..4 slots.

`integrate` below is a NumPy float64 restatement of the contract in include/wsocean.h ("Hydrostatic forces"): each
triangle clipped at depth 0 and the linear pressure integrated in closed form, summed with np.sum.  Two oracles use it:
  - `contract_oracle` takes the depths the contract defines (fp32 arms and world positions in the contract's order,
    heights from the surface-query host build at those positions), so only the float64 integration and the order of
    the sums differ from the library: records agree to one fp32 rounding (within 2 ulp, plus 2^-40 of the largest
    per-triangle term where a component cancels to near zero);
  - `float64_oracle` takes arms, world positions and heights (query_oracle, pos32=False) in float64 throughout; its
    gap to the library is bounded by an fp32 error model (`_gate`).  Worst observed ratio to the gate over the wave
    tests: 0.067 (test_host_body_waves, three cascades, RGBA32F).
The closed forms (Archimedes, a box at several drafts and heels against the wall-sided GZ formula, a single open
triangle) and an independent convex-polytope clip (scipy HalfspaceIntersection) check the integration itself.

CPU: the host build of the kernel body (tests/emu/emu_hydro.cpp, the same wso_hydro.cuh the sm_100a kernel compiles).
GPU (-m gpu): device records equal the host build's bit for bit on the library's own maps; a flat ocean made by the
library gives Archimedes; a one-hot swell pins the body / world convention; calls follow computes in stream order; and
the C ABI validates its arguments and keeps its state.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import test_surface_query as Q
from conftest import ROOT
from emu import driver as E

F32 = np.float32
DRY, PARTIAL, SUBMERGED, INVALID = 0, 1, 2, 3
RHO, G = 1025.0, 9.81
K = np.float64(F32(RHO)) * np.float64(F32(G))
U32 = 2.0 ** -24


# ---------------------------------------------------------------------------------------------------------------------
# host build of the hydrostatics body
# ---------------------------------------------------------------------------------------------------------------------
_SHIM = None


def _shim():
    """tests/emu/emu_hydro.cpp, compiled once per session into a temporary directory (the tree may be read-only)."""
    global _SHIM
    if _SHIM is None:
        out = os.path.join(tempfile.mkdtemp(prefix="wso_emuh_"), "libwsoemuh.so")
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-std=c++17", "-O2", "-w", "-ffp-contract=off", "-fPIC", "-shared", "-I", E.CSRC,
                               "-o", out, os.path.join(E.HERE, "emu_hydro.cpp")])
        L = C.CDLL(out)
        vp, u32 = C.c_void_p, C.c_uint32
        L.wso_emuh_hydro.argtypes = [C.c_int, u32, C.c_int, vp, vp, vp, vp, C.c_int, C.c_double, u32, vp, u32, vp, u32,
                                     vp, vp]
        L.wso_emuh_hydro.restype = C.c_int
        _SHIM = L
    return _SHIM


# struct wso_body, written out here so that the layout test compares two independent statements
BODY = np.dtype([("rotation", "<f4", (9,)), ("position", "<f4", (3,)), ("center", "<f4", (3,)), ("vertex_first", "<u4"),
                 ("vertex_count", "<u4"), ("triangle_first", "<u4"), ("triangle_count", "<u4"), ("unused", "<u4")])


def host_hydro(maps, A, L, bodies, vertices, triangles, I, density=RHO, gravity=G):
    """Host build: maps = [(disp, norm), ...] (float32, or float16 = RGBA16F) -> (n, 8) float32 records
    (force xyz, wetted area, torque xyz, status bits)."""
    half = maps[0][0].dtype == np.float16
    dt = np.float16 if half else F32
    disp = [np.ascontiguousarray(d, dt) for d, _ in maps]
    norm = [np.ascontiguousarray(g, dt) for _, g in maps]
    ns = len(disp)
    pd = (C.c_void_p * ns)(*[d.ctypes.data for d in disp])
    pn = (C.c_void_p * ns)(*[g.ctypes.data for g in norm])
    a = np.ascontiguousarray(A, F32)
    lt = np.ascontiguousarray(L, F32)
    b = np.ascontiguousarray(bodies, BODY)
    v = vec4(vertices)
    t = np.ascontiguousarray(triangles, np.uint32).reshape(-1, 3)
    out = np.zeros((b.shape[0], 8), F32)
    p = lambda x: x.ctypes.data_as(C.c_void_p)
    k = np.float64(F32(density)) * np.float64(F32(gravity))
    rc = _shim().wso_emuh_hydro(1 if half else 0, disp[0].shape[0], ns, C.cast(pd, C.c_void_p), C.cast(pn, C.c_void_p),
                                p(a), p(lt), int(I), float(k), b.shape[0], p(b), v.shape[0], p(v), t.shape[0], p(t),
                                p(out))
    assert rc == 0
    return out


def vec4(v):
    v = np.atleast_2d(np.asarray(v, F32))
    out = np.zeros((v.shape[0], 4), F32)
    out[:, :v.shape[1]] = v[:, :4]
    return out


def status_of(rec):
    return np.ascontiguousarray(rec[:, 7]).view(np.uint32)


def flat_maps(n=16, half=False):
    dt = np.float16 if half else F32
    return [(np.zeros((n, n, 4), dt), np.zeros((n, n, 4), dt))], [F32(1.0)], [F32(64.0)]


# ---------------------------------------------------------------------------------------------------------------------
# hulls and bodies
# ---------------------------------------------------------------------------------------------------------------------
def box(hx, hy, hz):
    """Closed box [-hx, hx] x [-hy, hy] x [-hz, hz]: 8 vertices, 12 triangles wound counter-clockwise from outside."""
    v = np.array([[x, y, z] for x in (-hx, hx) for y in (-hy, hy) for z in (-hz, hz)], np.float64)
    quads = [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4), (1, 5, 7, 3)]
    t = []
    for a, b, c, d in quads:
        t += [(a, b, c), (a, c, d)]
    return v, orient(v, np.array(t, np.uint32))


def icosphere(r, subdiv=3):
    """Icosphere of radius r: 20 * 4^subdiv triangles (1280 at subdiv 3), outward winding."""
    p = (1 + 5 ** 0.5) / 2
    v = [(-1, p, 0), (1, p, 0), (-1, -p, 0), (1, -p, 0), (0, -1, p), (0, 1, p), (0, -1, -p), (0, 1, -p), (p, 0, -1),
         (p, 0, 1), (-p, 0, -1), (-p, 0, 1)]
    f = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6),
         (7, 1, 8), (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10),
         (8, 6, 7), (9, 8, 1)]
    v = [np.array(x, np.float64) / np.linalg.norm(x) for x in v]
    for _ in range(subdiv):
        mid = {}

        def m(a, b):
            key = (min(a, b), max(a, b))
            if key not in mid:
                c = v[a] + v[b]
                v.append(c / np.linalg.norm(c))
                mid[key] = len(v) - 1
            return mid[key]

        nf = []
        for a, b, c in f:
            ab, bc, ca = m(a, b), m(b, c), m(c, a)
            nf += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
        f = nf
    v = np.array(v) * r
    return v, orient(v, np.array(f, np.uint32))


def orient(v, t):
    """Flip triangles whose (b - a) x (c - a) points towards the centroid (convex hulls only)."""
    c = v.mean(0)
    n = np.cross(v[t[:, 1]] - v[t[:, 0]], v[t[:, 2]] - v[t[:, 0]])
    flip = np.einsum("ij,ij->i", n, v[t].mean(1) - c) < 0
    t = t.copy()
    t[flip] = t[flip][:, [0, 2, 1]]
    return t


def volume_centroid(v, t):
    """Volume and centroid of a closed, outward-wound mesh (tetrahedra from the origin), float64."""
    a, b, c = v[t[:, 0]], v[t[:, 1]], v[t[:, 2]]
    dv = np.einsum("ij,ij->i", a, np.cross(b, c)) / 6
    return dv.sum(), (dv[:, None] * (a + b + c) / 4).sum(0) / dv.sum()


def rot(axis, ang):
    axis = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    x, y, z = axis
    c, s = np.cos(ang), np.sin(ang)
    return np.array([[c + x * x * (1 - c), x * y * (1 - c) - z * s, x * z * (1 - c) + y * s],
                     [y * x * (1 - c) + z * s, c + y * y * (1 - c), y * z * (1 - c) - x * s],
                     [z * x * (1 - c) - y * s, z * y * (1 - c) + x * s, c + z * z * (1 - c)]])


def random_rotation(rng):
    q = rng.standard_normal(4)
    q /= np.linalg.norm(q)
    return rot(q[1:], 2 * np.arccos(np.clip(q[0], -1, 1))) if np.linalg.norm(q[1:]) > 0 else np.eye(3)


def body(R=np.eye(3), t=(0, 0, 0), c=(0, 0, 0), vf=0, vc=0, tf=0, tc=0):
    b = np.zeros(1, BODY)
    b["rotation"] = np.asarray(R, F32).reshape(9)
    b["position"] = np.asarray(t, F32)
    b["center"] = np.asarray(c, F32)
    b["vertex_first"], b["vertex_count"], b["triangle_first"], b["triangle_count"] = vf, vc, tf, tc
    return b


def pack(hulls):
    """[(vertices, triangles), ...] -> (vertices, triangles, [(vf, vc, tf, tc), ...]) concatenated."""
    vs, ts, ranges = [], [], []
    nv = nt = 0
    for v, t in hulls:
        vs.append(np.asarray(v, F32))
        ts.append(np.asarray(t, np.uint32))
        ranges.append((nv, len(v), nt, len(t)))
        nv += len(v)
        nt += len(t)
    return np.concatenate(vs), np.concatenate(ts), ranges


# ---------------------------------------------------------------------------------------------------------------------
# the float64 integration and the two oracles
# ---------------------------------------------------------------------------------------------------------------------
def _cross_pt(p, dp, q, dq):
    u = dp / (dp - dq)
    return p + u[:, None] * (q - p)


def _subs(P, D):
    """Wet sub-triangles of triangles P (m, 3, 3) with depths D (m, 3): -> (k, 3, 3) points, (k, 3) depths."""
    wet = D > 0
    nw = wet.sum(1)
    out_p, out_d = [P[nw == 3]], [D[nw == 3]]
    for lone, count in ((True, 1), (False, 2)):
        sel = np.nonzero(nw == count)[0]
        if sel.size == 0:
            continue
        ia = np.argmax(wet[sel] == lone, axis=1)
        order = (ia[:, None] + np.arange(3)[None, :]) % 3
        p = np.take_along_axis(P[sel], order[:, :, None], 1)
        d = np.take_along_axis(D[sel], order, 1)
        a, b, c = p[:, 0], p[:, 1], p[:, 2]
        da, db, dc = d[:, 0], d[:, 1], d[:, 2]
        z = np.zeros_like(da)
        if lone:
            out_p.append(np.stack([a, _cross_pt(a, da, b, db), _cross_pt(a, da, c, dc)], 1))
            out_d.append(np.stack([da, z, z], 1))
        else:
            xba, xca = _cross_pt(b, db, a, da), _cross_pt(c, dc, a, da)
            out_p += [np.stack([xba, b, xca], 1), np.stack([b, c, xca], 1)]
            out_d += [np.stack([z, db, z], 1), np.stack([db, dc, z], 1)]
    return np.concatenate(out_p), np.concatenate(out_d)


def integrate(arms, depths, tris, k=K):
    """float64: -> force (3), torque (3) about the arms' origin, wetted area, the largest per-triangle |term| (F, tau)."""
    P, D = _subs(np.asarray(arms, np.float64)[tris], np.asarray(depths, np.float64)[tris])
    S = 0.5 * np.cross(P[:, 1] - P[:, 0], P[:, 2] - P[:, 0])
    sd = D.sum(1)
    f = -(sd / 3)[:, None] * S
    g = np.einsum("ki,kij->kj", D, P) + sd[:, None] * P.sum(1)
    tau = -np.cross(g, S) / 12
    area = np.sqrt((S * S).sum(1))
    big = (k * np.abs(f).max(initial=0.0), k * np.abs(tau).max(initial=0.0))
    return k * f.sum(0), k * tau.sum(0), area.sum(), big


def _rot32(R, x):
    """R x per row as the contract rounds it: fl(fl(fl(R_i0 x0) + fl(R_i1 x1)) + fl(R_i2 x2))."""
    R = np.asarray(R, F32)
    return np.stack([(R[i, 0] * x[:, 0] + R[i, 1] * x[:, 1]) + R[i, 2] * x[:, 2] for i in range(3)], 1).astype(F32)


def contract_arms(b, v):
    """fp32 arms and world positions of body b's vertices v (n, 3), in the contract's order."""
    R = np.asarray(b["rotation"], F32).reshape(3, 3)
    c = np.asarray(b["center"], F32).reshape(1, 3)
    t = np.asarray(b["position"], F32).reshape(3)
    cw = (t + _rot32(R, c)[0]).astype(F32)
    arm = _rot32(R, (np.asarray(v, F32)[:, :3] - c).astype(F32))
    return arm, (cw + arm).astype(F32)


def contract_oracle(maps, A, L, b, v, t, I):
    """Depths as the contract rounds them (heights: the surface-query host build at the fp32 world positions)."""
    arm, world = contract_arms(b, v)
    disp = [d for d, _ in maps]
    norm = [g for _, g in maps]
    h = Q.host_query(disp, norm, A, L, [F32(0)] * len(maps), world[:, [0, 2]], I)[:, 0]
    depth = (h - world[:, 1]).astype(F32)
    return integrate(arm, depth, t), arm, depth


def float64_oracle(maps, A, L, b, v, t, I):
    """Arms, world positions and heights in float64 (query_oracle with pos32=False)."""
    R = np.asarray(b["rotation"], np.float64).reshape(3, 3)
    c = np.asarray(b["center"], np.float64).reshape(3)
    tw = np.asarray(b["position"], np.float64).reshape(3)
    arm = (np.asarray(v, np.float64)[:, :3] - c) @ R.T
    world = tw + R @ c + arm
    h = Q.query_oracle(maps, A, L, [0.0] * len(maps), world[:, [0, 2]], I, pos32=False)["height"]
    return integrate(arm, h - world[:, 1], t), arm, world


def _ulp(x):
    return np.spacing(np.abs(np.asarray(x, F32))).astype(np.float64)


def assert_contract(rec, ref, what=""):
    """rec (8,) float32 against integrate()'s float64 result: within 2 ulp, plus 2^-40 of the largest term."""
    f, tau, area, (bf, bt) = ref
    for got, want, big in ((rec[0:3], f, bf), (rec[4:7], tau, bt), (rec[3:4], [area], area)):
        err = np.abs(np.asarray(got, np.float64) - want)
        lim = 2 * _ulp(want) + 2.0 ** -40 * big
        assert np.all(err <= lim), f"{what}: {got} vs {want} (err {err}, limit {lim})"


# ---------------------------------------------------------------------------------------------------------------------
# CPU: closed forms on flat water
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("half", [False, True], ids=["rgba32f", "rgba16f"])
def test_box_drafts_flat(half):
    """Upright box (4 x 2 x 6 m) at drafts 0.25 .. 2: F = (0, rho g V_sub, 0), tau = (c_B - c_w) x F."""
    maps, A, L = flat_maps(half=half)
    v, t = box(2.0, 1.0, 3.0)
    c = np.array([0.25, -0.5, 0.75])
    for draft in (0.25, 0.5, 1.0, 1.75):
        pos = np.array([3.5, 1.0 - draft, -1.25])
        b = body(t=pos, c=c, vc=8, tc=12)
        r = host_hydro(maps, A, L, b, v, t, 4)[0]
        V = 4.0 * 6.0 * draft
        F = np.array([0, K * V, 0])
        cB = pos + np.array([0, -1.0 + draft / 2, 0])
        cw = pos + c
        tau = np.cross(cB - cw, F)
        assert status_of(r[None])[0] == PARTIAL
        assert abs(r[1] - F[1]) <= 4 * _ulp(F[1]) and r[0] == 0 and r[2] == 0
        assert np.allclose(r[4:7], tau, rtol=4e-7, atol=4e-7 * F[1])
        assert np.isclose(r[3], 4 * 6 + 2 * (4 + 6) * draft, rtol=4e-7)        # bottom + wet sides


@pytest.mark.parametrize("hull", ["box", "icosphere"])
def test_archimedes_submerged(hull):
    v, t = box(1.5, 0.75, 2.25) if hull == "box" else icosphere(2.0)
    V, cen = volume_centroid(v.astype(F32).astype(np.float64), t)
    maps, A, L = flat_maps()
    rng = np.random.default_rng(1)
    for _ in range(6):
        R = random_rotation(rng)
        b = body(R=R, t=(rng.uniform(-100, 100), -rng.uniform(5, 40), rng.uniform(-100, 100)), c=cen, vc=len(v),
                 tc=len(t))
        r = host_hydro(maps, A, L, b, v, t, 0)[0]
        assert status_of(r[None])[0] == SUBMERGED
        assert np.isclose(r[1], K * V, rtol=2e-6)
        assert np.abs(r[[0, 2]]).max() <= 2e-6 * K * V
        # about the centroid the pressure has no moment (fp32 arms: a few ulp of F times the hull size)
        assert np.abs(r[4:7]).max() <= 1e-5 * K * V * 2.0


def test_dry_body():
    maps, A, L = flat_maps()
    v, t = icosphere(1.0, 1)
    b = body(R=random_rotation(np.random.default_rng(2)), t=(5, 1.5, 5), vc=len(v), tc=len(t))
    r = host_hydro(maps, A, L, b, v, t, 4)[0]
    assert status_of(r[None])[0] == DRY
    assert np.all(r[:7] == 0) and not np.any(np.signbit(r[:7]))


def test_single_open_triangle():
    """One wet triangle: F = -rho g * mean depth * S, tau = -(rho g / 12) (g x S) about c."""
    maps, A, L = flat_maps()
    v = np.array([[0.0, -1.0, 0.0], [2.0, -3.0, 0.5], [0.5, -2.0, 1.5]])
    for tri in ([0, 1, 2], [0, 2, 1]):
        b = body(c=(0.25, -1.5, 0.5), vc=3, tc=1)
        r = host_hydro(maps, A, L, b, v, np.array([tri]), 0)[0]
        p = v[tri]
        S = 0.5 * np.cross(p[1] - p[0], p[2] - p[0])
        F = -K * (-p[:, 1]).mean() * S
        assert status_of(r[None])[0] == SUBMERGED
        assert np.allclose(r[0:3], F, rtol=1e-6, atol=1e-6 * np.abs(F).max())
        assert np.isclose(r[3], np.linalg.norm(S), rtol=1e-6)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: heeled and arbitrary poses on flat water
# ---------------------------------------------------------------------------------------------------------------------
def _clip_below(vw):
    """Volume and centroid of conv(vw) cut at y <= 0 (scipy halfspaces, independent of the library's clipping)."""
    from scipy.spatial import ConvexHull, HalfspaceIntersection
    hull = ConvexHull(vw)
    from scipy.optimize import linprog
    hs = np.vstack([hull.equations, [[0, 1, 0, 0]]])
    # an interior point: the centre of the largest ball inside (A x + b <= 0)
    norm = np.linalg.norm(hs[:, :3], axis=1)
    lp = linprog([0, 0, 0, -1], A_ub=np.hstack([hs[:, :3], norm[:, None]]), b_ub=-hs[:, 3],
                 bounds=[(None, None)] * 3 + [(0, None)])
    sub = ConvexHull(HalfspaceIntersection(hs, lp.x[:3]).intersections)
    pts = sub.points
    o = pts.mean(0)
    vol, mom = 0.0, np.zeros(3)
    for s in sub.simplices:
        a, b, c = pts[s]
        dv = abs(np.dot(a - o, np.cross(b - o, c - o))) / 6
        vol += dv
        mom += dv * (a + b + c + o) / 4
    return vol, mom / vol


@pytest.mark.parametrize("hull", ["box", "icosphere"])
def test_heeled_against_polytope_clip(hull):
    v, t = box(2.0, 1.0, 3.0) if hull == "box" else icosphere(2.0, 2)
    maps, A, L = flat_maps()
    rng = np.random.default_rng(5 if hull == "box" else 6)
    for _ in range(8):
        R = random_rotation(rng)
        c = rng.uniform(-0.5, 0.5, 3)
        pos = np.array([rng.uniform(-50, 50), rng.uniform(-0.8, 0.8), rng.uniform(-50, 50)])
        b = body(R=R, t=pos, c=c, vc=len(v), tc=len(t))
        r = host_hydro(maps, A, L, b, v, t, 4)[0].astype(np.float64)
        arm, world = contract_arms(b[0], v)
        vol, cB = _clip_below(world.astype(np.float64))
        assert status_of(r[None].astype(F32))[0] == PARTIAL
        assert np.isclose(r[1], K * vol, rtol=2e-5)
        assert np.abs(r[[0, 2]]).max() <= 2e-5 * K * vol
        cw = (np.asarray(b["position"], np.float64) + R.astype(F32) @ np.asarray(b["center"][0], np.float64))[0]
        tau = np.cross(cB - cw, [0, K * vol, 0])
        assert np.allclose(r[4:7], tau, atol=4e-5 * K * vol * 3.0)


@pytest.mark.parametrize("theta_deg", [3.0, 8.0, 15.0, -11.0])
def test_wall_sided_righting_arm(theta_deg):
    """Box L x B x D = 10 x 4 x 3 at draft T = 1.2, G at KG = 1.6, heeled by theta about its long (x) axis around the
    waterline centre: GZ = sin(theta) (GM + BM tan^2(theta) / 2) while deck and bilge stay on their sides."""
    Lb, B, D, T, KG = 10.0, 4.0, 3.0, 1.2, 1.6
    th = np.radians(theta_deg)
    assert T + B / 2 * abs(np.tan(th)) < D and T - B / 2 * abs(np.tan(th)) > 0
    v, t = box(Lb / 2, D / 2, B / 2)
    v = v + [0, D / 2, 0]                               # keel at y = 0
    R = rot([1, 0, 0], th)
    W = np.array([0.0, T, 0.0])
    maps, A, L = flat_maps()
    b = body(R=R, t=-R @ W, c=(0, KG, 0), vc=8, tc=12)
    r = host_hydro(maps, A, L, b, v, t, 0)[0].astype(np.float64)
    V = Lb * B * T
    BM, KB = B * B / (12 * T), T / 2
    GZ = np.sin(th) * (KB + BM - KG + 0.5 * BM * np.tan(th) ** 2)
    assert np.isclose(r[1], K * V, rtol=1e-5)
    # righting moment: restoring, about the heel axis (x)
    assert np.isclose(r[4], -K * V * GZ, rtol=1e-4, atol=1e-5 * K * V)
    assert abs(r[5]) <= 1e-5 * K * V and abs(r[6]) <= 1e-5 * K * V


# ---------------------------------------------------------------------------------------------------------------------
# CPU: invariances
# ---------------------------------------------------------------------------------------------------------------------
def test_reversed_winding_negates():
    v, t = icosphere(1.5, 2)
    maps, A, L = flat_maps()
    rng = np.random.default_rng(9)
    for _ in range(6):
        b = body(R=random_rotation(rng), t=(rng.uniform(-9, 9), rng.uniform(-1, 1), rng.uniform(-9, 9)),
                 c=rng.uniform(-0.3, 0.3, 3), vc=len(v), tc=len(t))
        fwd = host_hydro(maps, A, L, b, v, t, 0)[0].astype(np.float64)
        rev = host_hydro(maps, A, L, b, v, t[:, ::-1], 0)[0].astype(np.float64)
        scale = np.abs(fwd[:3]).max() * 2.0
        assert np.allclose(rev[[0, 1, 2, 4, 5, 6]], -fwd[[0, 1, 2, 4, 5, 6]], rtol=1e-6, atol=1e-6 * scale)
        assert rev[3] == pytest.approx(fwd[3], rel=1e-6)


def _subdivide(v, t):
    v = list(map(tuple, v))
    idx = {p: i for i, p in enumerate(v)}

    def mid(a, b):
        p = tuple((np.asarray(v[a]) + np.asarray(v[b])) / 2)
        if p not in idx:
            idx[p] = len(v)
            v.append(p)
        return idx[p]

    nt = []
    for a, b, c in t:
        ab, bc, ca = mid(a, b), mid(b, c), mid(c, a)
        nt += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
    return np.array(v), np.array(nt, np.uint32)


def test_subdivision_keeps_force():
    v, t = box(2.0, 1.0, 3.0)
    v2, t2 = _subdivide(*_subdivide(v, t))
    maps, A, L = flat_maps()
    for R in (np.eye(3), rot([0, 1, 0], np.pi / 2)):
        for y in (0.75, 0.0, -0.375):
            R = np.round(R)
            b1 = body(R=R, t=(1.5, y, -2.5), vc=len(v), tc=len(t))
            b2 = body(R=R, t=(1.5, y, -2.5), vc=len(v2), tc=len(t2))
            r1 = host_hydro(maps, A, L, b1, v, t, 0)[0]
            r2 = host_hydro(maps, A, L, b2, v2, t2, 0)[0]
            assert np.all(np.abs(r1[:3].astype(np.float64) - r2[:3]) <= 2 * _ulp(np.abs(r1[:3]).max()))
            assert r1[3] == pytest.approx(r2[3], rel=1e-6)


def test_rotation_about_y_rotates_torque():
    v, t = icosphere(1.5, 2)
    maps, A, L = flat_maps()
    rng = np.random.default_rng(11)
    for _ in range(6):
        R0 = random_rotation(rng)
        pos = np.array([rng.uniform(-9, 9), rng.uniform(-1, 1), rng.uniform(-9, 9)])
        c = rng.uniform(-0.5, 0.5, 3)
        Ry = rot([0, 1, 0], rng.uniform(0, 2 * np.pi))
        r0 = host_hydro(maps, A, L, body(R=R0, t=pos, c=c, vc=len(v), tc=len(t)), v, t, 0)[0].astype(np.float64)
        r1 = host_hydro(maps, A, L, body(R=Ry @ R0, t=Ry @ pos, c=c, vc=len(v), tc=len(t)), v, t, 0)[0].astype(
            np.float64)
        scale = abs(r0[1])
        assert np.allclose(r1[:3], Ry @ r0[:3], atol=2e-5 * scale)
        assert np.allclose(r1[4:7], Ry @ r0[4:7], atol=2e-5 * scale * 1.5)
        assert r1[3] == pytest.approx(r0[3], rel=2e-5)


@pytest.mark.parametrize("half", [False, True], ids=["rgba32f", "rgba16f"])
def test_tile_shift_invariance(half):
    rng = np.random.default_rng(13)
    n, Lt = 64, F32(64.0)
    maps, A, _ = Q._random_cascades(rng, n, [Lt], half)
    v, t = box(2.0, 1.0, 3.0)
    perm = np.array([[0, 0, 1], [0, 1, 0], [-1, 0, 0]])   # exact rotation about y
    for R in (np.eye(3), perm):
        base = np.array([12.5, 0.25, -7.75])
        recs = []
        for kx, kz in ((0, 0), (1, 0), (-3, 2), (16, -16)):
            b = body(R=R, t=base + [kx * 64.0, 0, kz * 64.0], c=(0.5, 0.25, -0.75), vc=8, tc=12)
            recs.append(host_hydro(maps, A, [Lt], b, v, t, 4)[0])
        for r in recs[1:]:
            assert np.array_equal(r.view(np.uint32), recs[0].view(np.uint32))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: waves
# ---------------------------------------------------------------------------------------------------------------------
def _gate(maps, A, L, b, v, t, arm, world):
    """fp32 error model of the record against float64_oracle, u = 2^-24.  Per vertex: the world position is off by about
    2u |world| (two roundings), which moves the sampled height by s * that (s = sum over cascades of |A_s| times the
    steepest texel-to-texel step of D.y over the texel spacing); the height sum and the depth add 2u (sum |A_s| + |y|);
    the arm is off by e_y = 2u |arm|.  The pressure integral changes by k (e_d + d_max * 2 e_y / shortest edge) sum |S|,
    the torque by that times the largest arm plus k d_max sum |S| e_y."""
    s = 0.0
    for (d, _), a, l in zip(maps, A, L):
        dy = np.asarray(d[..., 1], np.float64)
        n = dy.shape[0]
        st = max(np.abs(np.diff(dy, axis=ax, append=dy.take([0], axis=ax))).max() for ax in (0, 1))
        s += abs(float(a)) * st / (float(l) / n)
    amp = sum(abs(float(a)) for a in A)
    e_d = 2 * U32 * s * np.abs(world[:, [0, 2]]).max() + 2 * U32 * (amp + np.abs(world[:, 1]).max())
    rmax = np.linalg.norm(arm, axis=1).max()
    e_y = 2 * U32 * rmax
    p = np.asarray(v, np.float64)[t]
    edge = min(np.linalg.norm(p[:, 1] - p[:, 0], axis=1).min(), np.linalg.norm(p[:, 2] - p[:, 0], axis=1).min())
    S = 0.5 * np.linalg.norm(np.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0]), axis=1).sum()
    dmax = amp + np.abs(world[:, 1]).max()
    gF = K * (e_d + dmax * 2 * e_y / edge) * S
    return gF, gF * rmax + K * dmax * S * e_y


@pytest.mark.parametrize("half", [False, True], ids=["rgba32f", "rgba16f"])
@pytest.mark.parametrize("ns", [1, 2, 3, 4])
def test_host_body_waves(ns, half):
    rng = np.random.default_rng(40 + 2 * ns + half)
    n = 64
    lengths = [F32(l) for l in (200.0, 61.0, 17.3, 5.1)[:ns]]
    maps, A, _ = Q._random_cascades(rng, n, lengths, half)
    hulls = [box(2.0, 1.0, 3.0), icosphere(1.5, 2), box(8.0, 1.5, 1.25)]
    vs, ts, ranges = pack(hulls)
    amp = sum(float(a) for a in A)
    worst = 0.0
    for I in (0, 4):
        bl = []
        for k in range(24):
            vf, vc, tf, tc = ranges[k % 3]
            y = rng.uniform(-amp - 1.5, amp + 1.5)
            bl.append(body(R=random_rotation(rng), t=(rng.uniform(-400, 400), y, rng.uniform(-400, 400)),
                           c=rng.uniform(-0.5, 0.5, 3), vf=vf, vc=vc, tf=tf, tc=tc))
        bodies = np.concatenate(bl)
        rec = host_hydro(maps, A, lengths, bodies, vs, ts, I)
        st = status_of(rec)
        assert np.sum(st == PARTIAL) >= 8, st
        for i, b in enumerate(bodies):
            vf, vc, tf, tc = (int(b[f]) for f in ("vertex_first", "vertex_count", "triangle_first", "triangle_count"))
            v, t = vs[vf:vf + vc], ts[tf:tf + tc]
            ref, arm, depth = contract_oracle(maps, A, lengths, b, v, t, I)
            what = f"ns={ns} I={I} body {i}"
            assert_contract(rec[i], ref, what)
            wet = depth > 0
            assert st[i] == (DRY if not wet.any() else SUBMERGED if wet.all() else PARTIAL), what
            (f64, t64, a64, _), arm64, world64 = float64_oracle(maps, A, lengths, b, v, t, I)
            gF, gT = _gate(maps, A, lengths, b, v, t, arm64, world64)
            eF = np.abs(rec[i, 0:3] - f64).max()
            eT = np.abs(rec[i, 4:7] - t64).max()
            assert eF <= gF and eT <= gT, f"{what}: {eF:.3e} / {gF:.3e}, {eT:.3e} / {gT:.3e}"
            worst = max(worst, eF / gF, eT / gT)
    print(f"worst ratio to the gate: {worst:.3f}")


# ---------------------------------------------------------------------------------------------------------------------
# CPU: validation, layouts, adaptor
# ---------------------------------------------------------------------------------------------------------------------
def test_invalid_bodies_leave_neighbours_alone():
    maps, A, L = flat_maps()
    vb, tb = box(1.0, 1.0, 1.0)
    vs, ts, ranges = pack([(vb, tb), (vb, np.array([[0, 1, 8]])), icosphere(1.0, 1)])
    good = [body(t=(0, 0.25, 0), c=(0.5, 0, 0), vc=8, tc=12), body(R=rot([1, 1, 0], 0.3), t=(4, -0.5, 2), vf=9,
                                                                      vc=42, tf=13, tc=80)]
    nan = np.float32(np.nan)
    bad = [body(vf=8, vc=1, tf=12, tc=1),                        # index 8 >= vertex_count (range of 1)
           body(vc=0, tc=0),                                     # no vertex
           body(vc=4097, tc=12),                                 # too many vertices
           body(vc=8, tc=65537),                                 # too many triangles
           body(vf=50, vc=12, tc=12),                            # vertex range past the array
           body(vc=8, tf=90, tc=12),                             # triangle range past the array
           body(R=np.full((3, 3), nan), vc=8, tc=12),
           body(t=(0, np.inf, 0), vc=8, tc=12),
           body(c=(nan, 0, 0), vc=8, tc=12)]
    ref = host_hydro(maps, A, L, np.concatenate(good), vs, ts, 0)
    assert np.all(status_of(ref) == PARTIAL)
    mixed = np.concatenate([good[0]] + bad + [good[1]])
    rec = host_hydro(maps, A, L, mixed, vs, ts, 0)
    assert np.array_equal(rec[[0, -1]].view(np.uint32), ref.view(np.uint32))
    mid = rec[1:-1]
    assert np.all(status_of(mid) == INVALID)
    assert np.all(np.isnan(mid[:, :7]))
    # a non-finite vertex
    vs2 = vs.copy()
    vs2[3, 1] = np.inf
    rec = host_hydro(maps, A, L, np.concatenate([good[0], good[1]]), vs2, ts, 0)
    assert status_of(rec)[0] == INVALID and np.array_equal(rec[1].view(np.uint32), ref[1].view(np.uint32))


def test_dtypes_match_the_c_structs():
    import watersurfacerendering_b200 as W
    from watersurfacerendering_b200 import _lib as L
    assert W.BODY_DTYPE == BODY and W.BODY_DTYPE.itemsize == 80
    assert W.HYDRO_RESULT_DTYPE.itemsize == 32
    assert W.HYDRO_RESULT_DTYPE.names == ("force", "wetted_area", "torque", "status")
    assert (L.WSO_HYDRO_DRY, L.WSO_HYDRO_PARTIAL, L.WSO_HYDRO_SUBMERGED, L.WSO_HYDRO_INVALID) == \
        (DRY, PARTIAL, SUBMERGED, INVALID)
    assert C.sizeof(L.WsoHydroParams) == 16
    src = r'''
#include <stddef.h>
#include "wsocean.h"
_Static_assert(sizeof(wso_body) == 80, "");
_Static_assert(offsetof(wso_body, position) == 36 && offsetof(wso_body, center) == 48, "");
_Static_assert(offsetof(wso_body, vertex_first) == 60 && offsetof(wso_body, triangle_count) == 72, "");
_Static_assert(sizeof(wso_hydro_result) == 32 && offsetof(wso_hydro_result, torque) == 16, "");
_Static_assert(offsetof(wso_hydro_result, status) == 28 && sizeof(wso_hydro_params) == 16, "");
'''
    assert [BODY.fields[f][1] for f in ("position", "center", "vertex_first", "triangle_count")] == [36, 48, 60, 72]
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "s.c")
        with open(p, "w") as f:
            f.write(src)
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        subprocess.check_call([cc, "-std=c11", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), p])


def test_adaptor_hydrostatics_compiles(tmp_path):
    src = tmp_path / "h.cpp"
    src.write_text(r'''
#include <vector>
#include "wso_tessendorf_adaptor.hpp"
float use(WSTessendorf& m) {
    std::vector<float> v = {-1, -1, -1, 0, 1, -1, -1, 0, 0, 1, -1, 0, 0, -1, 1, 0};
    std::vector<uint32_t> t = {0, 2, 1, 0, 1, 3, 0, 3, 2, 1, 2, 3};
    wso_body b = {{1, 0, 0, 0, 1, 0, 0, 0, 1}, {0, 0, 0}, {0, 0, 0}, 0, 4, 0, 4, 0};
    wso_hydro_result out;
    wso_hydro_params p = {1025.0f, 9.81f, 4u, 0u};
    m.Hydrostatics(&b, 1, v.data(), 4, t.data(), 4, &out, p);
    return out.force[1] + out.torque[0] + out.wetted_area + (out.status == WSO_HYDRO_PARTIAL ? 1.0f : 0.0f);
}
''')
    gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([gxx, "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)])


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
CASCADE_L = (1000.0, 250.0, 61.0, 17.3)


def _ocean(W, n, ncasc, fmt, seed=3):
    ws = W.WSTessendorf(n, CASCADE_L[0], max_tiles=ncasc, max_slots=ncasc)
    ws.set_map_format(fmt)
    for t in range(ncasc):
        ws.SetTileLength(CASCADE_L[t], t)
        ws.Prepare(seed=seed + t, tile=t)
    ws.compute_batch(np.full(ncasc, 7.25, F32), tiles=np.arange(ncasc, dtype=np.uint32))
    return ws


def _rows(rec):
    return np.ascontiguousarray(rec).view(F32).reshape(-1, 8)


def gpu_scene(rng, amp, count):
    """Mixed hulls (box, icosphere, long barge), instanced ranges, invalid bodies mixed in."""
    hulls = [box(2.0, 1.0, 3.0), icosphere(2.0, 3), box(40.0, 2.0, 6.0), (box(1, 1, 1)[0], np.array([[0, 1, 9]]))]
    vs, ts, ranges = pack(hulls)
    bl = []
    for k in range(count):
        j = k % 7
        if j == 6:
            bl.append(body(vf=ranges[3][0], vc=8, tf=ranges[3][2], tc=1) if k % 2 else body(vc=0))
            continue
        vf, vc, tf, tc = ranges[j % 3]
        bl.append(body(R=random_rotation(rng), t=(rng.uniform(-3000, 3000), rng.uniform(-amp - 2, amp + 2),
                                                  rng.uniform(-3000, 3000)), c=rng.uniform(-0.5, 0.5, 3),
                       vf=vf, vc=vc, tf=tf, tc=tc))
    return np.concatenate(bl), vs, ts


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["rgba32f", "rgba16f"])
def test_device_equals_host_build(fmt):
    import watersurfacerendering_b200 as W
    rng = np.random.default_rng(17)
    n = 512
    for ncasc in (1, 2, 3, 4):
        ws = _ocean(W, n, ncasc, fmt)
        try:
            slots = tuple(range(ncasc))
            maps, A = Q._maps_of(ws, ncasc)
            lengths = [F32(l) for l in CASCADE_L[:ncasc]]
            bodies, vs, ts = gpu_scene(rng, sum(float(a) for a in A), 2100)
            for I in (0, 4):
                dev = _rows(ws.hydrostatics(bodies, vs, ts, slots=slots, iterations=I))
                host = host_hydro(maps, A, lengths, bodies, vs, ts, I)
                what = f"{fmt} cascades={ncasc} I={I}"
                assert np.array_equal(dev.view(np.uint32), host.view(np.uint32)), what + ": device and host build differ"
                st = status_of(dev)
                assert np.sum(st == PARTIAL) >= 200 and np.sum(st == INVALID) == 300, what
        finally:
            ws.close()


@pytest.mark.gpu
def test_flat_ocean_archimedes():
    """An all-zero spectrum gives all-zero maps; then a submerged hull feels rho g V and a floating box its draft."""
    import watersurfacerendering_b200 as W
    n, L = 256, 500.0
    with W.WSTessendorf(n, L) as ws:
        ws.ImportH0(np.zeros((n, n, 5), F32))
        ws.compute_batch([3.0])
        d, g = ws.copy_map(0, 0), ws.copy_map(1, 0)
        assert not np.any(d[..., :3]) and not np.any(g[..., :2])
        v, t = icosphere(2.0, 3)
        V, cen = volume_centroid(v.astype(F32).astype(np.float64), t)
        vb, tb = box(2.0, 1.0, 3.0)
        vs, ts, ranges = pack([(v, t), (vb, tb)])
        rng = np.random.default_rng(3)
        bl = [body(R=random_rotation(rng), t=(rng.uniform(-900, 900), -rng.uniform(3, 30), rng.uniform(-900, 900)),
                   c=cen, vc=len(v), tc=len(t)) for _ in range(64)]
        bl.append(body(t=(10.5, 0.5, -3.25), vf=ranges[1][0], vc=8, tf=ranges[1][2], tc=12))
        r = _rows(ws.hydrostatics(np.concatenate(bl), vs, ts, iterations=4))
        assert np.all(status_of(r[:64]) == SUBMERGED)
        assert np.allclose(r[:64, 1], K * V, rtol=2e-6)
        assert np.abs(r[:64, 4:7]).max() <= 1e-5 * K * V * 2.0
        assert abs(r[64, 1] - K * 4 * 6 * 0.5) <= 4 * _ulp(K * 12)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["rgba32f", "rgba16f"])
def test_convention_pin_one_hot(fmt):
    """One-hot spectrum: h = H cos(kx x + kz z) with kx = 2 pi 5 / L, kz = 2 pi 3 / L (test_surface_query's convention
    pin), lambda = 0.  A 60 m barge across a wavelength at several headings: force and torque equal the float64
    integral of the closed-form heights within the bilinear bound."""
    import watersurfacerendering_b200 as W
    n, L = 256, 400.0
    m0, n0 = n // 2 + 3, n // 2 + 5
    h0 = np.zeros((n, n, 5), F32)
    re, im = 0.75, -0.4
    h0[m0, n0] = (re, im, re, -im, 0.0)
    kx, kz = 2 * np.pi * 5 / L, 2 * np.pi * 3 / L
    H = 2 * re
    delta = L / n
    bound = ((kx * delta) ** 2 + (kz * delta) ** 2) / 8 * H + (2e-3 * H if fmt == "rgba16f" else 2e-5 * H)
    v, t = _subdivide(*_subdivide(*box(30.0, 2.0, 4.0)))
    with W.WSTessendorf(n, L) as ws:
        ws.set_map_format(fmt)
        ws.SetLambda(0.0)
        ws.ImportH0(h0)
        ws.compute_batch([0.0])
        rng = np.random.default_rng(8)
        bl = [body(R=rot([0, 1, 0], rng.uniform(0, 2 * np.pi)) @ rot([1, 0, 0], rng.uniform(-0.1, 0.1)),
                   t=(rng.uniform(-L, 2 * L), rng.uniform(-0.5, 0.5), rng.uniform(-L, 2 * L)), c=(0.5, -0.5, 0.25),
                   vc=len(v), tc=len(t)) for _ in range(32)]
        bodies = np.concatenate(bl)
        r = _rows(ws.hydrostatics(bodies, v, t, iterations=0))
        for i, b in enumerate(bodies):
            arm, world = contract_arms(b, v)
            arm, world = arm.astype(np.float64), world.astype(np.float64)
            h = H * np.cos(kx * world[:, 0] + kz * world[:, 2])
            f, tau, area, _ = integrate(arm, h - world[:, 1], t)
            wet_area = area + 2 * 60.0 * 4.0
            assert np.abs(r[i, 0:3] - f).max() <= K * bound * wet_area * 2, i
            assert np.abs(r[i, 4:7] - tau).max() <= K * bound * wet_area * 2 * 31.0, i
            assert np.abs(f[1]) > 0.1 * K * 60 * 8 * 0.5


def _torch():
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available()
    return torch


@pytest.mark.gpu
def test_stream_order_without_host_sync():
    torch = _torch()
    import watersurfacerendering_b200 as W
    n, t1, t2 = 512, 3.5, 41.0
    rng = np.random.default_rng(2)
    bodies, vs, ts = gpu_scene(rng, 3.0, 1024)
    v4 = vec4(vs)
    tb = torch.from_numpy(bodies.view(np.uint8).copy()).cuda()
    tv = torch.from_numpy(v4).cuda()
    tt = torch.from_numpy(ts.astype(np.int32)).cuda()
    kw = dict(slots=(0, 1), iterations=4)
    with W.WSTessendorf(n, 1000.0, max_tiles=2, max_slots=2) as ws:
        ws.SetTileLength(61.0, 1)
        ws.Prepare(seed=17)
        ws.Prepare(seed=18, tile=1)
        stream = torch.cuda.Stream()
        ws.set_stream(stream.cuda_stream)
        tiles = np.array([0, 1], np.uint32)
        refs = []
        for tm in (t1, t2):
            ws.compute_batch([tm, tm], tiles=tiles)
            ws.sync()
            refs.append(_rows(ws.hydrostatics(bodies, vs, ts, **kw)))
        torch.cuda.synchronize()
        o1 = torch.empty((len(bodies), 8), dtype=torch.float32, device="cuda")
        o2 = torch.empty_like(o1)
        args = (tb.data_ptr(), len(bodies), tv.data_ptr(), len(v4), tt.data_ptr(), len(ts))
        k0 = ws.stats()["kernel_launches"]
        ws.compute_batch([t1, t1], tiles=tiles)
        k1 = ws.stats()["kernel_launches"]
        ws.hydrostatics_device(*args, o1.data_ptr(), **kw)
        assert ws.stats()["kernel_launches"] == k1 + 1
        ws.compute_batch([t2, t2], tiles=tiles)
        ws.hydrostatics_device(*args, o2.data_ptr(), **kw)
        assert ws.stats()["kernel_launches"] == 2 * (k1 - k0) + k0 + 2
        ws.sync()
        assert np.array_equal(o1.cpu().numpy().view(np.uint32), refs[0].view(np.uint32))
        assert np.array_equal(o2.cpu().numpy().view(np.uint32), refs[1].view(np.uint32))
        assert not np.array_equal(refs[0], refs[1])
        ws.set_stream(None)


@pytest.mark.gpu
def test_errors_state_and_launch_count():
    torch = _torch()
    import watersurfacerendering_b200 as W
    from watersurfacerendering_b200 import _lib as L
    lib = L.load()
    v, t = box(1.0, 30.0, 2.0)     # crosses the waterline whatever the waves
    b = body(t=(0, 0, 0), vc=8, tc=12)
    with W.WSTessendorf(256, 500.0, max_slots=3) as ws:
        ws.Prepare(seed=1)

        def expect_invalid(fn, *a, **k):
            k0 = ws.stats()["kernel_launches"]
            with pytest.raises(L.WsoError) as e:
                fn(*a, **k)
            assert e.value.status == L.WSO_ERR_INVALID_ARG
            assert lib.wso_last_error(ws._h)
            assert ws.stats()["kernel_launches"] == k0

        expect_invalid(ws.hydrostatics, b, v, t)                       # slot 0 holds no frame yet
        ws.compute_batch([1.0])
        good = _rows(ws.hydrostatics(b, v, t))
        assert status_of(good)[0] == PARTIAL
        expect_invalid(ws.hydrostatics, b, v, t, slots=(1,))
        expect_invalid(ws.hydrostatics, b, v, t, slots=(3,))
        expect_invalid(ws.hydrostatics, b, v, t, slots=())
        for bad in (dict(density=-1.0), dict(density=np.inf), dict(density=np.nan), dict(gravity=-9.81),
                    dict(gravity=np.inf), dict(iterations=17)):
            expect_invalid(ws.hydrostatics, b, v, t, **bad)
        sl = np.zeros(1, np.uint32)
        slp = sl.ctypes.data_as(C.c_void_p)
        bd = torch.from_numpy(b.view(np.uint8).copy()).cuda()
        vd = torch.from_numpy(vec4(v)).cuda()
        td = torch.from_numpy(t.astype(np.int32)).cuda()
        out = torch.zeros((8 + 4,), dtype=torch.float32, device="cuda")
        bp, vp, tp, op = (C.c_void_p(x.data_ptr()) for x in (bd, vd, td, out))
        pr = L.WsoHydroParams(1025.0, 9.81, 4, 0)
        k0 = ws.stats()["kernel_launches"]
        assert lib.wso_hydrostatics(ws._h, 1, slp, C.byref(pr), 1, bp, 8, vp, 12, tp, op) == L.WSO_OK
        ws.sync()
        assert np.array_equal(out[:8].cpu().numpy().view(np.uint32), good.reshape(-1).view(np.uint32))
        prr = L.WsoHydroParams(1025.0, 9.81, 4, 1)
        for args in ((ws._h, 1, slp, None, 1, bp, 8, vp, 12, tp, op),
                     (ws._h, 1, slp, C.byref(prr), 1, bp, 8, vp, 12, tp, op),            # reserved != 0
                     (ws._h, 1, None, C.byref(pr), 1, bp, 8, vp, 12, tp, op),
                     (ws._h, 1, slp, C.byref(pr), 1, None, 8, vp, 12, tp, op),
                     (ws._h, 1, slp, C.byref(pr), 1, bp, 8, None, 12, tp, op),
                     (ws._h, 1, slp, C.byref(pr), 1, bp, 8, vp, 12, None, op),
                     (ws._h, 1, slp, C.byref(pr), 1, bp, 8, vp, 12, tp, None),
                     (ws._h, 1, slp, C.byref(pr), 1, C.c_void_p(bd.data_ptr() + 8), 8, vp, 12, tp, op),
                     (ws._h, 1, slp, C.byref(pr), 1, bp, 8, C.c_void_p(vd.data_ptr() + 4), 12, tp, op),
                     (ws._h, 1, slp, C.byref(pr), 1, bp, 8, vp, 12, C.c_void_p(td.data_ptr() + 2), op),
                     (ws._h, 1, slp, C.byref(pr), 1, bp, 8, vp, 12, tp, C.c_void_p(out.data_ptr() + 4)),
                     (ws._h, 1, slp, C.byref(pr), 2 ** 31, bp, 8, vp, 12, tp, op)):
            assert lib.wso_hydrostatics(*args) == L.WSO_ERR_INVALID_ARG
        assert lib.wso_hydrostatics(None, 1, slp, C.byref(pr), 1, bp, 8, vp, 12, tp, op) == L.WSO_ERR_INVALID_ARG
        assert lib.wso_hydrostatics_host(ws._h, 1, slp, C.byref(pr), 1, None, 8, None, 12, None, None) == \
            L.WSO_ERR_INVALID_ARG
        # n_bodies == 0 launches nothing (and still checks its arguments)
        assert lib.wso_hydrostatics(ws._h, 1, slp, C.byref(pr), 0, None, 0, None, 0, None, None) == L.WSO_OK
        assert lib.wso_hydrostatics(ws._h, 1, slp, None, 0, None, 0, None, 0, None, None) == L.WSO_ERR_INVALID_ARG
        assert ws.stats()["kernel_launches"] == k0 + 1
        # the state is unchanged: the same call gives the same record
        assert np.array_equal(_rows(ws.hydrostatics(b, v, t)).view(np.uint32), good.view(np.uint32))
        # bad bodies are records, not errors
        r = _rows(ws.hydrostatics(np.concatenate([b, body(vc=0), b]), v, t))
        assert list(status_of(r)) == [PARTIAL, INVALID, PARTIAL] and np.all(np.isnan(r[1, :7]))
        ws.set_map_format("rgba16f")
        expect_invalid(ws.hydrostatics, b, v, t)
        ws.compute_batch([1.0])
        assert status_of(_rows(ws.hydrostatics(b, v, t)))[0] == PARTIAL
