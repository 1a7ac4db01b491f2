import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


class GoldenCase(dict):
    """The arrays of one fixture case; ``files`` lists their names like np.load's NpzFile."""

    @property
    def files(self):
        return list(self)


def load_golden(name):
    """One case, merged from <name>.npz and its parts <name>.1.npz, ... (make_golden.py keeps each file under 1 MB)."""
    g = GoldenCase()
    for f in sorted(os.listdir(GOLDEN)):
        if f == name + ".npz" or (f.startswith(name + ".") and f.endswith(".npz")):
            with np.load(os.path.join(GOLDEN, f)) as z:
                g.update((k, z[k]) for k in z.files)
    p = g["params"]
    params = dict(tile_size=int(p[0]), tile_length=float(p[1]), wind_x=float(p[2]), wind_y=float(p[3]),
                  wind_speed=float(p[4]), phillips_const=float(p[5]), damping=float(p[6]),
                  anim_period=float(p[7]), lam=float(p[8]))
    return g, params


def h0_struct(h0_5):
    """(N,N,5) fp32 -> structured array in the reference's 20-byte record layout."""
    from oracle.port import H0_DTYPE
    a = np.ascontiguousarray(h0_5, np.float32)
    return a.view(H0_DTYPE).reshape(a.shape[0], a.shape[1])


def rel_l2(a, b):
    dt = np.complex128 if (np.iscomplexobj(a) or np.iscomplexobj(b)) else np.float64
    a = np.asarray(a, dt)
    b = np.asarray(b, dt)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


# Parity gate (BASELINE.json north_star): per map channel rel-L2 <= 1e-5 and
# max-abs <= 1e-4 * (channel max - min) versus the oracle fed the same h0.
REL_L2_TOL = 1e-5
MAX_ABS_TOL = 1e-4
# amplitude / min / max of the height field (SURVEY.md §8d)
SCALAR_REL_TOL = 1e-6


def assert_maps_close(disp, norm, disp_ref, norm_ref, what="", skip_w=False):
    """skip_w: the Jacobian switch is on (disp.w carries J, checked by the caller)."""
    for name, got, ref in (("disp", disp, disp_ref), ("norm", norm, norm_ref)):
        for c in range(4):
            g, r = got[..., c], ref[..., c]
            rng = float(r.max() - r.min())
            if name == "disp" and c == 3:
                assert skip_w or np.all(g == 1.0), f"{what} disp.w must be exactly 1.0"
                continue
            e2 = rel_l2(g, r)
            emax = float(np.max(np.abs(g.astype(np.float64) - r.astype(np.float64))))
            assert e2 <= REL_L2_TOL, f"{what} {name}[{c}] rel-L2 {e2:.3e} > {REL_L2_TOL}"
            assert emax <= MAX_ABS_TOL * rng, f"{what} {name}[{c}] max-abs {emax:.3e} > {MAX_ABS_TOL}*{rng:.3e}"


@pytest.fixture(scope="session")
def ref_available():
    from oracle import refmodel
    return refmodel.available()
