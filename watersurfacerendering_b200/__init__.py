"""watersurfacerendering_b200 — B200-native Tessendorf wave synthesis (the hot path of
kentril0/WaterSurfaceRendering's `WSTessendorf`), hand-written sm_100a CUDA behind a C ABI.

    from watersurfacerendering_b200 import WSTessendorf
    ws = WSTessendorf(512, 1000.0); ws.Prepare(seed=1234); A = ws.ComputeWaves(1.5)
"""
from . import _lib  # noqa: F401
from ._lib import (WSO_SPECTRUM_JONSWAP, WSO_SPECTRUM_PHILLIPS, WSO_SPECTRUM_PIERSON_MOSKOWITZ,  # noqa: F401
                   WSO_SPECTRUM_TMA)
from .surface import (BODY_DTYPE, H0_DTYPE, HYDRO_RESULT_DTYPE, RAY_HIT_DTYPE, SURFACE_SAMPLE_DTYPE,  # noqa: F401
                      PinnedBuffer, WSTessendorf, make_spectrum, spectrum_h0)

__all__ = ["WSTessendorf", "PinnedBuffer", "H0_DTYPE", "SURFACE_SAMPLE_DTYPE", "RAY_HIT_DTYPE", "BODY_DTYPE",
           "HYDRO_RESULT_DTYPE", "make_spectrum",
           "spectrum_h0", "WSO_SPECTRUM_PHILLIPS", "WSO_SPECTRUM_PIERSON_MOSKOWITZ", "WSO_SPECTRUM_JONSWAP",
           "WSO_SPECTRUM_TMA"]
