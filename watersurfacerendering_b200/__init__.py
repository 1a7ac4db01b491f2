"""watersurfacerendering_b200 — B200-native Tessendorf wave synthesis (the hot path of
kentril0/WaterSurfaceRendering's `WSTessendorf`), hand-written sm_100a CUDA behind a C ABI.

    from watersurfacerendering_b200 import WSTessendorf
    ws = WSTessendorf(512, 1000.0); ws.Prepare(seed=1234); A = ws.ComputeWaves(1.5)
"""
from . import _lib  # noqa: F401
from .surface import H0_DTYPE, RAY_HIT_DTYPE, SURFACE_SAMPLE_DTYPE, PinnedBuffer, WSTessendorf  # noqa: F401

__all__ = ["WSTessendorf", "PinnedBuffer", "H0_DTYPE", "SURFACE_SAMPLE_DTYPE", "RAY_HIT_DTYPE"]
