"""rtb200 — B200-native replacement for raytracer-server's per-pixel radiance loop.

Python is only the host glue here (ctypes over the C ABI in include/rtb200.h); every sample is
computed by hand-written sm_100a kernels in librtb200.so.  Import name: ``raytracer_server_b200``
(the directory carries the repository's hyphenated name; see raytracer_server_b200.py).
"""
from ._abi import (ACCEL_LBVH, ACCEL_OCTREE_REFERENCE, EST_MIS_BALANCE, EST_MIS_DEAD, EST_NEE, LIB_PATH, RTB_ECANCELLED, RTB_ECUDA, RTB_EINVAL, RTB_EIO, RTB_EMESH,
                   RTB_ENOLIGHT, RTB_EPARSE, RTB_EUNSUPPORTED, RTB_OK, Adaptive, Params, SceneInfo, Stats)
from .host import LoadTomlError, RenderJob, RtbError, Scene, fp32_peak_tflops, make_adaptive, make_params, sample_pixel

__all__ = ["Scene", "RenderJob", "sample_pixel", "make_params", "make_adaptive", "Adaptive", "LoadTomlError", "RtbError", "Params", "SceneInfo",
           "Stats", "fp32_peak_tflops", "LIB_PATH", "EST_NEE", "EST_MIS_DEAD", "EST_MIS_BALANCE", "ACCEL_LBVH", "ACCEL_OCTREE_REFERENCE"]
