"""ctypes view of include/rtb200.h — the binding a host in any language would write.

The library is mandatory: importing this module without librtb200.so raises, and every compute
entry point fails with RTB_ECUDA when no CUDA device is present (there is no CPU fallback).
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "librtb200.so")

RTB_OK = 0
RTB_EIO = -1
RTB_EPARSE = -2
RTB_EMESH = -3
RTB_ENOLIGHT = -4
RTB_EUNSUPPORTED = -5
RTB_ECUDA = -6
RTB_EINVAL = -7
RTB_ESTOPPED = -8
RTB_ECANCELLED = 1

EST_NEE = 0
EST_MIS_DEAD = 1
EST_MIS_BALANCE = 2
EST_NEE_ALL_LIGHTS = 3
ACCEL_LBVH = 0
ACCEL_OCTREE_REFERENCE = 1


class Params(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("spp", C.c_int32), ("estimator", C.c_int32),
                ("seed", C.c_uint64), ("rank", C.c_int32), ("world", C.c_int32), ("pool_paths", C.c_int32),
                ("accel", C.c_int32), ("tuning", C.c_int32 * 4)]


class Adaptive(C.Structure):
    _fields_ = [("target_levels", C.c_float), ("pass_spp", C.c_int32), ("min_spp", C.c_int32), ("reserved", C.c_int32)]


class Denoise(C.Structure):
    _fields_ = [("levels", C.c_int32), ("sigma_color", C.c_float), ("sigma_normal", C.c_float), ("sigma_depth", C.c_float),
                ("reserved", C.c_int32 * 4)]


class SceneInfo(C.Structure):
    _fields_ = [("n_objects", C.c_int32), ("n_planes", C.c_int32), ("n_spheres", C.c_int32), ("n_meshes", C.c_int32),
                ("n_triangles", C.c_int32), ("light_object", C.c_int32), ("bvh_nodes", C.c_int32),
                ("bvh_leaves", C.c_int32), ("device", C.c_int32), ("bvh_depth", C.c_int32), ("octree_nodes", C.c_int32), ("octree_tri_refs", C.c_int32),
                ("bvh_min", C.c_float * 3), ("bvh_max", C.c_float * 3), ("camera_pos", C.c_float * 3),
                ("camera_dir", C.c_float * 3), ("build_ms", C.c_double)]


class Stats(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("rays_primary", C.c_uint64), ("rays_extension", C.c_uint64),
                ("rays_shadow", C.c_uint64), ("iterations", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("bvh_node_visits", C.c_uint64), ("bvh_tri_tests", C.c_uint64), ("render_ms", C.c_double),
                ("extend_ms", C.c_double), ("bin_ms", C.c_double), ("generate_ms", C.c_double),
                ("resolve_ms", C.c_double), ("shade_ms", C.c_double), ("rays_bvh", C.c_uint64),
                ("shadow_bvh", C.c_uint64), ("paths_queued", C.c_uint64), ("first_record_ms", C.c_double), ("wall_ms", C.c_double)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class ObjectDesc(C.Structure):
    _fields_ = [("emitted", C.c_double * 3), ("brdf", C.c_int32), ("geometry", C.c_int32), ("k", C.c_double * 3),
                ("color_d", C.c_double * 3), ("color_s", C.c_double * 3), ("pos", C.c_double * 3), ("n", C.c_double * 3),
                ("r", C.c_double), ("triangles", C.POINTER(C.c_float)), ("n_triangles", C.c_int64)]


class SceneDesc(C.Structure):
    _fields_ = [("camera_pos", C.c_double * 3), ("camera_dir", C.c_double * 3), ("n_objects", C.c_int32),
                ("reserved", C.c_int32), ("objects", C.POINTER(ObjectDesc))]


class ObjectInfo(C.Structure):
    _fields_ = [("brdf", C.c_int32), ("geometry", C.c_int32), ("n_triangles", C.c_int32), ("first_triangle", C.c_int32),
                ("emitted", C.c_double * 3), ("k", C.c_double * 3), ("color_d", C.c_double * 3),
                ("color_s", C.c_double * 3), ("pos", C.c_double * 3), ("n", C.c_double * 3), ("r", C.c_double),
                ("bb_min", C.c_double * 3), ("bb_max", C.c_double * 3), ("surface_area", C.c_double)]


EXPORTS = [
    "rtb_last_error", "rtb_scene_load_toml", "rtb_scene_load_toml_string", "rtb_scene_create", "rtb_scene_destroy", "rtb_scene_get_info", "rtb_scene_object",
    "rtb_scene_upload", "rtb_scene_triangles", "rtb_render", "rtb_local_pixels", "rtb_tile_map", "rtb_render_device",
    "rtb_untile_device", "rtb_get_stats", "rtb_job_begin", "rtb_job_next", "rtb_job_next_messages", "rtb_job_next_frame", "rtb_job_cancel",
    "rtb_job_end", "rtb_trace_primary", "rtb_trace_rays", "rtb_sample_radiance", "rtb_fp32_peak",
    "rtb_untile_device_async", "rtb_job_stats", "rtb_sample_pixels", "rtb_trace_rays_accel", "rtb_scene_octree_stats", "rtb_scene_export", "rtb_scene_import",
    "rtb_render_adaptive", "rtb_job_begin_adaptive",
    "rtb_render_denoised", "rtb_job_begin_denoised", "rtb_scene_gbuffer", "rtb_denoise_image",
    "rtb_scene_lights",
]

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python raytracer-server_b200/build.py` "
                          "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, ip, fp = C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_float)
    L.rtb_last_error.restype = C.c_char_p
    L.rtb_scene_load_toml.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.POINTER(vp)]
    L.rtb_scene_load_toml_string.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.POINTER(vp)]
    L.rtb_scene_create.argtypes = [C.POINTER(SceneDesc), C.c_int, C.POINTER(vp)]
    L.rtb_scene_destroy.argtypes = [vp]
    L.rtb_scene_destroy.restype = None
    L.rtb_scene_get_info.argtypes = [vp, C.POINTER(SceneInfo)]
    L.rtb_scene_object.argtypes = [vp, C.c_int32, C.POINTER(ObjectInfo)]
    L.rtb_scene_upload.argtypes = [vp, C.POINTER(C.c_uint64)]
    L.rtb_scene_triangles.argtypes = [vp, fp, C.c_int64]
    L.rtb_scene_triangles.restype = C.c_int64
    L.rtb_scene_lights.argtypes = [vp, ip, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int64]
    L.rtb_scene_lights.restype = C.c_int64
    L.rtb_render.argtypes = [vp, C.POINTER(Params), C.POINTER(C.c_uint8), ip]
    L.rtb_local_pixels.argtypes = [C.POINTER(Params)]
    L.rtb_local_pixels.restype = C.c_int64
    L.rtb_tile_map.argtypes = [C.POINTER(Params), ip, C.c_int64]
    L.rtb_tile_map.restype = C.c_int64
    L.rtb_render_device.argtypes = [vp, C.POINTER(Params), vp, vp, ip]
    L.rtb_untile_device.argtypes = [C.POINTER(Params), vp, C.c_int64, vp, C.c_int]
    L.rtb_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.rtb_job_begin.argtypes = [vp, C.POINTER(Params), C.c_int32, C.POINTER(vp)]
    L.rtb_render_adaptive.argtypes = [vp, C.POINTER(Params), C.POINTER(Adaptive), C.POINTER(C.c_uint8), ip, fp, ip]
    L.rtb_job_begin_adaptive.argtypes = [vp, C.POINTER(Params), C.POINTER(Adaptive), C.POINTER(vp)]
    L.rtb_render_denoised.argtypes = [vp, C.POINTER(Params), C.POINTER(Adaptive), C.POINTER(Denoise), C.POINTER(C.c_uint8), ip, fp, ip]
    L.rtb_job_begin_denoised.argtypes = [vp, C.POINTER(Params), C.c_int32, C.POINTER(Adaptive), C.POINTER(Denoise), C.POINTER(vp)]
    L.rtb_scene_gbuffer.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, fp, fp, fp, ip]
    L.rtb_denoise_image.argtypes = [C.c_int, C.c_int32, C.c_int32, C.POINTER(Denoise), fp, fp, fp, fp, fp, ip, fp]
    L.rtb_job_next.argtypes = [vp, C.POINTER(C.c_uint16), C.POINTER(C.c_uint16), C.POINTER(C.c_uint8),
                               C.POINTER(C.c_uint8)]
    L.rtb_job_next_messages.argtypes = [vp, C.POINTER(C.c_uint8), C.c_int64, C.c_int32, C.POINTER(C.c_int64)]
    L.rtb_job_next_frame.argtypes = [vp, C.POINTER(C.c_uint8), ip]
    L.rtb_job_cancel.argtypes = [vp]
    L.rtb_job_end.argtypes = [vp]
    L.rtb_trace_primary.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_float, ip, ip, fp]
    L.rtb_trace_rays.argtypes = [vp, C.c_int64, fp, fp, ip, ip, fp, C.POINTER(C.c_uint64)]
    L.rtb_sample_radiance.argtypes = [vp, C.POINTER(Params), C.c_int64, ip, ip, ip, fp]
    L.rtb_fp32_peak.argtypes = [C.c_int, C.POINTER(C.c_double)]
    L.rtb_untile_device_async.argtypes = [C.POINTER(Params), vp, C.c_int64, vp, C.c_int, vp]
    L.rtb_job_stats.argtypes = [vp, C.POINTER(Stats)]
    L.rtb_sample_pixels.argtypes = [vp, C.POINTER(Params), C.c_int64, ip, ip, fp]
    L.rtb_scene_export.argtypes = [vp, vp, C.c_int64]
    L.rtb_scene_export.restype = C.c_int64
    L.rtb_scene_import.argtypes = [vp, C.c_int64, C.c_int, C.POINTER(vp)]
    L.rtb_scene_octree_stats.argtypes = [vp, C.c_int32, C.POINTER(C.c_int64)]
    L.rtb_trace_rays_accel.argtypes = [vp, C.c_int32, C.c_int64, fp, fp, ip, ip, fp]
    for name in EXPORTS:
        fn = getattr(L, name)
        if fn.restype is C.c_int:
            fn.restype = C.c_int
    _lib = L
    return L


def last_error() -> str:
    return (lib().rtb_last_error() or b"").decode(errors="replace")
