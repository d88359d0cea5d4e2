"""ctypes binding of libtracer_cuda.so (include/tracer_cuda.h).

The library is built in-tree by ``esctp1raytracer_b200/csrc/Makefile`` (see
``__graft_entry__.build``).  There is no fallback: if the shared object is
missing, or no CUDA device is present, calls raise ``TracerError``.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtracer_cuda.so")

# every symbol include/tracer_cuda.h declares (checked by tests/test_abi.py)
ABI_SYMBOLS = [
    "tracer_cuda_abi_version", "tracer_cuda_init", "tracer_cuda_shutdown", "tracer_cuda_last_error",
    "tracer_cuda_device_info", "tracer_cuda_render", "tracer_cuda_scene_create", "tracer_cuda_scene_destroy",
    "tracer_cuda_render_scene", "tracer_cuda_last_stats", "tracer_band_row_count", "tracer_cuda_assemble_bands",
    "tracer_mt19937_faceids", "tracer_cuda_fp32_peak", "tracer_camera_lookat",
    "tracer_cuda_init_multi", "tracer_cuda_multi_gpu_count", "tracer_cuda_render_multi", "tracer_cuda_scene_create_multi",
    "tracer_cuda_scene_destroy_multi", "tracer_cuda_render_scene_multi", "tracer_cuda_last_stats_multi",
    "tracer_cuda_scene_update", "tracer_cuda_scene_update_multi", "tracer_cuda_render_views",
]
# include/tracer_host.h
HOST_SYMBOLS = ["tracer_scene_load_obj", "tracer_scene_host_flat", "tracer_scene_host_free", "tracer_host_last_error",
                "tracer_write_ppm", "tracer_scene_flatten_sorted", "tracer_scene_host_origin"]


class TracerError(RuntimeError):
    pass


class SceneFlat(C.Structure):
    _fields_ = [
        ("n_geoms", C.c_int32), ("geom_tri_offset", C.POINTER(C.c_int32)), ("tri_verts", C.POINTER(C.c_float)),
        ("tri_normals", C.POINTER(C.c_float)), ("geom_has_normals", C.POINTER(C.c_int32)),
        ("geom_material", C.POINTER(C.c_float)), ("n_lights", C.c_int32), ("light_geom", C.POINTER(C.c_int32)),
        ("n_spheres", C.c_int32), ("sphere_cr", C.POINTER(C.c_float)), ("sphere_material", C.POINTER(C.c_float)),
    ]


class CameraC(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("lower_left_corner", C.c_float * 3), ("horizontal", C.c_float * 3),
                ("vertical", C.c_float * 3)]


# int32_t (*row_hits_exchange)(void *user, int32_t height, int32_t *row_hits)
ROW_HITS_EXCHANGE = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_int32, C.POINTER(C.c_int32))


class RenderOpts(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("rng_mode", C.c_int32), ("seed", C.c_uint32), ("faceid", C.POINTER(C.c_int32)),
        ("band_rows", C.c_int32), ("band_index", C.c_int32), ("band_count", C.c_int32),
        ("rgb_out_is_device", C.c_int32), ("cuda_stream", C.c_void_p),
        ("exhaustive_strict", C.c_int32), ("samples_per_pixel", C.c_int32),
        ("rays_per_thread", C.c_int32), ("shadow_chunks", C.c_int32), ("bundle_cull", C.c_int32),
        ("out_tri", C.POINTER(C.c_int32)), ("out_t", C.POINTER(C.c_float)), ("out_v", C.POINTER(C.c_float)),
        ("out_occ_tri", C.POINTER(C.c_int32)), ("out_rgb", C.POINTER(C.c_float)), ("accel", C.c_int32),
        ("row_hits_exchange", ROW_HITS_EXCHANGE), ("row_hits_user", C.c_void_p),
        ("crop_x", C.c_int32), ("crop_y", C.c_int32), ("crop_w", C.c_int32), ("crop_h", C.c_int32),
    ]


class SceneUpdate(C.Structure):
    """tracer_scene_update; the array pointers are plain addresses (host or device, per data_is_device)"""
    _fields_ = [
        ("struct_size", C.c_uint32), ("data_is_device", C.c_int32), ("cuda_stream", C.c_void_p),
        ("tri_first", C.c_int32), ("tri_count", C.c_int32), ("tri_verts", C.c_void_p), ("tri_normals", C.c_void_p),
        ("geom_material", C.c_void_p), ("sphere_cr", C.c_void_p), ("sphere_material", C.c_void_p),
    ]


class FrameStats(C.Structure):
    _fields_ = [
        ("ms_total", C.c_double), ("ms_primary", C.c_double), ("ms_shadow", C.c_double), ("ms_other", C.c_double),
        ("n_pixels", C.c_int64), ("n_primary_rays", C.c_int64), ("n_shadow_rays", C.c_int64),
        ("tests_primary", C.c_int64), ("tests_shadow", C.c_int64), ("tests_shadow_ref", C.c_int64),
        ("strict_evals", C.c_int64), ("filter_misses", C.c_int64), ("kernel_launches", C.c_int32),
        ("n_sms", C.c_int32), ("flop_primary", C.c_double), ("flop_shadow", C.c_double),
        ("flop_primary_edges", C.c_double), ("flop_shadow_edges", C.c_double), ("pipeline_errors", C.c_int64),
    ]

    def asdict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class DeviceInfo(C.Structure):
    _fields_ = [("name", C.c_char * 128), ("sm_count", C.c_int32), ("cc_major", C.c_int32), ("cc_minor", C.c_int32),
                ("clock_khz", C.c_int32), ("total_mem", C.c_int64), ("l2_bytes", C.c_int64)]


_lib = None


def load():
    """Load the shared library (no device needed for this step)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TracerError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    lib.tracer_cuda_last_error.restype = C.c_char_p
    lib.tracer_cuda_init.argtypes = [C.c_int]
    lib.tracer_cuda_device_info.argtypes = [C.POINTER(DeviceInfo)]
    lib.tracer_cuda_scene_create.argtypes = [C.POINTER(SceneFlat), C.POINTER(C.c_void_p)]
    lib.tracer_cuda_scene_destroy.argtypes = [C.c_void_p]
    lib.tracer_cuda_scene_destroy.restype = None
    lib.tracer_cuda_render_scene.argtypes = [C.c_void_p, C.POINTER(CameraC), C.c_int32, C.c_int32,
                                             C.POINTER(RenderOpts), C.c_void_p]
    lib.tracer_cuda_render.argtypes = [C.POINTER(SceneFlat), C.POINTER(CameraC), C.c_int32, C.c_int32,
                                       C.POINTER(RenderOpts), C.c_void_p]
    lib.tracer_cuda_last_stats.argtypes = [C.c_void_p, C.POINTER(FrameStats)]
    lib.tracer_cuda_render_views.argtypes = [C.c_void_p, C.POINTER(CameraC), C.c_int32, C.c_int32, C.c_int32,
                                             C.POINTER(RenderOpts), C.c_void_p]
    lib.tracer_cuda_init_multi.argtypes = [C.c_int]
    lib.tracer_cuda_scene_create_multi.argtypes = [C.POINTER(SceneFlat), C.POINTER(C.c_void_p)]
    lib.tracer_cuda_scene_destroy_multi.argtypes = [C.c_void_p]
    lib.tracer_cuda_scene_destroy_multi.restype = None
    lib.tracer_cuda_render_scene_multi.argtypes = [C.c_void_p, C.POINTER(CameraC), C.c_int32, C.c_int32,
                                                   C.POINTER(RenderOpts), C.c_void_p]
    lib.tracer_cuda_render_multi.argtypes = [C.POINTER(SceneFlat), C.POINTER(CameraC), C.c_int32, C.c_int32,
                                             C.POINTER(RenderOpts), C.c_void_p]
    lib.tracer_cuda_last_stats_multi.argtypes = [C.c_void_p, C.POINTER(FrameStats)]
    lib.tracer_cuda_scene_update.argtypes = [C.c_void_p, C.POINTER(SceneUpdate)]
    lib.tracer_cuda_scene_update_multi.argtypes = [C.c_void_p, C.POINTER(SceneUpdate)]
    lib.tracer_band_row_count.argtypes = [C.c_int32] * 4
    lib.tracer_band_row_count.restype = C.c_int32
    lib.tracer_cuda_assemble_bands.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                               C.c_int32, C.c_void_p]
    lib.tracer_mt19937_faceids.argtypes = [C.POINTER(SceneFlat), C.c_int32, C.c_int32, C.c_uint32,
                                           C.POINTER(C.c_uint8), C.POINTER(C.c_int32)]
    lib.tracer_cuda_fp32_peak.argtypes = [C.c_int32, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.tracer_camera_lookat.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_float,
                                         C.c_float, C.POINTER(CameraC)]
    lib.tracer_camera_lookat.restype = None
    lib.tracer_scene_load_obj.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
    lib.tracer_scene_host_flat.argtypes = [C.c_void_p]
    lib.tracer_scene_host_flat.restype = C.POINTER(SceneFlat)
    lib.tracer_scene_host_free.argtypes = [C.c_void_p]
    lib.tracer_scene_host_free.restype = None
    lib.tracer_host_last_error.restype = C.c_char_p
    lib.tracer_scene_flatten_sorted.argtypes = [C.POINTER(SceneFlat), C.POINTER(C.c_void_p)]
    lib.tracer_scene_host_origin.argtypes = [C.c_void_p, C.POINTER(C.POINTER(C.c_int32)), C.POINTER(C.POINTER(C.c_int32))]
    lib.tracer_write_ppm.argtypes = [C.c_char_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32]
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise TracerError(f"tracer_cuda error {rc}: {load().tracer_cuda_last_error().decode()}")
