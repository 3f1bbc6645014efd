"""ctypes binding of libfirework_b200.so (include/firework_b200.h).  No torch types cross this boundary.

The library is the product; there is no Python / CPU fallback.  If it is missing or a CUDA device is not
available, calls fail loudly.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FW_LIB_PATH", os.path.join(_HERE, "libfirework_b200.so"))


class FwParams(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("samples", C.c_uint32),
                ("sample_begin", C.c_uint32), ("sample_count", C.c_uint32), ("use_bvh", C.c_uint32),
                ("gamma", C.c_float), ("cam_pos", C.c_float * 3), ("look_at", C.c_float * 3),
                ("vfov", C.c_float), ("aperture", C.c_float), ("focus_dist", C.c_float), ("seed", C.c_uint64)]


class FwStats(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("rays", C.c_uint64), ("launches", C.c_uint64),
                ("ms_device", C.c_double), ("ms_extend", C.c_double), ("extend_launches", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class FwAdaptive(C.Structure):
    _fields_ = [("min_samples", C.c_uint32), ("threshold", C.c_float), ("floor", C.c_float)]


class FwAdaptiveResult(C.Structure):
    _fields_ = [("rounds", C.c_uint32), ("samples", C.c_uint64), ("active", C.c_uint32 * 32)]


class FwAov(C.Structure):
    _fields_ = [("albedo", C.c_void_p), ("normal", C.c_void_p), ("depth", C.c_void_p), ("object", C.c_void_p)]


class FwDenoise(C.Structure):
    _fields_ = [("iterations", C.c_uint32), ("aov_samples", C.c_uint32), ("sigma_luminance", C.c_float),
                ("sigma_depth", C.c_float), ("sigma_albedo", C.c_float)]


class FireworkError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"firework_b200 error {code}: {msg}")
        self.code = code


# every symbol include/firework_b200.h declares (tests check that the library exports all of them)
EXPORTS = [
    "fw_scene_from_yaml", "fw_scene_from_file", "fw_scene_destroy", "fw_scene_num_assets", "fw_scene_asset_path",
    "fw_scene_asset_kind", "fw_scene_set_image", "fw_scene_set_hdr", "fw_scene_build_host", "fw_scene_commit", "fw_scene_num_objects",
    "fw_scene_num_nodes", "fw_scene_device_bytes", "fw_scene_top_leaf_order", "fw_scene_object_aabb", "fw_scene_mesh_leaf_order", "fw_scene_linear_program", "fw_scene_bvh_nodes", "fw_render",
    "fw_render_accumulate_device", "fw_resolve_device", "fw_primary_rays", "fw_first_hit", "fw_scatter_step",
    "fw_scatter_step_keyed",    "fw_env_sample", "fw_texture_sample", "fw_material_texture", "fw_camera", "fw_last_error", "fw_version",
    "fw_device_count", "fw_measure_peaks", "fw_selftest_shared_division", "fw_obj_load", "fw_obj_num_models",
    "fw_obj_model_name", "fw_obj_model_sizes", "fw_obj_model_copy", "fw_obj_destroy", "fw_hdr_load", "fw_hdr_free", "fw_image_load", "fw_image_free", "fw_png_write", "fw_set_profiling", "fw_set_batch_paths", "fw_release_cached_memory", "fw_texture_store_stats",
    "fw_resolve_host", "fw_render_multi", "fw_scene_walk_info", "fw_first_hit_wavefront", "fw_render_adaptive",
    "fw_render_aov", "fw_denoise_host", "fw_render_denoised", "fw_trace_rays", "fw_trace_rays_device",
]

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FireworkError(-100, f"{LIB_PATH} is missing: run `python -m firework_b200.build` "
                                      "(there is no CPU fallback)")
        if "FW_NCCL_LIB" not in os.environ:
            # fw_render_multi dlopens NCCL on first use; if PyTorch's bundled (newer) copy exists, use that one so that a
            # later `import torch` in the same process finds the libnccl.so.2 it was built against (one library per SONAME)
            try:
                import importlib.util
                spec = importlib.util.find_spec("nvidia.nccl")
                for d in (spec.submodule_search_locations if spec else []):
                    cand = os.path.join(d, "lib", "libnccl.so.2")
                    if os.path.exists(cand):
                        os.environ["FW_NCCL_LIB"] = cand
                        break
            except Exception:
                pass
        L = C.CDLL(LIB_PATH)
        L.fw_last_error.restype = C.c_char_p
        L.fw_version.restype = C.c_char_p
        L.fw_scene_asset_path.restype = C.c_char_p
        L.fw_scene_asset_path.argtypes = [C.c_void_p, C.c_int]
        L.fw_scene_from_yaml.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_void_p)]
        L.fw_scene_from_file.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
        L.fw_scene_destroy.argtypes = [C.c_void_p]
        L.fw_obj_load.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
        L.fw_obj_num_models.argtypes = [C.c_void_p]
        L.fw_obj_model_name.argtypes = [C.c_void_p, C.c_int]
        L.fw_obj_model_name.restype = C.c_char_p
        L.fw_obj_model_sizes.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.fw_obj_model_copy.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.fw_obj_destroy.argtypes = [C.c_void_p]
        L.fw_obj_destroy.restype = None
        L.fw_hdr_load.argtypes = [C.c_char_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.POINTER(C.c_float))]
        L.fw_hdr_free.argtypes = [C.POINTER(C.c_float)]
        L.fw_hdr_free.restype = None
        L.fw_image_load.argtypes = [C.c_char_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.POINTER(C.c_uint8))]
        L.fw_image_free.argtypes = [C.POINTER(C.c_uint8)]
        L.fw_image_free.restype = None
        L.fw_png_write.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.c_void_p]
        L.fw_texture_store_stats.argtypes = [C.c_void_p]
        L.fw_scene_destroy.restype = None
        for name in ("fw_scene_num_assets", "fw_scene_num_objects", "fw_scene_num_nodes"):
            getattr(L, name).argtypes = [C.c_void_p]
        L.fw_scene_asset_kind.argtypes = [C.c_void_p, C.c_int]
        L.fw_scene_set_image.argtypes = [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_void_p]
        L.fw_scene_set_hdr.argtypes = [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_void_p]
        L.fw_scene_commit.argtypes = [C.c_void_p, C.c_int]
        L.fw_scene_build_host.argtypes = [C.c_void_p]
        L.fw_scene_device_bytes.argtypes = [C.c_void_p]
        L.fw_scene_device_bytes.restype = C.c_uint64
        L.fw_scene_top_leaf_order.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.fw_scene_object_aabb.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.fw_scene_mesh_leaf_order.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        L.fw_scene_bvh_nodes.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        if hasattr(L, "fw_scene_linear_program"):   # absent only in older builds used for A/B timing
            L.fw_scene_linear_program.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.fw_render.argtypes = [C.c_void_p, C.POINTER(FwParams), C.c_void_p, C.c_void_p, C.POINTER(FwStats)]
        L.fw_render_accumulate_device.argtypes = [C.c_void_p, C.POINTER(FwParams), C.c_void_p, C.c_void_p, C.POINTER(FwStats)]
        L.fw_resolve_device.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_void_p, C.c_void_p]
        L.fw_primary_rays.argtypes = [C.c_void_p, C.POINTER(FwParams), C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
        L.fw_first_hit.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint32] + [C.c_void_p] * 13
        L.fw_first_hit_wavefront.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32] + [C.c_void_p] * 7
        L.fw_scatter_step.argtypes = [C.c_void_p, C.c_uint32] + [C.c_void_p] * 8 + [C.c_uint32] + [C.c_void_p] * 6
        L.fw_scatter_step_keyed.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32] + [C.c_void_p] * 16
        L.fw_env_sample.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
        L.fw_texture_sample.argtypes = [C.c_void_p, C.c_int, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.fw_material_texture.argtypes = [C.c_void_p, C.c_int]
        L.fw_camera.argtypes = [C.POINTER(FwParams), C.c_void_p]
        L.fw_measure_peaks.argtypes = [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.fw_set_profiling.argtypes = [C.c_void_p, C.c_int]
        L.fw_set_batch_paths.argtypes = [C.c_void_p, C.c_uint64]
        L.fw_scene_walk_info.argtypes = [C.c_void_p, C.c_void_p]
        L.fw_resolve_host.argtypes = [C.c_int, C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_void_p]
        L.fw_render_multi.argtypes = [C.c_void_p, C.POINTER(FwParams), C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                      C.POINTER(FwStats), C.POINTER(C.c_double)]
        if hasattr(L, "fw_render_adaptive"):        # absent only in older builds used for A/B timing
            L.fw_render_adaptive.argtypes = [C.c_void_p, C.POINTER(FwParams), C.POINTER(FwAdaptive)] + [C.c_void_p] * 4 + \
                                            [C.POINTER(FwStats), C.POINTER(FwAdaptiveResult)]
        if hasattr(L, "fw_render_denoised"):        # absent only in older builds used for A/B timing
            L.fw_render_aov.argtypes = [C.c_void_p, C.POINTER(FwParams), C.POINTER(FwAov), C.POINTER(FwStats)]
            L.fw_denoise_host.argtypes = [C.c_int, C.c_uint32, C.c_uint32] + [C.c_void_p] * 5 + [C.POINTER(FwDenoise), C.c_void_p, C.c_void_p]
            L.fw_render_denoised.argtypes = [C.c_void_p, C.POINTER(FwParams), C.POINTER(FwDenoise)] + [C.c_void_p] * 4 + \
                                            [C.POINTER(FwAov), C.POINTER(FwStats)]
        if hasattr(L, "fw_trace_rays"):             # absent only in older builds used for A/B timing
            trace = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_uint64, C.c_int,
                     C.c_void_p]
            L.fw_trace_rays.argtypes = trace + [C.POINTER(FwStats)]
            L.fw_trace_rays_device.argtypes = trace + [C.c_void_p, C.POINTER(FwStats)]
        _lib = L
    return _lib


def check(rc: int) -> int:
    if rc < 0:
        raise FireworkError(rc, lib().fw_last_error().decode("utf-8", "replace"))
    return rc


def ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)
