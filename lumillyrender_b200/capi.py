"""ctypes mirror of include/lumilly.h — the only way Python touches the product.

The library is built in-tree by lumillyrender_b200/build.py (nvcc, sm_100a).  There is no Python or CPU
implementation of the render path: if the shared library is missing and cannot be built, import fails
loudly; if no CUDA device is present, every compute call raises LumillyError(LR_ERR_NO_DEVICE).
"""
import ctypes as C
import os

from . import build as _build

LR_OK = 0
LR_ERR_INVALID, LR_ERR_NO_DEVICE, LR_ERR_CUDA, LR_ERR_IO, LR_ERR_PARSE, LR_ERR_UNSUPPORTED = -1, -2, -3, -4, -5, -6
LR_MAT_LAMBERT, LR_MAT_PHONG, LR_MAT_BLINN_PHONG, LR_MAT_GGX, LR_MAT_IDEAL_REFRACTION = range(5)
LR_CAM_IDEAL_PINHOLE, LR_CAM_PINHOLE, LR_CAM_THIN_LENS, LR_CAM_OMNIDIRECTIONAL = range(4)
LR_SKY_UNIFORM, LR_SKY_IBL = 0, 1
LR_INTEGRATOR_PT, LR_INTEGRATOR_PT_DIRECT = 0, 1
LR_AOV_NORMAL, LR_AOV_DEPTH = 0, 1
LR_BVH_HOST, LR_BVH_DEVICE = 0, 1

f32, i32, u64, i64 = C.c_float, C.c_int32, C.c_uint64, C.c_int64


class LrMaterial(C.Structure):
    _fields_ = [("type", i32), ("color", f32 * 3), ("emission", f32 * 3), ("param0", f32), ("param1", f32)]


class LrTriangle(C.Structure):
    _fields_ = [("p0", f32 * 3), ("p1", f32 * 3), ("p2", f32 * 3), ("material", i32), ("prim_id", i32)]


class LrSphere(C.Structure):
    _fields_ = [("center", f32 * 3), ("radius", f32), ("material", i32), ("prim_id", i32)]


class LrCamera(C.Structure):
    _fields_ = [("type", i32), ("width", i32), ("height", i32), ("forward", f32 * 3), ("right", f32 * 3), ("up", f32 * 3),
                ("position", f32 * 3), ("aperture_position", f32 * 3), ("sensor_size", f32 * 2), ("aperture_radius", f32),
                ("aperture_sensor_distance", f32), ("sensor_pixel_area", f32), ("sensor_sensitivity", f32), ("focus_distance", f32)]


class LrSky(C.Structure):
    _fields_ = [("type", i32), ("color", f32 * 3), ("pixels", C.POINTER(f32)), ("n_pixels", i64), ("height", i32),
                ("longitude_offset", f32)]


class LrBvhNode(C.Structure):
    _fields_ = [("f", f32 * 12), ("c", i32 * 2), ("n", i32 * 2)]


class LrSceneDesc(C.Structure):
    _fields_ = [("materials", C.POINTER(LrMaterial)), ("n_materials", i32), ("triangles", C.POINTER(LrTriangle)), ("n_triangles", i32),
                ("spheres", C.POINTER(LrSphere)), ("n_spheres", i32), ("nodes", C.POINTER(LrBvhNode)), ("n_nodes", i32),
                ("bvh_depth", i32), ("n_flat_triangles", i32), ("camera", LrCamera), ("sky", LrSky)]


class LrRenderParams(C.Structure):
    _fields_ = [("integrator", i32), ("spp_begin", i32), ("spp_count", i32), ("depth", i32), ("depth_limit", i32),
                ("no_direct_emitter", i32), ("seed", u64), ("crop_x", i32), ("crop_y", i32), ("crop_w", i32), ("crop_h", i32),
                ("splits", i32), ("count_traversal", i32)]


class LrStats(C.Structure):
    _fields_ = [("rays", u64), ("samples", u64), ("nodes_visited", u64), ("tris_tested", u64), ("spheres_tested", u64),
                ("nonfinite_samples", u64), ("gate_retraces", u64), ("flat_tris_tested", u64), ("flat_boxes_tested", u64),
                ("kernel_ms", f32), ("launches", i32), ("splits", i32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class LrSceneConfig(C.Structure):
    _fields_ = [("samples", i32), ("depth", i32), ("depth_limit", i32), ("no_direct_emitter", i32), ("threads", i32),
                ("integrator", i32), ("width", i32), ("height", i32), ("output", i32), ("gamma", f32), ("n_prims", i32),
                ("n_emitters", i32), ("bvh_build_seconds", f32), ("bvh_builder", i32), ("bvh_device_kernel_ms", f32)]


class LumillyError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("liblumilly_b200 error %d: %s" % (code, message))
        self.code = code
        self.message = message


_PF = C.POINTER(f32)
_PI = C.POINTER(i32)
_VP = C.c_void_p

# name -> (restype, argtypes); every entry point include/lumilly.h declares
SIGNATURES = {
    "lr_abi_version": (C.c_int, []),
    "lr_init": (C.c_int, [C.c_int]),
    "lr_shutdown": (None, []),
    "lr_last_error": (C.c_char_p, []),
    "lr_device_info": (C.c_int, [_PI, _PI, _PI, C.c_char_p, C.c_int]),
    "lr_scene_create": (C.c_int, [C.POINTER(LrSceneDesc), C.POINTER(_VP)]),
    "lr_scene_destroy": (None, [_VP]),
    "lr_scene_bytes": (C.c_int, [_VP, C.POINTER(u64)]),
    "lr_render": (C.c_int, [_VP, C.POINTER(LrRenderParams), _PF, _PF, C.POINTER(LrStats)]),
    "lr_render_accumulate_device": (C.c_int, [_VP, C.POINTER(LrRenderParams), _VP, _VP, _VP]),
    "lr_stats_fetch": (C.c_int, [_VP, _VP, C.POINTER(LrStats)]),
    "lr_shard_range": (C.c_int, [i32, i32, i32, i32, _PI, _PI]),
    "lr_render_multi": (C.c_int, [C.POINTER(LrSceneDesc), C.POINTER(LrRenderParams), i32, _PI, _PF, _PF, C.POINTER(LrStats)]),
    "lr_render_aov": (C.c_int, [_VP, C.POINTER(LrRenderParams), i32, _PF]),
    "lr_film_create": (C.c_int, [_VP, C.POINTER(LrRenderParams), i32, C.POINTER(_VP)]),
    "lr_film_render": (C.c_int, [_VP, i32, C.POINTER(LrStats)]),
    "lr_film_info": (C.c_int, [_VP, _PI, _PI, _PI, _PI]),
    "lr_film_read": (C.c_int, [_VP, _PF, _PF]),
    "lr_film_save": (C.c_int, [_VP, C.c_char_p]),
    "lr_film_load": (C.c_int, [_VP, C.c_char_p, C.POINTER(_VP)]),
    "lr_film_destroy": (None, [_VP]),
    "lr_multi_scene_create": (C.c_int, [C.POINTER(LrSceneDesc), i32, _PI, C.POINTER(_VP)]),
    "lr_multi_render": (C.c_int, [_VP, C.POINTER(LrRenderParams), _PF, _PF, C.POINTER(LrStats)]),
    "lr_multi_scene_destroy": (None, [_VP]),
    "lr_multi_film_create": (C.c_int, [_VP, C.POINTER(LrRenderParams), i32, C.POINTER(_VP)]),
    "lr_multi_film_render": (C.c_int, [_VP, i32, C.POINTER(LrStats)]),
    "lr_multi_film_info": (C.c_int, [_VP, _PI, _PI, _PI, _PI]),
    "lr_multi_film_read": (C.c_int, [_VP, _PF, _PF]),
    "lr_multi_film_save": (C.c_int, [_VP, C.c_char_p]),
    "lr_multi_film_load": (C.c_int, [_VP, C.c_char_p, C.POINTER(_VP)]),
    "lr_multi_film_destroy": (None, [_VP]),
    "lr_film_render_adaptive": (C.c_int, [_VP, i32, f32, i32, _PI, C.POINTER(LrStats)]),
    "lr_film_spp_map": (C.c_int, [_VP, _PI]),
    "lr_multi_film_render_adaptive": (C.c_int, [_VP, i32, f32, i32, _PI, C.POINTER(LrStats)]),
    "lr_multi_film_spp_map": (C.c_int, [_VP, _PI]),
    "lr_trace_primary": (C.c_int, [_VP, f32, f32, f32, f32, _PI, _PF]),
    "lr_trace_rays": (C.c_int, [_VP, i64, _PF, _PF, _PI, _PF, _PF]),
    "lr_trace_rays_query": (C.c_int, [_VP, i64, _PF, _PF, i32, _PI, _PF, _PF]),
    "lr_measure_l2_read_gbs": (C.c_int, [u64, C.c_int, _PF]),
    "lr_measure_hbm_read_gbs": (C.c_int, [u64, C.c_int, _PF]),
    "lr_host_scene_load": (C.c_int, [C.c_char_p, C.c_char_p, i32, i32, C.POINTER(_VP)]),
    "lr_host_scene_desc": (C.POINTER(LrSceneDesc), [_VP]),
    "lr_host_scene_config": (C.c_int, [_VP, C.POINTER(LrSceneConfig)]),
    "lr_host_scene_free": (None, [_VP]),
    "lr_host_scene_rebuild_bvh": (C.c_int, [_VP, i32]),
    "lr_host_scene_from_arrays": (C.c_int, [C.POINTER(LrMaterial), i32, C.POINTER(LrTriangle), i32, C.POINTER(LrSphere), i32,
                                            C.POINTER(LrCamera), C.POINTER(LrSky), C.POINTER(_VP)]),
    "lr_camera_ideal_pinhole": (C.c_int, [_PF, f32, i32, i32, C.POINTER(LrCamera)]),
    "lr_camera_thin_lens": (C.c_int, [_PF, f32, f32, f32, i32, i32, C.POINTER(LrCamera)]),
    "lr_camera_omnidirectional": (C.c_int, [_PF, i32, i32, C.POINTER(LrCamera)]),
    "lr_camera_pinhole": (C.c_int, [_PF, _PF, _PF, i32, i32, f32, C.POINTER(LrCamera)]),
    "lr_matrix_unit": (None, [_PF]),
    "lr_matrix_translate": (None, [_PF, _PF]),
    "lr_matrix_scale": (None, [_PF, _PF]),
    "lr_matrix_axis_angle": (None, [_PF, f32, _PF]),
    "lr_matrix_look_at": (None, [_PF, _PF, _PF, _PF]),
    "lr_matrix_mul": (None, [_PF, _PF, _PF]),
    "lr_matrix_apply": (None, [_PF, _PF, _PF]),
    "lr_save_png": (C.c_int, [C.c_char_p, _PF, i32, i32, f32]),
    "lr_save_hdr": (C.c_int, [C.c_char_p, _PF, i32, i32]),
    "lr_load_hdr": (C.c_int, [C.c_char_p, C.POINTER(_PF), _PI, _PI]),
    "lr_free": (None, [_VP]),
}

_lib = None


def library_path():
    return _build.LIB


def load_library():
    """Loads (building first if needed) liblumilly_b200.so.  Raises if it cannot be had: no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("LUMILLY_LIB")            # development: A/B a variant build (tools/ab.py)
    if path:
        if not os.path.exists(path):
            raise FileNotFoundError(path)
    else:
        path = _build.LIB
    if path == _build.LIB and (not os.path.exists(path) or os.environ.get("LUMILLY_REBUILD")):
        _build.build_library(force=bool(os.environ.get("LUMILLY_REBUILD")))
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError = the library does not export what the header declares
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != LR_OK:
        msg = load_library().lr_last_error()
        raise LumillyError(rc, msg.decode("utf-8", "replace") if msg else "")
    return rc
