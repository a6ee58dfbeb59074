"""ctypes view of include/rttnw_b200.h and the loader of librttnw_b200.so.

The product has no CPU path: if the CUDA library is missing, `load()` raises —
nothing here (or anywhere in this package) falls back to the oracle or numpy.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# RTTNW_B200_LIB: an alternative build of the same library (kernel tuning experiments)
LIB_PATH = os.environ.get("RTTNW_B200_LIB") or os.path.join(_HERE, "lib", "librttnw_b200.so")

RTX_OK = 0
RTX_MISS = -1

# rtx_node_kind
NODE_SPHERE, NODE_MOVING_SPHERE, NODE_RECT_XY, NODE_RECT_XZ, NODE_RECT_YZ, NODE_CUBE = 1, 2, 3, 4, 5, 6
NODE_LIST, NODE_BVH, NODE_TRANSLATE, NODE_ROTATE_Y, NODE_MEDIUM = 7, 8, 9, 10, 11
# rtx_material_kind
MAT_LAMBERTIAN, MAT_METAL, MAT_DIELECTRIC, MAT_DIFFUSE_LIGHT, MAT_ISOTROPIC = 1, 2, 3, 4, 5
# rtx_texture_kind
TEX_SOLID, TEX_CHECKER, TEX_NOISE, TEX_IMAGE = 1, 2, 3, 4


class Node(C.Structure):
    _fields_ = [("kind", C.c_int32), ("material", C.c_int32), ("child", C.c_int32),
                ("n_children", C.c_int32), ("f", C.c_double * 10)]


class Material(C.Structure):
    _fields_ = [("kind", C.c_int32), ("texture", C.c_int32), ("albedo", C.c_double * 3),
                ("param", C.c_double)]


class Texture(C.Structure):
    _fields_ = [("kind", C.c_int32), ("a", C.c_int32), ("b", C.c_int32), ("_pad", C.c_int32),
                ("f", C.c_double * 4)]


class Perlin(C.Structure):
    _fields_ = [("ranvec", (C.c_double * 3) * 256), ("perm_x", C.c_int32 * 256),
                ("perm_y", C.c_int32 * 256), ("perm_z", C.c_int32 * 256)]


class Image(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("rgba", C.POINTER(C.c_uint8))]


class Camera(C.Structure):
    _fields_ = [("lookfrom", C.c_double * 3), ("lookat", C.c_double * 3), ("view_up", C.c_double * 3),
                ("vertical_fov", C.c_double), ("aspect_ratio", C.c_double), ("aperture", C.c_double),
                ("focus_distance", C.c_double), ("open_time", C.c_double), ("close_time", C.c_double)]


class SceneDesc(C.Structure):
    _fields_ = [("nodes", C.POINTER(Node)), ("n_nodes", C.c_int32), ("root", C.c_int32),
                ("children", C.POINTER(C.c_int32)), ("n_children", C.c_int32), ("n_materials", C.c_int32),
                ("materials", C.POINTER(Material)), ("textures", C.POINTER(Texture)),
                ("n_textures", C.c_int32), ("n_perlins", C.c_int32), ("perlins", C.POINTER(Perlin)),
                ("images", C.POINTER(Image)), ("n_images", C.c_int32), ("_pad", C.c_int32),
                ("background", C.c_double * 3), ("camera", Camera)]


class Ray(C.Structure):
    _fields_ = [("origin", C.c_double * 3), ("direction", C.c_double * 3), ("time", C.c_double),
                ("t_min", C.c_double), ("t_max", C.c_double), ("xi", C.c_double)]


class Hit(C.Structure):
    _fields_ = [("prim_id", C.c_int32), ("material", C.c_int32), ("front_face", C.c_int32),
                ("_pad", C.c_int32), ("t", C.c_double), ("p", C.c_double * 3),
                ("normal", C.c_double * 3), ("u", C.c_double), ("v", C.c_double)]


class TraceStats(C.Structure):
    _fields_ = [("rays", C.c_double), ("box_tests", C.c_double), ("node_visits", C.c_double),
                ("sphere_tests", C.c_double), ("rect_tests", C.c_double),
                ("instance_enters", C.c_double), ("medium_tests", C.c_double)]


class RenderParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("spp_begin", C.c_int32),
                ("spp_count", C.c_int32), ("max_depth", C.c_int32), ("_pad", C.c_int32),
                ("seed", C.c_uint64)]


class SceneDefaults(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("samples", C.c_int32),
                ("max_depth", C.c_int32), ("name", C.c_char_p)]


class AdaptiveParams(C.Structure):
    _fields_ = [("threshold", C.c_double), ("min_spp", C.c_int32), ("step_spp", C.c_int32)]


class AdaptiveStats(C.Structure):
    _fields_ = [("path_samples", C.c_int64), ("rounds", C.c_int32), ("tiles", C.c_int32),
                ("tiles_converged", C.c_int32), ("tiles_at_max", C.c_int32)]


class DenoiseParams(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("sigma_normal", C.c_float), ("sigma_albedo", C.c_float),
                ("sigma_luminance", C.c_float)]


class Environment(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("rgb", C.POINTER(C.c_float)), ("rotation_y", C.c_double),
                ("scale", C.c_double * 3)]


assert C.sizeof(Node) == 96 and C.sizeof(Material) == 40 and C.sizeof(Texture) == 48
assert C.sizeof(Ray) == 80 and C.sizeof(Hit) == 88 and C.sizeof(RenderParams) == 32
assert C.sizeof(AdaptiveParams) == 16 and C.sizeof(AdaptiveStats) == 24 and C.sizeof(DenoiseParams) == 16
assert C.sizeof(Environment) == 48

# numpy views of the two bulk records (same memory layout as the C structs)
RAY_DTYPE = [("origin", "<f8", 3), ("direction", "<f8", 3), ("time", "<f8"), ("t_min", "<f8"),
             ("t_max", "<f8"), ("xi", "<f8")]
HIT_DTYPE = [("prim_id", "<i4"), ("material", "<i4"), ("front_face", "<i4"), ("_pad", "<i4"),
             ("t", "<f8"), ("p", "<f8", 3), ("normal", "<f8", 3), ("u", "<f8"), ("v", "<f8")]

# name -> (restype, argtypes); every symbol include/rttnw_b200.h declares
_P = C.c_void_p
SIGNATURES = {
    "rtx_abi_version": (C.c_int, []),
    "rtx_last_error": (C.c_char_p, []),
    "rtx_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "rtx_ctx_create": (C.c_int, [C.c_int, _P, C.POINTER(_P)]),
    "rtx_ctx_destroy": (C.c_int, [_P]),
    "rtx_ctx_sync": (C.c_int, [_P]),
    "rtx_ctx_set_async": (C.c_int, [_P, C.c_int]),
    "rtx_ctx_stream": (_P, [_P]),
    "rtx_ctx_set_bvh_builder": (C.c_int, [_P, C.c_int]),
    "rtx_ctx_kernel_launches": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "rtx_ctx_set_profiling": (C.c_int, [_P, C.c_int]),
    "rtx_ctx_profile_read": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.c_int]),
    "rtx_ctx_measure_l2_read": (C.c_int, [_P, C.c_uint64, C.c_int, C.POINTER(C.c_double)]),
    "rtx_scene_create": (C.c_int, [_P, C.POINTER(SceneDesc), C.POINTER(_P)]),
    "rtx_scene_destroy": (C.c_int, [_P]),
    "rtx_cache_trim": (C.c_int, [C.c_int]),
    "rtx_scene_info": (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                 C.POINTER(C.c_int64)]),
    "rtx_trace_rays": (C.c_int, [_P, _P, C.c_int64, _P, _P]),
    "rtx_trace_rays_device": (C.c_int, [_P, _P, C.c_int64, _P, _P]),
    "rtx_trace_rays_stats": (C.c_int, [_P, _P, C.c_int64, _P, C.POINTER(TraceStats)]),
    "rtx_render": (C.c_int, [_P, _P, C.POINTER(RenderParams), _P, _P]),
    "rtx_render_counted": (C.c_int, [_P, _P, C.POINTER(RenderParams), _P, C.POINTER(TraceStats)]),
    "rtx_render_adaptive": (C.c_int, [_P, _P, C.POINTER(RenderParams), C.POINTER(AdaptiveParams), _P, _P,
                                      C.POINTER(AdaptiveStats)]),
    "rtx_adaptive_error": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, _P]),
    "rtx_render_aov": (C.c_int, [_P, _P, C.POINTER(RenderParams), _P, _P, _P]),
    "rtx_denoise": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, C.POINTER(DenoiseParams), _P]),
    "rtx_tonemap_rgba8": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, C.c_int]),
    "rtx_reduce_tonemap_peers": (C.c_int, [_P, _P, C.POINTER(_P), C.c_int32, C.c_int32, C.c_int32, _P]),
    "rtx_reduce_tonemap_slice": (C.c_int, [_P, C.POINTER(_P), C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    "rtx_comm_unique_id": (C.c_int, [C.POINTER(C.c_uint8 * 128)]),
    "rtx_comm_create": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_uint8 * 128), C.POINTER(_P)]),
    "rtx_comm_wrap": (C.c_int, [_P, C.POINTER(_P)]),
    "rtx_comm_destroy": (C.c_int, [_P]),
    "rtx_accum_reduce": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32]),
    "rtx_malloc": (C.c_int, [_P, C.c_size_t, C.POINTER(_P)]),
    "rtx_free": (C.c_int, [_P, _P]),
    "rtx_memset_zero": (C.c_int, [_P, _P, C.c_size_t]),
    "rtx_memcpy_h2d": (C.c_int, [_P, _P, _P, C.c_size_t]),
    "rtx_memcpy_d2h": (C.c_int, [_P, _P, _P, C.c_size_t]),
    "rtx_memcpy_d2d": (C.c_int, [_P, _P, _P, C.c_size_t]),
    "rtx_ipc_export": (C.c_int, [_P, _P, C.POINTER(C.c_uint8 * 64)]),
    "rtx_ipc_open": (C.c_int, [_P, C.POINTER(C.c_uint8 * 64), C.POINTER(_P)]),
    "rtx_ipc_close": (C.c_int, [_P, _P]),
    "rtx_builtin_scene_defaults": (C.c_int, [C.c_int, C.POINTER(SceneDefaults)]),
    "rtx_builtin_scene": (C.c_int, [C.c_int, C.c_uint64, C.c_char_p, C.POINTER(C.POINTER(SceneDesc))]),
    "rtx_scene_desc_free": (C.c_int, [C.POINTER(SceneDesc)]),
    "rtx_flatten_check": (C.c_int, [C.POINTER(SceneDesc), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                    C.POINTER(C.c_int32)]),
    "rtx_png_read_rgba8": (C.c_int, [C.c_char_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                     C.POINTER(C.POINTER(C.c_uint8))]),
    "rtx_png_write_rgba8": (C.c_int, [C.c_char_p, C.c_int32, C.c_int32, _P]),
    "rtx_pfm_write": (C.c_int, [C.c_char_p, C.c_int32, C.c_int32, C.c_int32, _P]),
    "rtx_scene_set_environment": (C.c_int, [_P, _P, C.POINTER(Environment)]),
    "rtx_pfm_read": (C.c_int, [C.c_char_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                               C.POINTER(C.POINTER(C.c_float))]),
    "rtx_hdr_read": (C.c_int, [C.c_char_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.POINTER(C.c_float))]),
    "rtx_buffer_free": (C.c_int, [_P]),
}


class RtxError(RuntimeError):
    pass


_lib = None


def load() -> C.CDLL:
    """Loads librttnw_b200.so (built by `make` / __graft_entry__.build()). Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RtxError(
            f"{LIB_PATH} is missing: the CUDA library has not been built (run `make` at the repo "
            "root or __graft_entry__.build()). rttnw_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.rtx_abi_version() != 1:
        raise RtxError("librttnw_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != RTX_OK:
        msg = load().rtx_last_error()
        raise RtxError(f"rtx status {status}: {msg.decode() if msg else '?'}")
