"""ctypes mirror of include/rtp.h (struct layouts, enums, prototypes).

Plain plumbing: nothing here computes. The shared library is loaded lazily by `load()`;
`declare()` applies the same prototypes to any library exporting the rtp_* symbols.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

ABI_VERSION = 3
MISS = 0xFFFFFFFF

# rtp_status
OK, ERR_INVALID, ERR_IO, ERR_FORMAT, ERR_CUDA, ERR_NOMEM, ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5, -6
# rtp_hittable_kind
HITTABLE_SPHERE, HITTABLE_TRIANGLE, HITTABLE_LIST, HITTABLE_BVH = 0, 1, 2, 3
# rtp_scatter_kind / rtp_absorb_kind / rtp_emit_kind / rtp_texture_kind / rtp_root_kind
SCATTER_NONE, SCATTER_LAMBERT, SCATTER_METAL, SCATTER_DIELECTRIC = 0, 1, 2, 3
ABSORB_BLACKBODY, ABSORB_WHITEBODY, ABSORB_ALBEDO, ABSORB_ALBEDO_MAP = 0, 1, 2, 3
EMIT_NONE, EMIT_DEBUG_NORMALS, EMIT_COLOR, EMIT_SKY_GRADIENT, EMIT_SKY_SPHERE = 0, 1, 2, 3, 4
TEXTURE_MISSING, TEXTURE_DEBUG_UVS, TEXTURE_SOLID, TEXTURE_IMAGE, TEXTURE_CHECKER, TEXTURE_NOISE, TEXTURE_PERLIN = range(7)
ROOT_BVH, ROOT_LIST = 0, 1
RENDER_RAW_SUMS, RENDER_COUNTERS, RENDER_TRANSPARENT = 1, 2, 4
RNG_STREAM_PATH, RNG_STREAM_RAYS = 0, 1

# numpy views of the POD records that travel in bulk
RAY_DTYPE = np.dtype([("origin", "<f8", 3), ("direction", "<f8", 3), ("t_min", "<f8"), ("t_max", "<f8")])
HIT_DTYPE = np.dtype([("leaf", "<u4"), ("material", "<u4"), ("t", "<f8")])
HIT_FULL_DTYPE = np.dtype(
    [("leaf", "<u4"), ("material", "<u4"), ("t", "<f8"), ("position", "<f8", 3), ("normal", "<f8", 3), ("uv", "<f8", 2)]
)
VERTEX_DTYPE = np.dtype([("position", "<f8", 3), ("normal", "<f8", 3), ("uv", "<f8", 2)])
HITTABLE_DTYPE = np.dtype(
    [("kind", "<u4"), ("material", "<u4"), ("mesh", "<u4"), ("triangle", "<u4"), ("center", "<f8", 3), ("radius", "<f8")]
)
assert RAY_DTYPE.itemsize == 64 and HIT_DTYPE.itemsize == 16 and HIT_FULL_DTYPE.itemsize == 80
assert VERTEX_DTYPE.itemsize == 64 and HITTABLE_DTYPE.itemsize == 48


class Mesh(C.Structure):
    _fields_ = [
        ("vertices", C.c_void_p),
        ("indices", C.c_void_p),
        ("n_vertices", C.c_uint32),
        ("n_indices", C.c_uint32),
        ("material", C.c_uint32),
        ("_pad", C.c_uint32),
    ]


class Emit(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("texture", C.c_uint32), ("rgb", C.c_double * 3)]


class Material(C.Structure):
    _fields_ = [
        ("scatter", C.c_uint32),
        ("absorb", C.c_uint32),
        ("absorb_texture", C.c_uint32),
        ("_pad", C.c_uint32),
        ("scatter_param", C.c_double),
        ("absorb_rgb", C.c_double * 3),
        ("emit", Emit),
    ]


class Texture(C.Structure):
    _fields_ = [
        ("kind", C.c_uint32),
        ("width", C.c_uint32),
        ("height", C.c_uint32),
        ("odd", C.c_uint32),
        ("even", C.c_uint32),
        ("_pad", C.c_uint32),
        ("seed", C.c_int64),
        ("rgb", C.c_double * 3),
        ("rgba", C.c_void_p),
    ]


class SceneDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_uint32),
        ("root_kind", C.c_uint32),
        ("meshes", C.POINTER(Mesh)),
        ("hittables", C.c_void_p),
        ("materials", C.POINTER(Material)),
        ("textures", C.POINTER(Texture)),
        ("n_meshes", C.c_uint32),
        ("n_hittables", C.c_uint32),
        ("n_materials", C.c_uint32),
        ("n_textures", C.c_uint32),
        ("background", Emit),
        ("nested", C.c_void_p),
        ("n_nested", C.c_uint32),
        ("_pad", C.c_uint32),
    ]


class Camera(C.Structure):
    _fields_ = [
        ("aspect_ratio", C.c_double),
        ("fov", C.c_double),
        ("focal_dist", C.c_double),
        ("lens_radius", C.c_double),
        ("orientation", C.c_double * 9),
        ("position", C.c_double * 3),
    ]


class RenderParams(C.Structure):
    _fields_ = [
        ("width", C.c_uint32),
        ("height", C.c_uint32),
        ("num_samples", C.c_uint32),
        ("max_bounce", C.c_uint32),
        ("seed", C.c_uint64),
        ("sample_begin", C.c_uint32),
        ("sample_end", C.c_uint32),
        ("tile_x", C.c_uint32),
        ("tile_y", C.c_uint32),
        ("tile_w", C.c_uint32),
        ("tile_h", C.c_uint32),
        ("flags", C.c_uint32),
        ("device_mask", C.c_uint32),
        ("row_offset", C.c_uint32),
        ("row_stride", C.c_uint32),
    ]


class AdaptiveParams(C.Structure):
    _fields_ = [
        ("min_samples", C.c_uint32),
        ("max_samples", C.c_uint32),
        ("batch", C.c_uint32),
        ("_pad", C.c_uint32),
        ("abs_tol", C.c_double),
        ("rel_tol", C.c_double),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("rays", C.c_uint64),
        ("paths", C.c_uint64),
        ("node_visits", C.c_uint64),
        ("triangle_tests", C.c_uint64),
        ("sphere_tests", C.c_uint64),
        ("leaf_gates", C.c_uint64),
        ("conservative_violations", C.c_uint64),
        ("device_ms", C.c_double),
        ("kernel_launches", C.c_uint64),
        ("order_rewalks", C.c_uint64),
        ("trace_ms", C.c_double),
        ("shade_ms", C.c_double),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class SceneInfo(C.Structure):
    _fields_ = [
        ("n_leaves", C.c_uint32),
        ("n_nodes", C.c_uint32),
        ("depth", C.c_uint32),
        ("root_kind", C.c_uint32),
        ("device_bytes", C.c_uint64),
        ("culling_depth", C.c_uint32),
        ("any_order", C.c_uint32),
        ("n_big", C.c_uint32),
        ("free_tree_depth", C.c_uint32),
    ]


class AnyTables(C.Structure):
    _fields_ = [
        ("n_big", C.c_uint32),
        ("big", C.c_uint32 * 8),
        ("any_spheres", C.c_uint32),
        ("any_E", C.c_double),
        ("any_A", C.c_double),
        ("any_C", C.c_double),
        ("any_R", C.c_double),
        ("scene_mag", C.c_double),
        ("cull", C.c_float * 6),
    ]


class Image(C.Structure):
    _fields_ = [("rgba", C.c_void_p), ("width", C.c_uint32), ("height", C.c_uint32)]


# every symbol include/rtp.h declares: name -> (restype, argtypes)
_P = C.POINTER
PROTOTYPES = {
    "rtp_init": (C.c_int, [C.c_int]),
    "rtp_device_count": (C.c_int, [_P(C.c_int)]),
    "rtp_last_error": (C.c_char_p, []),
    "rtp_abi_version": (C.c_uint32, []),
    "rtp_host_alloc": (C.c_int, [C.c_size_t, _P(C.c_void_p)]),
    "rtp_host_free": (None, [C.c_void_p]),
    "rtp_obj_load": (C.c_int, [C.c_char_p, _P(Mesh)]),
    "rtp_mesh_free": (None, [_P(Mesh)]),
    "rtp_tga_load": (C.c_int, [C.c_char_p, _P(Image)]),
    "rtp_tga_save": (C.c_int, [_P(Image), C.c_char_p]),
    "rtp_image_free": (None, [_P(Image)]),
    "rtp_camera_lookat": (C.c_int, [_P(C.c_double), _P(C.c_double), _P(C.c_double), _P(Camera)]),
    "rtp_frame_to_srgb8": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "rtp_split_in_tiles": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_size_t, _P(C.c_size_t)]),
    "rtp_scene_create": (C.c_int, [_P(SceneDesc), _P(C.c_void_p)]),
    "rtp_scene_create_multi": (C.c_int, [_P(SceneDesc), C.c_uint32, _P(C.c_void_p)]),
    "rtp_scene_devices": (C.c_int, [C.c_void_p, _P(C.c_uint32)]),
    "rtp_scene_destroy": (None, [C.c_void_p]),
    "rtp_scene_get_info": (C.c_int, [C.c_void_p, _P(SceneInfo)]),
    "rtp_bvh_build_order": (C.c_int, [_P(SceneDesc), C.c_void_p, C.c_size_t, _P(SceneInfo)]),
    "rtp_bvh_culled_set": (C.c_int, [_P(SceneDesc), _P(C.c_float), _P(C.c_uint32), _P(C.c_uint32)]),
    "rtp_scene_leaf_order": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "rtp_trace_closest": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, _P(Stats)]),
    "rtp_trace_closest_full": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, _P(Stats)]),
    "rtp_trace_closest_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "rtp_trace_closest_device_counted": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, _P(Stats)]),
    "rtp_trace_occluded": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, _P(Stats)]),
    "rtp_trace_occluded_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "rtp_trace_occluded_device_counted": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, _P(Stats)]),
    "rtp_camera_rays_device": (C.c_int, [_P(Camera), C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "rtp_camera_rays": (C.c_int, [_P(Camera), C.c_uint32, C.c_uint32, C.c_void_p]),
    "rtp_render": (C.c_int, [C.c_void_p, _P(Camera), _P(RenderParams), C.c_void_p, C.c_void_p, _P(Stats)]),
    "rtp_render_device": (C.c_int, [C.c_void_p, _P(Camera), _P(RenderParams), C.c_void_p, C.c_void_p, _P(Stats), C.c_void_p]),
    "rtp_render_aov": (C.c_int, [C.c_void_p, _P(Camera), _P(RenderParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, _P(Stats)]),
    "rtp_render_aov_device": (
        C.c_int, [C.c_void_p, _P(Camera), _P(RenderParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, _P(Stats), C.c_void_p]
    ),
    "rtp_render_adaptive": (C.c_int, [C.c_void_p, _P(Camera), _P(RenderParams), _P(AdaptiveParams), C.c_void_p, C.c_void_p, C.c_void_p, _P(Stats)]),
    "rtp_render_adaptive_device": (
        C.c_int, [C.c_void_p, _P(Camera), _P(RenderParams), _P(AdaptiveParams), C.c_void_p, C.c_void_p, C.c_void_p, _P(Stats), C.c_void_p]
    ),
    "rtp_render_srgb8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rtp_trace_camera": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "rtp_rng_draws": (C.c_int, [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]),
    "rtp_probe_fp64": (C.c_int, [C.POINTER(C.c_double)]),
    "rtp_scene_digest": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "rtp_scene_any_tables": (C.c_int, [C.c_void_p, _P(AnyTables)]),
}

# RTP_B200_LIB: another build of the same library (kernel A/B runs from tools/); it is still this product's CUDA library
LIB_PATH = os.environ.get("RTP_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "librtp_b200.so")
_lib = None


def load():
    """Load librtp_b200.so. Fails loudly when the library has not been built — there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(raytracing-potato_b200 has no CPU or pure-Python fallback)"
            )
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def ptr(a: np.ndarray):
    return C.c_void_p(a.ctypes.data)
