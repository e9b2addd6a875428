"""ctypes wrapper of the CPU oracle (oracle/rtp_oracle.c). TEST INFRASTRUCTURE ONLY.

Loaded by tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs — never by the product.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import rtp_b200
from rtp_b200 import _abi as A
from rtp_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB = os.path.join(ORACLE_DIR, "_build", "liboracle.so")
_lib = None


def build():
    subprocess.run(["make", "-C", ORACLE_DIR], check=True, stdout=subprocess.DEVNULL)


def lib():
    global _lib
    if _lib is None:
        src = os.path.join(ORACLE_DIR, "rtp_oracle.c")
        if not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(src):
            build()
        L = C.CDLL(LIB)
        P = C.POINTER
        sigs = {
            "orc_last_error": (C.c_char_p, []),
            "orc_philox4x32_10": (None, [C.c_void_p, C.c_void_p, C.c_void_p]),
            "orc_rng_draws": (None, [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]),
            "orc_obj_load": (C.c_int, [C.c_char_p, P(A.Mesh)]),
            "orc_mesh_free": (None, [P(A.Mesh)]),
            "orc_tga_load": (C.c_int, [C.c_char_p, P(A.Image)]),
            "orc_tga_save": (C.c_int, [P(A.Image), C.c_char_p]),
            "orc_image_free": (None, [P(A.Image)]),
            "orc_camera_lookat": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, P(A.Camera)]),
            "orc_frame_to_srgb8": (None, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]),
            "orc_split_in_tiles": (C.c_size_t, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_size_t]),
            "orc_scene_create": (C.c_int, [P(A.SceneDesc), P(C.c_void_p)]),
            "orc_scene_destroy": (None, [C.c_void_p]),
            "orc_scene_get_info": (C.c_int, [C.c_void_p, P(A.SceneInfo)]),
            "orc_scene_leaf_order": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
            "orc_scene_node": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
            "orc_scene_root": (C.c_uint32, [C.c_void_p]),
            "orc_aabb_collide": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
            "orc_trace_closest": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, P(A.Stats)]),
            "orc_camera_rays": (None, [P(A.Camera), C.c_uint32, C.c_uint32, C.c_void_p]),
            "orc_render": (C.c_int, [C.c_void_p, P(A.Camera), P(A.RenderParams), C.c_void_p, C.c_void_p, C.c_int, P(A.Stats)]),
            "orc_trace_one": (C.c_int, [C.c_void_p, P(A.Camera), P(A.RenderParams), C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, P(C.c_int), P(C.c_uint32)]),
            "orc_texture_sample": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
            "orc_noise_integer": (C.c_int64, [C.c_int64, C.c_int64, C.c_int64, C.c_int64]),
            "orc_scene_set_libm": (C.c_int, [C.c_void_p, C.c_int]),
            "orc_device_atan2_n": (None, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
            "orc_device_asin_n": (None, [C.c_void_p, C.c_size_t, C.c_void_p]),
        }
        for name, (res, args) in sigs.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


class OracleError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"oracle error {code}: {msg}")
        self.code = code


def _check(rc):
    if rc != 0:
        raise OracleError(rc, (lib().orc_last_error() or b"").decode())


def philox(ctr, key):
    c = np.asarray(ctr, dtype=np.uint32)
    k = np.asarray(key, dtype=np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    lib().orc_philox4x32_10(A.ptr(c), A.ptr(k), A.ptr(out))
    return out


def rng_draws(seed, lo, hi, stream, first, n):
    out = np.empty(n, dtype=np.float64)
    lib().orc_rng_draws(seed, lo, hi, stream, first, n, A.ptr(out))
    return out


def obj_load(path) -> api.Mesh:
    m = A.Mesh()
    _check(lib().orc_obj_load(path.encode(), C.byref(m)))
    v = np.empty(m.n_vertices, dtype=A.VERTEX_DTYPE)
    ix = np.empty(m.n_indices, dtype=np.uint32)
    if m.n_vertices:
        C.memmove(v.ctypes.data, m.vertices, v.nbytes)
    if m.n_indices:
        C.memmove(ix.ctypes.data, m.indices, ix.nbytes)
    lib().orc_mesh_free(C.byref(m))
    return api.Mesh(v, ix, 0)


def tga_load(path) -> np.ndarray:
    img = A.Image()
    _check(lib().orc_tga_load(path.encode(), C.byref(img)))
    out = np.empty((img.height, img.width, 4), dtype=np.uint8)
    if out.nbytes:
        C.memmove(out.ctypes.data, img.rgba, out.nbytes)
    lib().orc_image_free(C.byref(img))
    return out


def tga_save(image, path):
    image = np.ascontiguousarray(image, dtype=np.uint8)
    img = A.Image(image.ctypes.data, image.shape[1], image.shape[0])
    _check(lib().orc_tga_save(C.byref(img), path.encode()))


def lookat(position, target, up) -> A.Camera:
    cam = A.Camera()
    p, t, u = (np.asarray(x, dtype=np.float64) for x in (position, target, up))
    _check(lib().orc_camera_lookat(A.ptr(p), A.ptr(t), A.ptr(u), C.byref(cam)))
    return cam


def to_srgb_u8(frame):
    frame = np.ascontiguousarray(frame, dtype=np.float64)
    h, w = frame.shape[:2]
    out = np.empty((h, w, 4), dtype=np.uint8)
    lib().orc_frame_to_srgb8(A.ptr(frame), w, h, A.ptr(out))
    return out


def split_in_tiles(fw, fh, tw, th):
    n = lib().orc_split_in_tiles(fw, fh, tw, th, None, 0)
    out = np.zeros((n, 4), dtype=np.uint32)
    lib().orc_split_in_tiles(fw, fh, tw, th, A.ptr(out), n)
    return out


def aabb_collide(bmin, bmax, ray) -> bool:
    bmin = np.asarray(bmin, dtype=np.float64)
    bmax = np.asarray(bmax, dtype=np.float64)
    r = np.asarray(ray, dtype=np.float64).reshape(8)
    return bool(lib().orc_aabb_collide(A.ptr(bmin), A.ptr(bmax), A.ptr(r)))


def device_atan2(y, x) -> np.ndarray:
    """CUDA's double atan2 (the oracle's transcription of libdevice), elementwise over broadcast arrays."""
    y, x = (np.array(a, dtype=np.float64) for a in np.broadcast_arrays(y, x))
    out = np.empty(y.shape, dtype=np.float64)
    lib().orc_device_atan2_n(A.ptr(y), A.ptr(x), y.size, A.ptr(out))
    return out


def device_asin(x) -> np.ndarray:
    """CUDA's double asin (the oracle's transcription of libdevice), elementwise."""
    x = np.array(x, dtype=np.float64)
    out = np.empty(x.shape, dtype=np.float64)
    lib().orc_device_asin_n(A.ptr(x), x.size, A.ptr(out))
    return out


def camera_rays(camera: api.Camera, width, height) -> np.ndarray:
    out = np.empty(width * height, dtype=A.RAY_DTYPE)
    cc = camera.to_c()
    lib().orc_camera_rays(C.byref(cc), width, height, A.ptr(out))
    return out


class Scene:
    """Oracle twin of rtp_b200.api.Scene.

    libm picks the atan2 / asin of sphere and sky uv: "host" is the C library's (the reference's), "device" is CUDA's,
    with which the device's images are equal to the oracle's bit for bit."""

    def __init__(self, scene: api.ExampleScene, libm="host"):
        desc, keep = api.build_desc(scene)
        h = C.c_void_p()
        _check(lib().orc_scene_create(C.byref(desc), C.byref(h)))
        self._h = h
        self.camera = scene.camera
        _check(lib().orc_scene_set_libm(h, {"host": 0, "device": 1}[libm]))

    def close(self):
        if self._h:
            lib().orc_scene_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self):
        i = A.SceneInfo()
        _check(lib().orc_scene_get_info(self._h, C.byref(i)))
        return i

    def leaf_order(self):
        n = self.info().n_leaves
        out = np.zeros(n, dtype=np.uint32)
        _check(lib().orc_scene_leaf_order(self._h, A.ptr(out), n))
        return out

    def node(self, k):
        aabb = np.zeros(6)
        lrl = np.zeros(3, dtype=np.uint32)
        _check(lib().orc_scene_node(self._h, k, A.ptr(aabb), A.ptr(lrl)))
        return aabb, lrl

    def root(self):
        return lib().orc_scene_root(self._h)

    def hit_full(self, rays, mode=0, threads=None, stats=False):
        rays = api._as_rays(rays)
        hits = np.empty(len(rays), dtype=A.HIT_FULL_DTYPE)
        st = A.Stats()
        threads = threads or os.cpu_count() or 1
        _check(lib().orc_trace_closest(self._h, A.ptr(rays), len(rays), A.ptr(hits), mode, threads, C.byref(st)))
        return (hits, st) if stats else hits

    def hit(self, rays, mode=0, threads=None):
        f = self.hit_full(rays, mode, threads)
        out = np.empty(len(f), dtype=A.HIT_DTYPE)
        out["leaf"], out["material"], out["t"] = f["leaf"], f["material"], f["t"]
        return out

    def render(self, width, height, num_samples, max_bounce=8, seed=1, camera=None, sample_range=None, tile=None, flags=0, threads=None, rows=None):
        cam = camera or self.camera
        cam = api.Camera(width / height, cam.fov, cam.focal_dist, cam.lens_radius, cam.transformation)
        p = api.render_params(width, height, num_samples, max_bounce, seed,
                              sample_range[0] if sample_range else 0, sample_range[1] if sample_range else None, tile, flags, rows)
        rgbf = np.zeros((height, width, 3), dtype=np.float64)
        fg = np.zeros((height, width), dtype=np.float64)
        st = A.Stats()
        cc = cam.to_c()
        threads = threads or os.cpu_count() or 1
        _check(lib().orc_render(self._h, C.byref(cc), C.byref(p), A.ptr(rgbf), A.ptr(fg), threads, C.byref(st)))
        return rgbf, fg, st

    def trace_one(self, width, height, i, j, s, max_bounce=8, seed=1, camera=None):
        cam = camera or self.camera
        cam = api.Camera(width / height, cam.fov, cam.focal_dist, cam.lens_radius, cam.transformation)
        p = api.render_params(width, height, 1, max_bounce, seed)
        rgb = np.zeros(3)
        hit = C.c_int(0)
        nr = C.c_uint32(0)
        cc = cam.to_c()
        _check(lib().orc_trace_one(self._h, C.byref(cc), C.byref(p), i, j, s, A.ptr(rgb), C.byref(hit), C.byref(nr)))
        return rgb, bool(hit.value), nr.value

    def texture_sample(self, tid, position, uv):
        pos = np.asarray(position, dtype=np.float64)
        uvv = np.asarray(uv, dtype=np.float64)
        out = np.zeros(3)
        _check(lib().orc_texture_sample(self._h, tid, A.ptr(pos), A.ptr(uvv), A.ptr(out)))
        return out
