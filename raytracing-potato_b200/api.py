"""Host-side mirror of the reference crate's scene / render interface, over the C ABI.

Names follow /root/reference/src: `Mesh`, `Vertex` arrays, `obj.load`, `tga.load/save`,
`Transformation.lookat`, `Camera`, `Scatter`/`Absorb`/`Emit`/`Material`, `Texture`, `Hittable`,
`SceneData`, `ExampleScene`, `Multisampler`-style render parameters. A `Scene` is the device-resident
replacement for `Hittable::Bvh(Bvh::new(..))` / `Hittable::List(..)` plus its `SceneData`:
`Scene.hit` is the batched `Hittable::hit` (bvh.rs:121-124) and `Scene.render` the worker loop of
main.rs:61-92. All compute happens in librtp_b200.so on the GPU; this module only marshals.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

from . import _abi as A


class RtpError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"rtp error {code}: {message}")
        self.code = code
        self.message = message


def _check(lib, rc: int):
    if rc != A.OK:
        raise RtpError(rc, (lib.rtp_last_error() or b"").decode("utf-8", "replace"))


def _vec3(v) -> np.ndarray:
    a = np.asarray(v, dtype=np.float64).reshape(3)
    return a


def rgb(r: float, g: float, b: float) -> np.ndarray:
    """utility.rs:198-200"""
    return np.array([r, g, b], dtype=np.float64)


# ------------------------------------------------------------------------------ mesh.rs ----------


@dataclass
class Mesh:
    """mesh.rs:18-22. `vertices` has dtype VERTEX_DTYPE, `indices` is uint32 (3 per face)."""

    vertices: np.ndarray
    indices: np.ndarray
    material: int = 0

    def iter_triangles(self) -> np.ndarray:
        """mesh.rs:32-34: TriangleId = 3*i"""
        return np.arange(0, len(self.indices) // 3, dtype=np.uint32) * 3

    @staticmethod
    def from_arrays(positions, normals=None, uvs=None, indices=None, material: int = 0) -> "Mesh":
        positions = np.asarray(positions, dtype=np.float64).reshape(-1, 3)
        v = np.zeros(len(positions), dtype=A.VERTEX_DTYPE)
        v["position"] = positions
        if normals is not None:
            v["normal"] = np.asarray(normals, dtype=np.float64).reshape(-1, 3)
        if uvs is not None:
            v["uv"] = np.asarray(uvs, dtype=np.float64).reshape(-1, 2)
        if indices is None:
            indices = np.arange(len(positions), dtype=np.uint32)
        return Mesh(v, np.ascontiguousarray(indices, dtype=np.uint32).reshape(-1), material)


class obj:
    @staticmethod
    def load(path: str) -> Mesh:
        """mesh.rs:145-183 obj::load"""
        lib = A.load()
        m = A.Mesh()
        _check(lib, lib.rtp_obj_load(path.encode(), C.byref(m)))
        try:
            v = np.empty(m.n_vertices, dtype=A.VERTEX_DTYPE)
            ix = np.empty(m.n_indices, dtype=np.uint32)
            if m.n_vertices:
                C.memmove(v.ctypes.data, m.vertices, v.nbytes)
            if m.n_indices:
                C.memmove(ix.ctypes.data, m.indices, ix.nbytes)
            return Mesh(v, ix, int(m.material))
        finally:
            lib.rtp_mesh_free(C.byref(m))


# ------------------------------------------------------------------------------ image.rs ---------


class tga:
    @staticmethod
    def load(path: str) -> np.ndarray:
        """image.rs:73-114 → uint8 array [height, width, 4], row 0 = bottom"""
        lib = A.load()
        img = A.Image()
        _check(lib, lib.rtp_tga_load(path.encode(), C.byref(img)))
        try:
            out = np.empty((img.height, img.width, 4), dtype=np.uint8)
            if out.nbytes:
                C.memmove(out.ctypes.data, img.rgba, out.nbytes)
            return out
        finally:
            lib.rtp_image_free(C.byref(img))

    @staticmethod
    def save(image: np.ndarray, path: str) -> None:
        """image.rs:116-137"""
        lib = A.load()
        image = np.ascontiguousarray(image, dtype=np.uint8)
        img = A.Image(image.ctypes.data, image.shape[1], image.shape[0])
        _check(lib, lib.rtp_tga_save(C.byref(img), path.encode()))


def split_in_tiles(full_width: int, full_height: int, tile_width: int, tile_height: int) -> np.ndarray:
    """image.rs:151-167 → uint32 [n, 4] rows of (offset_i, offset_j, width, height)"""
    lib = A.load()
    n = C.c_size_t(0)
    _check(lib, lib.rtp_split_in_tiles(full_width, full_height, tile_width, tile_height, None, 0, C.byref(n)))
    out = np.zeros((n.value, 4), dtype=np.uint32)
    _check(lib, lib.rtp_split_in_tiles(full_width, full_height, tile_width, tile_height, A.ptr(out), n.value, C.byref(n)))
    return out


def to_srgb_u8(frame: np.ndarray) -> np.ndarray:
    """utility.rs:212-220 over a [H, W, 3] float64 frame → [H, W, 4] uint8"""
    lib = A.load()
    frame = np.ascontiguousarray(frame, dtype=np.float64)
    h, w = frame.shape[:2]
    out = np.empty((h, w, 4), dtype=np.uint8)
    _check(lib, lib.rtp_frame_to_srgb8(A.ptr(frame), w, h, A.ptr(out)))
    return out


# ------------------------------------------------------------------------------ utility.rs / render.rs


@dataclass
class Transformation:
    """utility.rs:160-163; orientation columns are x, y, z"""

    orientation: np.ndarray  # [3,3], orientation[:, c] = column c
    position: np.ndarray

    @staticmethod
    def lookat(position, target, up) -> "Transformation":
        """utility.rs:172-177 (x = up × z is not normalised)"""
        lib = A.load()
        cam = A.Camera()
        p, t, u = _vec3(position), _vec3(target), _vec3(up)
        dp = C.POINTER(C.c_double)
        _check(lib, lib.rtp_camera_lookat(p.ctypes.data_as(dp), t.ctypes.data_as(dp), u.ctypes.data_as(dp), C.byref(cam)))
        m = np.array(list(cam.orientation), dtype=np.float64).reshape(3, 3).T.copy()  # stored column-major
        return Transformation(m, np.array(list(cam.position), dtype=np.float64))


@dataclass
class Camera:
    """render.rs:19-25"""

    aspect_ratio: float
    fov: float
    focal_dist: float
    lens_radius: float
    transformation: Transformation

    def to_c(self) -> A.Camera:
        c = A.Camera()
        c.aspect_ratio, c.fov, c.focal_dist, c.lens_radius = self.aspect_ratio, self.fov, self.focal_dist, self.lens_radius
        m = np.asarray(self.transformation.orientation, dtype=np.float64)
        for col in range(3):
            for row in range(3):
                c.orientation[3 * col + row] = m[row, col]
        for k in range(3):
            c.position[k] = float(self.transformation.position[k])
        return c


# ------------------------------------------------------------------------------ material.rs / texture.rs


@dataclass
class Scatter:
    kind: int
    param: float = 0.0

    NONE = None  # filled below
    Lambert = None

    @staticmethod
    def Metal(fuzziness: float) -> "Scatter":
        return Scatter(A.SCATTER_METAL, float(fuzziness))

    @staticmethod
    def Dielectric(refraction_index: float) -> "Scatter":
        return Scatter(A.SCATTER_DIELECTRIC, float(refraction_index))


Scatter.NONE = Scatter(A.SCATTER_NONE)
Scatter.Lambert = Scatter(A.SCATTER_LAMBERT)


@dataclass
class Absorb:
    kind: int
    color: np.ndarray = field(default_factory=lambda: np.zeros(3))
    texture: int = 0

    BlackBody = None
    WhiteBody = None

    @staticmethod
    def Albedo(color) -> "Absorb":
        return Absorb(A.ABSORB_ALBEDO, _vec3(color))

    @staticmethod
    def AlbedoMap(texture_id: int) -> "Absorb":
        return Absorb(A.ABSORB_ALBEDO_MAP, np.zeros(3), int(texture_id))


Absorb.BlackBody = Absorb(A.ABSORB_BLACKBODY)
Absorb.WhiteBody = Absorb(A.ABSORB_WHITEBODY)


@dataclass
class Emit:
    kind: int
    color: np.ndarray = field(default_factory=lambda: np.zeros(3))
    texture: int = 0

    NONE = None
    DebugNormals = None
    SkyGradient = None

    @staticmethod
    def Color(color) -> "Emit":
        return Emit(A.EMIT_COLOR, _vec3(color))

    @staticmethod
    def SkySphere(texture_id: int) -> "Emit":
        return Emit(A.EMIT_SKY_SPHERE, np.zeros(3), int(texture_id))

    def to_c(self) -> A.Emit:
        e = A.Emit()
        e.kind, e.texture = self.kind, self.texture
        for k in range(3):
            e.rgb[k] = float(self.color[k])
        return e


Emit.NONE = Emit(A.EMIT_NONE)
Emit.DebugNormals = Emit(A.EMIT_DEBUG_NORMALS)
Emit.SkyGradient = Emit(A.EMIT_SKY_GRADIENT)


@dataclass
class Material:
    """material.rs:86-100"""

    scatter: Scatter
    absorb: Absorb
    emit: Emit

    @staticmethod
    def new(scatter: Scatter, absorb: Absorb, emit: Emit) -> "Material":
        return Material(scatter, absorb, emit)


@dataclass
class Texture:
    """texture.rs:10-18"""

    kind: int
    color: np.ndarray = field(default_factory=lambda: np.zeros(3))
    image: Optional[np.ndarray] = None  # [h, w, 4] uint8, row 0 = bottom
    odd: int = 0
    even: int = 0
    seed: int = 0

    Missing = None
    DebugUVs = None

    @staticmethod
    def Solid(color) -> "Texture":
        return Texture(A.TEXTURE_SOLID, _vec3(color))

    @staticmethod
    def Image(image: np.ndarray) -> "Texture":
        return Texture(A.TEXTURE_IMAGE, image=np.ascontiguousarray(image, dtype=np.uint8))

    @staticmethod
    def Checker(odd: int, even: int) -> "Texture":
        return Texture(A.TEXTURE_CHECKER, odd=int(odd), even=int(even))

    @staticmethod
    def Noise(seed: int) -> "Texture":
        return Texture(A.TEXTURE_NOISE, seed=int(seed))

    @staticmethod
    def Perlin(seed: int) -> "Texture":
        return Texture(A.TEXTURE_PERLIN, seed=int(seed))


Texture.Missing = Texture(A.TEXTURE_MISSING)
Texture.DebugUVs = Texture(A.TEXTURE_DEBUG_UVS)


# ------------------------------------------------------------------------------ hittable.rs ------


class Hittable:
    """hittable.rs:10-15. Primitive lists are numpy arrays of HITTABLE_DTYPE so that multi-million
    triangle scenes marshal without Python objects."""

    @staticmethod
    def Sphere(center, radius: float, material: int) -> np.ndarray:
        h = np.zeros(1, dtype=A.HITTABLE_DTYPE)
        h["kind"], h["material"], h["center"], h["radius"] = A.HITTABLE_SPHERE, material, _vec3(center), radius
        return h

    @staticmethod
    def Triangle(triangle: int, mesh: int) -> np.ndarray:
        h = np.zeros(1, dtype=A.HITTABLE_DTYPE)
        h["kind"], h["mesh"], h["triangle"] = A.HITTABLE_TRIANGLE, mesh, triangle
        return h

    @staticmethod
    def triangles_of(mesh: Mesh, mesh_id: int) -> np.ndarray:
        """`bunny.iter_triangles().map(|tid| Hittable::Triangle{triangle: tid, mesh})` (example_scenes.rs:322-324)"""
        tids = mesh.iter_triangles()
        h = np.zeros(len(tids), dtype=A.HITTABLE_DTYPE)
        h["kind"], h["mesh"], h["triangle"] = A.HITTABLE_TRIANGLE, mesh_id, tids
        return h

    @staticmethod
    def concat(parts: Sequence[np.ndarray]) -> np.ndarray:
        return np.concatenate(list(parts)) if len(parts) else np.zeros(0, dtype=A.HITTABLE_DTYPE)


class NestedPool:
    """Items of nested containers (`Hittable::List(vec)` / `Hittable::Bvh(Bvh::new(vec))` used as an item of another
    container, hittable.rs:13-14). `List(items)` / `Bvh(items)` store the items in the pool and return the one-element
    hittable that names them; hand `pool.array()` to ExampleScene(nested=...)."""

    def __init__(self):
        self._parts: List[np.ndarray] = []
        self._n = 0

    def _add(self, kind: int, items: np.ndarray) -> np.ndarray:
        items = np.ascontiguousarray(items, dtype=A.HITTABLE_DTYPE)
        h = np.zeros(1, dtype=A.HITTABLE_DTYPE)
        h["kind"], h["mesh"], h["triangle"] = kind, self._n, len(items)
        self._parts.append(items)
        self._n += len(items)
        return h

    def List(self, items: np.ndarray) -> np.ndarray:
        return self._add(A.HITTABLE_LIST, items)

    def Bvh(self, items: np.ndarray) -> np.ndarray:
        return self._add(A.HITTABLE_BVH, items)

    def array(self) -> np.ndarray:
        return Hittable.concat(self._parts)


@dataclass
class SceneData:
    """render.rs:10-14"""

    material_table: List[Material]
    texture_table: List[Texture]
    mesh_table: List[Mesh]


@dataclass
class ExampleScene:
    """example_scenes.rs:14-19. root = ("bvh" | "list", hittables)"""

    camera: Camera
    scene_data: SceneData
    root_kind: str
    hittables: np.ndarray
    background: Emit
    nested: Optional[np.ndarray] = None  # items of nested List / Bvh hittables (NestedPool.array())


def build_desc(scene: ExampleScene):
    """Marshal an ExampleScene into an rtp_scene_desc. Returns (desc, keepalive)."""
    keep = []
    sd = scene.scene_data
    meshes = (A.Mesh * max(len(sd.mesh_table), 1))()
    for i, m in enumerate(sd.mesh_table):
        v = np.ascontiguousarray(m.vertices, dtype=A.VERTEX_DTYPE)
        ix = np.ascontiguousarray(m.indices, dtype=np.uint32)
        keep += [v, ix]
        meshes[i] = A.Mesh(v.ctypes.data, ix.ctypes.data, len(v), len(ix), m.material, 0)
    mats = (A.Material * max(len(sd.material_table), 1))()
    for i, m in enumerate(sd.material_table):
        c = A.Material()
        c.scatter, c.scatter_param = m.scatter.kind, m.scatter.param
        c.absorb, c.absorb_texture = m.absorb.kind, m.absorb.texture
        for k in range(3):
            c.absorb_rgb[k] = float(m.absorb.color[k])
        c.emit = m.emit.to_c()
        mats[i] = c
    texs = (A.Texture * max(len(sd.texture_table), 1))()
    for i, t in enumerate(sd.texture_table):
        c = A.Texture()
        c.kind, c.odd, c.even, c.seed = t.kind, t.odd, t.even, t.seed
        for k in range(3):
            c.rgb[k] = float(t.color[k])
        if t.kind == A.TEXTURE_IMAGE:
            img = np.ascontiguousarray(t.image, dtype=np.uint8)
            keep.append(img)
            c.height, c.width = img.shape[0], img.shape[1]
            c.rgba = img.ctypes.data
        texs[i] = c
    hit = np.ascontiguousarray(scene.hittables, dtype=A.HITTABLE_DTYPE)
    nested = np.ascontiguousarray(scene.nested if scene.nested is not None else np.zeros(0, dtype=A.HITTABLE_DTYPE), dtype=A.HITTABLE_DTYPE)
    keep += [meshes, mats, texs, hit, nested]
    d = A.SceneDesc()
    d.abi_version = A.ABI_VERSION
    d.root_kind = {"bvh": A.ROOT_BVH, "list": A.ROOT_LIST}[scene.root_kind]
    d.meshes = C.cast(meshes, C.POINTER(A.Mesh))
    d.hittables = hit.ctypes.data if len(hit) else None
    d.materials = C.cast(mats, C.POINTER(A.Material))
    d.textures = C.cast(texs, C.POINTER(A.Texture))
    d.n_meshes, d.n_hittables = len(sd.mesh_table), len(hit)
    d.n_materials, d.n_textures = len(sd.material_table), len(sd.texture_table)
    d.background = scene.background.to_c()
    d.nested = nested.ctypes.data if len(nested) else None
    d.n_nested = len(nested)
    return d, keep


def render_params(width, height, num_samples, max_bounce=8, seed=1, sample_begin=0, sample_end=None, tile=None, flags=0,
                  rows=None, device_mask=0) -> A.RenderParams:
    """rows = (row_offset, row_stride): only every row_stride-th row of the tile rectangle, starting at row_offset"""
    p = A.RenderParams()
    if rows is not None:
        p.row_offset, p.row_stride = rows
    p.device_mask = device_mask
    p.width, p.height, p.num_samples, p.max_bounce, p.seed = width, height, num_samples, max_bounce, seed
    p.sample_begin = sample_begin
    p.sample_end = num_samples if sample_end is None else sample_end
    if tile is not None:
        p.tile_x, p.tile_y, p.tile_w, p.tile_h = tile
    p.flags = flags
    return p


def adaptive_params(min_samples, max_samples, batch, abs_tol=0.0, rel_tol=0.01) -> A.AdaptiveParams:
    """the stop rule of rtp_render_adaptive (include/rtp.h)"""
    a = A.AdaptiveParams()
    a.min_samples, a.max_samples, a.batch, a.abs_tol, a.rel_tol = min_samples, max_samples, batch, abs_tol, rel_tol
    return a


# ------------------------------------------------------------------------------ device scene -----


def init(device: int = 0) -> None:
    lib = A.load()
    _check(lib, lib.rtp_init(device))


def device_count() -> int:
    lib = A.load()
    n = C.c_int(0)
    rc = lib.rtp_device_count(C.byref(n))
    return n.value if rc == A.OK else 0


def rng_draws(seed: int, index_lo: int, index_hi: int, stream: int, first: int, n: int) -> np.ndarray:
    lib = A.load()
    out = np.empty(n, dtype=np.float64)
    _check(lib, lib.rtp_rng_draws(seed, index_lo, index_hi, stream, first, n, A.ptr(out)))
    return out


def bvh_build_order(scene: ExampleScene):
    """`Bvh::new` on the host only (bvh.rs:70-91): (leaf ids in DFS order, SceneInfo). No device needed."""
    lib = A.load()
    desc, keep = build_desc(scene)
    info = A.SceneInfo()
    _check(lib, lib.rtp_bvh_build_order(C.byref(desc), None, 0, C.byref(info)))  # n_leaves: primitives after nested containers are flattened
    out = np.zeros(max(info.n_leaves, 1), dtype=np.uint32)
    _check(lib, lib.rtp_bvh_build_order(C.byref(desc), A.ptr(out), len(out), C.byref(info)))
    return out[: info.n_leaves], info


def bvh_culled_set(scene: ExampleScene):
    """rtp_bvh_culled_set, host only: (culled-set box as float32 [min xyz, max xyz], leaves of the order-free tree, big ones among them)"""
    lib = A.load()
    desc, keep = build_desc(scene)
    box = (C.c_float * 6)()
    leaves, big = C.c_uint32(0), C.c_uint32(0)
    _check(lib, lib.rtp_bvh_culled_set(C.byref(desc), box, C.byref(leaves), C.byref(big)))
    return np.array(box[:], dtype=np.float32), leaves.value, big.value


class PinnedBuffer:
    """Page-locked host array from rtp_host_alloc, exposed as a numpy array."""

    def __init__(self, shape, dtype):
        lib = A.load()
        self._lib = lib
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        p = C.c_void_p()
        _check(lib, lib.rtp_host_alloc(n, C.byref(p)))
        self._ptr = p
        buf = (C.c_char * max(n, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self._ptr:
            self.array = None
            self._lib.rtp_host_free(self._ptr)
            self._ptr = None


class Scene:
    """Device-resident scene: the replacement for `ExampleScene.root` + `scene_data` + `background`."""

    def __init__(self, scene: ExampleScene, device_mask: int = 0):
        """device_mask != 0: replicate the scene on those CUDA devices (rtp_scene_create_multi); render() / hit() then fan out"""
        self._lib = A.load()
        desc, keep = build_desc(scene)
        h = C.c_void_p()
        if device_mask:
            _check(self._lib, self._lib.rtp_scene_create_multi(C.byref(desc), device_mask, C.byref(h)))
        else:
            _check(self._lib, self._lib.rtp_scene_create(C.byref(desc), C.byref(h)))
        del keep
        self._h = h
        self.camera = scene.camera

    def close(self):
        if getattr(self, "_h", None):
            self._lib.rtp_scene_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def handle(self):
        return self._h

    def digest(self):
        """structural digests of the device-resident build (rtp_scene_digest): equal for equal trees, whatever built them"""
        out = (C.c_uint64 * 4)()
        _check(self._lib, self._lib.rtp_scene_digest(self._h, out))
        return tuple(int(x) for x in out)

    def any_tables(self) -> A.AnyTables:
        """the any-order walk's scene tables (rtp_scene_any_tables): big primitives, slack constants, scene magnitude, culled-set box"""
        t = A.AnyTables()
        _check(self._lib, self._lib.rtp_scene_any_tables(self._h, C.byref(t)))
        return t

    def devices(self) -> int:
        """bit d set = the scene holds a replica on CUDA device d"""
        m = C.c_uint32(0)
        _check(self._lib, self._lib.rtp_scene_devices(self._h, C.byref(m)))
        return m.value

    def info(self) -> A.SceneInfo:
        i = A.SceneInfo()
        _check(self._lib, self._lib.rtp_scene_get_info(self._h, C.byref(i)))
        return i

    def leaf_order(self) -> np.ndarray:
        n = self.info().n_leaves
        out = np.zeros(n, dtype=np.uint32)
        _check(self._lib, self._lib.rtp_scene_leaf_order(self._h, A.ptr(out), n))
        return out

    # -- batched Hittable::hit (bvh.rs:121-124 / hittable.rs:110-120) --
    def hit(self, rays: np.ndarray, out: Optional[np.ndarray] = None, stats: bool = False):
        rays = _as_rays(rays)
        hits = out if out is not None else np.empty(len(rays), dtype=A.HIT_DTYPE)
        st = A.Stats()
        _check(self._lib, self._lib.rtp_trace_closest(self._h, A.ptr(rays), len(rays), A.ptr(hits), C.byref(st) if stats else None))
        return (hits, st) if stats else hits

    def hit_camera(self, camera: Camera, width: int, height: int, out: Optional[np.ndarray] = None, stats: bool = False):
        """main.rs:67-77 at pixel centres: Camera::shoot + Hittable::hit per pixel, rays generated on the device (rtp_trace_camera)"""
        hits = out if out is not None else np.empty(width * height, dtype=A.HIT_DTYPE)
        st = A.Stats()
        cc = camera.to_c()
        _check(self._lib, self._lib.rtp_trace_camera(self._h, C.byref(cc), width, height, A.ptr(hits), C.byref(st) if stats else None))
        return (hits, st) if stats else hits

    def hit_full(self, rays: np.ndarray) -> np.ndarray:
        rays = _as_rays(rays)
        hits = np.empty(len(rays), dtype=A.HIT_FULL_DTYPE)
        _check(self._lib, self._lib.rtp_trace_closest_full(self._h, A.ptr(rays), len(rays), A.ptr(hits), None))
        return hits

    def hit_device(self, d_rays: int, n: int, d_hits: int, stream: int = 0) -> None:
        _check(self._lib, self._lib.rtp_trace_closest_device(self._h, d_rays, n, d_hits, stream))

    def hit_device_counted(self, d_rays: int, n: int, d_hits: int) -> A.Stats:
        st = A.Stats()
        _check(self._lib, self._lib.rtp_trace_closest_device_counted(self._h, d_rays, n, d_hits, C.byref(st)))
        return st

    # -- scene.hit(ray).is_some() (hittable.rs:18-25, bvh.rs:121-124): does the ray hit anything in [t_min, t_max] --
    def occluded(self, rays: np.ndarray, out: Optional[np.ndarray] = None, stats: bool = False):
        """bool array, one entry per ray: equal to hit(rays)["leaf"] != MISS; the walk stops at the first accepted leaf"""
        rays = _as_rays(rays)
        occ = out if out is not None else np.empty(len(rays), dtype=np.bool_)
        assert occ.dtype == np.bool_ and occ.flags.c_contiguous and len(occ) >= len(rays), "out must be a contiguous bool array"
        st = A.Stats()
        _check(self._lib, self._lib.rtp_trace_occluded(self._h, A.ptr(rays), len(rays), A.ptr(occ), C.byref(st) if stats else None))
        return (occ, st) if stats else occ

    def occluded_device(self, d_rays: int, n: int, d_out: int, stream: int = 0) -> None:
        """d_out: n bytes of device memory, 1 = occluded, 0 = not"""
        _check(self._lib, self._lib.rtp_trace_occluded_device(self._h, d_rays, n, d_out, stream))

    def occluded_device_counted(self, d_rays: int, n: int, d_out: int) -> A.Stats:
        st = A.Stats()
        _check(self._lib, self._lib.rtp_trace_occluded_device_counted(self._h, d_rays, n, d_out, C.byref(st)))
        return st

    # -- main.rs:61-92 --
    def render(self, width: int, height: int, num_samples: int, max_bounce: int = 8, seed: int = 1, camera: Optional[Camera] = None,
               sample_range=None, tile=None, flags: int = 0, out=None, foreground: bool = True, rows=None, device_mask: int = 0):
        """out: an [h, w, 3] f64 array, or a pair (rgb [h, w, 3], foreground [h, w] or None) of caller buffers (e.g. pinned)"""
        cam = camera or self.camera
        cam = Camera(width / height, cam.fov, cam.focal_dist, cam.lens_radius, cam.transformation)  # main.rs:22 overrides the aspect
        p = render_params(width, height, num_samples, max_bounce, seed,
                          sample_range[0] if sample_range else 0, sample_range[1] if sample_range else None, tile, flags, rows, device_mask)
        if isinstance(out, tuple):
            rgbf, fg = out
        else:
            rgbf = out if out is not None else np.zeros((height, width, 3), dtype=np.float64)
            fg = np.zeros((height, width), dtype=np.float64) if foreground else None
        st = A.Stats()
        cc = cam.to_c()
        _check(self._lib, self._lib.rtp_render(self._h, C.byref(cc), C.byref(p), A.ptr(rgbf), A.ptr(fg) if fg is not None else None, C.byref(st)))
        return rgbf, fg, st

    def render_aov(self, width: int, height: int, num_samples: int, max_bounce: int = 8, seed: int = 1, camera: Optional[Camera] = None,
                   sample_range=None, tile=None, flags: int = 0, out=None, foreground: bool = True, rows=None, device_mask: int = 0):
        """render() plus each pixel's mean first-vertex albedo and normal, the guide buffers of a denoiser (rtp_render_aov). Returns
        (rgb [h, w, 3], foreground [h, w], albedo [h, w, 3], normal [h, w, 3], stats); rgb and foreground are render()'s bits.
        out: a 4-tuple (rgb, foreground, albedo, normal) of caller buffers, any but rgb may be None"""
        cam = camera or self.camera
        cam = Camera(width / height, cam.fov, cam.focal_dist, cam.lens_radius, cam.transformation)  # main.rs:22 overrides the aspect
        p = render_params(width, height, num_samples, max_bounce, seed,
                          sample_range[0] if sample_range else 0, sample_range[1] if sample_range else None, tile, flags, rows, device_mask)
        if out is not None:
            rgbf, fg, albedo, normal = out
        else:
            rgbf = np.zeros((height, width, 3), dtype=np.float64)
            fg = np.zeros((height, width), dtype=np.float64) if foreground else None
            albedo = np.zeros((height, width, 3), dtype=np.float64)
            normal = np.zeros((height, width, 3), dtype=np.float64)
        st = A.Stats()
        cc = cam.to_c()
        opt = lambda a: A.ptr(a) if a is not None else None  # noqa: E731
        _check(self._lib, self._lib.rtp_render_aov(self._h, C.byref(cc), C.byref(p), A.ptr(rgbf), opt(fg), opt(albedo), opt(normal), C.byref(st)))
        return rgbf, fg, albedo, normal, st

    def render_aov_device(self, params: A.RenderParams, camera: Camera, d_rgb: int, d_fg: int = 0, d_albedo: int = 0, d_normal: int = 0,
                          stream: int = 0, stats: bool = False):
        """rtp_render_aov_device: device buffers on the scene's first device; asynchronous on `stream` unless stats"""
        st = A.Stats()
        cc = camera.to_c()
        _check(self._lib, self._lib.rtp_render_aov_device(self._h, C.byref(cc), C.byref(params), d_rgb, d_fg or None, d_albedo or None,
                                                          d_normal or None, C.byref(st) if stats else None, stream or None))
        return st

    def render_srgb8(self, width: int, height: int, num_samples: int, max_bounce: int = 8, seed: int = 1, camera: Optional[Camera] = None,
                     tile=None, transparent_background: bool = False, out: Optional[np.ndarray] = None, rows=None, device_mask: int = 0):
        """main.rs:61-122: render + tile merge + to_srgb_u8 with the output stage on the device; [height, width, 4] uint8, ready for tga.save"""
        cam = camera or self.camera
        cam = Camera(width / height, cam.fov, cam.focal_dist, cam.lens_radius, cam.transformation)
        p = render_params(width, height, num_samples, max_bounce, seed, 0, None, tile, A.RENDER_TRANSPARENT if transparent_background else 0, rows, device_mask)
        rgba = out if out is not None else np.zeros((height, width, 4), dtype=np.uint8)
        st = A.Stats()
        cc = cam.to_c()
        _check(self._lib, self._lib.rtp_render_srgb8(self._h, C.byref(cc), C.byref(p), A.ptr(rgba), C.byref(st)))
        return rgba, st

    def render_adaptive(self, width: int, height: int, min_samples: int, max_samples: int, batch: int, abs_tol: float = 0.0, rel_tol: float = 0.01,
                        max_bounce: int = 8, seed: int = 1, camera: Optional[Camera] = None, tile=None, rows=None, raw_sums: bool = False,
                        device_mask: int = 0, out=None, counters: bool = False):
        """render() that stops each pixel once the standard error of its mean luminance is at most abs_tol + rel_tol * |mean|
        (rtp_render_adaptive). Returns (rgb [h, w, 3], foreground [h, w], samples [h, w] uint32, stats): every pixel equals
        render(samples[p], sample_range=(0, samples[p])) at p. out: a triple (rgb, foreground or None, samples or None) of caller
        buffers; pixels outside the tile and rows are left as they are."""
        cam = camera or self.camera
        cam = Camera(width / height, cam.fov, cam.focal_dist, cam.lens_radius, cam.transformation)  # main.rs:22 overrides the aspect
        p = render_params(width, height, 0, max_bounce, seed, 0, 0, tile,
                          (A.RENDER_RAW_SUMS if raw_sums else 0) | (A.RENDER_COUNTERS if counters else 0), rows, device_mask)
        a = adaptive_params(min_samples, max_samples, batch, abs_tol, rel_tol)
        if out is not None:
            rgbf, fg, samples = out
        else:
            rgbf = np.zeros((height, width, 3), dtype=np.float64)
            fg = np.zeros((height, width), dtype=np.float64)
            samples = np.zeros((height, width), dtype=np.uint32)
        st = A.Stats()
        cc = cam.to_c()
        _check(self._lib, self._lib.rtp_render_adaptive(self._h, C.byref(cc), C.byref(p), C.byref(a), A.ptr(rgbf),
                                                        A.ptr(fg) if fg is not None else None, A.ptr(samples) if samples is not None else None,
                                                        C.byref(st)))
        return rgbf, fg, samples, st

    def render_adaptive_device(self, params: A.RenderParams, adaptive: A.AdaptiveParams, camera: Camera, d_rgb: int, d_fg: int = 0,
                               d_samples: int = 0, stream: int = 0, stats: bool = False):
        """rtp_render_adaptive_device: device buffers on the scene's first device; returns when the frame is done"""
        st = A.Stats()
        cc = camera.to_c()
        _check(self._lib, self._lib.rtp_render_adaptive_device(self._h, C.byref(cc), C.byref(params), C.byref(adaptive), d_rgb, d_fg or None,
                                                               d_samples or None, C.byref(st) if stats else None, stream or None))
        return st

    def render_device(self, params: A.RenderParams, camera: Camera, d_rgb: int, d_fg: int = 0, stream: int = 0, stats: bool = False):
        st = A.Stats()
        cc = camera.to_c()
        _check(self._lib, self._lib.rtp_render_device(self._h, C.byref(cc), C.byref(params), d_rgb, d_fg or None, C.byref(st) if stats else None, stream or None))
        return st


def _as_rays(rays: np.ndarray) -> np.ndarray:
    if rays.dtype == A.RAY_DTYPE:
        return np.ascontiguousarray(rays)
    a = np.ascontiguousarray(rays, dtype=np.float64)
    assert a.ndim == 2 and a.shape[1] == 8, "rays must be RAY_DTYPE or float64 [n, 8]"
    return a.view(A.RAY_DTYPE).reshape(-1)


def camera_rays(camera: Camera, width: int, height: int) -> np.ndarray:
    """Pixel-centre primary rays, i fastest (render.rs:32-52 with lens 0)."""
    lib = A.load()
    out = np.empty(width * height, dtype=A.RAY_DTYPE)
    cc = camera.to_c()
    _check(lib, lib.rtp_camera_rays(C.byref(cc), width, height, A.ptr(out)))
    return out


def camera_rays_device(camera: Camera, width: int, height: int, d_rays: int, stream: int = 0) -> None:
    lib = A.load()
    cc = camera.to_c()
    _check(lib, lib.rtp_camera_rays_device(C.byref(cc), width, height, d_rays, stream or None))
