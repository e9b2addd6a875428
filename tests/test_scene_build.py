"""The device scene build (rtp_build.cu device_build_scene) against the host build (rtp_host.cpp flatten_scene) and the oracle,
beyond triangle meshes: sphere fields, several outsized primitives with tied extents, clusters of identical triangles deep enough
for the SAH's median fallback, scenes whose median extent is 0, sizes around the device-build threshold and scene magnitudes on
both sides of the f32-culling limit. Each scene is built three ways (RTP_DEVICE_BUILD=1, RTP_DEVICE_BUILD=0, the oracle) and must
give the same leaf order, trees (rtp_scene_digest, order-free tree included), plan (rtp_scene_info), any-order tables (equal to a
numpy restatement of prepare_any_order), hits and image. Also: the irregular-box fallback, validation errors (the same message,
naming the smallest failing index, from both builds) and device-built arrays replicated on a second device."""
import contextlib
import os

import numpy as np
import pytest

import oracle
from rtp_b200 import _abi as A
from rtp_b200 import api, assets, scenes
from rtp_b200.api import Absorb, Camera, Emit, Hittable, Material, Mesh, Scatter, SceneData, Transformation, rgb
from test_any_setup_cull import big_leaves, f32_down, f32_up, leaf_boxes
from test_gpu_parity import IMG_FRAC, IMG_RMSE, image_report

MISS = A.MISS
W, H = 96, 54


@contextlib.contextmanager
def env(**kv):
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: str(v) for k, v in kv.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


# ---------------------------------------------------------------------------------------------------------------------------------
# scenes

MATERIALS = [
    Material.new(Scatter.Lambert, Absorb.Albedo(rgb(0.8, 0.3, 0.3)), Emit.NONE),
    Material.new(Scatter.Metal(0.1), Absorb.Albedo(rgb(0.8, 0.8, 0.6)), Emit.NONE),
    Material.new(Scatter.Dielectric(1.5), Absorb.WhiteBody, Emit.NONE),
    Material.new(Scatter.Lambert, Absorb.Albedo(rgb(0.5, 0.5, 0.5)), Emit.NONE),  # ground
]


def _camera(position, target):
    return Camera(1.0, np.pi / 4, 1.0, 0.0, Transformation.lookat(position, target, [0.0, 1.0, 0.0]))


def sphere_field(n, seed=7, ground=True):
    """n leaves: a seeded grid of spheres of varied radii on the ground sphere (r = 1000), which is the last leaf"""
    rng = np.random.default_rng(seed)
    m = n - 1 if ground else n
    side = int(np.ceil(np.sqrt(max(m, 1))))
    k = np.arange(m)
    r = rng.uniform(0.05, 0.24, m)
    h = np.zeros(m, dtype=A.HITTABLE_DTYPE)
    h["kind"], h["material"], h["radius"] = A.HITTABLE_SPHERE, k % 3, r
    h["center"][:, 0] = (k % side - side / 2) * 0.5 + rng.uniform(-0.02, 0.02, m)
    h["center"][:, 1] = r
    h["center"][:, 2] = (k // side - side / 2) * 0.5 + rng.uniform(-0.02, 0.02, m)
    parts = [h] + ([Hittable.Sphere([0.0, -1000.0, -1.0], 1000.0, 3)] if ground else [])
    span = side * 0.5
    cam = _camera([-0.3 * span - 2.0, 0.25 * span + 2.0, 0.6 * span + 2.0], [0.0, 0.0, 0.0])
    return api.ExampleScene(cam, SceneData(list(MATERIALS), [], []), "bvh", Hittable.concat(parts), Emit.SkyGradient)


def field_with_outsized():
    """bunny_field(8, 4) plus 12 spheres of radius 40 and a floor of 2 triangles of equal extent: 15 outsized primitives (with
    the ground sphere), 5 of the 8 big ones picked among 12 exact ties"""
    sc = scenes.bunny_field(8, 4)
    floor = Mesh.from_arrays([[-150.0, -0.001, -150.0], [150.0, -0.001, -150.0], [150.0, -0.001, 150.0], [-150.0, -0.001, 150.0]],
                             indices=[0, 1, 2, 0, 2, 3], material=len(sc.scene_data.material_table))
    sc.scene_data.material_table.append(MATERIALS[0])
    sc.scene_data.mesh_table.append(floor)
    ring = [Hittable.Sphere([100.0 * np.cos(a), 40.0, 100.0 * np.sin(a)], 40.0, k % 4) for k, a in enumerate(np.linspace(0, 2 * np.pi, 12, endpoint=False))]
    sc.hittables = Hittable.concat([sc.hittables] + ring + [Hittable.triangles_of(floor, len(sc.scene_data.mesh_table) - 1)])
    return sc


def cluster(copies):
    """`copies` of one bunny triangle: every cut of a range costs the same up to rounding, so the SAH build cuts where rounding
    puts the first minimum and the tree grows as deep as the median fallback past 192 levels allows. 4-wide depth: 58 for 300
    copies (in-order walk, f32 culling), 65 for 1,000, 105 for 70,000 (above 96: exact f64 walk)"""
    mesh = assets.bunny()
    p = mesh.vertices["position"][mesh.indices[30:33]]
    centre, size = p.mean(axis=0), (p.max(axis=0) - p.min(axis=0)).max()
    cam = _camera(centre + np.array([0.0, 0.0, 8.0 * size]), centre)
    return api.ExampleScene(cam, SceneData(list(MATERIALS), [], [mesh]), "bvh", np.repeat(Hittable.Triangle(30, 0), copies), Emit.SkyGradient)


def bunny_with_cluster(copies):
    sc = scenes.bunny_lambert()
    sc.hittables = Hittable.concat([sc.hittables, np.repeat(sc.hittables[:1], copies)])
    return sc


def zero_extent():
    """more than half of the leaves are points (zero-radius spheres, triangles with three equal vertices): median extent 0, so
    every primitive of non-zero extent is outsized"""
    rng = np.random.default_rng(11)
    base = sphere_field(3001, seed=3)  # 3,000 spheres + ground
    pts = rng.uniform(-10, 10, (3000, 3))
    pts[:, 1] = np.abs(pts[:, 1])
    z = np.zeros(3000, dtype=A.HITTABLE_DTYPE)
    z["kind"], z["material"], z["center"], z["radius"] = A.HITTABLE_SPHERE, 1, pts, 0.0
    pos = np.repeat(rng.uniform(-10, 10, (3000, 3)), 3, axis=0)
    mesh = Mesh.from_arrays(pos, indices=np.arange(9000), material=0)
    base.scene_data.mesh_table.append(mesh)
    base.hittables = Hittable.concat([base.hittables, z, Hittable.triangles_of(mesh, 0)])
    return base


def translated_field(mag):
    """bunny_field(4, 2) moved along x so that the largest |coordinate| of a leaf box (the ground sphere's +x face) is `mag`"""
    sc = scenes.bunny_field(4, 2)
    shift = mag - 1000.0
    for m in sc.scene_data.mesh_table:
        m.vertices = m.vertices.copy()
        m.vertices["position"][:, 0] += shift
    h = sc.hittables.copy()
    sph = h["kind"] == A.HITTABLE_SPHERE
    h["center"][sph, 0] += shift
    sc.hittables = h
    span = 8.0
    sc.camera = _camera([shift - 0.35 * span, 0.3 * span + 2.0, 0.75 * span + 2.0], [shift, 0.5, 0.0])
    return sc


SCENES = {
    "S1_more_balls": scenes.more_balls_optimized,
    "S2_sphere_field_70k": lambda: sphere_field(70001),
    "S3_field_outsized_ties": field_with_outsized,
    "S4_cluster_300": lambda: cluster(300),
    "S4_cluster_1000": lambda: cluster(1000),
    "S4_cluster_70000": lambda: cluster(70000),
    "S4_bunny_cluster_300": lambda: bunny_with_cluster(300),
    "S5_zero_extent": zero_extent,
    "S6_n2": lambda: sphere_field(2),
    "S6_n3": lambda: sphere_field(3),
    "S6_n65535": lambda: sphere_field(65535),
    "S6_n65536": lambda: sphere_field(65536),
    "S6_n65537": lambda: sphere_field(65537),
    "S6_n131071": lambda: sphere_field(131071),
    "S7_mag_below_1e15": lambda: translated_field(1e15 - 0.5),
    "S7_mag_above_1e15": lambda: translated_field(1e15 + 0.5),
}


def test_scene_magnitudes_straddle_the_f32_culling_limit():
    for name, below in (("S7_mag_below_1e15", True), ("S7_mag_above_1e15", False)):
        lo, hi = leaf_boxes(SCENES[name]())
        mag = np.maximum(np.abs(lo), np.abs(hi)).max()
        assert (mag <= 1e15) == below and abs(mag - 1e15) <= 1.0, (name, mag)


def test_outsized_primitives_outnumber_the_big_slots_with_ties():
    lo, hi = leaf_boxes(field_with_outsized())
    ext = (hi - lo).max(axis=1)
    cap = 16.0 * np.sort(ext)[len(ext) // 2]
    assert (ext > cap).sum() == 15 and len(big_leaves(lo, hi)) == 8
    assert (ext[big_leaves(lo, hi)] == 80.0).sum() == 5  # five of the twelve tied spheres
    lo, hi = leaf_boxes(zero_extent())
    assert np.sort((hi - lo).max(axis=1))[len(lo) // 2] == 0.0


# ---------------------------------------------------------------------------------------------------------------------------------
# numpy restatement of prepare_any_order (rtp_host.cpp)


def expected_tables(sc, order, eligible):
    lo, hi = leaf_boxes(sc)
    n = len(lo)
    slot = np.empty(n, dtype=np.int64)
    slot[order] = np.arange(n)
    mag = np.maximum(np.abs(lo), np.abs(hi)).max(axis=1)
    want = dict(n_big=0, big=[0] * 8, any_spheres=0, any_E=0.0, any_A=0.0, any_C=0.0, any_R=0.0, scene_mag=float(mag.max()),
                cull=[np.inf] * 3 + [-np.inf] * 3)
    if not eligible:
        return want
    ext = (hi - lo).max(axis=1)
    cap = 16.0 * np.sort(ext)[n // 2]
    over = np.flatnonzero(ext > cap)
    over = over[np.lexsort((slot[over], -ext[over]))][:8]  # extent descending, slot ascending
    kind = sc.hittables["kind"].astype(np.int64)
    small = np.ones(n, dtype=bool)
    small[over] = False
    tri, sph = small & (kind == A.HITTABLE_TRIANGLE), small & (kind == A.HITTABLE_SPHERE)
    grow = 1.0 + 1e-12
    want.update(n_big=len(over), big=[int(slot[b] | (kind[b] << 31)) for b in over] + [0] * (8 - len(over)),
                any_spheres=int(sph.any()), any_E=ext[tri].max(initial=0.0) * grow, any_A=mag[tri].max(initial=0.0) * grow,
                any_C=mag[sph].max(initial=0.0) * grow, any_R=(0.5 * ext[sph]).max(initial=0.0) * grow)
    if small.any():  # rtp_host.cpp round_out of the union of the boxes that are not big
        ulo, uhi = lo[small].min(axis=0), hi[small].max(axis=0)
        r = np.ldexp(np.maximum(np.abs(ulo), np.abs(uhi)), -21)
        want["cull"] = list(f32_down(ulo - r).astype(np.float64)) + list(f32_up(uhi + r).astype(np.float64))
    return want


def tables_of(g):
    t = g.any_tables()
    return dict(n_big=t.n_big, big=list(t.big), any_spheres=t.any_spheres, any_E=t.any_E, any_A=t.any_A, any_C=t.any_C, any_R=t.any_R,
                scene_mag=t.scene_mag, cull=[float(x) for x in t.cull])


# ---------------------------------------------------------------------------------------------------------------------------------
# rays


def rays_of(origin, direction, t_min=1e-3, t_max=np.inf):
    r = np.zeros(len(origin), dtype=A.RAY_DTYPE)
    r["origin"], r["direction"], r["t_min"], r["t_max"] = origin, direction, t_min, t_max
    return r


def probe_rays(sc, n_incoherent, seed=5):
    """the camera's primary rays, incoherent rays aimed at the box of the primitives that are not big, and axis-parallel rays
    along the faces of that box and of the boxes of sampled leaves"""
    lo, hi = leaf_boxes(sc)
    small = np.setdiff1d(np.arange(len(lo)), big_leaves(lo, hi))
    if len(small) == 0:
        small = np.arange(len(lo))
    blo, bhi = lo[small].min(axis=0), hi[small].max(axis=0)
    c = sc.camera
    primary = oracle.camera_rays(Camera(W / H, c.fov, c.focal_dist, 0.0, c.transformation), W, H)
    rng = np.random.default_rng(seed)
    centre, radius = 0.5 * (blo + bhi), max(1.5 * 0.5 * np.linalg.norm(bhi - blo), 1.0)
    u = rng.normal(size=(n_incoherent, 3))
    origin = centre + radius * u / np.linalg.norm(u, axis=1, keepdims=True)
    d = blo + rng.uniform(size=(n_incoherent, 3)) * (bhi - blo) - origin
    incoherent = rays_of(origin, d / np.linalg.norm(d, axis=1, keepdims=True))
    o, dirs = [], []
    sample = rng.choice(small, min(200, len(small)), replace=False)
    boxes = np.unique(np.vstack([np.hstack([blo, bhi]), np.hstack([lo[sample], hi[sample]])]), axis=0)  # a cluster's copies share one box
    for b_lo, b_hi in zip(boxes[:, :3], boxes[:, 3:]):
        far = 1.0 + (b_hi - b_lo).max()
        for a in range(3):
            b, cc = (a + 1) % 3, (a + 2) % 3
            for vb in (b_lo[b], b_hi[b], 0.5 * (b_lo[b] + b_hi[b])):
                for vc in (b_lo[cc], b_hi[cc], 0.5 * (b_lo[cc] + b_hi[cc])):
                    for s in (1.0, -1.0):
                        p = np.zeros(3)
                        p[a], p[b], p[cc] = (b_lo[a] - far) if s > 0 else (b_hi[a] + far), vb, vc
                        q = np.zeros(3)
                        q[a] = s
                        o.append(p), dirs.append(q)
    axis = rays_of(np.array(o), np.array(dirs))
    return np.concatenate([primary, incoherent, axis])


def retrace_rays(rays, hits):
    """rays that hit, traced again with t_max = t (the hit stays) and t_max = nextafter(t, 0)"""
    k = np.flatnonzero(hits["leaf"] != MISS)[:25000]
    a, b = rays[k].copy(), rays[k].copy()
    a["t_max"] = hits["t"][k]
    b["t_max"] = np.nextafter(hits["t"][k], 0.0)
    return np.concatenate([a, b])


def assert_hits_equal(got, want):
    assert (got["leaf"] == want["leaf"]).all(), np.flatnonzero(got["leaf"] != want["leaf"])[:10]
    assert (got["material"] == want["material"]).all()
    assert got["t"].tobytes() == want["t"].tobytes(), np.flatnonzero(got["t"] != want["t"])[:10]


def assert_full_equal(got, want, kind_of_leaf):
    assert_hits_equal(got, want)
    hit = want["leaf"] != MISS
    kind = np.full(len(want), -1)
    kind[hit] = kind_of_leaf[want["leaf"][hit]]
    tri, sph = kind == A.HITTABLE_TRIANGLE, kind == A.HITTABLE_SPHERE
    for f in ("position", "normal", "uv"):
        assert got[f][tri].tobytes() == want[f][tri].tobytes(), f
    for f in ("position", "normal"):
        assert got[f][sph].tobytes() == want[f][sph].tobytes(), f
    # sphere uv goes through atan2 / asin: CUDA and glibc may differ by an ulp or two (test_full_hit_record)
    assert np.allclose(got["uv"][sph], want["uv"][sph], rtol=0, atol=1e-14)


# ---------------------------------------------------------------------------------------------------------------------------------
# the three builds of one scene, shared by the tests of that scene


class Built:
    def __init__(self, name):
        self.name = name
        self.sc = SCENES[name]()
        with env(RTP_DEVICE_BUILD=1):
            self.dev = api.Scene(self.sc)
        with env(RTP_DEVICE_BUILD=0):
            self.host = api.Scene(self.sc)
        self.o = oracle.Scene(self.sc)
        n = len(self.sc.hittables)
        # every ray of a cluster tests every copy (their boxes are equal): fewer incoherent rays keep the oracle's share in seconds
        self.rays = probe_rays(self.sc, int(min(50000, 2e8 / n)))
        self.want = self.o.hit_full(self.rays)
        self.rays = np.concatenate([self.rays, retrace_rays(self.rays, self.want)])
        self.want = np.concatenate([self.want, self.o.hit_full(self.rays[len(self.want):])])

    def close(self):
        self.dev.close(); self.host.close(); self.o.close()


@pytest.fixture(scope="module", params=list(SCENES))
def built(request, gpu):
    b = Built(request.param)
    yield b
    b.close()


@pytest.mark.gpu
def test_same_build(built):
    order = built.o.leaf_order()
    assert (built.dev.leaf_order() == order).all() and (built.host.leaf_order() == order).all()
    assert built.dev.digest() == built.host.digest()
    idev, ihost, iorc = built.dev.info(), built.host.info(), built.o.info()
    for f in ("n_leaves", "n_nodes", "depth", "culling_depth", "any_order", "n_big", "free_tree_depth"):
        assert getattr(idev, f) == getattr(ihost, f), (f, getattr(idev, f), getattr(ihost, f))
    assert (idev.n_leaves, idev.n_nodes, idev.depth) == (iorc.n_leaves, iorc.n_nodes, iorc.depth)
    n = len(built.sc.hittables)
    # the host rule of the order-free tree (RTP_FREE_TREE unset): every any-order scene below 262,144 leaves has one
    if ihost.culling_depth <= 48 and ihost.n_big < n:
        assert idev.free_tree_depth > 0


@pytest.mark.gpu
def test_same_tables(built):
    tdev, thost = tables_of(built.dev), tables_of(built.host)
    assert tdev == thost
    info = built.host.info()
    want = expected_tables(built.sc, built.o.leaf_order(), eligible=info.culling_depth <= 48)
    assert tdev == want
    assert info.n_big == want["n_big"]


@pytest.mark.gpu
def test_same_hits(built):
    import torch

    rays, want = built.rays, built.want
    kind_of_leaf = built.sc.hittables["kind"].astype(np.int64)
    d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 8)).cuda()
    d_hits = torch.empty((len(rays), 2), dtype=torch.float64, device="cuda")
    for g in (built.dev, built.host):
        hits = g.hit(rays)
        assert_hits_equal(hits, want)
        assert_full_equal(g.hit_full(rays), want, kind_of_leaf)
        assert (g.occluded(rays) == (hits["leaf"] != MISS)).all()
        st = g.hit_device_counted(d_rays.data_ptr(), len(rays), d_hits.data_ptr())
        assert_hits_equal(d_hits.cpu().numpy().view(A.HIT_DTYPE).reshape(-1), want)
        assert st.conservative_violations == 0


@pytest.mark.gpu
def test_same_image(built):
    io, fo, _ = built.o.render(W, H, 2, max_bounce=8, seed=1)
    ig, fg, _ = built.dev.render(W, H, 2, max_bounce=8, seed=1)
    ih, fh, _ = built.host.render(W, H, 2, max_bounce=8, seed=1)
    rep = image_report(ig, io)
    assert rep["rmse"] <= IMG_RMSE and rep["differing"] <= max(1, IMG_FRAC * rep["pixels"]), rep
    assert (fg == fo).all()
    assert ig.tobytes() == ih.tobytes() and fg.tobytes() == fh.tobytes()


# ---------------------------------------------------------------------------------------------------------------------------------
# the irregular-box fallback and validation errors


@pytest.mark.gpu
def test_inverted_box_hands_the_scene_to_the_host_build(gpu):
    """a sphere of negative radius has an inverted box: the device build returns the scene to the host path, which keeps the
    reference topology and the in-order walk"""
    sc = sphere_field(70000)
    sc.hittables = sc.hittables.copy()
    sc.hittables["radius"][1234] = -0.2
    with env(RTP_DEVICE_BUILD=1):
        g = api.Scene(sc)
    with env(RTP_DEVICE_BUILD=0):
        gh = api.Scene(sc)
    o = oracle.Scene(sc)
    assert (g.leaf_order() == o.leaf_order()).all() and (gh.leaf_order() == o.leaf_order()).all()
    assert g.digest() == gh.digest()
    ig, ih = g.info(), gh.info()
    for f in ("n_leaves", "n_nodes", "depth", "culling_depth", "any_order", "n_big", "free_tree_depth"):
        assert getattr(ig, f) == getattr(ih, f), f
    assert ig.any_order == 0 and ig.n_big == 0
    assert tables_of(g) == tables_of(gh)
    rays = probe_rays(sc, 20000)
    want = o.hit(rays)
    assert_hits_equal(g.hit(rays), want)
    assert_hits_equal(gh.hit(rays), want)
    g.close(); gh.close(); o.close()


def bad_scene(n, faults):
    """sphere field of n leaves plus one small mesh; faults: {index: "nan" | "material" | "triangle"}"""
    sc = sphere_field(n)
    mesh = Mesh.from_arrays([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0]], indices=[0, 1, 2], material=0)
    sc.scene_data.mesh_table.append(mesh)
    h = sc.hittables.copy()
    for i, what in faults.items():
        if what == "nan":
            h["center"][i, 1] = np.nan
        elif what == "material":
            h["material"][i] = len(sc.scene_data.material_table)
        else:
            h[i] = Hittable.Triangle(3, 0)[0]  # the mesh has one triangle (ids 0..2 of its index array)
    sc.hittables = h
    return sc


MESSAGES = {"nan": "NaN bounding-box centroid in hittable {}", "material": "sphere material out of range", "triangle": "triangle id out of range"}

# Host validation of a scene of >= 262,144 hittables runs in contiguous chunks on the host cores. 9,000 lies at the end of the first
# chunk and 150,000 at the start of a later one for every worker count that divides 300,000 into chunks of >= 9,375 (1 to 32
# workers, 7 aside): the later chunk meets its fault first.
FAULTS = [
    (70000, {12345: "nan"}),
    (70000, {12345: "material"}),
    (70000, {12345: "triangle"}),
    (300000, {150000: "nan"}),
    (300000, {150000: "material"}),
    (300000, {150000: "triangle"}),
    (300000, {9000: "material", 150000: "nan"}),
    (300000, {9000: "nan", 150000: "material"}),
    (300000, {9000: "triangle", 150000: "nan"}),
]


def _fault_id(case):
    n, faults = case
    return f"{n}-" + "-".join(f"{w}@{i}" for i, w in sorted(faults.items()))


def expected_message(faults):
    i = min(faults)
    return MESSAGES[faults[i]].format(i)


@pytest.mark.parametrize("case", FAULTS, ids=_fault_id)
def test_host_validation_reports_the_smallest_failing_index(case):
    """host only (rtp_bvh_build_order): the error of the smallest failing index, whatever chunk of the parallel validation
    finds its fault first"""
    n, faults = case
    sc = bad_scene(n, faults)
    for _ in range(3):
        with pytest.raises(api.RtpError) as e:
            api.bvh_build_order(sc)
        assert e.value.code == A.ERR_INVALID and e.value.message == expected_message(faults)


@pytest.mark.gpu
@pytest.mark.parametrize("case", FAULTS, ids=_fault_id)
def test_both_builds_reject_the_same_hittable(gpu, case):
    n, faults = case
    sc = bad_scene(n, faults)
    for device_build in (1, 0):
        with env(RTP_DEVICE_BUILD=device_build):
            with pytest.raises(api.RtpError) as e:
                api.Scene(sc)
        assert e.value.code == A.ERR_INVALID and e.value.message == expected_message(faults), (device_build, e.value.message)
    with pytest.raises(oracle.OracleError):
        oracle.Scene(sc)
    # the library is still usable: a valid scene afterwards builds both ways and traces
    good = sphere_field(70000)
    rays = probe_rays(good, 2000)
    o = oracle.Scene(good)
    want = o.hit(rays)
    for device_build in (1, 0):
        with env(RTP_DEVICE_BUILD=device_build):
            with api.Scene(good) as g:
                assert_hits_equal(g.hit(rays), want)
    o.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# device-built arrays on two devices (device_scene_upload adopts them on the building device and copies them peer to peer)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["S2_sphere_field_70k", "S3_field_outsized_ties"])
@pytest.mark.parametrize("mask", [0b11, 0b10])
def test_device_built_scene_on_two_devices(gpu, name, mask):
    if api.device_count() < 2:
        pytest.skip("needs two GPUs")
    sc = SCENES[name]()
    rays = probe_rays(sc, 20000)
    with env(RTP_DEVICE_BUILD=1):
        one = api.Scene(sc)
        many = api.Scene(sc, device_mask=mask)  # bound to device 0 (the gpu fixture); 0b10 builds on device 1 alone
    assert many.devices() == mask
    assert one.digest() == many.digest()
    assert one.hit(rays).tobytes() == many.hit(rays).tobytes()
    assert one.hit_full(rays).tobytes() == many.hit_full(rays).tobytes()
    i1, f1, _ = one.render(W, H, 2, max_bounce=8, seed=1)
    i2, f2, _ = many.render(W, H, 2, max_bounce=8, seed=1)
    assert i1.tobytes() == i2.tobytes() and f1.tobytes() == f2.tobytes()
    one.close(); many.close()
