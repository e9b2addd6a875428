"""Set-up cull of the any-order walk (DESIGN.md §4b "Big primitives"): after its big-primitive tests a ray tests the culled-set
box, the union of the boxes of every primitive that is not big, against its window; rejected, it is done without a walk. The
order-free tree holds only the primitives that are not big. CPU half: the host tables and an f32 restatement of the decision that
must never reject a ray whose oracle hit is a leaf inside the box. GPU half: bit parity with the cull on and off, and fewer nodes."""
import numpy as np
import pytest

import oracle
from rtp_b200 import _abi as A
from rtp_b200 import api, scenes

SCENES = ["bunny_lambert", "demo", "more_balls_optimized"]


def leaf_boxes(sc):
    """exact f64 box of every hittable of a flat scene, indexed by LeafId (hittable.rs:124-140)"""
    h = sc.hittables
    lo, hi = np.empty((len(h), 3)), np.empty((len(h), 3))
    sph = h["kind"] == A.HITTABLE_SPHERE
    lo[sph] = h["center"][sph] - h["radius"][sph, None]
    hi[sph] = h["center"][sph] + h["radius"][sph, None]
    for k in np.flatnonzero(~sph):
        m = sc.scene_data.mesh_table[h["mesh"][k]]
        p = m.vertices["position"][m.indices[h["triangle"][k]:h["triangle"][k] + 3]]
        lo[k], hi[k] = p.min(axis=0), p.max(axis=0)
    return lo, hi


def big_leaves(lo, hi):
    """prepare_any_order's rule: extent above 16 x the median extent, the eight largest of them"""
    ext = (hi - lo).max(axis=1)
    cap = 16.0 * np.sort(ext)[len(ext) // 2]
    over = np.flatnonzero(ext > cap)
    over = over[np.lexsort((over, -ext[over]))]
    return np.sort(over[:8])


@pytest.mark.parametrize("name", SCENES)
def test_free_tree_holds_no_big_leaf_and_the_box_holds_every_other(name):
    sc = getattr(scenes, name)()
    _, info = api.bvh_build_order(sc)
    box, free_leaves, free_big = api.bvh_culled_set(sc)
    lo, hi = leaf_boxes(sc)
    big = big_leaves(lo, hi)
    assert len(big) == info.n_big >= 1
    assert free_big == 0 and free_leaves == info.n_leaves - info.n_big
    small = np.setdiff1d(np.arange(len(lo)), big)
    assert (box[:3].astype(np.float64) <= lo[small].min(axis=0)).all()
    assert (box[3:].astype(np.float64) >= hi[small].max(axis=0)).all()
    # rounded out like a culling-tree box: no wider than 2^-20 of the magnitude plus one f32 step
    mag = np.maximum(np.abs(lo[small].min(axis=0)), np.abs(hi[small].max(axis=0)))
    assert (lo[small].min(axis=0) - box[:3] <= mag * 2.0 ** -20 + 1e-30).all()
    assert (box[3:] - hi[small].max(axis=0) <= mag * 2.0 ** -20 + 1e-30).all()
    # the big primitives are what the box leaves out (the ground sphere of r = 1000 reaches y = -2000)
    assert not ((box[:3] <= lo[big]) & (box[3:] >= hi[big])).all(axis=1).any()


def f32_down(x):
    """largest float32 <= x (x float64)"""
    f = x.astype(np.float32)
    return np.where(f.astype(np.float64) > x, np.nextafter(f, np.float32(-np.inf)), f)


def f32_up(x):
    f = x.astype(np.float32)
    return np.where(f.astype(np.float64) < x, np.nextafter(f, np.float32(np.inf)), f)


def fma32(a, b, c):
    # the exact product of two floats fits a double; the sum is rounded twice, which can move the result by one f32 step at most,
    # three orders of magnitude below the 2^-21 margin of the culling box
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def setup_rejects(rays, box, t_win):
    """trace_any_kernel's set-up decision in numpy: the culling constants of walker_start and the culled-set box test with the window
    top t_win (True: the ray is done without a walk)"""
    o, d = rays["origin"], rays["direction"]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        inv = 1.0 / d
        p = o * inv
        k = np.abs(p) * 2.0 ** -21 + 1e-37
        i32 = inv.astype(np.float32)
        cl, ch = f32_down(-p - k), f32_up(-p + k)
        neg = inv < 0.0
        near = np.where(neg, box[3:], box[:3]).astype(np.float32)
        far = np.where(neg, box[:3], box[3:]).astype(np.float32)
        n = np.maximum(fma32(near, i32, cl).max(axis=1), f32_down(rays["t_min"]))
        f = np.minimum(fma32(far, i32, ch).min(axis=1), f32_up(t_win))
    eligible = np.isfinite(o).all(axis=1) & (np.abs(inv) >= 1e-15).all(axis=1) & (np.abs(inv) <= 1e15).all(axis=1)
    return ~(f >= n), eligible


@pytest.mark.parametrize("batch", ["c2", "c3"])
def test_setup_decision_never_rejects_a_ray_that_hits_inside_the_box(batch):
    """at the bench's own sizes: the full 1920x1080 primary batch (C2) and 2^16 incoherent rays (C3) of the bunny scene"""
    sc = scenes.bunny_lambert()
    if batch == "c2":
        cam = api.Camera(1920 / 1080, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
        rays = oracle.camera_rays(cam, 1920, 1080)
    else:
        rays = scenes.incoherent_rays(1 << 16)
    box, _, _ = api.bvh_culled_set(sc)
    lo, hi = leaf_boxes(sc)
    big = big_leaves(lo, hi)
    o = oracle.Scene(sc)
    want = o.hit(rays)
    o.close()
    hit = want["leaf"] != 0xFFFFFFFF
    small_hit = hit & ~np.isin(want["leaf"], big)
    # the kernel's window after the big tests is min(t_max, t_big + 2 slack) >= the oracle's t of a ray whose hit is not big:
    # testing with the smaller window t = the oracle's t is the stricter check
    t_win = np.where(hit, want["t"], rays["t_max"])
    rejected, eligible = setup_rejects(rays, box, t_win)
    assert small_hit.sum() > 0
    assert not (rejected & eligible & small_hit).any(), np.flatnonzero(rejected & eligible & small_hit)[:10]
    if batch == "c2":  # the mechanism: most primary rays end on the ground sphere in front of the bunny's box
        assert (rejected & eligible).mean() > 0.5, (rejected & eligible).mean()


# ---------------------------------------------------------------------------------------------------------------------------------


def _equal_bits(got, want):
    assert (got["leaf"] == want["leaf"]).all(), np.flatnonzero(got["leaf"] != want["leaf"])[:10]
    assert (got["material"] == want["material"]).all()
    assert got["t"].tobytes() == want["t"].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("free_tree", ["0", "1"])
@pytest.mark.parametrize("setup_cull", ["0", "1"])
@pytest.mark.parametrize("name", SCENES + ["field"])
def test_setup_cull_returns_the_reference_hits(gpu, monkeypatch, name, setup_cull, free_tree):
    import torch

    monkeypatch.setenv("RTP_TRAVERSAL", "any")
    monkeypatch.setenv("RTP_ANY_SETUP_CULL", setup_cull)
    monkeypatch.setenv("RTP_FREE_TREE", free_tree)
    sc = scenes.bunny_field(4, 2) if name == "field" else getattr(scenes, name)()
    cam = api.Camera(16 / 9, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    rays = np.concatenate([oracle.camera_rays(cam, 480, 270), scenes.incoherent_rays(60000, seed=5)])
    o = oracle.Scene(sc)
    want = o.hit(rays)
    g = api.Scene(sc)
    d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 8)).cuda()
    d_hits = torch.empty((len(rays), 2), dtype=torch.float64, device="cuda")
    st = g.hit_device_counted(d_rays.data_ptr(), len(rays), d_hits.data_ptr())
    _equal_bits(d_hits.cpu().numpy().view(A.HIT_DTYPE).reshape(-1), want)
    _equal_bits(g.hit(rays), want)
    assert st.conservative_violations == 0
    g.close(); o.close()


@pytest.mark.gpu
def test_setup_cull_lowers_the_node_visits_of_the_primary_batch(gpu, monkeypatch):
    import torch

    sc = scenes.bunny_lambert()
    cam = api.Camera(1920 / 1080, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    d_rays = torch.empty((1920 * 1080, 8), dtype=torch.float64, device="cuda")
    api.camera_rays_device(cam, 1920, 1080, d_rays.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    d_hits = torch.empty((1920 * 1080, 2), dtype=torch.float64, device="cuda")
    visits, hits = {}, {}
    for cull in ("0", "1"):
        monkeypatch.setenv("RTP_ANY_SETUP_CULL", cull)
        g = api.Scene(sc)
        st = g.hit_device_counted(d_rays.data_ptr(), 1920 * 1080, d_hits.data_ptr())
        assert st.conservative_violations == 0 and st.order_rewalks == 0
        visits[cull], hits[cull] = st.node_visits, d_hits.cpu().numpy().tobytes()
        g.close()
    assert hits["0"] == hits["1"]
    assert visits["1"] < visits["0"], visits
