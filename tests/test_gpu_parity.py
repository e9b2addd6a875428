"""GPU parity proper: the CUDA path, called through the C ABI, against the CPU oracle on the same inputs.

Bar (BASELINE.json north_star): closest-hit ids bit-exact; triangle t within 4 ULP (we assert 0 ULP, since the
kernels keep the reference's operation order unfused); images per pixel within the stated tolerance.
"""
import math

import numpy as np
import pytest

import oracle
from rtp_b200 import _abi as A
from rtp_b200 import api, assets, scenes
from rtp_b200.api import rgb

pytestmark = pytest.mark.gpu

MISS = 0xFFFFFFFF


def ulp_diff(a, b):
    """distance in units in the last place between two float64 arrays (same-sign finite values)"""
    ia = a.view(np.int64).astype(np.int64)
    ib = b.view(np.int64).astype(np.int64)
    return np.abs(ia - ib)


def assert_hits_equal(g, o, what=""):
    assert (g["leaf"] == o["leaf"]).all(), f"{what}: {(g['leaf'] != o['leaf']).sum()} leaf ids differ"
    assert (g["material"] == o["material"]).all(), what
    hit = o["leaf"] != MISS
    assert (g["t"][hit].view(np.uint64) == o["t"][hit].view(np.uint64)).all(), \
        f"{what}: t differs, max ulp {ulp_diff(g['t'][hit], o['t'][hit]).max()}"
    assert np.isinf(g["t"][~hit]).all()


@pytest.fixture(scope="module")
def bunny_pair(gpu):
    sc = scenes.bunny_lambert()
    return sc, api.Scene(sc), oracle.Scene(sc)


def primary(sc, w, h):
    cam = api.Camera(w / h, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    return cam


def test_scene_layout_matches_oracle(bunny_pair):
    sc, g, o = bunny_pair
    gi, oi = g.info(), o.info()
    assert (gi.n_leaves, gi.n_nodes, gi.depth) == (oi.n_leaves, oi.n_nodes, oi.depth) == (4969, 9937, 14)
    assert (g.leaf_order() == o.leaf_order()).all()


def test_camera_rays_bit_exact(bunny_pair):
    sc, g, o = bunny_pair
    cam = primary(sc, 1920, 1080)
    rg = api.camera_rays(cam, 1920, 1080)
    ro = oracle.camera_rays(cam, 1920, 1080)
    assert rg.tobytes() == ro.tobytes()


def test_c2_primary_batch_bit_exact(bunny_pair):
    """BASELINE config C2: 1920x1080 coherent camera rays vs the bunny BVH"""
    sc, g, o = bunny_pair
    rays = oracle.camera_rays(primary(sc, 1920, 1080), 1920, 1080)
    hg, st = g.hit(rays, stats=True)
    ho, so = o.hit_full(rays, stats=True)
    assert_hits_equal(hg, ho, "C2")
    assert st.rays == len(rays)
    frac = (ho["leaf"] < 4968).mean()
    assert 0.15 < frac < 0.19


def test_trace_camera_equals_ray_batch(bunny_pair):
    """rtp_trace_camera (rays generated on the device from the camera, only hits return) == rtp_trace_closest on the same
    pixel-centre rays == the oracle; odd sizes exercise the chunk boundaries of the copy pipeline"""
    sc, g, o = bunny_pair
    for (w, h) in ((1920, 1080), (1000, 333), (7, 3)):
        cam = primary(sc, w, h)
        hc = g.hit_camera(cam, w, h)
        assert_hits_equal(hc, o.hit(oracle.camera_rays(cam, w, h)), f"camera {w}x{h}")


def test_c3_incoherent_subset_bit_exact(bunny_pair):
    """BASELINE config C3 (first 2^20 rays of the 2^24 stream)"""
    sc, g, o = bunny_pair
    rays = scenes.incoherent_rays(1 << 20)
    assert_hits_equal(g.hit(rays), o.hit(rays), "C3")


def test_full_hit_record(bunny_pair):
    sc, g, o = bunny_pair
    rays = oracle.camera_rays(primary(sc, 320, 180), 320, 180)
    hg = g.hit_full(rays)
    ho = o.hit_full(rays)
    assert (hg["leaf"] == ho["leaf"]).all()
    tri = ho["leaf"] < 4968
    for f in ("t", "position", "normal", "uv"):
        assert hg[f][tri].tobytes() == ho[f][tri].tobytes(), f
    sph = ho["leaf"] == 4968
    for f in ("t", "position", "normal"):
        assert hg[f][sph].tobytes() == ho[f][sph].tobytes(), f
    # sphere uv goes through atan2/asin: CUDA and glibc may differ by an ulp or two
    assert np.allclose(hg["uv"][sph], ho["uv"][sph], rtol=0, atol=1e-14)


def test_counters_match_oracle(bunny_pair, monkeypatch):
    """Work counters. With the reference's own median-split topology on the device (RTP_TREE=reference) the kernel performs
    exactly the oracle's AABB::collide evaluations; with the default SAH culling tree it visits fewer nodes but must run
    exactly the same primitive tests (the same leaves get through their own slab gate, in the same order)."""
    sc, g, o = bunny_pair
    import torch

    rays = oracle.camera_rays(primary(sc, 640, 360), 640, 360)
    d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 8)).cuda()
    d_hits = torch.empty((len(rays), 2), dtype=torch.float64, device="cuda")
    ho, so = o.hit_full(rays, stats=True)
    monkeypatch.setenv("RTP_TRAVERSAL", "inorder")  # the reference's visiting order on the SAH culling tree
    gi = api.Scene(sc)
    st = gi.hit_device_counted(d_rays.data_ptr(), len(rays), d_hits.data_ptr())
    assert (st.rays, st.triangle_tests, st.sphere_tests) == (so.rays, so.triangle_tests, so.sphere_tests)
    assert 0 < st.node_visits < so.node_visits
    assert st.conservative_violations == 0  # the f32 culling test never rejected a box the exact f64 test accepts
    gi.close()
    sa = g.hit_device_counted(d_rays.data_ptr(), len(rays), d_hits.data_ptr())  # default: the any-order walk (front to back)
    assert sa.rays == so.rays and 0 < sa.node_visits < st.node_visits and sa.triangle_tests < st.triangle_tests
    assert sa.conservative_violations == 0 and sa.order_rewalks <= len(rays) // 1000
    monkeypatch.setenv("RTP_TREE", "reference")
    monkeypatch.setenv("RTP_F32_CULLING", "0")  # exact f64 slab tests only: the node-visit count must equal the oracle's
    gr = api.Scene(sc)
    monkeypatch.delenv("RTP_TREE")
    monkeypatch.delenv("RTP_F32_CULLING")
    sr = gr.hit_device_counted(d_rays.data_ptr(), len(rays), d_hits.data_ptr())
    assert (sr.rays, sr.node_visits, sr.triangle_tests, sr.sphere_tests) == (so.rays, so.node_visits, so.triangle_tests, so.sphere_tests)
    hits = d_hits.cpu().numpy().view(A.HIT_DTYPE).reshape(-1)
    assert (hits["leaf"] == ho["leaf"]).all() and hits["t"].tobytes() == ho["t"].tobytes()
    gr.close()


@pytest.mark.parametrize("kernel,tree,f32,order", [("simple", "reference", 1, "any"), ("simple", "sah", 1, "any"), ("persist", "reference", 1, "any"),
                                                   ("persist", "sah", 0, "any"), ("persist", "reference", 0, "any"), ("persist", "sah", 1, "inorder"),
                                                   ("persist", "reference", 1, "inorder")])
def test_kernel_and_tree_variants_agree(gpu, monkeypatch, kernel, tree, f32, order):
    """every (kernel, culling tree, visiting order) combination returns the oracle's hits: the baseline one-thread-per-ray kernel,
    the persistent wavefront kernel, the reference topology and the SAH-over-rank-order topology, walked in the reference's
    order or front to back"""
    monkeypatch.setenv("RTP_TRACE_KERNEL", kernel)
    monkeypatch.setenv("RTP_TREE", tree)
    monkeypatch.setenv("RTP_F32_CULLING", str(f32))
    monkeypatch.setenv("RTP_TRAVERSAL", order)
    sc = scenes.bunny_lambert()
    g, o = api.Scene(sc), oracle.Scene(sc)
    rays = np.concatenate([oracle.camera_rays(primary(sc, 480, 270), 480, 270), scenes.incoherent_rays(50000, seed=5), edge_rays().view(A.RAY_DTYPE).reshape(-1)])
    assert_hits_equal_bits(g.hit(rays), o.hit(rays))
    g.close(); o.close()


def assert_hits_equal_bits(g, o):
    assert (g["leaf"] == o["leaf"]).all() and (g["material"] == o["material"]).all() and g["t"].tobytes() == o["t"].tobytes()


def edge_rays():
    r = []
    def add(o, d, tmin=1e-3, tmax=np.inf):
        r.append(list(o) + list(d) + [tmin, tmax])
    for d in ([1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1], [0, -1, 1e-300], [1, 1, 0], [0.0, -0.0, -1.0]):
        for o in ([0, 0.5, 3], [-3, 0.5, 0], [0, 5, 0], [-0.168, 0.768, 5], [0.60779, 1.53609, 0.58715], [0, -0.00078, 0]):
            add(o, d)
    add([0, 0.5, 3], [np.nan, 0, -1])
    add([0, 0.5, 3], [0, 0, 0])
    add([np.nan, 0.5, 3], [0, 0, -1])
    add([0, 0.5, 3], [0, 0, -1], 1e-3, 1.0)      # t_max before the bunny
    add([0, 0.5, 3], [0, 0, -1], 5.0, 1.0)       # t_min > t_max
    add([0, 0.5, 3], [0, 0, -1], 1e-3, np.nan)
    add([0, 0.5, 3], [0, 0, -1], np.nan, np.inf)
    add([0, 0.5, 3], [0, 0, -np.inf])
    add([0, 0.5, 3], [0, 0, -1e-310])            # denormal direction
    add([0, 0.5, 3], [0, 0, -1e300])
    add([1e300, 0.5, 3], [-1, 0, 0])
    add([0, 2000, 0], [0, -1, 0])
    add([0, -999.9999, -1], [0.3, 1, 0.2])       # from inside the ground sphere
    return np.array(r, dtype=np.float64)


def test_edge_rays(bunny_pair):
    sc, g, o = bunny_pair
    rays = edge_rays()
    hg, ho = g.hit(rays), o.hit(rays)
    assert (hg["leaf"] == ho["leaf"]).all(), np.nonzero(hg["leaf"] != ho["leaf"])
    assert hg["t"].tobytes() == ho["t"].tobytes()


@pytest.mark.parametrize("n", [0, 1, 31, 127, 129, (1 << 18) - 1, (1 << 18) + 1])
def test_ragged_batch_sizes(bunny_pair, n):
    sc, g, o = bunny_pair
    rays = scenes.incoherent_rays(n, seed=7)
    hg = g.hit(rays)
    assert len(hg) == n
    if n:
        assert_hits_equal(hg, o.hit(rays), f"n={n}")


def test_exact_tmax_is_accepted(bunny_pair):
    """hittable.rs:99 rejects only t > t_max: re-tracing with t_max = t returns the same primitive"""
    sc, g, o = bunny_pair
    rays = scenes.incoherent_rays(20000, seed=11)
    h = g.hit(rays)
    hit = h["leaf"] != MISS
    r2 = rays[hit].copy()
    r2["t_max"] = h["t"][hit]
    h2 = g.hit(r2)
    assert (h2["leaf"] == h["leaf"][hit]).all() and h2["t"].tobytes() == h["t"][hit].tobytes()
    r2["t_max"] = np.nextafter(h["t"][hit], 0.0)
    h3 = g.hit(r2)
    assert (h3["t"] < h["t"][hit]).sum() == 0  # nothing closer existed
    assert_hits_equal(h3, o.hit(r2), "shrunk t_max")


@pytest.mark.parametrize("name", ["bunny_triangles_only", "glass_bunny", "demo", "three_balls", "two_balls", "earth", "one_triangle", "more_balls",
                                  "more_balls_optimized"])
def test_other_scenes_closest_hit(gpu, name):
    sc = getattr(scenes, name)()
    g, o = api.Scene(sc), oracle.Scene(sc)
    rays = oracle.camera_rays(primary(sc, 384, 216), 384, 216)
    assert_hits_equal(g.hit(rays), o.hit(rays), name)
    g.close(); o.close()


def image_report(a, b):
    d = np.abs(a - b)
    return dict(max=float(d.max()), rmse=float(np.sqrt((d * d).mean())), differing=int((a != b).any(axis=-1).sum()), pixels=a.shape[0] * a.shape[1])


# Tolerance for image parity. The integrator reproduces the oracle's arithmetic order, RNG stream and sample
# summation order, so pixels are expected bit-identical; the only operations not bit-pinned are atan2/asin
# (CUDA libm vs glibc, <= 2 ulp), which can move a texture lookup across a texel boundary. We therefore require
# RMSE <= 1e-6 and at most 0.1% of pixels differing at all.
IMG_RMSE = 1e-6
IMG_FRAC = 1e-3


@pytest.mark.parametrize("name,w,h,spp", [
    ("bunny_lambert", 320, 180, 4), ("bunny", 160, 90, 2), ("glass_bunny", 160, 90, 4), ("demo", 192, 108, 4),
    ("three_balls", 128, 128, 8), ("two_balls", 128, 128, 4), ("earth", 128, 128, 4), ("one_triangle", 128, 128, 2),
    ("more_balls_optimized", 160, 160, 2), ("more_balls", 48, 48, 1),
])
def test_render_matches_oracle(gpu, name, w, h, spp):
    sc = getattr(scenes, name)()
    g, o = api.Scene(sc), oracle.Scene(sc)
    ig, fg, sg = g.render(w, h, spp, max_bounce=8, seed=1)
    io, fo, so = o.render(w, h, spp, max_bounce=8, seed=1)
    rep = image_report(ig, io)
    assert rep["rmse"] <= IMG_RMSE and rep["differing"] <= max(1, IMG_FRAC * rep["pixels"]), rep
    assert (fg == fo).all()
    assert sg.paths == so.paths == w * h * spp
    assert abs(int(sg.rays) - int(so.rays)) <= 8 * max(1, rep["differing"]) * spp, (sg.rays, so.rays)
    g.close(); o.close()


def test_c1_config_reduced_spp(gpu):
    """BASELINE config C1 geometry and resolution (640x360, depth 8) at 2 spp so the oracle finishes in seconds"""
    sc = scenes.bunny_lambert()
    g, o = api.Scene(sc), oracle.Scene(sc)
    ig, fg, sg = g.render(640, 360, 2, seed=1)
    io, fo, so = o.render(640, 360, 2, seed=1)
    rep = image_report(ig, io)
    assert rep["rmse"] <= IMG_RMSE and rep["differing"] <= IMG_FRAC * rep["pixels"], rep
    assert sg.rays == so.rays or rep["differing"] > 0


@pytest.mark.parametrize("name,depth", [("demo", 8), ("glass_bunny", 1), ("glass_bunny", 2), ("glass_bunny", 12), ("bunny_lambert", 40), ("three_balls", 3)])
def test_wavefront_equals_one_thread_per_path_integrator(gpu, monkeypatch, name, depth):
    """the wavefront integrator (queues in HBM, persistent traversal, f32 culling) and the baseline one-thread-per-path kernel
    (exact f64 walk) are two implementations of main.rs:70-83: every pixel, the foreground mask and the ray count agree bit for bit"""
    sc = getattr(scenes, name)()
    g = api.Scene(sc)
    iw, fw, sw = g.render(160, 90, 3, max_bounce=depth, seed=7)
    monkeypatch.setenv("RTP_RENDER_KERNEL", "simple")
    gs = api.Scene(sc)
    monkeypatch.delenv("RTP_RENDER_KERNEL")
    i1, f1, s1 = gs.render(160, 90, 3, max_bounce=depth, seed=7)
    assert iw.tobytes() == i1.tobytes() and fw.tobytes() == f1.tobytes()
    assert sw.rays == s1.rays and sw.paths == s1.paths
    g.close(); gs.close()


def test_tail_mode_equals_wavefront(gpu, monkeypatch):
    """small launches finish in ONE tail-mode launch of the traversal kernel (shading in place); it must return the bits of
    the trace/shade pairs."""
    sc = scenes.demo()
    monkeypatch.setenv("RTP_TAIL_THRESHOLD", "0")
    g0 = api.Scene(sc)
    ref, fref, sref = g0.render(200, 120, 3, max_bounce=8, seed=11)
    monkeypatch.setenv("RTP_TAIL_THRESHOLD", "1000000")
    g = api.Scene(sc)
    img, fg, st = g.render(200, 120, 3, max_bounce=8, seed=11)
    assert img.tobytes() == ref.tobytes() and fg.tobytes() == fref.tobytes() and st.rays == sref.rays
    g.close()
    g0.close()


def test_tiles_and_sample_ranges(gpu):
    sc = scenes.bunny_lambert()
    g = api.Scene(sc)
    w, h, spp = 96, 64, 6
    full, ffg, _ = g.render(w, h, spp, seed=3)
    # tiles: stitched result is bit-identical (main.rs:36 tiling is only a work partition)
    stitched = np.zeros_like(full)
    for (oi, oj, tw, th) in api.split_in_tiles(w, h, 32, 32):
        g.render(w, h, spp, seed=3, tile=(int(oi), int(oj), int(tw), int(th)), out=stitched)
    assert stitched.tobytes() == full.tobytes()
    # sample ranges: raw sums over [0,2) + [2,6) reproduce the frame up to f64 re-association
    a, _, _ = g.render(w, h, spp, seed=3, sample_range=(0, 2), flags=A.RENDER_RAW_SUMS)
    b, _, _ = g.render(w, h, spp, seed=3, sample_range=(2, 6), flags=A.RENDER_RAW_SUMS)
    assert np.allclose((a + b) / spp, full, rtol=1e-14, atol=1e-15)


def test_errors_are_reported_not_thrown(gpu):
    sc = scenes.one_triangle()
    sc.scene_data.mesh_table[0].material = 9
    with pytest.raises(api.RtpError) as e:
        api.Scene(sc)
    assert e.value.code == A.ERR_INVALID
    g = api.Scene(scenes.one_triangle())
    with pytest.raises(api.RtpError) as e:
        g.render(16, 16, 1, max_bounce=0)  # assert!(depth >= 1), render.rs:97
    assert e.value.code == A.ERR_INVALID


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE sizes, through size-independent properties (the oracle finishes only subsets of these in seconds)
# ---------------------------------------------------------------------------------------------------------------------

def _device_hits(g, d_rays):
    import torch

    d_hits = torch.empty((d_rays.shape[0], 2), dtype=torch.float64, device="cuda")
    g.hit_device(d_rays.data_ptr(), d_rays.shape[0], d_hits.data_ptr())
    torch.cuda.synchronize()
    return d_hits


def test_c3_full_16m_rays_two_algorithms_agree(gpu, monkeypatch):
    """BASELINE config C3 at full size: all 2^24 incoherent rays. The production kernel (4-wide f32-culled walk, persistent
    warps) and the exact f64 pre-order walk of the reference topology in the one-thread-per-ray kernel are different
    algorithms over different trees; they must agree bit for bit on every ray, and with the oracle on every 1021st ray."""
    import torch

    sc = scenes.bunny_lambert()
    g = api.Scene(sc)
    monkeypatch.setenv("RTP_TRACE_KERNEL", "simple")
    monkeypatch.setenv("RTP_TREE", "reference")
    ge = api.Scene(sc)
    monkeypatch.delenv("RTP_TRACE_KERNEL"); monkeypatch.delenv("RTP_TREE")
    o = oracle.Scene(sc)
    n, chunk = 1 << 24, 1 << 22
    kinds = np.zeros(3, dtype=np.int64)
    for first in range(0, n, chunk):
        rays = scenes.incoherent_rays(chunk, first=first)
        d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 8)).cuda()
        a, b = _device_hits(g, d_rays), _device_hits(ge, d_rays)
        assert bool((a.view(torch.int64) == b.view(torch.int64)).all()), first
        hg = a.cpu().numpy().view(A.HIT_DTYPE).reshape(-1)
        sub = slice(first % 1021, chunk, 1021)
        assert_hits_equal_bits(hg[sub], o.hit(rays[sub]))
        kinds += [int((hg["leaf"] < 4968).sum()), int((hg["leaf"] == 4968).sum()), int((hg["leaf"] == A.MISS).sum())]
    frac = kinds / n
    assert 0.30 < frac[0] < 0.42 and 0.50 < frac[1] < 0.64 and 0.03 < frac[2] < 0.12, frac  # SURVEY.md §8d: ~36 / 57 / 8 %
    g.close(); ge.close(); o.close()


def test_c4_full_resolution_frame_properties(gpu):
    """BASELINE config C4 geometry at 1920x1080 (1 of its 256 spp): tiling is only a work partition (main.rs:36), so 32x32
    tiles stitched through the tail-mode path equal the whole-frame wavefront render bit for bit; a sample-range split
    reproduces the frame up to f64 re-association; and the oracle agrees on a 96x54 crop rendered as its own tile."""
    sc = scenes.demo()
    g, o = api.Scene(sc), oracle.Scene(sc)
    w, h = 1920, 1080
    full, ffg, st = g.render(w, h, 2, seed=5)
    assert st.paths == w * h * 2 and st.rays >= st.paths
    stitched = np.zeros_like(full)
    for (oi, oj, tw, th) in api.split_in_tiles(w, h, 256, 256):
        g.render(w, h, 2, seed=5, tile=(int(oi), int(oj), int(tw), int(th)), out=stitched)
    assert stitched.tobytes() == full.tobytes()
    a, _, _ = g.render(w, h, 2, seed=5, sample_range=(0, 1), flags=A.RENDER_RAW_SUMS)
    b, _, _ = g.render(w, h, 2, seed=5, sample_range=(1, 2), flags=A.RENDER_RAW_SUMS)
    assert np.allclose((a + b) / 2, full, rtol=1e-14, atol=1e-15)
    tile = (900, 500, 96, 54)
    ref = np.zeros_like(full)
    o_img, _, _ = o.render(w, h, 2, seed=5, tile=tile)
    crop = (slice(tile[1], tile[1] + tile[3]), slice(tile[0], tile[0] + tile[2]))
    rep = image_report(full[crop], o_img[crop])
    assert rep["rmse"] <= IMG_RMSE and rep["differing"] <= max(1, IMG_FRAC * rep["pixels"]), rep
    g.close(); o.close()


def test_c5_reduced_bunny_field_matches_oracle(gpu):
    """BASELINE config C5 scene generator at 8x4 copies (158,977 leaves): closest hits and a small render vs the oracle. The full
    64x32 field (10.2 M triangles, 5 GiB) is exercised by tools/c5_run.py, which checks the f32-culled walk against the exact walk."""
    sc = scenes.bunny_field(8, 4)
    g, o = api.Scene(sc), oracle.Scene(sc)
    assert g.info().n_leaves == o.info().n_leaves == 8 * 4 * 4968 + 1
    assert (g.leaf_order() == o.leaf_order()).all()
    cam = api.Camera(16 / 9, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    rays = oracle.camera_rays(cam, 640, 360)
    rng = np.random.default_rng(3)
    shuffled = rays.copy()
    shuffled["direction"] = rays["direction"][rng.permutation(len(rays))]
    both = np.concatenate([rays, shuffled])
    assert_hits_equal_bits(g.hit(both), o.hit(both))
    ig, fg, sg = g.render(160, 90, 2, seed=2)
    io, fo, so = o.render(160, 90, 2, seed=2)
    rep = image_report(ig, io)
    assert rep["rmse"] <= IMG_RMSE and rep["differing"] <= max(1, IMG_FRAC * rep["pixels"]), rep
    g.close(); o.close()


def test_nan_uv_samples_texel_row_zero_like_rust(gpu):
    """`Hit::at_infinity` takes asin(dir.y) of a NON-unit direction (utility.rs:93-100; the camera basis is scaled by |up x z|,
    utility.rs:174). With a long `up` vector dir.y exceeds 1, asin is NaN, f64::clamp keeps NaN and `NaN as u32` is 0
    (texture.rs:40-49): those pixels read texel row 0. CUDA's cvt maps NaN to 0x80000000 instead — regression for that."""
    from rtp_b200.api import Camera, Transformation

    sc = scenes.bunny_lambert()
    sc.camera = Camera(1.0, sc.camera.fov, 1.0, 0.0, Transformation.lookat([0.0, 0.3, 2.0], [0.0, 2.5, 0.0], [0.0, 3.0, 0.0]))
    g, o = api.Scene(sc), oracle.Scene(sc)
    cam = api.Camera(1.0, sc.camera.fov, 1.0, 0.0, sc.camera.transformation)
    rays = oracle.camera_rays(cam, 64, 64)
    assert (np.abs(rays["direction"][:, 1]) > 1.0).any()  # the premise: asin gets arguments outside [-1, 1]
    ig, fg, _ = g.render(64, 64, 2, seed=4)
    io, fo, _ = o.render(64, 64, 2, seed=4)
    rep = image_report(ig, io)
    assert rep["rmse"] <= IMG_RMSE and rep["differing"] <= max(1, IMG_FRAC * rep["pixels"]), rep
    g.close(); o.close()


@pytest.mark.parametrize("name", ["bunny_lambert", "demo", "one_triangle"])
def test_output_stage_on_device(gpu, name):
    """main.rs:110-122 on the device (rtp_render_srgb8): the RGBA8 frame equals to_srgb_u8 of the f64 frame byte for byte —
    against this library's own f64 frame and against the oracle's (where the oracle's frame is bit-identical); the transparent
    background variant writes alpha = (255 * foreground) as u8; tiles stitch."""
    sc = getattr(scenes, name)()
    g, o = api.Scene(sc), oracle.Scene(sc)
    w, h, spp = 240, 135, 3
    frame, fg, _ = g.render(w, h, spp, seed=6)
    rgba, st = g.render_srgb8(w, h, spp, seed=6)
    assert rgba.tobytes() == api.to_srgb_u8(frame).tobytes()
    assert st.paths == w * h * spp
    io, fo, _ = o.render(w, h, spp, seed=6)
    same = (io == frame).all(axis=-1)
    assert same.mean() > 0.999
    assert (rgba[same] == oracle.to_srgb_u8(io)[same]).all()
    ta, _ = g.render_srgb8(w, h, spp, seed=6, transparent_background=True)
    assert (ta[..., :3] == rgba[..., :3]).all()
    assert (ta[..., 3] == np.minimum(255.0 * fg, 255.0).astype(np.uint8)).all()
    stitched = np.zeros_like(rgba)
    for (oi, oj, tw, th) in api.split_in_tiles(w, h, 64, 64):
        g.render_srgb8(w, h, spp, seed=6, tile=(int(oi), int(oj), int(tw), int(th)), out=stitched)
    assert stitched.tobytes() == rgba.tobytes()
    g.close(); o.close()


@pytest.mark.parametrize("name", ["bunny_lambert", "demo", "field", "ties"])
def test_device_bvh_order_equals_reference_order(gpu, monkeypatch, name):
    """§8f: `Bvh::new`'s depth-first leaf order computed on the GPU (rtp_build.cu: one segmented radix sort per depth) equals the
    host build and the oracle leaf for leaf, including scenes where thousands of median splits straddle equal centroid keys
    (ties go to the smaller LeafId) and keys of -0.0 / +0.0."""
    if name == "field":
        sc = scenes.bunny_field(8, 4)
    elif name == "ties":
        # a 24x24x3 lattice of identical small triangles (every centroid key repeats many times) plus mirrored copies
        # whose keys are -0.0 and +0.0 on one axis
        pos, idx = [], []
        for k, (x, y, z) in enumerate((x, y, z) for x in range(-12, 12) for y in range(-12, 12) for z in (-1, 0, 1)):
            base = len(pos)
            pos += [[x, y, float(z)], [x + 0.5, y, float(z)], [x, y + 0.5, float(z)]]
            idx += [base, base + 1, base + 2]
        pos += [[-1.0, 0.0, 5.0], [1.0, 0.0, 5.0], [0.0, 0.0, 6.0], [1.0, -0.0, 5.0], [-1.0, -0.0, 5.0], [0.0, -0.0, 6.0]]
        idx += [len(pos) - 6, len(pos) - 5, len(pos) - 4, len(pos) - 3, len(pos) - 2, len(pos) - 1]
        mesh = api.Mesh.from_arrays(pos, indices=idx, material=0)
        sc = scenes.one_triangle()
        sc.scene_data.mesh_table[:] = [mesh]
        sc.hittables = api.Hittable.triangles_of(mesh, 0)
    else:
        sc = getattr(scenes, name)()
    monkeypatch.setenv("RTP_DEVICE_BUILD", "1")
    g = api.Scene(sc)
    monkeypatch.setenv("RTP_DEVICE_BUILD", "0")
    gh = api.Scene(sc)
    o = oracle.Scene(sc)
    assert (g.leaf_order() == o.leaf_order()).all() and (gh.leaf_order() == o.leaf_order()).all()
    # the whole build runs on the device now (leaf boxes, order, SAH culling tree, records, 4-wide collapse, any-order tables):
    # equal to the host build node for node and record for record (rtp_scene_digest), with the same plan
    assert g.digest() == gh.digest(), (g.digest(), gh.digest())
    ig, ih = g.info(), gh.info()
    for f in ("n_leaves", "n_nodes", "depth", "culling_depth", "n_big"):
        assert getattr(ig, f) == getattr(ih, f), f
    assert (ig.any_order != 0) == (ih.any_order != 0)
    cam = api.Camera(1.0, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    rays = oracle.camera_rays(cam, 96, 96)
    assert_hits_equal_bits(g.hit(rays), o.hit(rays))
    g.close(); gh.close(); o.close()


def test_thin_lens_camera(gpu):
    """render.rs:32-52 with lens_radius > 0: the UnitDisk rejection loop (randomness.rs:21-34) now feeds the ray origin, so the
    per-path draw count varies; GPU and oracle must stay on the same stream (depth-of-field frame, closest hits of lens rays)"""
    from rtp_b200.api import Camera

    sc = scenes.demo()
    c = sc.camera
    sc.camera = Camera(c.aspect_ratio, c.fov, 3.2, 0.08, c.transformation)
    g, o = api.Scene(sc), oracle.Scene(sc)
    ig, fg, sg = g.render(192, 108, 4, seed=8)
    io, fo, so = o.render(192, 108, 4, seed=8)
    rep = image_report(ig, io)
    assert rep["rmse"] <= IMG_RMSE and rep["differing"] <= max(1, IMG_FRAC * rep["pixels"]), rep
    assert (fg == fo).all() and sg.paths == so.paths
    sharp, _, _ = g.render(192, 108, 4, seed=8, camera=Camera(c.aspect_ratio, c.fov, 3.2, 0.0, c.transformation))
    assert not np.array_equal(sharp, ig)  # the lens does something
    g.close(); o.close()


@pytest.mark.parametrize("scale,shift", [(1.0, 0.0), (1e9, 3e12), (1e-9, 0.0), (1e6, -7e13), (1e-3, 4e14)])
def test_f32_culling_error_budget_at_extreme_magnitudes(gpu, scale, shift):
    """DESIGN.md §4 at the edges of its preconditions: the bunny scaled / translated so that coordinates reach 1e12..1e14 (where
    an f32 ulp is thousands of units and the culling boxes inflate accordingly) or shrink to 1e-9, and rays whose direction
    components span 13 orders of magnitude. The conservative test may stop culling, but it must never reject a box the exact
    test accepts (violation counter 0) and the hits must stay the oracle's bits."""
    import torch

    sc = scenes.bunny_triangles_only()
    m = sc.scene_data.mesh_table[0]
    m.vertices["position"] = m.vertices["position"] * scale + shift
    g, o = api.Scene(sc), oracle.Scene(sc)
    rng = np.random.default_rng(11)
    n = 60000
    lo, hi = m.vertices["position"].min(axis=0), m.vertices["position"].max(axis=0)
    centre, ext = 0.5 * (lo + hi), (hi - lo).max()
    origin = centre + rng.normal(size=(n, 3)) * ext * 2.0
    target = lo + rng.random((n, 3)) * (hi - lo)
    d = target - origin
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d[: n // 4] *= 10.0 ** rng.uniform(-12, 12, size=(n // 4, 1))                 # non-unit directions, |d| from 1e-12 to 1e12
    skew = slice(n // 4, n // 2)
    d[skew] *= 10.0 ** rng.uniform(-13, 0, size=(n // 4, 3))                     # components 13 orders of magnitude apart
    rays = np.zeros(n, dtype=A.RAY_DTYPE)
    rays["origin"], rays["direction"], rays["t_min"], rays["t_max"] = origin, d, 1e-3 * min(scale, 1.0), np.inf
    assert_hits_equal_bits(g.hit(rays), o.hit(rays))
    d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 8)).cuda()
    d_hits = torch.empty((n, 2), dtype=torch.float64, device="cuda")
    st = g.hit_device_counted(d_rays.data_ptr(), n, d_hits.data_ptr())
    assert st.conservative_violations == 0 and st.node_visits > 0
    g.close(); o.close()


def test_frames_split_into_several_launches_sum_in_sample_order(gpu, monkeypatch):
    """a frame whose paths exceed the per-launch budget (C4: 64 launches of 4 spp) is traced in several launches whose samples
    are added to the per-pixel sums in sample order (main.rs:78-87): forcing 1, 2 or 3 spp per launch must not change a bit"""
    sc = scenes.glass_bunny()
    g = api.Scene(sc)
    w, h, spp = 96, 54, 7
    ref, fref, sref = g.render(w, h, spp, seed=12)
    for budget in (w * h, 2 * w * h, 3 * w * h + 5):
        monkeypatch.setenv("RTP_PATH_BUDGET", str(budget))
        img, fg, st = g.render(w, h, spp, seed=12)
        assert img.tobytes() == ref.tobytes() and fg.tobytes() == fref.tobytes() and st.rays == sref.rays
        assert st.kernel_launches > sref.kernel_launches
    monkeypatch.delenv("RTP_PATH_BUDGET")
    g.close()


@pytest.mark.parametrize("kind", ["one_sphere_bvh", "one_triangle_bvh", "empty_list", "one_sphere_list"])
def test_degenerate_scene_sizes(gpu, kind):
    """the smallest scenes: a Bvh over a single leaf (the culling tree is one node with one child), and List roots with zero and
    one primitive (every ray of the empty list misses and shades the background)"""
    sc = scenes.one_triangle()
    if kind == "one_sphere_bvh":
        sc.hittables = api.Hittable.Sphere([0.0, 0.0, 0.0], 0.7, 1)
    elif kind == "one_triangle_bvh":
        sc.hittables = api.Hittable.Triangle(0, 0)
    elif kind == "empty_list":
        sc.root_kind, sc.hittables = "list", sc.hittables[:0]
    else:
        sc.root_kind, sc.hittables = "list", api.Hittable.Sphere([0.0, 0.0, 0.0], 0.7, 1)
    sc.hittables = np.atleast_1d(sc.hittables)
    g, o = api.Scene(sc), oracle.Scene(sc)
    cam = api.Camera(1.0, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    rays = oracle.camera_rays(cam, 64, 64)
    assert_hits_equal_bits(g.hit(rays), o.hit(rays))
    ig, fg, sg = g.render(48, 48, 3, seed=2)
    io, fo, so = o.render(48, 48, 3, seed=2)
    rep = image_report(ig, io)
    assert rep["rmse"] <= IMG_RMSE and rep["differing"] <= max(1, IMG_FRAC * rep["pixels"]), rep
    assert (fg == fo).all() and sg.rays == so.rays
    g.close(); o.close()


def test_exact_ties_and_degenerate_primitives(gpu):
    """coincident triangles hit at exactly the same t: the reference keeps the LATER one in depth-first order (bvh.rs:108,111 and
    hittable.rs:99 accept t == t_max). Every triangle of a small grid appears three times, plus zero-area triangles, a
    zero-radius and a negative-radius sphere and a sphere nested exactly inside another; ids must be the oracle's."""
    pos, idx = [], []
    for k, (x, y) in enumerate((x, y) for x in range(-6, 6) for y in range(-6, 6)):
        for _ in range(3):  # the same triangle three times, with its own vertices
            base = len(pos)
            pos += [[x, y, 0.0], [x + 1.0, y, 0.0], [x, y + 1.0, 0.25 * ((x + y) % 3)]]
            idx += [base, base + 1, base + 2]
    base = len(pos)
    pos += [[0.0, 0.0, 1.0], [1.0, 1.0, 1.0], [2.0, 2.0, 1.0], [3.0, 0.0, 1.0], [3.0, 0.0, 1.0], [3.0, 0.0, 1.0]]  # collinear, and a point
    idx += [base, base + 1, base + 2, base + 3, base + 4, base + 5]
    mesh = api.Mesh.from_arrays(pos, indices=idx, material=0)
    sc = scenes.one_triangle()
    sc.scene_data.mesh_table[:] = [mesh]
    sc.hittables = api.Hittable.concat([api.Hittable.triangles_of(mesh, 0), api.Hittable.Sphere([0.5, 0.5, 2.0], 0.0, 1),
                                        api.Hittable.Sphere([-2.0, 1.0, 2.0], -0.5, 1), api.Hittable.Sphere([2.0, -2.0, 1.5], 0.6, 1),
                                        api.Hittable.Sphere([2.0, -2.0, 1.5], 0.6, 0)])
    g, o = api.Scene(sc), oracle.Scene(sc)
    rng = np.random.default_rng(5)
    n = 40000
    rays = np.zeros(n, dtype=A.RAY_DTYPE)
    rays["origin"] = np.stack([rng.uniform(-7, 7, n), rng.uniform(-7, 7, n), np.full(n, 5.0)], axis=1)
    target = np.stack([rng.uniform(-6, 6, n), rng.uniform(-6, 6, n), np.zeros(n)], axis=1)
    d = target - rays["origin"]
    rays["direction"] = d / np.linalg.norm(d, axis=1, keepdims=True)
    rays["direction"][: n // 8] = [0.0, 0.0, -1.0]  # axis-parallel: the exact walk
    rays["t_min"], rays["t_max"] = 1e-3, np.inf
    hg, ho = g.hit(rays), o.hit(rays)
    assert_hits_equal_bits(hg, ho)
    tri_hits = ho["leaf"][ho["leaf"] < len(idx) // 3 - 2]
    assert len(tri_hits) > n // 4
    for root in ("bvh", "list"):
        sc.root_kind = root
        gl, ol = api.Scene(sc), oracle.Scene(sc)
        assert_hits_equal_bits(gl.hit(rays[:8000]), ol.hit(rays[:8000]))
        gl.close(); ol.close()
    g.close(); o.close()
    # non-finite geometry: an infinite-radius sphere and a triangle with a vertex at infinity (infinite, not NaN, centroids)
    sc.root_kind = "bvh"
    good = sc.hittables
    sc.hittables = api.Hittable.concat([good, api.Hittable.Sphere([0.0, 0.0, -3.0], np.inf, 1)])
    with pytest.raises(api.RtpError) as e:  # its centroid is inf - inf = NaN: partial_cmp().unwrap() panics (bvh.rs:63)
        api.Scene(sc)
    assert e.value.code == A.ERR_INVALID
    pos2 = pos + [[0.0, 0.0, 1.5], [np.inf, 0.0, 1.5], [0.0, 1.0, 1.5]]
    idx2 = idx + [len(pos), len(pos) + 1, len(pos) + 2]
    mesh2 = api.Mesh.from_arrays(pos2, indices=idx2, material=0)
    sc.scene_data.mesh_table[:] = [mesh2]
    sc.hittables = api.Hittable.concat([api.Hittable.triangles_of(mesh2, 0), good[good["kind"] == 0]])
    gi, oi = api.Scene(sc), oracle.Scene(sc)
    hgi, hoi = gi.hit(rays[:8000]), oi.hit(rays[:8000])
    assert (hgi["leaf"] == hoi["leaf"]).all()
    both_nan = np.isnan(hgi["t"]) & np.isnan(hoi["t"])  # a NaN t is accepted by hittable.rs:99 (every comparison is false); payload bits are not pinned
    assert ((hgi["t"].view(np.uint64) == hoi["t"].view(np.uint64)) | both_nan).all()
    gi.close(); oi.close()


def test_material_and_texture_zoo(gpu):
    """every Scatter / Absorb / Emit / Texture variant at unusual parameters in one scene, rendered against the oracle: metal with
    fuzz 5 (most reflections end below the surface and are absorbed, material.rs:141-150), dielectrics of index 0.5, 1.0 and 2.4
    (total internal reflection both ways, utility.rs:110-119), WhiteBody / BlackBody, emissive DebugNormals / Color / SkySphere
    used as a SURFACE emit, Missing / DebugUVs / Solid / Image / Noise / Perlin textures and a checker of checkers; a triangle
    mesh with per-vertex uvs carries an AlbedoMap."""
    from rtp_b200.api import Absorb, Camera, Emit, Hittable, Material, Mesh, SceneData, Scatter, Texture, Transformation, ExampleScene

    textures = [Texture.Image(assets.earthmap()), Texture.Missing, Texture.DebugUVs, Texture.Solid(rgb(0.9, 0.2, 0.1)), Texture.Noise(7), Texture.Perlin(-3),
                Texture.Checker(4, 5), Texture.Checker(6, 3), Texture.Image(assets.sky_panorama(2, 256, 128))]
    materials = [
        Material.new(Scatter.Metal(5.0), Absorb.Albedo(rgb(0.9, 0.9, 0.9)), Emit.NONE),
        Material.new(Scatter.Dielectric(0.5), Absorb.WhiteBody, Emit.NONE),
        Material.new(Scatter.Dielectric(1.0), Absorb.Albedo(rgb(0.9, 1.0, 0.9)), Emit.NONE),
        Material.new(Scatter.Dielectric(2.4), Absorb.WhiteBody, Emit.Color(rgb(0.01, 0.0, 0.02))),
        Material.new(Scatter.Lambert, Absorb.AlbedoMap(7), Emit.NONE),
        Material.new(Scatter.Lambert, Absorb.AlbedoMap(0), Emit.NONE),
        Material.new(Scatter.NONE, Absorb.BlackBody, Emit.SkySphere(8)),
        Material.new(Scatter.NONE, Absorb.BlackBody, Emit.DebugNormals),
        Material.new(Scatter.Lambert, Absorb.AlbedoMap(2), Emit.NONE),
        Material.new(Scatter.Metal(0.0), Absorb.AlbedoMap(1), Emit.NONE),
        Material.new(Scatter.Lambert, Absorb.BlackBody, Emit.NONE),
        Material.new(Scatter.Lambert, Absorb.AlbedoMap(4), Emit.NONE),
    ]
    quad = Mesh.from_arrays([[-4.0, 0.0, -4.0], [4.0, 0.0, -4.0], [4.0, 0.0, 4.0], [-4.0, 0.0, 4.0]], normals=[[0.0, 1.0, 0.0]] * 4,
                            uvs=[[0.0, 0.0], [1.0, 0.0], [1.0, 1.0], [0.0, 1.0]], indices=[0, 2, 1, 0, 3, 2], material=5)
    parts = [Hittable.triangles_of(quad, 0)]
    for k in range(11):
        ang = 2.0 * math.pi * k / 11.0
        parts.append(Hittable.Sphere([2.2 * math.cos(ang), 0.5, 2.2 * math.sin(ang)], 0.5, k if k < 5 else k + 1))
    parts.append(Hittable.Sphere([0.0, 0.8, 0.0], 0.8, 3))
    cam = Camera(1.0, 1.0, 1.0, 0.0, Transformation.lookat([0.0, 4.0, 6.0], [0.0, 0.3, 0.0], [0.0, 1.0, 0.0]))
    sc = ExampleScene(cam, SceneData(materials, textures, [quad]), "bvh", Hittable.concat(parts), Emit.SkyGradient)
    g, o = api.Scene(sc), oracle.Scene(sc)
    ig, fg, sg = g.render(200, 200, 6, max_bounce=12, seed=21)
    io, fo, so = o.render(200, 200, 6, max_bounce=12, seed=21)
    rep = image_report(ig, io)
    # the DebugUVs texture turns the sphere uv — atan2 / asin, the two operations CUDA and glibc do not share bit for bit — into a
    # COLOUR, so here the ulp shows up in pixel values instead of (rarely) moving a texel: bound the size, not the count
    assert rep["rmse"] <= 1e-12 and rep["max"] <= 1e-12, rep
    assert (fg == fo).all() and sg.rays == so.rays
    assert sg.rays / sg.paths > 1.5  # the zoo really bounces
    g.close(); o.close()


def test_parameter_limits_and_concurrent_callers(gpu):
    """argument errors come back as status codes (render.rs:97's assert, tile bounds, depth limit), and one scene serves several host
    threads at once (the reference shares its scene between 4 workers through an Arc, main.rs:40,51)"""
    import threading

    sc = scenes.bunny_lambert()
    g, o = api.Scene(sc), oracle.Scene(sc)
    for kw in (dict(max_bounce=0), dict(max_bounce=129), dict(tile=(90, 0, 16, 16)), dict(tile=(0, 0, 65, 1)), dict(sample_range=(3, 2))):
        with pytest.raises(api.RtpError):
            g.render(64, 48, 2, **kw)
    img128, _, st = g.render(32, 24, 1, max_bounce=128, seed=3)
    assert st.paths == 32 * 24
    cam = api.Camera(4 / 3, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    rays = oracle.camera_rays(cam, 400, 300)
    want = o.hit(rays)
    frame_ref, _, _ = g.render(80, 60, 2, seed=9)
    errors = []

    def worker(k):
        try:
            for _ in range(5):
                if k % 2:
                    assert_hits_equal_bits(g.hit(rays), want)
                else:
                    f, _, _ = g.render(80, 60, 2, seed=9)
                    assert f.tobytes() == frame_ref.tobytes()
        except Exception as exc:  # noqa: BLE001
            errors.append(repr(exc))

    threads = [threading.Thread(target=worker, args=(k,)) for k in range(4)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errors, errors
    g.close(); o.close()


# ---------------------------------------------------------------------------------------------
# any-order walk (DESIGN.md §4b): front-to-back traversal with distance culling must return the in-order bits
# ---------------------------------------------------------------------------------------------

def _mixed_rays(sc, n_inc=60000, seed=9):
    return np.concatenate([oracle.camera_rays(primary(sc, 480, 270), 480, 270), scenes.incoherent_rays(n_inc, seed=seed),
                           edge_rays().view(A.RAY_DTYPE).reshape(-1)])


@pytest.mark.parametrize("free_tree", ["0", "1"])
@pytest.mark.parametrize("name", ["bunny_lambert", "bunny_triangles_only", "glass_bunny", "demo", "one_triangle", "field"])
def test_any_order_walk_returns_the_reference_hits(gpu, monkeypatch, name, free_tree):
    """RTP_TRAVERSAL=any forces the any-order walk on every eligible ray of the scene; hits must be the oracle's bit for bit,
    no conservative-culling violation may be counted, and the walk must actually be cheaper than the in-order one"""
    monkeypatch.setenv("RTP_FREE_TREE", free_tree)  # 1: the any-order lanes walk a second tree over the Morton order of the leaves
    sc = scenes.bunny_field(4, 2) if name == "field" else getattr(scenes, name)()
    rays = _mixed_rays(sc)
    if name == "field":
        cam = api.Camera(16 / 9, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
        rays = np.concatenate([oracle.camera_rays(cam, 480, 270), rays])
    import torch

    o = oracle.Scene(sc)
    want = o.hit(rays)
    d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 8)).cuda()
    d_hits = torch.empty((len(rays), 2), dtype=torch.float64, device="cuda")
    monkeypatch.setenv("RTP_TRAVERSAL", "inorder")
    g0 = api.Scene(sc)
    s0 = g0.hit_device_counted(d_rays.data_ptr(), len(rays), d_hits.data_ptr())
    assert_hits_equal_bits(d_hits.cpu().numpy().view(A.HIT_DTYPE).reshape(-1), want)
    assert_hits_equal_bits(g0.hit(rays), want)
    monkeypatch.setenv("RTP_TRAVERSAL", "any")
    g1 = api.Scene(sc)
    s1 = g1.hit_device_counted(d_rays.data_ptr(), len(rays), d_hits.data_ptr())
    assert_hits_equal_bits(d_hits.cpu().numpy().view(A.HIT_DTYPE).reshape(-1), want)
    assert_hits_equal_bits(g1.hit(rays), want)
    assert s0.conservative_violations == 0 and s1.conservative_violations == 0
    assert s0.order_rewalks == 0
    assert s1.order_rewalks <= len(rays) // 1000, s1.order_rewalks  # organic meshes: abnormal leaves are ulp-level coincidences
    if name not in ("one_triangle",):
        assert s1.node_visits < s0.node_visits, (s1.node_visits, s0.node_visits)
    g0.close(); g1.close(); o.close()


@pytest.mark.parametrize("free_tree", ["0", "1"])
def test_any_order_walk_axis_aligned_geometry_and_exact_ties(gpu, monkeypatch, free_tree):
    """axis-aligned triangles have boxes of zero thickness, so their computed t falls below their own box entry about half the
    time (abnormal leaves): those rays must be walked again in the reference's order and still return the oracle's bits.
    Every triangle appears twice (exact ties: the later one in depth-first order wins), one ground sphere is the big primitive."""
    pos, idx = [], []
    def quad(p0, e1, e2):
        for _ in range(2):
            b = len(pos)
            p0a, e1a, e2a = np.array(p0, float), np.array(e1, float), np.array(e2, float)
            pos.extend([list(p0a), list(p0a + e1a), list(p0a + e1a + e2a), list(p0a + e2a)])
            idx.extend([b, b + 1, b + 2, b, b + 2, b + 3])
    for x in range(-4, 4):
        for y in range(-4, 4):
            quad([x, y, 0.0], [1, 0, 0], [0, 1, 0])             # floor tiles in z = 0
            if (x + y) % 3 == 0:
                quad([x, y, 0.0], [1, 0, 0], [0, 0, 0.75])      # walls in y = const
                quad([x, y, 0.0], [0, 1, 0], [0, 0, 0.5])       # walls in x = const
            if (x * y) % 5 == 0:
                quad([x, y, 0.3], [0.7, 0.1, 0.2], [-0.1, 0.6, 0.15])  # slanted panels
    mesh = api.Mesh.from_arrays(pos, indices=idx, material=0)
    sc = scenes.one_triangle()
    sc.scene_data.mesh_table[:] = [mesh]
    sc.hittables = api.Hittable.concat([api.Hittable.triangles_of(mesh, 0), api.Hittable.Sphere([0.0, 0.0, -1000.0], 999.5, 1)])
    rng = np.random.default_rng(11)
    n = 60000
    rays = np.zeros(n, dtype=A.RAY_DTYPE)
    rays["origin"] = np.stack([rng.uniform(-5, 5, n), rng.uniform(-5, 5, n), rng.uniform(0.5, 6.0, n)], axis=1)
    target = np.stack([rng.uniform(-4, 4, n), rng.uniform(-4, 4, n), rng.uniform(-0.2, 0.6, n)], axis=1)
    d = target - rays["origin"]
    rays["direction"] = d / np.linalg.norm(d, axis=1, keepdims=True)
    rays["t_min"], rays["t_max"] = 1e-3, np.inf
    rays["t_max"][: n // 10] = rng.uniform(0.5, 8.0, n // 10)  # finite t_max, some before the first hit
    # rays aimed exactly at grid vertices and along tile edges: several triangles answer with the same t
    k = n // 10
    rays["origin"][k:2 * k] = [0.25, 0.5, 4.0]
    vert = np.stack([rng.integers(-4, 5, k), rng.integers(-4, 5, k), np.zeros(k)], axis=1).astype(np.float64)
    rays["direction"][k:2 * k] = vert - rays["origin"][k:2 * k]
    o = oracle.Scene(sc)
    want = o.hit(rays)
    import torch

    monkeypatch.setenv("RTP_TRAVERSAL", "any")
    monkeypatch.setenv("RTP_FREE_TREE", free_tree)
    g = api.Scene(sc)
    assert_hits_equal_bits(g.hit(rays), want)
    d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 8)).cuda()
    d_hits = torch.empty((len(rays), 2), dtype=torch.float64, device="cuda")
    st = g.hit_device_counted(d_rays.data_ptr(), len(rays), d_hits.data_ptr())
    assert_hits_equal_bits(d_hits.cpu().numpy().view(A.HIT_DTYPE).reshape(-1), want)
    assert st.conservative_violations == 0
    assert st.order_rewalks > n // 100, st.order_rewalks  # the fallback is exercised, not merely present
    assert (want["leaf"] != MISS).mean() > 0.9
    # the same through the integrator (wavefront and tail-mode launches walk with the same lanes)
    ig, fg, sg = g.render(96, 64, 2, seed=4)
    io, fo, so = o.render(96, 64, 2, seed=4)
    rep = image_report(ig, io)
    assert rep["rmse"] <= IMG_RMSE and rep["differing"] <= max(1, IMG_FRAC * rep["pixels"]), rep
    g.close(); o.close()


@pytest.mark.parametrize("name,w,h,spp", [("demo", 160, 90, 4), ("glass_bunny", 128, 96, 2)])
def test_any_order_walk_renders_match_oracle(gpu, monkeypatch, name, w, h, spp):
    monkeypatch.setenv("RTP_TRAVERSAL", "any")
    sc = getattr(scenes, name)()
    g, o = api.Scene(sc), oracle.Scene(sc)
    ig, fg, sg = g.render(w, h, spp, seed=3)
    io, fo, so = o.render(w, h, spp, seed=3)
    rep = image_report(ig, io)
    assert rep["rmse"] <= IMG_RMSE and rep["differing"] <= max(1, IMG_FRAC * rep["pixels"]), rep
    assert sg.rays == so.rays or rep["differing"] > 0
    ig2, _, _ = g.render(w, h, spp, seed=3, tile=(32, 16, 32, 32))  # a 32x32 tile runs as one tail-mode launch
    assert np.array_equal(ig2[16:48, 32:64], ig[16:48, 32:64])
    g.close(); o.close()


def test_any_order_stack_overflow_hands_the_ray_to_the_in_order_walk(gpu, monkeypatch):
    """the any-order stack is capped per lane; a lane that cannot postpone three more children defers its ray to the in-order
    kernel (second launch over the defer list; inside the integrator: the shading thread's exact walk). With the cap forced down
    to four entries most incoherent rays overflow: same bits, many deferred rays."""
    import torch

    monkeypatch.setenv("RTP_TRAVERSAL", "any")
    sc = scenes.bunny_lambert()
    rays = _mixed_rays(sc)
    o = oracle.Scene(sc)
    want = o.hit(rays)
    d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 8)).cuda()
    d_hits = torch.empty((len(rays), 2), dtype=torch.float64, device="cuda")
    for cap, some in (("1", True), ("12", None), ("48", False)):
        monkeypatch.setenv("RTP_ANY_CAP", cap)
        g = api.Scene(sc)
        st = g.hit_device_counted(d_rays.data_ptr(), len(rays), d_hits.data_ptr())
        assert_hits_equal_bits(d_hits.cpu().numpy().view(A.HIT_DTYPE).reshape(-1), want)
        assert_hits_equal_bits(g.hit(rays), want)
        assert st.conservative_violations == 0
        if some is True:
            assert st.order_rewalks > 0, st.order_rewalks
        if some is False:
            assert st.order_rewalks <= len(rays) // 1000, st.order_rewalks
        ig, fg, sg = g.render(64, 48, 2, seed=8)
        io, fo, so = o.render(64, 48, 2, seed=8)
        rep = image_report(ig, io)
        assert rep["rmse"] <= IMG_RMSE and rep["differing"] <= max(1, IMG_FRAC * rep["pixels"]), rep
        g.close()
    o.close()


@pytest.mark.parametrize("name", ["bunny_lambert", "demo"])
def test_any_order_walk_unusual_rays(gpu, monkeypatch, name):
    """rays at the edge of the any-order walk's preconditions: zero and negative t_min (not eligible), finite t_max before,
    inside and behind the geometry, directions with one tiny component (huge 1/d: large slack, or outside the f32 walk), unnormalised
    directions, distant origins (large |o|: large slack), origins on the geometry. Both visiting orders must return the oracle's bits."""
    import torch

    sc = getattr(scenes, name)()
    rng = np.random.default_rng(77)
    n = 80000
    base = scenes.incoherent_rays(n, seed=21)
    rays = base.copy()
    k = n // 10
    rays["t_min"][0 * k:1 * k] = 0.0
    rays["t_min"][1 * k:2 * k] = -rng.uniform(0.0, 5.0, k)
    rays["t_max"][2 * k:3 * k] = rng.uniform(0.0, 6.0, k)
    tiny = rng.choice([1e-5, 1e-9, 1e-13, 1e-15, 3e-16, 1e-17, 1e-30], k)
    axis = rng.integers(0, 3, k)
    d = rays["direction"][3 * k:4 * k].copy()
    d[np.arange(k), axis] = tiny * rng.choice([-1.0, 1.0], k)
    rays["direction"][3 * k:4 * k] = d
    rays["direction"][4 * k:5 * k] *= rng.choice([1e-6, 1e-3, 1e3, 1e6], k)[:, None]
    far = rng.choice([1e2, 1e4, 1e7, 1e10], k)[:, None]
    o = rays["origin"][5 * k:6 * k] * far
    rays["origin"][5 * k:6 * k] = o
    tgt = rng.uniform([-0.9, 0.0, -0.6], [0.6, 1.5, 0.58], (k, 3))
    rays["direction"][5 * k:6 * k] = tgt - o
    # origins on the geometry: the hit points of other rays, new directions, the reference's own scatter epsilon
    orc = oracle.Scene(sc)
    first = orc.hit(base[6 * k:8 * k])
    ok = first["leaf"] != MISS
    p = base["origin"][6 * k:8 * k] + first["t"][:, None] * base["direction"][6 * k:8 * k]
    p[~ok] = base["origin"][6 * k:8 * k][~ok]
    rays["origin"][6 * k:8 * k] = p
    nd = rng.normal(size=(2 * k, 3))
    rays["direction"][6 * k:8 * k] = nd / np.linalg.norm(nd, axis=1, keepdims=True)
    rays["t_min"][6 * k:8 * k] = 1e-3
    rays["t_min"][8 * k:9 * k] = rng.uniform(0.0, 4.0, k)  # t_min inside the scene
    rays["t_max"][8 * k:9 * k] = rays["t_min"][8 * k:9 * k] + rng.uniform(0.0, 2.0, k)
    want = orc.hit(rays)
    d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 8)).cuda()
    d_hits = torch.empty((len(rays), 2), dtype=torch.float64, device="cuda")
    for order in ("any", "inorder"):
        monkeypatch.setenv("RTP_TRAVERSAL", order)
        g = api.Scene(sc)
        st = g.hit_device_counted(d_rays.data_ptr(), len(rays), d_hits.data_ptr())
        assert_hits_equal_bits(d_hits.cpu().numpy().view(A.HIT_DTYPE).reshape(-1), want)
        assert_hits_equal_bits(g.hit(rays), want)
        assert st.conservative_violations == 0
        g.close()
    assert (want["leaf"] != MISS).mean() > 0.3
    orc.close()


@pytest.mark.parametrize("name", ["more_balls_optimized", "two_balls", "earth", "one_triangle", "sphere_soup"])
def test_any_order_walk_on_sphere_scenes(gpu, monkeypatch, name):
    """spheres that are not outsized stay in the culled set, covered by the sphere term of the slack bound (any_slack): sphere-heavy
    scenes walked front to back must return the in-order bits, from outside, from inside the geometry and with grazing rays"""
    import torch

    rng = np.random.default_rng(31)
    if name == "sphere_soup":  # overlapping, nested and touching spheres of very different sizes, duplicates included
        n = 600
        c = rng.uniform(-6, 6, (n, 3))
        r = np.exp(rng.uniform(np.log(0.02), np.log(1.5), n))
        parts = [api.Hittable.Sphere(c[k], float(r[k]), k % 3) for k in range(n)] + [api.Hittable.Sphere(c[k], float(r[k]), 1) for k in range(0, n, 7)]
        mats = [api.Material.new(api.Scatter.Lambert, api.Absorb.WhiteBody, api.Emit.NONE), api.Material.new(api.Scatter.Metal(0.2), api.Absorb.WhiteBody, api.Emit.NONE),
                api.Material.new(api.Scatter.Dielectric(1.5), api.Absorb.WhiteBody, api.Emit.NONE)]
        sc = api.ExampleScene(scenes._bunny_camera(), api.SceneData(mats, [], []), "bvh", api.Hittable.concat(parts), api.Emit.SkyGradient)
        centres, radii, reach = c, r, 8.0
    else:
        sc = getattr(scenes, name)()
        sph = sc.hittables[sc.hittables["kind"] == A.HITTABLE_SPHERE]
        small = sph[sph["radius"] < 100.0] if (sph["radius"] < 100.0).any() else sph
        centres, radii, reach = small["center"], small["radius"], float(np.abs(small["center"]).max() + small["radius"].max() + 2.0)
    cam = api.Camera(1.0, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    m = 30000
    rays = np.zeros(m, dtype=A.RAY_DTYPE)
    o = rng.normal(size=(m, 3))
    o = o / np.linalg.norm(o, axis=1, keepdims=True) * rng.uniform(0.2, 1.0, (m, 1)) * reach
    o[:, 1] = np.abs(o[:, 1]) + 0.05
    pick = rng.integers(0, len(centres), m)
    # aim at a sphere, half of the rays at its silhouette (grazing: delta ~ 0)
    tgt = centres[pick] + rng.normal(size=(m, 3)) * radii[pick][:, None] * 0.6
    side = rng.normal(size=(m, 3))
    to_c = centres[pick] - o
    side -= (side * to_c).sum(axis=1, keepdims=True) * to_c / (to_c * to_c).sum(axis=1, keepdims=True)
    side /= np.linalg.norm(side, axis=1, keepdims=True)
    graze = centres[pick] + side * radii[pick][:, None] * (1.0 + rng.choice([0.0, 1e-15, -1e-15, 1e-9, -1e-9, 1e-4], m))[:, None]
    tgt[m // 2:] = graze[m // 2:]
    d = tgt - o
    rays["origin"], rays["direction"] = o, d / np.linalg.norm(d, axis=1, keepdims=True)
    rays["t_min"], rays["t_max"] = 1e-3, np.inf
    rays = np.concatenate([oracle.camera_rays(cam, 160, 160), rays])
    orc = oracle.Scene(sc)
    want = orc.hit(rays)
    d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 8)).cuda()
    d_hits = torch.empty((len(rays), 2), dtype=torch.float64, device="cuda")
    visits = {}
    for order in ("inorder", "any"):
        monkeypatch.setenv("RTP_TRAVERSAL", order)
        g = api.Scene(sc)
        assert g.info().any_order == (0 if order == "inorder" else 1)
        st = g.hit_device_counted(d_rays.data_ptr(), len(rays), d_hits.data_ptr())
        assert_hits_equal_bits(d_hits.cpu().numpy().view(A.HIT_DTYPE).reshape(-1), want)
        assert st.conservative_violations == 0
        assert st.order_rewalks <= len(rays) // 200, st.order_rewalks
        visits[order] = st.node_visits
        if order == "any":
            ig, fg, sg = g.render(96, 96, 2, seed=6)
            io, fo, so = orc.render(96, 96, 2, seed=6)
            rep = image_report(ig, io)
            assert rep["rmse"] <= IMG_RMSE and rep["differing"] <= max(1, IMG_FRAC * rep["pixels"]), rep
        g.close()
    if name in ("more_balls_optimized", "sphere_soup"):
        assert visits["any"] < visits["inorder"], visits
    assert (want["leaf"] != MISS).mean() > 0.3
    orc.close()


def test_c5_full_field_sampled_rays_equal_oracle(gpu):
    """BASELINE config C5 at FULL size: the 2,048-copy bunny field (10,174,464 triangles + ground sphere, 20,348,929 reference nodes),
    built on the device. Every 499th ray of the 3840x2160 primary batch, a direction-shuffled (incoherent) set and a set of
    bounce-like rays starting on the geometry are traced on the GPU and by the oracle (its own Bvh::new over all 10 M leaves):
    leaf ids and t bit for bit; the counted pass reports no conservative-culling violation; a small tile of the 4K frame
    renders to the oracle's pixels."""
    sc = scenes.bunny_field(64, 32)
    g = api.Scene(sc)
    info = g.info()
    assert info.n_leaves == 10_174_465 and info.n_nodes == 2 * 10_174_465 - 1 and info.any_order != 0
    o = oracle.Scene(sc)
    assert o.info().depth == info.depth
    W, H = 3840, 2160
    cam = api.Camera(W / H, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    primary = api.camera_rays(cam, W, H)[::499].copy()
    rng = np.random.default_rng(5)
    shuffled = primary.copy()
    shuffled["direction"] = primary["direction"][rng.permutation(len(primary))]
    hp = o.hit_full(primary)
    hit = hp["leaf"] != 0xFFFFFFFF
    bounce = primary[hit][:6000].copy()  # leave the first hit point in a random direction of the upper hemisphere
    d = rng.normal(size=(len(bounce), 3))
    d[:, 1] = np.abs(d[:, 1])
    bounce["origin"], bounce["direction"] = hp["position"][hit][:6000], d / np.linalg.norm(d, axis=1, keepdims=True)
    for name, rays in (("primary", primary), ("shuffled", shuffled), ("bounce", bounce)):
        got, st = g.hit(rays, stats=True)
        want = o.hit(rays)
        assert (got["leaf"] == want["leaf"]).all(), name
        assert got["t"].tobytes() == want["t"].tobytes(), name
        assert (got["material"] == want["material"]).all(), name
    d_rays = np.ascontiguousarray(np.concatenate([primary, shuffled, bounce]))
    import torch

    dr = torch.from_numpy(d_rays.view(np.float64).reshape(-1, 8)).cuda()
    dh = torch.empty((len(d_rays), 2), dtype=torch.float64, device="cuda")
    c = g.hit_device_counted(dr.data_ptr(), len(d_rays), dh.data_ptr())
    assert c.conservative_violations == 0 and c.rays == len(d_rays)
    tile = (1900, 700, 24, 16)
    ig, fg, _ = g.render(W, H, 2, max_bounce=8, seed=1, tile=tile)
    io, fo, _ = o.render(W, H, 2, max_bounce=8, seed=1, tile=tile)
    sl = (slice(tile[1], tile[1] + tile[3]), slice(tile[0], tile[0] + tile[2]))
    assert np.sqrt(((ig[sl] - io[sl]) ** 2).mean()) <= IMG_RMSE and (fg[sl] == fo[sl]).all()
    g.close(); o.close()


def test_many_concurrent_launches_on_many_streams(gpu):
    """rtp_trace_closest_device from more streams than the library has launch slots (8): every launch owns a work queue and a defer
    list for its lifetime (a slot's next user waits on the event of its last launch), so launches in flight on different streams never
    share them. 24 streams x 4 rounds of different batches — primary, incoherent, and one with axis-parallel rays that are deferred
    to the in-order kernel — must each return the bits of the same batch traced alone."""
    import torch

    sc = scenes.bunny_lambert()
    cam = api.Camera(16 / 9, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    primary = api.camera_rays(cam, 320, 180)
    axis = primary[:20000].copy()
    axis["direction"][::3] = [0.0, -1.0, 0.0]  # not eligible for the f32 walk: deferred
    batches = [primary, scenes.incoherent_rays(70000), axis, scenes.incoherent_rays(30000, first=10 ** 6)]
    with api.Scene(sc) as g:
        d_rays = [torch.from_numpy(b.view(np.float64).reshape(-1, 8)).cuda() for b in batches]
        want = []
        for r in d_rays:
            h = torch.empty((r.shape[0], 2), dtype=torch.float64, device="cuda")
            g.hit_device(r.data_ptr(), r.shape[0], h.data_ptr(), torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            want.append(h.clone())
        streams = [torch.cuda.Stream() for _ in range(24)]
        outs = [[torch.empty_like(want[k % len(batches)]) for k in range(4)] for _ in streams]
        torch.cuda.synchronize()
        for rnd in range(4):
            for s_i, st in enumerate(streams):
                k = (s_i + rnd) % len(batches)
                out = outs[s_i][rnd]
                if out.shape != want[k].shape:
                    outs[s_i][rnd] = out = torch.empty_like(want[k])
                g.hit_device(d_rays[k].data_ptr(), d_rays[k].shape[0], out.data_ptr(), st.cuda_stream)
        torch.cuda.synchronize()
        for rnd in range(4):
            for s_i in range(len(streams)):
                k = (s_i + rnd) % len(batches)
                assert bool((outs[s_i][rnd].view(torch.int64) == want[k].view(torch.int64)).all()), (s_i, rnd, k)
