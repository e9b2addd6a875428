"""The occlusion query rtp_trace_occluded* (`scene.hit(ray).is_some()`, hittable.rs:18-25, bvh.rs:121-124).

The claim (DESIGN.md §2c): up to the first accept of the reference's sequential process every test is made with T = ray.t_max,
so the answer is Some iff some primitive passes its gate and its test at T = ray.t_max, whatever the order in which primitives are
examined; a walk with T fixed may therefore stop at the first accepted leaf. The CPU tests check this on the literal restatements
(any-hit walks in both child orders against `hit(ray) is not None`); the GPU tests check that the product returns, for every ray,
exactly the bit `rtp_trace_closest(..).leaf != RTP_MISS`, and the oracle's where the closest-hit tests use it."""
import ctypes as C

import numpy as np
import pytest

import oracle
from rtp_b200 import _abi as A
from rtp_b200 import api, scenes
from test_bvh_restatement import MISS, LiteralBvh, div, soup_rays, soup_scene
from test_gpu_parity import edge_rays as edge_rays_f64
from test_nested_hittables import LiteralNested, nested_scene

# ---------------------------------------------------------------------------------------------------------------------
# CPU: the claim on the literal restatements
# ---------------------------------------------------------------------------------------------------------------------


def literal_any(lit, ray, reverse):
    """LiteralBvh.hit_node with t_max fixed at ray.t_max and a return at the first accept; `reverse` visits right before left"""
    o = [float(x) for x in ray["origin"]]
    d = [float(x) for x in ray["direction"]]
    inv = [div(1.0, d[k]) for k in range(3)]
    t_min, t_max = float(ray["t_min"]), float(ray["t_max"])

    def walk(node):
        nd = lit.nodes[node]
        if not nd[1].collide(o, inv, t_min, t_max):
            return False
        if nd[0] == "leaf":
            return lit.hit_leaf(lit.sc.hittables[nd[2]], o, d, t_min, t_max) is not None
        return any(walk(k) for k in ((nd[3], nd[2]) if reverse else (nd[2], nd[3])))

    return walk(lit.root)


def nested_any(lit, ray, reverse):
    """the same over LiteralNested: every container (List items, nested Bvh children) ends at its first accept"""
    o = [float(x) for x in ray["origin"]]
    d = [float(x) for x in ray["direction"]]
    t_min, t_max = float(ray["t_min"]), float(ray["t_max"])
    order = (lambda xs: list(xs)[::-1]) if reverse else list

    def hit_any(node):  # hittable.rs:18-25
        if node.kind == "prim":
            return lit.hit_leaf(node.record, o, d, t_min, t_max) is not None
        if node.kind == "list":
            return any(hit_any(x) for x in order(node.items))
        if id(node) not in lit.bvhs:
            lit.bvhs[id(node)] = lit.new_bvh(node.items)
        return bvh_any(lit.bvhs[id(node)])

    def bvh_any(bvh):
        nodes, root, items = bvh
        inv = [div(1.0, d[k]) for k in range(3)]

        def walk(n):
            nd = nodes[n]
            if not nd[1].collide(o, inv, t_min, t_max):
                return False
            if nd[0] == "leaf":
                return hit_any(items[nd[2]])
            return any(walk(k) for k in order((nd[2], nd[3])))

        return walk(root)

    if lit.root_kind == "bvh":
        return bvh_any(lit.root_bvh)
    return any(hit_any(x) for x in order(lit.tree))


def with_tmax_at_hits(rays, t):
    """the rays that hit, twice: t_max = the hit's t (the hit is still accepted) and t_max = nextafter(t, 0)"""
    hit = ~np.isinf(t)
    a, b = rays[hit].copy(), rays[hit].copy()
    a["t_max"] = t[hit]
    b["t_max"] = np.nextafter(t[hit], 0.0)
    return a, b


def literal_t(lit, rays):
    out = np.full(len(rays), np.inf)
    for k, r in enumerate(rays):
        h = lit.hit(r)
        if h is not None:
            out[k] = h[0][0]
    return out


@pytest.mark.parametrize("seed,n_tri,dup", [(1, 120, True), (2, 257, False), (3, 40, True)])
def test_first_accept_answers_the_literal_bvh(seed, n_tri, dup):
    lit = LiteralBvh(soup_scene(seed, n_tri, dup))
    rays = soup_rays(seed + 30, 600)
    t = literal_t(lit, rays)
    a, b = with_tmax_at_hits(rays, t)
    assert len(a) > len(rays) // 3
    for batch in (rays, a, b):
        for r in batch:
            want = lit.hit(r) is not None
            assert literal_any(lit, r, False) == want and literal_any(lit, r, True) == want


@pytest.mark.parametrize("seed,root_kind", [(1, "bvh"), (2, "list"), (3, "bvh"), (4, "list")])
def test_first_accept_answers_the_literal_nested_scene(seed, root_kind):
    sc, tree = nested_scene(seed, root_kind)
    lit = LiteralNested(sc, root_kind, tree)
    rays = soup_rays(seed + 40, 300)
    t = literal_t(lit, rays)
    a, b = with_tmax_at_hits(rays, t)
    for batch in (rays, a, b):
        for r in batch:
            want = lit.hit(r) is not None
            assert nested_any(lit, r, False) == want and nested_any(lit, r, True) == want


def test_null_arguments_are_rejected_without_a_device():
    lib = A.load()
    st = A.Stats()
    assert lib.rtp_trace_occluded(None, None, 4, None, C.byref(st)) == A.ERR_INVALID
    assert lib.rtp_trace_occluded_device(None, None, 4, None, None) == A.ERR_INVALID
    assert lib.rtp_trace_occluded_device_counted(None, None, 4, None, C.byref(st)) == A.ERR_INVALID
    assert lib.rtp_trace_occluded(None, None, 0, None, None) == A.ERR_INVALID  # a NULL scene, whatever n


# ---------------------------------------------------------------------------------------------------------------------
# GPU: bit for bit the closest hit's `leaf != MISS`
# ---------------------------------------------------------------------------------------------------------------------


def primary(sc, w, h):
    return api.Camera(w / h, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)


def check(g, rays, want=None):
    """g.occluded(rays) == (g.hit(rays).leaf != MISS) [== (want.leaf != MISS)]; returns the occlusion array"""
    occ = g.occluded(rays)
    assert occ.dtype == np.bool_ and len(occ) == len(rays)
    closest = g.hit(rays)["leaf"] != MISS
    assert (occ == closest).all(), np.nonzero(occ != closest)[0][:10]
    if want is not None:
        assert (occ == (want["leaf"] != MISS)).all()
    return occ


def edge_rays():
    return edge_rays_f64().view(A.RAY_DTYPE).reshape(-1)


def mixed_rays(sc):
    return np.concatenate([oracle.camera_rays(primary(sc, 240, 135), 240, 135), scenes.incoherent_rays(20000, seed=5), edge_rays()])


def shadow_rays(sc, g, w, h, light=(1.0, 4.0, 2.0)):
    """from every primary hit toward a point light: d = light - p, t_min = 1e-3, t_max = 1 (tools/occlusion_probe.py, workload a)"""
    full = g.hit_full(api.camera_rays(primary(sc, w, h), w, h))
    p = full["position"][full["leaf"] != MISS]
    r = np.zeros(len(p), dtype=A.RAY_DTYPE)
    r["origin"], r["direction"], r["t_min"], r["t_max"] = p, np.asarray(light) - p, 1e-3, 1.0
    return r


@pytest.fixture(scope="module")
def bunny(gpu):
    sc = scenes.bunny_lambert()
    g, o = api.Scene(sc), oracle.Scene(sc)
    yield sc, g, o
    g.close(); o.close()


@pytest.mark.gpu
def test_c2_and_c3_batches(bunny):
    sc, g, o = bunny
    c2 = oracle.camera_rays(primary(sc, 1920, 1080), 1920, 1080)
    occ, st = g.occluded(c2, stats=True)
    assert (occ == (o.hit(c2)["leaf"] != MISS)).all() and (occ == (g.hit(c2)["leaf"] != MISS)).all()
    assert st.rays == len(c2) and st.kernel_launches >= 1 and st.device_ms > 0
    c3 = scenes.incoherent_rays(1 << 20)
    check(g, c3, o.hit(c3))


@pytest.mark.gpu
def test_shadow_rays_from_primary_hits(bunny):
    sc, g, o = bunny
    r = shadow_rays(sc, g, 480, 270)
    occ = check(g, r, o.hit(r))
    assert 0.01 < occ.mean() < 0.99  # both answers occur


@pytest.mark.gpu
def test_edge_rays_and_tmax_at_the_hit(bunny):
    sc, g, o = bunny
    check(g, edge_rays(), o.hit(edge_rays()))
    inc = scenes.incoherent_rays(20000, seed=11)
    a, _ = with_tmax_at_hits(inc, g.hit(inc)["t"])
    assert g.occluded(a).all()  # t_max = t: hittable.rs:99 rejects only t > t_max (test_gpu_parity.test_exact_tmax_is_accepted)
    # with t_max = t a leaf whose computed t lies below its own box entry is no longer reached: the exact bit is the reference's
    rays = np.concatenate([inc, shadow_rays(sc, g, 160, 90)])
    for r in with_tmax_at_hits(rays, g.hit(rays)["t"]):
        check(g, r, o.hit(r))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["bunny_triangles_only", "glass_bunny", "demo", "three_balls", "two_balls", "earth", "one_triangle", "more_balls",
                                  "more_balls_optimized"])
def test_other_scenes(gpu, name):
    sc = getattr(scenes, name)()
    with api.Scene(sc) as g:
        o = oracle.Scene(sc)
        rays = oracle.camera_rays(primary(sc, 384, 216), 384, 216)
        check(g, rays, o.hit(rays))
        check(g, mixed_rays(sc))
        o.close()


@pytest.mark.gpu
@pytest.mark.parametrize("seed,root_kind", [(1, "bvh"), (2, "list"), (3, "bvh"), (4, "list")])
def test_nested_scenes(gpu, monkeypatch, seed, root_kind):
    sc, _ = nested_scene(seed, root_kind)
    o = oracle.Scene(sc)
    rays = soup_rays(seed + 20, 6000)
    want = o.hit(rays)
    a, b = with_tmax_at_hits(rays, want["t"])
    for env in ({}, {"RTP_TRAVERSAL": "inorder"}, {"RTP_TRACE_KERNEL": "simple"}, {"RTP_F32_CULLING": "0"}):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        with api.Scene(sc) as g:
            check(g, rays, want)
            check(g, a, o.hit(a))
            check(g, b, o.hit(b))
        for k in env:
            monkeypatch.delenv(k)
    o.close()


def axis_aligned_tie_scene():
    """every quad twice (exact t ties) in axis-aligned planes (zero-thickness boxes), a few slanted panels, a ground sphere"""
    pos, idx = [], []

    def quad(p0, e1, e2):
        for _ in range(2):
            b = len(pos)
            p0a, e1a, e2a = np.array(p0, float), np.array(e1, float), np.array(e2, float)
            pos.extend([p0a, p0a + e1a, p0a + e1a + e2a, p0a + e2a])
            idx.extend([b, b + 1, b + 2, b, b + 2, b + 3])

    for x in range(-4, 4):
        for y in range(-4, 4):
            quad([x, y, 0.0], [1, 0, 0], [0, 1, 0])
            if (x + y) % 3 == 0:
                quad([x, y, 0.0], [1, 0, 0], [0, 0, 0.75])
                quad([x, y, 0.0], [0, 1, 0], [0, 0, 0.5])
            if (x * y) % 5 == 0:
                quad([x, y, 0.3], [0.7, 0.1, 0.2], [-0.1, 0.6, 0.15])
    mesh = api.Mesh.from_arrays(np.array(pos), indices=idx, material=0)
    sc = scenes.one_triangle()
    sc.scene_data.mesh_table[:] = [mesh]
    sc.hittables = api.Hittable.concat([api.Hittable.triangles_of(mesh, 0), api.Hittable.Sphere([0.0, 0.0, -1000.0], 999.5, 1)])
    rng = np.random.default_rng(11)
    n = 40000
    rays = np.zeros(n, dtype=A.RAY_DTYPE)
    rays["origin"] = np.stack([rng.uniform(-5, 5, n), rng.uniform(-5, 5, n), rng.uniform(0.5, 6.0, n)], axis=1)
    d = np.stack([rng.uniform(-4, 4, n), rng.uniform(-4, 4, n), rng.uniform(-0.2, 0.6, n)], axis=1) - rays["origin"]
    rays["direction"] = d / np.linalg.norm(d, axis=1, keepdims=True)
    rays["t_min"], rays["t_max"] = 1e-3, np.inf
    rays["t_max"][: n // 10] = rng.uniform(0.5, 8.0, n // 10)
    k = n // 10
    rays["origin"][k:2 * k] = [0.25, 0.5, 4.0]  # aimed at grid vertices: several triangles answer with the same t
    rays["direction"][k:2 * k] = np.stack([rng.integers(-4, 5, k), rng.integers(-4, 5, k), np.zeros(k)], axis=1) - rays["origin"][k:2 * k]
    rays["direction"][2 * k:3 * k] = [0.0, 0.0, -1.0]  # axis-parallel: the exact walk
    return sc, rays


@pytest.mark.gpu
def test_axis_aligned_ties_both_roots(gpu):
    sc, rays = axis_aligned_tie_scene()
    for root in ("bvh", "list"):
        sc.root_kind = root
        r = rays if root == "bvh" else rays[:8000]
        with api.Scene(sc) as g:
            o = oracle.Scene(sc)
            check(g, r, o.hit(r))
            o.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["one_sphere_bvh", "one_triangle_bvh", "empty_list", "one_sphere_list"])
def test_degenerate_scene_sizes(gpu, kind):
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
    with api.Scene(sc) as g:
        o = oracle.Scene(sc)
        rays = np.concatenate([oracle.camera_rays(primary(sc, 64, 64), 64, 64), edge_rays()])
        occ = check(g, rays, o.hit(rays))
        if kind == "empty_list":
            assert not occ.any()
        else:
            assert occ.any()
        o.close()


@pytest.mark.gpu
@pytest.mark.parametrize("scale,shift", [(1.0, 0.0), (1e9, 3e12), (1e-9, 0.0), (1e6, -7e13), (1e-3, 4e14)])
def test_f32_extreme_magnitudes(gpu, scale, shift):
    import torch

    sc = scenes.bunny_triangles_only()
    m = sc.scene_data.mesh_table[0]
    m.vertices["position"] = m.vertices["position"] * scale + shift
    rng = np.random.default_rng(12)
    n = 40000
    lo, hi = m.vertices["position"].min(axis=0), m.vertices["position"].max(axis=0)
    origin = 0.5 * (lo + hi) + rng.normal(size=(n, 3)) * (hi - lo).max() * 2.0
    d = lo + rng.random((n, 3)) * (hi - lo) - origin
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d[: n // 4] *= 10.0 ** rng.uniform(-12, 12, size=(n // 4, 1))
    d[n // 4: n // 2] *= 10.0 ** rng.uniform(-13, 0, size=(n // 4, 3))
    rays = np.zeros(n, dtype=A.RAY_DTYPE)
    rays["origin"], rays["direction"], rays["t_min"], rays["t_max"] = origin, d, 1e-3 * min(scale, 1.0), np.inf
    rays["t_max"][n // 2: 3 * n // 4] = rng.uniform(0.5, 4.0, n // 4) * (hi - lo).max()  # finite t_max, some short of the mesh
    with api.Scene(sc) as g:
        o = oracle.Scene(sc)
        check(g, rays, o.hit(rays))
        d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 8)).cuda()
        d_occ = torch.empty(n, dtype=torch.uint8, device="cuda")
        st = g.occluded_device_counted(d_rays.data_ptr(), n, d_occ.data_ptr())
        assert st.conservative_violations == 0 and st.node_visits > 0 and st.rays == n
        assert (d_occ.cpu().numpy().astype(bool) == (o.hit(rays)["leaf"] != MISS)).all()
        o.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"RTP_TRACE_KERNEL": "simple"}, {"RTP_TRAVERSAL": "inorder"}, {"RTP_TREE": "reference"}, {"RTP_F32_CULLING": "0"},
                                 {"RTP_TREE": "reference", "RTP_F32_CULLING": "0", "RTP_TRACE_KERNEL": "simple"}])
def test_switches(gpu, monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    sc = scenes.bunny_lambert()
    with api.Scene(sc) as g:
        rays = np.concatenate([mixed_rays(sc), shadow_rays(sc, g, 160, 90)])
        o = oracle.Scene(sc)
        check(g, rays, o.hit(rays))
        o.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 31, 129, (1 << 18) - 1, (1 << 18) + 1])
def test_ragged_batch_sizes(bunny, n):
    sc, g, o = bunny
    rays = scenes.incoherent_rays(n, seed=7)
    occ = g.occluded(rays)
    assert len(occ) == n
    if n:
        assert (occ == (o.hit(rays)["leaf"] != MISS)).all()


@pytest.mark.gpu
def test_multi_chunk_host_batch(gpu, monkeypatch):
    monkeypatch.setenv("RTP_CHUNK_LOG2", "12")  # 4096-ray chunks: 25 chunks through the three-stream pipeline
    sc = scenes.bunny_lambert()
    with api.Scene(sc) as g:
        rays = np.concatenate([scenes.incoherent_rays(60000, seed=3), shadow_rays(sc, g, 160, 90)])
        occ, st = g.occluded(rays, stats=True)
        assert (occ == (g.hit(rays)["leaf"] != MISS)).all()
        assert st.rays == len(rays) and st.kernel_launches == (len(rays) + 4095) // 4096


@pytest.mark.gpu
def test_device_output_bytes_sentinel_and_stream(bunny):
    import torch

    sc, g, o = bunny
    for n in (1, 31, 129, 70001):
        rays = np.concatenate([edge_rays(), scenes.incoherent_rays(n, seed=n)])[:n]
        want = (o.hit(rays)["leaf"] != MISS).astype(np.uint8)
        d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 8)).cuda()
        buf = torch.full((n + 1 + 64,), 0xAB, dtype=torch.uint8, device="cuda")  # d_out + 1: an odd device pointer, 64 canary bytes after
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())  # the rays and the sentinel fill land before the kernel
        with torch.cuda.stream(s):
            g.occluded_device(d_rays.data_ptr(), n, buf.data_ptr() + 1, s.cuda_stream)
        s.synchronize()
        got = buf.cpu().numpy()
        assert got[0] == 0xAB and (got[n + 1:] == 0xAB).all()
        assert np.isin(got[1:n + 1], (0, 1)).all() and (got[1:n + 1] == want).all()
        buf.fill_(0xAB)
        torch.cuda.synchronize()  # the counted call runs on the library's own stream, which does not wait for torch's
        st = g.occluded_device_counted(d_rays.data_ptr(), n, buf.data_ptr() + 1)
        got = buf.cpu().numpy()
        assert st.rays == n and st.conservative_violations == 0
        assert got[0] == 0xAB and (got[n + 1:] == 0xAB).all() and (got[1:n + 1] == want).all()
    g.occluded_device(0, 0, 0)  # n == 0: nothing to check, nothing touched
    assert g.occluded_device_counted(0, 0, 0).rays == 0


@pytest.mark.gpu
def test_long_lived_scene_interleaves_occlusion_and_closest_hit(gpu):
    import torch

    sc = scenes.bunny_lambert()
    rays = np.concatenate([oracle.camera_rays(primary(sc, 320, 180), 320, 180), scenes.incoherent_rays(30000, seed=21), edge_rays()])
    n = len(rays)
    with api.Scene(sc) as fresh:
        want_hits = fresh.hit(rays)
    want_occ = want_hits["leaf"] != MISS
    d_rays = torch.from_numpy(rays.view(np.float64).reshape(-1, 8)).cuda()
    streams = [torch.cuda.Stream() for _ in range(3)]
    with api.Scene(sc) as g:
        for rnd in range(3):
            occs = [torch.full((n,), 0xAB, dtype=torch.uint8, device="cuda") for _ in streams]
            hits = [torch.empty((n, 2), dtype=torch.float64, device="cuda") for _ in streams]
            torch.cuda.synchronize()
            for s, dh, do in zip(streams, hits, occs):  # device calls on three streams, occlusion and closest hit in turn
                if rnd % 2:
                    g.hit_device(d_rays.data_ptr(), n, dh.data_ptr(), s.cuda_stream)
                    g.occluded_device(d_rays.data_ptr(), n, do.data_ptr(), s.cuda_stream)
                else:
                    g.occluded_device(d_rays.data_ptr(), n, do.data_ptr(), s.cuda_stream)
                    g.hit_device(d_rays.data_ptr(), n, dh.data_ptr(), s.cuda_stream)
            torch.cuda.synchronize()
            for dh, do in zip(hits, occs):
                assert dh.cpu().numpy().view(A.HIT_DTYPE).reshape(-1).tobytes() == want_hits.tobytes()
                assert (do.cpu().numpy() == want_occ).all()
            assert (g.occluded(rays) == want_occ).all()  # host calls in between
            assert g.hit(rays).tobytes() == want_hits.tobytes()
            assert g.hit_device_counted(d_rays.data_ptr(), n, hits[0].data_ptr()).rays == n
            assert g.occluded_device_counted(d_rays.data_ptr(), n, occs[0].data_ptr()).rays == n
        assert g.hit(rays).tobytes() == want_hits.tobytes()


@pytest.mark.gpu
def test_two_devices_give_the_bytes_of_one(gpu, monkeypatch):
    if api.device_count() < 2:
        pytest.skip("needs two GPUs")
    monkeypatch.setenv("RTP_CHUNK_LOG2", "12")
    sc = scenes.demo()
    rays = np.concatenate([api.camera_rays(primary(sc, 160, 90), 160, 90), scenes.incoherent_rays(20000)])
    with api.Scene(sc) as one, api.Scene(sc, device_mask=3) as two:
        o1 = one.occluded(rays)
        o2, st = two.occluded(rays, stats=True)
        assert o1.tobytes() == o2.tobytes() and st.rays == len(rays)


@pytest.mark.gpu
def test_errors_are_reported_not_thrown(gpu):
    import torch

    g = api.Scene(scenes.one_triangle())
    lib = A.load()
    d = torch.empty(64, dtype=torch.float64, device="cuda")
    assert lib.rtp_trace_occluded(g.handle, None, 3, None, None) == A.ERR_INVALID
    assert lib.rtp_trace_occluded_device(g.handle, d.data_ptr(), 3, None, None) == A.ERR_INVALID
    assert lib.rtp_trace_occluded_device_counted(g.handle, d.data_ptr(), 3, d.data_ptr(), None) == A.ERR_INVALID
    assert lib.rtp_trace_occluded(g.handle, None, 0, None, None) == A.OK
    g.close()
    with pytest.raises(api.RtpError) as e:
        g.occluded(scenes.incoherent_rays(8))
    assert e.value.code == A.ERR_INVALID
