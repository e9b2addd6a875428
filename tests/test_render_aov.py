"""rtp_render_aov: rtp_render plus each pixel's mean first-vertex albedo and normal (include/rtp.h, DESIGN.md §6c).

The reference for the two buffers is `first_vertex_reference` below: the first segment of every path (main.rs:70-76) from the pure-Python
integrator of test_integrator_restatement, whose primary rays equal the oracle's path by path; its closest hit through the oracle's
`Hittable::hit` (Hit::normal, material, position, uv); the absorb of that material by the oracle's texture sampler; and the per-pixel
sums in sample order from 0.0. On the CPU it is checked against the pure-Python integrator's own first vertex; on the GPU the library's
buffers must equal it bit for bit, with the oracle's uv taken through CUDA's atan2 / asin where a texture is looked up by uv, and the
colour and foreground must be rtp_render's bytes.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle
from rtp_b200 import _abi as A
from rtp_b200 import api, scenes
from test_integrator_restatement import RAY_EPSILON, Restated, add, textured_scene, zoo_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "rtp.h")

SENTINEL = 0x7FF8_DEAD_BEEF_0003  # bits of a quiet NaN whose payload no computation produces
ZERO3 = (0.0, 0.0, 0.0)


class PrimaryRay(Restated):
    """the pure-Python integrator stopped before its first trace: path(i, j, s) leaves the jittered thin-lens ray in self.ray"""

    def shade(self, o, d, depth, rng, first):
        self.ray = (o, d)
        return ZERO3, False


def first_vertex_reference(sc, o, width, height, num_samples, seed=1, sample_range=None, flags=0):
    """(albedo [h, w, 3], normal [h, w, 3]) as rtp_render_aov defines them, for sample range [s0, s1) (default [0, num_samples)).
    o: an oracle.Scene of sc"""
    s0, s1 = sample_range or (0, num_samples)
    n = s1 - s0
    r = PrimaryRay(sc, width, height, 1, seed)
    rays = np.zeros((height, width, n), dtype=A.RAY_DTYPE)
    for j in range(height):
        for i in range(width):
            for k in range(n):
                r.path(i, j, s0 + k)
                rays[j, i, k] = (r.ray[0], r.ray[1], RAY_EPSILON, np.inf)  # render.rs:102 traces [RAY_EPSILON, inf)
    hits = o.hit_full(rays.reshape(-1)).reshape(height, width, n)
    hit = hits["leaf"] != A.MISS
    albedo = np.zeros((height, width, n, 3))
    mats = sc.scene_data.material_table
    for idx in zip(*np.nonzero(hit)):  # material.rs:74-81
        h, a = hits[idx], mats[int(hits[idx]["material"])].absorb
        if a.kind == A.ABSORB_WHITEBODY:
            albedo[idx] = 1.0
        elif a.kind == A.ABSORB_ALBEDO:
            albedo[idx] = [float(x) for x in a.color]
        elif a.kind == A.ABSORB_ALBEDO_MAP:
            albedo[idx] = o.texture_sample(a.texture, h["position"], h["uv"])
    normal = np.where(hit[..., None], hits["normal"], 0.0)
    sums = []
    for per_sample in (albedo, normal):
        acc = np.zeros((height, width, 3))
        for k in range(n):  # sample order, from 0.0
            acc = acc + per_sample[:, :, k]
        sums.append(acc if flags & A.RENDER_RAW_SUMS else acc / float(num_samples))
    return sums[0], sums[1]


# ------------------------------------------------------------------------------------------------------------ CPU ----


def test_prototypes_compile_against_the_ctypes_mirror(tmp_path):
    """include/rtp.h compiled as plain C: both entry points assign to pointers of the declared types; the ctypes mirror has their
    arity and struct arguments"""
    src = f"""#include "{HEADER}"
int (*render_aov)(rtp_scene*, const rtp_camera*, const rtp_render_params*, double*, double*, double*, double*, rtp_stats*) = rtp_render_aov;
int (*render_aov_device)(rtp_scene*, const rtp_camera*, const rtp_render_params*, double*, double*, double*, double*, rtp_stats*,
                         void*) = rtp_render_aov_device;
"""
    c = tmp_path / "protos.c"
    c.write_text(src)
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-c", "-o", str(tmp_path / "protos.o"), str(c)], check=True)
    for name, n in (("rtp_render_aov", 8), ("rtp_render_aov_device", 9)):
        res, args = A.PROTOTYPES[name]
        assert res == C.c_int and len(args) == n, name
        assert args[1] == C.POINTER(A.Camera) and args[2] == C.POINTER(A.RenderParams) and args[7] == C.POINTER(A.Stats), name


class FirstVertexRestated(Restated):
    """the pure-Python integrator, also reporting the first segment's closest hit: (absorb, Hit::normal), (0, 0, 0) twice on a miss"""

    def scene_hit(self, o, d, t_min, t_max):
        hit = super().scene_hit(o, d, t_min, t_max)
        if self.fv is None:
            if hit is None:
                self.fv = (ZERO3, ZERO3)
            else:
                (_, _, normal, uv), mid = hit
                self.fv = (self.absorb(self.sc.scene_data.material_table[mid].absorb, uv), normal)
        return hit

    def path(self, i, j, s):
        self.fv = None
        color, hit, rays = super().path(i, j, s)
        return color, hit, rays, self.fv


@pytest.mark.parametrize("name,depth", [("three_balls", 8), ("zoo", 8), ("zoo", 1), ("textured", 8)])
def test_reference_equals_python_restatement(name, depth):
    """the reference's per-pixel sums equal the pure-Python integrator's first vertex (its own List walk, hit_sphere and texture
    lookup), summed in sample order and divided by num_samples, bit for bit"""
    sc = {"three_balls": scenes.three_balls, "zoo": zoo_scene, "textured": textured_scene}[name]()
    w, h, spp, seed = 24, 16, 3, 5
    o = oracle.Scene(sc)
    albedo, normal = first_vertex_reference(sc, o, w, h, spp, seed=seed)
    r = FirstVertexRestated(sc, w, h, depth, seed)
    hits = 0
    for j in range(h):
        for i in range(w):
            a, n = ZERO3, ZERO3
            for s in range(spp):
                _, hit, _, (fa, fn) = r.path(i, j, s)
                a, n = add(a, fa), add(n, fn)
                hits += hit
            want_a = np.array([x / float(spp) for x in a])
            want_n = np.array([x / float(spp) for x in n])
            assert want_a.tobytes() == albedo[j, i].tobytes(), (i, j, want_a, albedo[j, i])
            assert want_n.tobytes() == normal[j, i].tobytes(), (i, j, want_n, normal[j, i])
    assert 0 < hits < w * h * spp  # both hits and misses are covered
    o.close()


# ------------------------------------------------------------------------------------------------------------ GPU ----

W, H, SPP, DEPTH, SEED = 64, 48, 2, 8, 3
EXAMPLES = ["three_balls", "more_balls", "more_balls_optimized", "two_balls", "earth", "one_triangle", "bunny", "glass_bunny"]


def nested(root_kind):
    from test_nested_hittables import nested_scene

    return nested_scene(3, root_kind)[0]


def make_scene(name):
    if name in ("zoo", "textured"):
        return zoo_scene() if name == "zoo" else textured_scene()
    if name.startswith("nested_"):
        return nested(name[len("nested_"):])
    return getattr(scenes, name)()


def assert_same_colour(g, w=W, h=H, spp=SPP, **kw):
    img, fg, albedo, normal, st = g.render_aov(w, h, spp, **kw)
    ref, fref, sref = g.render(w, h, spp, **kw)
    assert img.tobytes() == ref.tobytes() and fg.tobytes() == fref.tobytes()
    assert st.paths == sref.paths and st.rays == sref.rays
    return albedo, normal, st, sref


@pytest.mark.gpu
@pytest.mark.parametrize("name", EXAMPLES + ["demo", "bunny_lambert", "nested_bvh", "nested_list"])
def test_colour_and_foreground_are_rtp_render(gpu, name):
    with api.Scene(make_scene(name)) as g:
        albedo, normal, _, _ = assert_same_colour(g, max_bounce=DEPTH, seed=SEED)
        assert np.isfinite(albedo).all() and np.isfinite(normal).all()
        assert (normal != 0.0).any()


@pytest.mark.gpu
def test_small_frame_without_tail_mode(gpu):
    """32 x 32 x 16 = 16,384 paths: rtp_render runs one tail-mode launch, the AOV call trace/shade pairs; the same colour bytes"""
    with api.Scene(scenes.bunny_lambert()) as g:
        _, _, st, sref = assert_same_colour(g, 32, 32, 16, max_bounce=DEPTH, seed=SEED)
        assert sref.kernel_launches == 4  # generate, one tail-mode traversal, resolve, write
        assert st.kernel_launches > sref.kernel_launches


# scenes whose first-vertex albedo involves no uv-dependent lookup, and scenes whose albedo is a texture looked up by uv
EXACT = ["bunny_lambert", "three_balls", "one_triangle", "glass_bunny", "more_balls", "zoo", "nested_bvh", "nested_list"]
TEXTURED = ["textured", "earth", "demo"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", EXACT + TEXTURED)
def test_buffers_equal_the_oracle(gpu, name):
    sc = make_scene(name)
    o = oracle.Scene(sc, libm="device")
    with api.Scene(sc) as g:
        _, _, albedo, normal, _ = g.render_aov(W, H, SPP, max_bounce=DEPTH, seed=SEED)
    oa, on = first_vertex_reference(sc, o, W, H, SPP, seed=SEED)
    o.close()
    assert albedo.tobytes() == oa.tobytes()
    assert normal.tobytes() == on.tobytes()


@pytest.fixture(scope="module")
def demo(gpu):
    sc = scenes.demo()
    g = api.Scene(sc)
    yield sc, g, g.render_aov(W, H, 4, max_bounce=DEPTH, seed=SEED)
    g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["simple_kernel", "several_launches", "inorder"])
def test_buffers_are_the_same_whatever_the_path(demo, monkeypatch, variant):
    sc, _, ref = demo
    if variant == "simple_kernel":
        monkeypatch.setenv("RTP_RENDER_KERNEL", "simple")
    elif variant == "inorder":
        monkeypatch.setenv("RTP_TRAVERSAL", "inorder")
    else:
        monkeypatch.setenv("RTP_PATH_BUDGET", str(W * H + 5))  # one sample per launch: four launches
    with api.Scene(sc) as g:  # the switches are read when a scene is created; RTP_PATH_BUDGET at every call
        got = g.render_aov(W, H, 4, max_bounce=DEPTH, seed=SEED)
    for a, b in zip(got[:4], ref[:4]):
        assert a.tobytes() == b.tobytes()
    if variant == "several_launches":
        assert got[4].kernel_launches > ref[4].kernel_launches


@pytest.mark.gpu
@pytest.mark.parametrize("raw", [False, True])
def test_sample_range_equals_the_oracle(gpu, raw):
    sc = scenes.bunny_lambert()
    flags = A.RENDER_RAW_SUMS if raw else 0
    o = oracle.Scene(sc)
    want = first_vertex_reference(sc, o, W, H, 6, seed=SEED, sample_range=(2, 5), flags=flags)
    o.close()
    with api.Scene(sc) as g:
        got = g.render_aov(W, H, 6, max_bounce=DEPTH, seed=SEED, sample_range=(2, 5), flags=flags)
        ref = g.render(W, H, 6, max_bounce=DEPTH, seed=SEED, sample_range=(2, 5), flags=flags)
    for a, b in zip(got[:4], (*ref[:2], *want)):
        assert a.tobytes() == b.tobytes()


def sentinel_frame(w=W, h=H):
    return (np.full((h, w, 3), SENTINEL, dtype=np.uint64).view(np.float64), np.full((h, w), SENTINEL, dtype=np.uint64).view(np.float64),
            np.full((h, w, 3), SENTINEL, dtype=np.uint64).view(np.float64), np.full((h, w, 3), SENTINEL, dtype=np.uint64).view(np.float64))


def written(a):
    u = a.view(np.uint64)
    return (u != SENTINEL) if u.ndim == 2 else (u != SENTINEL).all(axis=-1)


@pytest.mark.gpu
@pytest.mark.parametrize("kw,mask", [
    (dict(tile=(9, 5, 37, 30)), (slice(5, 35), slice(9, 46))),
    (dict(tile=(4, 6, 50, 40), rows=(1, 3)), (slice(7, 46, 3), slice(4, 54))),
], ids=["tile", "tile_rows"])
def test_only_the_requested_pixels_are_written(demo, kw, mask):
    _, g, (ref_img, ref_fg, ref_a, ref_n, _) = demo
    out = sentinel_frame()
    g.render_aov(W, H, 4, max_bounce=DEPTH, seed=SEED, out=out, **kw)
    m = np.zeros((H, W), dtype=bool)
    m[mask] = True
    for buf, ref in zip(out, (ref_img, ref_fg, ref_a, ref_n)):
        assert (written(buf) == m).all()
        assert buf[m].tobytes() == ref[m].tobytes()


@pytest.mark.gpu
def test_null_buffers_are_accepted(demo):
    _, g, (ref_img, ref_fg, ref_a, ref_n, _) = demo
    img = np.zeros((H, W, 3))
    for fg, a, n in ((None, None, None), (None, np.zeros((H, W, 3)), None), (np.zeros((H, W)), None, np.zeros((H, W, 3)))):
        g.render_aov(W, H, 4, max_bounce=DEPTH, seed=SEED, out=(img, fg, a, n))
        assert img.tobytes() == ref_img.tobytes()
        for got, ref in ((fg, ref_fg), (a, ref_a), (n, ref_n)):
            assert got is None or got.tobytes() == ref.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("stats", [False, True])
def test_device_variant_on_a_stream(demo, stats):
    import torch

    sc, g, ref = demo
    n = W * H
    buf = torch.full((10 * n,), SENTINEL, dtype=torch.int64, device="cuda").view(torch.float64)
    p = api.render_params(W, H, 4, DEPTH, SEED)
    cam = api.Camera(W / H, sc.camera.fov, sc.camera.focal_dist, sc.camera.lens_radius, sc.camera.transformation)
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())  # the sentinel fill runs on the current stream
    base = buf.data_ptr()
    st = g.render_aov_device(p, cam, base, base + 3 * n * 8, base + 4 * n * 8, base + 7 * n * 8, stream.cuda_stream, stats=stats)
    stream.synchronize()
    a = buf.cpu().numpy()
    got = (a[:3 * n].reshape(H, W, 3), a[3 * n:4 * n].reshape(H, W), a[4 * n:7 * n].reshape(H, W, 3), a[7 * n:].reshape(H, W, 3))
    for x, y in zip(got, ref[:4]):
        assert x.tobytes() == y.tobytes()
    if stats:
        assert st.paths == ref[4].paths and st.rays == ref[4].rays and st.device_ms > 0.0


@pytest.mark.gpu
def test_one_scene_alternates_render_calls(gpu):
    """a long-lived scene serves rtp_render, rtp_render_aov and rtp_render_adaptive in turn (shared scratch, queues and staging
    frame); every result equals the same call on a fresh scene"""
    sc = scenes.demo()

    calls = [lambda g: g.render(W, H, 3, max_bounce=DEPTH, seed=SEED)[:2],
             lambda g: g.render_aov(W, H, 4, max_bounce=DEPTH, seed=SEED)[:4],
             lambda g: g.render_adaptive(W, H, 2, 6, 2, rel_tol=0.05, max_bounce=DEPTH, seed=SEED)[:3],
             lambda g: g.render_aov(32, 24, 2, max_bounce=3, seed=SEED + 1, tile=(3, 2, 20, 20))[:4],
             lambda g: g.render(96, 54, 2, max_bounce=DEPTH, seed=SEED)[:2]]
    with api.Scene(sc) as g:
        runs = [[call(g) for call in calls] for _ in range(2)]
    fresh = []
    for call in calls:
        with api.Scene(sc) as g:
            fresh.append(call(g))
    for run in runs:
        for got, want in zip(run, fresh):
            for a, b in zip(got, want):
                assert a.tobytes() == b.tobytes()


@pytest.mark.gpu
def test_two_devices_equal_one(gpu):
    if api.device_count() < 2:
        pytest.skip("needs two GPUs")
    with api.Scene(scenes.demo(), device_mask=0b11) as g:
        one = g.render_aov(W, H, 4, max_bounce=DEPTH, seed=SEED, device_mask=0b01)
        two = g.render_aov(W, H, 4, max_bounce=DEPTH, seed=SEED)
        for a, b in zip(one[:4], two[:4]):
            assert a.tobytes() == b.tobytes()
        assert one[4].paths == two[4].paths


INVALID = {
    "null_scene": dict(null="scene"),
    "null_camera": dict(null="camera"),
    "null_params": dict(null="params"),
    "null_rgb": dict(null="rgb"),
    "transparent_flag": dict(p=dict(flags=A.RENDER_TRANSPARENT)),
    "unknown_flag": dict(p=dict(flags=8)),
    "tile_outside_frame": dict(p=dict(tile_x=W - 4, tile_w=8)),
    "max_bounce_zero": dict(p=dict(max_bounce=0)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(INVALID))
@pytest.mark.parametrize("entry", ["host", "device"])
def test_invalid_arguments(demo, case, entry):
    sc, g, ref = demo
    spec = INVALID[case]
    p = api.render_params(W, H, 4, DEPTH, SEED)
    for k, v in spec.get("p", {}).items():
        setattr(p, k, v)
    cam = api.Camera(W / H, sc.camera.fov, sc.camera.focal_dist, sc.camera.lens_radius, sc.camera.transformation).to_c()
    null = spec.get("null")
    lib = A.load()
    scene = None if null == "scene" else g.handle
    cam_arg = None if null == "camera" else C.byref(cam)
    p_arg = None if null == "params" else C.byref(p)
    if entry == "host":
        rgb = np.zeros((H, W, 3))
        rc = lib.rtp_render_aov(scene, cam_arg, p_arg, None if null == "rgb" else A.ptr(rgb), None, None, None, None)
    else:
        import torch

        d = torch.zeros(3 * W * H, dtype=torch.float64, device="cuda")
        rc = lib.rtp_render_aov_device(scene, cam_arg, p_arg, None if null == "rgb" else d.data_ptr(), None, None, None, None, None)
        torch.cuda.synchronize()
    assert rc == A.ERR_INVALID, (lib.rtp_last_error() or b"").decode()
    got = g.render_aov(W, H, 4, max_bounce=DEPTH, seed=SEED)  # the scene is still usable
    for a, b in zip(got[:4], ref[:4]):
        assert a.tobytes() == b.tobytes()
