"""The render paths the benchmark times, and the state a scene keeps between render calls.

- rtp_render_device as bench.py calls it: one caller-owned device buffer (rgb of the whole frame, then foreground), rows dealt
  out over ranks, raw sums over sample ranges, repeated calls into the same buffer, a non-default stream, a small tile.
- Frames split into several wavefront launches, including a frame whose last launch is small enough for tail mode.
- Counted renders (RTP_RENDER_COUNTERS), which run the counting instantiations of every traversal and integrator kernel.
- One scene serving calls of changing shape: the integrator's queues are sized per call and must stay within their budget.
- The sRGB output stage when every pixel is borderline, so that the host fix-up list does all the work.

Equality against the library's own other paths is bit for bit; against the oracle it is the image tolerance of
test_gpu_parity.py. Device outputs are torch buffers filled with a NaN of a distinctive payload, with CANARY words of it past
their end, so that a stray write or a missing one shows.
"""
import numpy as np
import pytest

import oracle
from rtp_b200 import _abi as A
from rtp_b200 import api, scenes
from rtp_b200.api import Absorb, Camera, Emit, ExampleScene, Hittable, Material, Scatter, SceneData, Transformation
from test_gpu_parity import IMG_FRAC, IMG_RMSE, assert_hits_equal, image_report

pytestmark = pytest.mark.gpu

SENTINEL = 0x7FF8_DEAD_BEEF_0001  # bits of a quiet NaN whose payload no computation produces
CANARY = 64                        # sentinel words past the end of every device output


def sentinel_words(n):
    """a float64 device buffer of n words + CANARY, every word the sentinel"""
    import torch

    return torch.full((n + CANARY,), SENTINEL, dtype=torch.int64, device="cuda").view(torch.float64)


def unwritten(buf):
    """numpy bool per word of buf: still the sentinel"""
    import torch

    return buf.view(torch.int64).cpu().numpy() == SENTINEL


def frame_views(a, w, h):
    """bench.py's layout of a w x h frame in a flat array: (rgb [h, w, 3], foreground [h, w], the words past the frame)"""
    n = w * h
    return a[: 3 * n].reshape(h, w, 3), a[3 * n: 4 * n].reshape(h, w), a[4 * n:]


def camera_for(sc, w, h):
    """the camera Scene.render builds: the scene's camera with aspect = w / h (main.rs:22)"""
    c = sc.camera
    return Camera(w / h, c.fov, c.focal_dist, c.lens_radius, c.transformation)


def render_into(g, sc, buf, w, h, spp, depth=8, seed=1, stream=None, stats=False, **params):
    """one rtp_render_device call into buf (rgb, then foreground at word 3 * w * h), waited for"""
    import torch

    p = api.render_params(w, h, spp, depth, seed, **params)
    d_rgb = buf.data_ptr()
    d_fg = d_rgb + 3 * w * h * 8
    if stream is None:
        st = g.render_device(p, camera_for(sc, w, h), d_rgb, d_fg, stats=stats)
        torch.cuda.synchronize()
    else:
        stream.wait_stream(torch.cuda.current_stream())  # the sentinel fill runs on the current stream
        st = g.render_device(p, camera_for(sc, w, h), d_rgb, d_fg, stream.cuda_stream, stats=stats)
        stream.synchronize()
    return st


def assert_matches_oracle(img, fg, io, fo):
    rep = image_report(img, io)
    assert rep["rmse"] <= IMG_RMSE and rep["differing"] <= max(1, IMG_FRAC * rep["pixels"]), rep
    assert (fg == fo).all()


def wave_launches(depth):
    """kernels of one trace/shade launch of the integrator: generate, a traversal and a shade kernel per bounce, resolve"""
    return 2 + 2 * depth


TAIL_LAUNCHES = 3  # generate, ONE tail-mode traversal, resolve


# ---------------------------------------------------------------------------------------------------------------------
# 1. rtp_render_device as bench.py calls it
# ---------------------------------------------------------------------------------------------------------------------

W1, H1, SPP1, DEPTH1 = 320, 180, 4, 8  # 230,400 paths: one trace/shade launch of the wavefront integrator


@pytest.fixture(scope="module", params=["bunny_lambert", "three_balls"])
def bench_scene(request, gpu):
    """(scene, device scene, Scene.render's frame): the any-order BVH walk, and a List root under a thin lens"""
    sc = getattr(scenes, request.param)()
    g = api.Scene(sc)
    host = g.render(W1, H1, SPP1, max_bounce=DEPTH1, seed=1)
    yield sc, g, host
    g.close()


def test_render_device_full_frame(bench_scene):
    """a full-frame call equals Scene.render bit for bit and the oracle within tolerance; the warm-up and timed steps of the
    benchmark (three calls into one buffer), a call with stats and a call on another stream give the same bits"""
    import torch

    sc, g, (ih, fh, sh) = bench_scene
    w, h, spp = W1, H1, SPP1
    buf = sentinel_words(4 * w * h)
    render_into(g, sc, buf, w, h, spp)
    a = buf.cpu().numpy()
    rgb, fg, _ = frame_views(a, w, h)
    assert rgb.tobytes() == ih.tobytes() and fg.tobytes() == fh.tobytes()
    left = unwritten(buf)
    assert not left[: 4 * w * h].any() and left[4 * w * h:].all()
    o = oracle.Scene(sc)
    io, fo, _ = o.render(w, h, spp, max_bounce=DEPTH1, seed=1)
    o.close()
    assert_matches_oracle(rgb, fg, io, fo)

    first = buf.view(torch.int64).clone()
    for _ in range(2):
        render_into(g, sc, buf, w, h, spp)
        assert torch.equal(buf.view(torch.int64), first)

    st = render_into(g, sc, buf, w, h, spp, stats=True)
    assert torch.equal(buf.view(torch.int64), first)
    assert st.paths == w * h * spp and st.rays == sh.rays
    assert st.kernel_launches == wave_launches(DEPTH1) + 1  # one trace/shade launch, then the frame write
    assert 0 < st.trace_ms <= st.device_ms

    other = torch.cuda.Stream()
    buf2 = sentinel_words(4 * w * h)
    render_into(g, sc, buf2, w, h, spp, stream=other)
    assert torch.equal(buf2.view(torch.int64), first)


@pytest.mark.parametrize("n", [2, 3])
def test_render_device_rows_dealt_out(bench_scene, n):
    """the strong-scaling split: call r of n renders rows r::n into the full-frame buffer and writes nothing else; all n
    calls together give the one-call frame bit for bit"""
    sc, g, (ih, fh, _) = bench_scene
    w, h, spp = W1, H1, SPP1
    buf = sentinel_words(4 * w * h)
    row = np.arange(h)
    for r in range(n):
        render_into(g, sc, buf, w, h, spp, rows=(r, n))
        rgb_left, fg_left, tail_left = frame_views(unwritten(buf), w, h)
        done = row % n <= r
        assert not rgb_left[done].any() and rgb_left[~done].all(), r
        assert not fg_left[done].any() and fg_left[~done].all(), r
        assert tail_left.all()
    rgb, fg, _ = frame_views(buf.cpu().numpy(), w, h)
    assert rgb.tobytes() == ih.tobytes() and fg.tobytes() == fh.tobytes()


@pytest.mark.parametrize("n", [2, 4])
def test_render_device_sample_ranges(bench_scene, n):
    """the weak-scaling split: raw sums over sample ranges [r s, (r + 1) s) equal Scene.render of the same range bit for bit,
    and their sum over the ranges, divided by spp, is the frame up to f64 re-association"""
    sc, g, (ih, fh, _) = bench_scene
    w, h, spp = W1, H1, SPP1
    s = spp // n
    total, total_fg = np.zeros((h, w, 3)), np.zeros((h, w))
    for r in range(n):
        buf = sentinel_words(4 * w * h)
        render_into(g, sc, buf, w, h, spp, sample_begin=r * s, sample_end=(r + 1) * s, flags=A.RENDER_RAW_SUMS)
        rgb, fg, tail = frame_views(buf.cpu().numpy(), w, h)
        hr, hf, _ = g.render(w, h, spp, max_bounce=DEPTH1, seed=1, sample_range=(r * s, (r + 1) * s), flags=A.RENDER_RAW_SUMS)
        assert rgb.tobytes() == hr.tobytes() and fg.tobytes() == hf.tobytes(), r
        assert (tail.view(np.int64) == SENTINEL).all()
        total += rgb
        total_fg += fg
    assert np.allclose(total / spp, ih, rtol=1e-14, atol=1e-15)
    assert np.allclose(total_fg / spp, fh, rtol=1e-14, atol=1e-15)


def test_render_device_tile_is_one_tail_launch(bench_scene):
    """a 48 x 32 tile (6,144 paths) is finished by one tail-mode launch and writes its rectangle of the frame, nothing else"""
    sc, g, (ih, fh, _) = bench_scene
    w, h, spp = W1, H1, SPP1
    x, y, tw, th = tile = (101, 67, 48, 32)
    buf = sentinel_words(4 * w * h)
    st = render_into(g, sc, buf, w, h, spp, tile=tile, stats=True)
    assert st.paths == tw * th * spp and st.kernel_launches == TAIL_LAUNCHES + 1
    inside = np.zeros((h, w), dtype=bool)
    inside[y:y + th, x:x + tw] = True
    rgb_left, fg_left, tail_left = frame_views(unwritten(buf), w, h)
    assert not rgb_left[inside].any() and rgb_left[~inside].all()
    assert not fg_left[inside].any() and fg_left[~inside].all()
    assert tail_left.all()
    rgb, fg, _ = frame_views(buf.cpu().numpy(), w, h)
    assert rgb[inside].tobytes() == ih[inside].tobytes() and fg[inside].tobytes() == fh[inside].tobytes()


# ---------------------------------------------------------------------------------------------------------------------
# 2. frames split into several wavefront launches
# ---------------------------------------------------------------------------------------------------------------------

TAIL_THRESHOLD = 65536  # DeviceScene::tail_threshold: a launch of at most this many paths runs in tail mode

SPLITS = {  # frame size, spp, paths per launch (RTP_PATH_BUDGET) as a function of the pixel count
    "all_wave": (480, 270, 5, lambda npix: 2 * npix),        # 2 + 2 + 1 spp: 259,200 / 259,200 / 129,600 paths
    "wave_then_tail": (320, 180, 5, lambda npix: 2 * npix),  # 115,200 / 115,200 / 57,600 paths: the last launch in tail mode
    "uneven": (480, 270, 5, lambda npix: 3 * npix + 5),      # 3 + 2 spp
}


@pytest.mark.parametrize("case", list(SPLITS))
@pytest.mark.parametrize("name", ["bunny_lambert", "three_balls"])
def test_frame_split_into_several_launches(gpu, monkeypatch, name, case):
    """a frame traced in several launches adds their samples in sample order: the same bits as the one-launch frame, whether
    the launches are all trace/shade launches or the last one runs in tail mode"""
    w, h, spp, budget = SPLITS[case]
    npix, depth = w * h, 8
    sc = getattr(scenes, name)()
    g = api.Scene(sc)
    ref, fref, sref = g.render(w, h, spp, max_bounce=depth, seed=12)
    assert sref.kernel_launches == wave_launches(depth) + 1
    per_launch = budget(npix) // npix
    monkeypatch.setenv("RTP_PATH_BUDGET", str(budget(npix)))
    img, fg, st = g.render(w, h, spp, max_bounce=depth, seed=12)
    monkeypatch.delenv("RTP_PATH_BUDGET")
    assert img.tobytes() == ref.tobytes() and fg.tobytes() == fref.tobytes() and st.rays == sref.rays
    launches = [npix * min(per_launch, spp - s0) for s0 in range(0, spp, per_launch)]
    assert len(launches) > 1
    assert (launches[-1] <= TAIL_THRESHOLD) == (case == "wave_then_tail")
    assert st.kernel_launches == sum(TAIL_LAUNCHES if n <= TAIL_THRESHOLD else wave_launches(depth) for n in launches) + 1
    assert st.kernel_launches > sref.kernel_launches
    x, y, cw, ch = crop = (200, 100, 64, 48)
    o = oracle.Scene(sc)
    io, fo, _ = o.render(w, h, spp, max_bounce=depth, seed=12, tile=crop)
    o.close()
    sl = (slice(y, y + ch), slice(x, x + cw))
    assert_matches_oracle(img[sl], fg[sl], io[sl], fo[sl])
    g.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. counted renders
# ---------------------------------------------------------------------------------------------------------------------

COUNTED = [  # scene, frame, depth, environment at scene creation: the counting instantiation each case runs
    ("bunny_lambert", 320, 180, 4, 8, {}),                                 # trace_any_kernel<true, OUT_WAVE>
    ("bunny_lambert", 64, 48, 2, 8, {}),                                   # trace_persistent_kernel<true, OUT_TAIL, false>
    ("three_balls", 320, 180, 4, 8, {}),                                   # trace_persistent_kernel<true, OUT_WAVE, true>
    ("three_balls", 64, 48, 2, 8, {}),                                     # trace_persistent_kernel<true, OUT_TAIL, true>
    ("bunny_lambert", 320, 180, 4, 8, {"RTP_TRAVERSAL": "inorder"}),       # trace_persistent_kernel<true, OUT_WAVE, false>
    ("bunny_lambert", 160, 90, 2, 8, {"RTP_RENDER_KERNEL": "simple"}),     # render_paths_kernel<8, true>
    ("bunny_lambert", 160, 90, 2, 32, {"RTP_RENDER_KERNEL": "simple"}),    # render_paths_kernel<32, true>
    ("bunny_lambert", 160, 90, 2, 128, {"RTP_RENDER_KERNEL": "simple"}),   # render_paths_kernel<128, true>
]


@pytest.mark.parametrize("name,w,h,spp,depth,env", COUNTED,
                         ids=[f"{c[0]}-{c[1]}x{c[2]}-d{c[4]}-{'-'.join(c[5].values()) or 'default'}" for c in COUNTED])
def test_counted_render_changes_no_bit(gpu, monkeypatch, name, w, h, spp, depth, env):
    """RTP_RENDER_COUNTERS only adds counting: the image, the foreground and the ray count are those of the uncounted render,
    the f32 culling never rejected a box the exact test accepts, and the counters show the work of the scene's root"""
    sc = getattr(scenes, name)()
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    g = api.Scene(sc)  # the traversal and the integrator are chosen when the scene is created
    for k in env:
        monkeypatch.delenv(k)
    img, fg, st = g.render(w, h, spp, max_bounce=depth, seed=9)
    ic, fc, sc_ = g.render(w, h, spp, max_bounce=depth, seed=9, flags=A.RENDER_COUNTERS)
    assert ic.tobytes() == img.tobytes() and fc.tobytes() == fg.tobytes() and sc_.rays == st.rays
    assert sc_.paths == st.paths == w * h * spp
    assert (st.node_visits, st.triangle_tests, st.sphere_tests) == (0, 0, 0)  # uncounted: nothing but rays
    assert sc_.conservative_violations == 0
    if name == "bunny_lambert":
        assert sc_.node_visits > 0 and sc_.triangle_tests > 0
    else:
        assert sc_.node_visits == 0 and sc_.sphere_tests > 0  # a List root has no nodes
    g.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. one scene, calls of changing shape
# ---------------------------------------------------------------------------------------------------------------------

def test_one_scene_serves_calls_of_changing_shape(gpu):
    """The integrator's queues are kept between calls and grown on demand. A big shallow frame followed by a small deep one
    must not leave the scene holding (big capacity) x (deep stack) - 204 GB for 1080p x 16 spp followed by depth 128 - and
    whatever a call reallocates, every call returns what a fresh scene making only that call returns."""
    import torch

    sc = scenes.bunny_lambert()
    g, o = api.Scene(sc), oracle.Scene(sc)

    def fresh(call):
        with api.Scene(sc) as f:  # closed at once: the big frames hold about 8.5 GB of queues
            return call(f)

    def same(a, b):
        return all(x.tobytes() == y.tobytes() for x, y in zip(a[:2], b[:2])) and a[2].rays == b[2].rays

    def big(s):
        return s.render(1920, 1080, 16, max_bounce=1, seed=3)

    def deep(s):
        return s.render(64, 48, 2, max_bounce=128, seed=4)

    # 1, 2, 3: a full launch of depth 1, then a small one of depth 128, then the first again
    r1 = big(g)
    assert same(r1, fresh(big))
    del r1
    r2 = deep(g)
    assert same(r2, fresh(deep))
    io, fo, _ = o.render(64, 48, 2, max_bounce=128, seed=4)
    assert_matches_oracle(r2[0], r2[1], io, fo)
    r3 = big(g)
    assert same(r3, fresh(big))
    del r3

    # 4: a tile of a C1-sized frame
    tile = (100, 40, 200, 120)

    def tiled(s):
        return s.render(640, 360, 4, max_bounce=8, seed=5, tile=tile)

    r4 = tiled(g)
    assert same(r4, fresh(tiled))
    io, fo, _ = o.render(640, 360, 4, max_bounce=8, seed=5, tile=tile)
    sl = (slice(tile[1], tile[1] + tile[3]), slice(tile[0], tile[0] + tile[2]))
    assert_matches_oracle(r4[0][sl], r4[1][sl], io[sl], fo[sl])

    # 5: closest hits through the host-buffer calls: two pipeline chunks, the full hit record, camera rays
    rays = scenes.incoherent_rays((1 << 18) + 1, first=77)
    h5 = g.hit(rays)
    assert h5.tobytes() == fresh(lambda f: f.hit(rays)).tobytes()
    assert_hits_equal(h5, o.hit(rays), "hit")
    few = rays[:1000]
    hf = g.hit_full(few)
    assert hf.tobytes() == fresh(lambda f: f.hit_full(few)).tobytes()
    assert_hits_equal(hf, o.hit_full(few), "hit_full")
    cam = camera_for(sc, 7, 3)
    hc = g.hit_camera(cam, 7, 3)
    assert hc.tobytes() == fresh(lambda f: f.hit_camera(cam, 7, 3)).tobytes()
    assert_hits_equal(hc, o.hit(oracle.camera_rays(cam, 7, 3)), "hit_camera")

    # 6: device batches on three streams at once, into buffers with canary tails
    sizes = (1, 300_000, 129)
    batches = [scenes.incoherent_rays(n, first=1000 + 7 * n) for n in sizes]
    d_rays = [torch.from_numpy(b.view(np.float64).reshape(-1, 8)).cuda() for b in batches]
    outs = [sentinel_words(2 * n) for n in sizes]
    streams = [torch.cuda.Stream() for _ in sizes]
    for s, r, out, n in zip(streams, d_rays, outs, sizes):
        s.wait_stream(torch.cuda.current_stream())
        g.hit_device(r.data_ptr(), n, out.data_ptr(), s.cuda_stream)
    torch.cuda.synchronize()
    for b, r, out, n in zip(batches, d_rays, outs, sizes):
        left = unwritten(out)
        assert not left[: 2 * n].any() and left[2 * n:].all(), n
        ref = sentinel_words(2 * n)

        def one(f, r=r, ref=ref, n=n):
            f.hit_device(r.data_ptr(), n, ref.data_ptr())
            torch.cuda.synchronize()

        fresh(one)
        assert torch.equal(out.view(torch.int64), ref.view(torch.int64)), n
        if n < 1000:
            assert_hits_equal(out[: 2 * n].cpu().numpy().view(A.HIT_DTYPE), o.hit(b), f"hit_device {n}")

    # 7: the 8-bit output stage with a transparent background
    def srgb(s):
        return s.render_srgb8(200, 120, 3, max_bounce=8, seed=6, transparent_background=True)[0]

    r7 = srgb(g)
    assert r7.tobytes() == fresh(srgb).tobytes()
    io, fo, _ = o.render(200, 120, 3, max_bounce=8, seed=6)
    ref7 = oracle.to_srgb_u8(io)
    ref7[..., 3] = np.minimum(255.0 * fo, 255.0).astype(np.uint8)
    differ = (r7 != ref7).any(axis=-1)
    assert differ.sum() <= max(1, IMG_FRAC * differ.size)

    # 8: the deep call again
    assert same(deep(g), r2)
    g.close(); o.close()


# ---------------------------------------------------------------------------------------------------------------------
# 5. the sRGB fix-up list under load
# ---------------------------------------------------------------------------------------------------------------------

FIX_CAP = 65536  # pixels of one rtp_render_srgb8 call that the host fix-up list holds (rtp.h)


def borderline_scene():
    """Emissive spheres in a grid in front of the camera, on an emissive background. Every channel of every colour is
    (n / 255)^2.2 for a distinct level n in 1..254, so 255 x^(1/2.2) of a pixel that sees one colour is an integer to ~1e-12
    and the device sends it to the host fix-up list."""
    nx, ny = 8, 6
    levels = np.random.default_rng(5).permutation(np.arange(1, 255))[: 3 * (nx * ny + 1)].reshape(-1, 3)
    colours = (levels / 255.0) ** 2.2
    materials = [Material.new(Scatter.NONE, Absorb.BlackBody, Emit.Color(c)) for c in colours[1:]]
    spheres = [Hittable.Sphere([ix - 3.5, iy - 2.5, -4.0], 0.42, iy * nx + ix) for iy in range(ny) for ix in range(nx)]
    camera = Camera(4.0 / 3.0, np.pi / 2, 1.0, 0.0, Transformation.lookat([0.0, 0.0, 0.0], [0.0, 0.0, -1.0], [0.0, 1.0, 0.0]))
    return ExampleScene(camera, SceneData(materials, [], []), "bvh", Hittable.concat(spheres), Emit.Color(colours[0]))


@pytest.fixture(scope="module")
def borderline(gpu):
    sc = borderline_scene()
    g, o = api.Scene(sc), oracle.Scene(sc)
    yield sc, g, o
    g.close(); o.close()


@pytest.mark.parametrize("spp", [1, 2])
def test_srgb8_fixups_of_every_pixel(borderline, spp):
    """render_srgb8 equals to_srgb_u8 of the f64 frame (this library's and the oracle's), opaque and transparent, when the
    fix-up list holds every pixel (1 spp) or every pixel but the silhouettes (2 spp)"""
    sc, g, o = borderline
    w, h = 200, 150
    frame, fg, _ = g.render(w, h, spp)
    io, fo, _ = o.render(w, h, spp)
    assert frame.tobytes() == io.tobytes() and fg.tobytes() == fo.tobytes()  # emission only: exact sums
    y = 255.0 * frame ** (1.0 / 2.2)
    near = (np.abs(y - np.rint(y)) < 1e-9).any(axis=-1)
    assert near.all() if spp == 1 else near.mean() > 0.8  # the premise: the pixels are borderline
    rgba, st = g.render_srgb8(w, h, spp)
    assert rgba.tobytes() == api.to_srgb_u8(frame).tobytes()
    assert rgba.tobytes() == oracle.to_srgb_u8(io).tobytes()
    ta, _ = g.render_srgb8(w, h, spp, transparent_background=True)
    assert ta[..., :3].tobytes() == rgba[..., :3].tobytes()
    assert (ta[..., 3] == np.minimum(255.0 * fo, 255.0).astype(np.uint8)).all()
    assert (ta[..., 3] == 255).mean() < 0.9 and (ta[..., 3] == 0).mean() < 0.9  # spheres and background both seen


@pytest.mark.parametrize("part", ["tile", "rows", "tile_rows"])
def test_srgb8_fixups_land_on_their_own_pixels(borderline, part):
    """a tile or a row split writes only its own pixels, fix-ups included: the fix-up list holds frame pixel indices"""
    sc, g, o = borderline
    w, h = 200, 150
    full, _ = g.render_srgb8(w, h, 1)
    kw, mine = {}, np.zeros((h, w), dtype=bool)
    if part in ("tile", "tile_rows"):
        x, y, tw, th = kw["tile"] = (37, 21, 90, 60)
    else:
        x, y, tw, th = 0, 0, w, h
    if part in ("rows", "tile_rows"):
        kw["rows"] = (1, 3)
        mine[y + 1:y + th:3, x:x + tw] = True
    else:
        mine[y:y + th, x:x + tw] = True
    out = np.full((h, w, 4), 0xA5, dtype=np.uint8)
    g.render_srgb8(w, h, 1, out=out, **kw)
    assert (out[~mine] == 0xA5).all()
    assert out[mine].tobytes() == full[mine].tobytes()


def test_srgb8_fixup_cap(borderline):
    """a call with more than 65,536 borderline pixels is refused with RTP_ERR_UNSUPPORTED; the cap counts the pixels of the
    call, so a 200 x 200 tile of that frame succeeds, and the scene renders correctly afterwards"""
    sc, g, o = borderline
    w, h = 320, 240
    assert w * h > FIX_CAP
    with pytest.raises(api.RtpError) as e:
        g.render_srgb8(w, h, 1)
    assert e.value.code == A.ERR_UNSUPPORTED
    frame, _, _ = g.render(w, h, 1)
    x, y, tw, th = tile = (60, 20, 200, 200)
    assert tw * th <= FIX_CAP
    out = np.zeros((h, w, 4), dtype=np.uint8)
    g.render_srgb8(w, h, 1, tile=tile, out=out)
    assert out[y:y + th, x:x + tw].tobytes() == api.to_srgb_u8(frame)[y:y + th, x:x + tw].tobytes()
    small, _, _ = g.render(200, 150, 1)
    rgba, _ = g.render_srgb8(200, 150, 1)
    assert rgba.tobytes() == api.to_srgb_u8(small).tobytes()
