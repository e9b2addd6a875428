"""rtp_render_adaptive: rounds of samples over the pixels that have not converged (include/rtp.h, DESIGN.md §6b).

The reference for the stop decisions is `stop_counts` below, a numpy model of the stop rule that works on per-sample colours in the
rule's own operation order. On the CPU it is checked on oracle colours; on the GPU the library's decisions must equal the model
applied to the GPU's own per-sample colours (rtp_render of one-sample ranges with RTP_RENDER_RAW_SUMS: the GPU's atan2 / asin may
differ from the host libm by an ulp, so the oracle's colours are not the input for that check). The pixels themselves are checked
bit for bit against rtp_render at each pixel's own sample count.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle
from rtp_b200 import _abi as A
from rtp_b200 import api, scenes
from test_gpu_parity import IMG_FRAC, IMG_RMSE, image_report

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "rtp.h")

SENTINEL = 0x7FF8_DEAD_BEEF_0002  # bits of a quiet NaN whose payload no computation produces
SENTINEL_N = 0xFFFFFFFF           # samples_out words nobody wrote


def luminance(c):
    """Y_s = (0.2126 * r + 0.7152 * g) + 0.0722 * b, per sample"""
    return (0.2126 * c[..., 0] + 0.7152 * c[..., 1]) + 0.0722 * c[..., 2]


def stop_counts(colors, min_samples, max_samples, batch, abs_tol, rel_tol):
    """numpy model of the stop rule: colors [n_samples >= max_samples, H, W, 3] per-sample colours -> n_p [H, W]"""
    y = luminance(colors[:max_samples])
    shape = y.shape[1:]
    s1, s2 = np.zeros(shape), np.zeros(shape)
    counts = np.zeros(shape, dtype=np.uint32)
    live = np.ones(shape, dtype=bool)
    n, b = 0, min_samples
    with np.errstate(all="ignore"):
        while True:
            for s in range(n, n + b):
                s1 = np.where(live, s1 + y[s], s1)
                s2 = np.where(live, s2 + y[s] * y[s], s2)
            n += b
            nd = float(n)
            mean = s1 / nd
            var = (s2 - s1 * mean) / (nd - 1.0)
            tol = abs_tol + rel_tol * np.abs(mean)
            stop = (n >= max_samples) | ((n >= 2) & (var / nd <= tol * tol))
            counts[live & stop] = n
            live &= ~stop
            if not live.any() or n >= max_samples:
                return counts
            b = min(batch, max_samples - n)


# ------------------------------------------------------------------------------------------------------------ CPU ----


def test_adaptive_params_layout_matches_the_header(tmp_path):
    """compile include/rtp.h as plain C and compare sizeof / offsetof of rtp_adaptive_params with the ctypes mirror"""
    fields = ["min_samples", "max_samples", "batch", "abs_tol", "rel_tol"]
    src = ["#include <stdio.h>", "#include <stddef.h>", f'#include "{HEADER}"', "int main(void){",
           'printf("size %zu\\n", sizeof(rtp_adaptive_params));']
    src += [f'printf("{f} %zu\\n", offsetof(rtp_adaptive_params, {f}));' for f in fields]
    src.append("return 0;}")
    c = tmp_path / "layout.c"
    c.write_text("\n".join(src))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(c)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(A.AdaptiveParams) == 32
    for f in fields:
        assert int(got[f]) == getattr(A.AdaptiveParams, f).offset, f
    assert A.PROTOTYPES["rtp_render_adaptive"][1][3] == C.POINTER(A.AdaptiveParams)


@pytest.fixture(scope="module")
def oracle_samples():
    """per-sample colours of a 16 x 12 three_balls frame from the CPU oracle, [8, 12, 16, 3]"""
    sc = scenes.three_balls()
    o = oracle.Scene(sc)
    out = np.stack([o.render(16, 12, 1, max_bounce=8, seed=3, sample_range=(s, s + 1), flags=A.RENDER_RAW_SUMS)[0] for s in range(8)])
    o.close()
    return out


def test_model_min_equals_max(oracle_samples):
    assert (stop_counts(oracle_samples, 5, 5, 3, 1e9, 1e9) == 5).all()


@pytest.mark.parametrize("min_samples,batch,expect", [(1, 1, 2), (2, 3, 2), (3, 4, 3)])
def test_model_huge_tolerance_stops_at_the_first_allowed_count(oracle_samples, min_samples, batch, expect):
    """n >= 2 is needed for a variance: min_samples = 1 stops after the next round, any larger min_samples at min_samples"""
    assert (stop_counts(oracle_samples, min_samples, 8, batch, 1e100, 0.0) == expect).all()


def test_model_zero_tolerance_runs_noisy_pixels_to_max(oracle_samples):
    n = stop_counts(oracle_samples, 2, 8, 2, 0.0, 0.0)
    y = luminance(oracle_samples)
    noisy = (y[:2] != y[0]).any(axis=0)
    assert noisy.sum() > 0.5 * noisy.size
    assert (n[noisy] == 8).all()


def test_model_nan_sample_runs_its_pixel_to_max(oracle_samples):
    c = oracle_samples.copy()
    c[1, 5, 7, 0] = np.nan
    c[0, 2, 2, 2] = np.inf  # both inside round 1: a later one would come after the pixel has stopped
    n = stop_counts(c, 2, 8, 2, 1e100, 0.0)
    assert n[5, 7] == 8 and n[2, 2] == 8
    n[5, 7] = n[2, 2] = 2
    assert (n == 2).all()


# ------------------------------------------------------------------------------------------------------------ GPU ----

W, H, DEPTH, SEED = 64, 48, 8, 7
MIN, MAX, BATCH = 4, 32, 4


def per_sample_colors(g, w, h, n, seed=SEED, depth=DEPTH):
    """[n, h, w, 3]: the GPU's colour of every sample s < n (rtp_render of the range [s, s + 1), raw sums)"""
    return np.stack([g.render(w, h, 1, max_bounce=depth, seed=seed, sample_range=(s, s + 1), flags=A.RENDER_RAW_SUMS)[0] for s in range(n)])


class Case:
    """a scene with its GPU per-sample colours and a rel_tol for which the model gives at least three distinct counts, MIN and MAX
    among them"""

    def __init__(self, name):
        self.sc = getattr(scenes, name)()
        self.g = api.Scene(self.sc)
        self.colors = per_sample_colors(self.g, W, H, MAX)
        for rel in (0.3, 0.1, 0.03, 0.01, 0.003):
            n = stop_counts(self.colors, MIN, MAX, BATCH, 0.0, rel)
            if len(np.unique(n)) >= 3 and n.min() == MIN and n.max() == MAX:
                self.rel, self.model = rel, n
                break
        else:
            raise AssertionError(f"{name}: no tolerance gives three distinct sample counts")

    def render(self, **kw):
        return self.g.render_adaptive(W, H, MIN, MAX, BATCH, rel_tol=self.rel, max_bounce=DEPTH, seed=SEED, **kw)


@pytest.fixture(scope="module")
def cases(gpu):
    made = {}

    def get(name):
        if name not in made:
            made[name] = Case(name)
        return made[name]

    yield get
    for c in made.values():
        c.g.close()


def assert_equals_fixed_renders(g, img, fg, samples, mask, raw=False, w=W, h=H, seed=SEED, depth=DEPTH):
    """at every pixel of mask, rgb and fg equal rtp_render(num_samples = n_p, sample_range = [0, n_p)) bit for bit"""
    groups = np.unique(samples[mask])
    for n in groups:
        ref, fref, _ = g.render(w, h, int(n), max_bounce=depth, seed=seed, sample_range=(0, int(n)), flags=A.RENDER_RAW_SUMS if raw else 0)
        sel = mask & (samples == n)
        assert img[sel].tobytes() == ref[sel].tobytes(), f"rgb differs at n_p = {n}"
        assert fg[sel].tobytes() == fref[sel].tobytes(), f"foreground differs at n_p = {n}"
    return groups


def sentinel_frame(w=W, h=H):
    rgb = np.full((h, w, 3), SENTINEL, dtype=np.uint64).view(np.float64)
    fg = np.full((h, w), SENTINEL, dtype=np.uint64).view(np.float64)
    n = np.full((h, w), SENTINEL_N, dtype=np.uint32)
    return rgb, fg, n


def unwritten(rgb, fg, n):
    return (rgb.view(np.uint64) == SENTINEL).all(axis=-1) & (fg.view(np.uint64) == SENTINEL) & (n == SENTINEL_N)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["demo", "bunny_lambert"])
def test_every_pixel_equals_rtp_render_at_its_own_count(cases, name):
    c = cases(name)
    img, fg, n, st = c.render()
    assert (n == c.model).all(), "the device's stop decisions differ from the model on the device's own colours"
    groups = assert_equals_fixed_renders(c.g, img, fg, n, np.ones((H, W), dtype=bool))
    assert len(groups) >= 3 and groups[0] == MIN and groups[-1] == MAX
    assert st.paths == int(n.astype(np.uint64).sum())
    assert st.rays > 0 and st.kernel_launches > 0


VARIANTS = {
    "tile": dict(tile=(9, 5, 37, 30)),
    "rows": dict(rows=(1, 3)),
    "raw_sums": dict(raw_sums=True),
    "simple_kernel": dict(),
    "several_launches_per_round": dict(),
    "device_buffers": dict(),
}


def region(kw):
    """pixels a call with these parameters writes"""
    m = np.zeros((H, W), dtype=bool)
    if "tile" in kw:
        x, y, w, h = kw["tile"]
        m[y:y + h, x:x + w] = True
    elif "rows" in kw:
        off, stride = kw["rows"]
        m[off::stride, :] = True
    else:
        m[:] = True
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_variants_are_exact(cases, monkeypatch, variant):
    c = cases("demo")
    kw = VARIANTS[variant]
    mask = region(kw)
    g = c.g
    ref_launches = c.render()[3].kernel_launches
    if variant == "simple_kernel":
        monkeypatch.setenv("RTP_RENDER_KERNEL", "simple")  # read when a scene is created
        g = api.Scene(c.sc)
        monkeypatch.delenv("RTP_RENDER_KERNEL")
    if variant == "several_launches_per_round":
        monkeypatch.setenv("RTP_PATH_BUDGET", str(W * H + 7))  # round 1: 1 sample per launch; later rounds by their live count
    if variant == "device_buffers":
        import torch

        buf = torch.full((3 * W * H + W * H,), SENTINEL, dtype=torch.int64, device="cuda").view(torch.float64)
        nbuf = torch.full((W * H,), -1, dtype=torch.int32, device="cuda")
        p = api.render_params(W, H, 0, DEPTH, SEED, 0, 0)
        a = api.adaptive_params(MIN, MAX, BATCH, 0.0, c.rel)
        stream = torch.cuda.Stream()
        stream.wait_stream(torch.cuda.current_stream())  # the sentinel fill runs on the current stream
        st = g.render_adaptive_device(p, a, api.Camera(W / H, c.sc.camera.fov, c.sc.camera.focal_dist, c.sc.camera.lens_radius,
                                                       c.sc.camera.transformation),
                                      buf.data_ptr(), buf.data_ptr() + 3 * W * H * 8, nbuf.data_ptr(), stream.cuda_stream, stats=True)
        a_host = buf.cpu().numpy()  # the call is synchronous: no wait on the stream before reading
        img, fg = a_host[: 3 * W * H].reshape(H, W, 3), a_host[3 * W * H:].reshape(H, W)
        n = nbuf.cpu().numpy().view(np.uint32).reshape(H, W)
    else:
        out = sentinel_frame()
        img, fg, n, st = g.render_adaptive(W, H, MIN, MAX, BATCH, rel_tol=c.rel, max_bounce=DEPTH, seed=SEED, out=out, **kw)
    if variant == "several_launches_per_round":
        monkeypatch.delenv("RTP_PATH_BUDGET")
        assert st.kernel_launches > ref_launches
    assert (n[mask] == c.model[mask]).all()
    assert_equals_fixed_renders(g, img, fg, n, mask, raw=kw.get("raw_sums", False))
    if variant in ("tile", "rows"):
        assert unwritten(img, fg, n)[~mask].all() and not unwritten(img, fg, n)[mask].any()
    assert st.paths == int(n[mask].astype(np.uint64).sum())
    if g is not c.g:
        g.close()


@pytest.mark.gpu
def test_min_equal_max_is_rtp_render(gpu):
    sc = scenes.bunny_lambert()
    with api.Scene(sc) as g:
        img, fg, n, st = g.render_adaptive(W, H, 6, 6, 3, rel_tol=0.5, max_bounce=DEPTH, seed=SEED)
        ref, fref, sref = g.render(W, H, 6, max_bounce=DEPTH, seed=SEED)
        assert (n == 6).all()
        assert img.tobytes() == ref.tobytes() and fg.tobytes() == fref.tobytes()
        assert st.paths == sref.paths


@pytest.mark.gpu
def test_fixed_renders_around_an_adaptive_call_agree(cases):
    c = cases("bunny_lambert")
    before = c.g.render(96, 54, 3, max_bounce=DEPTH, seed=2)
    c.render()
    c.g.render_adaptive(W, H, 1, 5, 1, rel_tol=0.1, max_bounce=DEPTH, seed=SEED, tile=(3, 3, 20, 20))
    after = c.g.render(96, 54, 3, max_bounce=DEPTH, seed=2)
    assert before[0].tobytes() == after[0].tobytes() and before[1].tobytes() == after[1].tobytes()
    assert before[2].rays == after[2].rays


INVALID = {
    "min_zero": dict(a=(0, 8, 2, 0.0, 0.1)),
    "min_above_max": dict(a=(9, 8, 2, 0.0, 0.1)),
    "batch_zero": dict(a=(2, 8, 0, 0.0, 0.1)),
    "abs_tol_nan": dict(a=(2, 8, 2, float("nan"), 0.1)),
    "rel_tol_nan": dict(a=(2, 8, 2, 0.0, float("nan"))),
    "abs_tol_negative": dict(a=(2, 8, 2, -1e-9, 0.1)),
    "rel_tol_negative": dict(a=(2, 8, 2, 0.0, -0.1)),
    "abs_tol_inf": dict(a=(2, 8, 2, float("inf"), 0.1)),
    "rel_tol_inf": dict(a=(2, 8, 2, 0.0, float("inf"))),
    "num_samples": dict(p=dict(num_samples=4)),
    "sample_begin": dict(p=dict(sample_begin=1)),
    "sample_end": dict(p=dict(sample_end=4)),
    "transparent_flag": dict(p=dict(flags=A.RENDER_TRANSPARENT)),
    "unknown_flag": dict(p=dict(flags=8)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(INVALID))
@pytest.mark.parametrize("entry", ["host", "device"])
def test_invalid_arguments(cases, case, entry):
    c = cases("bunny_lambert")
    spec = INVALID[case]
    a = api.adaptive_params(*spec.get("a", (2, 8, 2, 0.0, 0.1)))
    p = api.render_params(W, H, 0, DEPTH, SEED, 0, 0)
    for k, v in spec.get("p", {}).items():
        setattr(p, k, v)
    cam = api.Camera(W / H, c.sc.camera.fov, c.sc.camera.focal_dist, c.sc.camera.lens_radius, c.sc.camera.transformation).to_c()
    lib = A.load()
    if entry == "host":
        rgb = np.zeros((H, W, 3))
        rc = lib.rtp_render_adaptive(c.g.handle, C.byref(cam), C.byref(p), C.byref(a), A.ptr(rgb), None, None, None)
    else:
        import torch

        d = torch.zeros(3 * W * H, dtype=torch.float64, device="cuda")
        rc = lib.rtp_render_adaptive_device(c.g.handle, C.byref(cam), C.byref(p), C.byref(a), d.data_ptr(), None, None, None, None)
    assert rc == A.ERR_INVALID, (lib.rtp_last_error() or b"").decode()
    # the scene is still usable
    img, fg, n, _ = c.g.render_adaptive(W, H, 2, 2, 1, max_bounce=DEPTH, seed=SEED)
    assert (n == 2).all()


@pytest.mark.gpu
def test_groups_match_the_oracle(cases):
    c = cases("demo")
    img, fg, n, _ = c.render()
    o = oracle.Scene(c.sc)
    for k in np.unique(n):
        io, fo, _ = o.render(W, H, int(k), max_bounce=DEPTH, seed=SEED, sample_range=(0, int(k)))
        sel = n == k
        rep = image_report(img[sel][None], io[sel][None])
        assert rep["rmse"] <= IMG_RMSE and rep["differing"] <= max(1, IMG_FRAC * rep["pixels"]), (k, rep)
        assert (fg[sel] == fo[sel]).all()
    o.close()


@pytest.mark.gpu
def test_two_devices_equal_one(gpu):
    if api.device_count() < 2:
        pytest.skip("needs two GPUs")
    sc = scenes.demo()
    with api.Scene(sc, device_mask=0b11) as g:
        one = g.render_adaptive(W, H, MIN, MAX, BATCH, rel_tol=0.03, max_bounce=DEPTH, seed=SEED, device_mask=0b01)
        two = g.render_adaptive(W, H, MIN, MAX, BATCH, rel_tol=0.03, max_bounce=DEPTH, seed=SEED)
        for a, b in zip(one[:3], two[:3]):
            assert a.tobytes() == b.tobytes()
        assert one[3].paths == two[3].paths
