"""Multi-GPU behind the C ABI (SURVEY.md 8e, VERDICT r1 item 5): a scene made by rtp_scene_create_multi lives on several devices and
ONE rtp_render / rtp_trace_closest call fans out to them — rows of the frame round-robin over the devices, ray chunks round-robin
over the devices, no exchange between them — with results bit-identical to one device. Also the row split of rtp_render_params
(row_offset / row_stride) that one-process-per-GPU hosts use. Tests that need two devices skip on a one-GPU box; the
one-device ones exercise the same code paths with a mask of one device."""
import numpy as np
import pytest

import oracle
from rtp_b200 import _abi as A
from rtp_b200 import api, scenes

pytestmark = pytest.mark.gpu


def two_gpus():
    if api.device_count() < 2:
        pytest.skip("needs two GPUs")


def test_row_split_covers_the_frame_bit_for_bit(gpu):
    sc = scenes.demo()
    w, h, spp = 96, 53, 3
    with api.Scene(sc) as g:
        full, full_fg, st_full = g.render(w, h, spp, max_bounce=6, seed=5)
        for stride in (2, 3, 8):
            img = np.full((h, w, 3), np.nan)
            fg = np.full((h, w), np.nan)
            paths = 0
            for off in range(stride):
                _, _, st = g.render(w, h, spp, max_bounce=6, seed=5, out=(img, fg), rows=(off, stride))
                assert st.paths == len(range(h)[off::stride]) * w * spp
                paths += st.paths
            assert paths == st_full.paths
            assert img.tobytes() == full.tobytes() and fg.tobytes() == full_fg.tobytes()
        # a tile rectangle with a row split: only the rows of the split INSIDE the rectangle are written
        img = np.zeros((h, w, 3))
        g.render(w, h, spp, max_bounce=6, seed=5, out=(img, None), tile=(8, 5, 40, 20), rows=(1, 4))
        want = np.zeros_like(img)
        want[6:25:4, 8:48] = full[6:25:4, 8:48]
        assert img.tobytes() == want.tobytes()
        # the 8-bit output stage follows the same split
        rgba_full, _ = g.render_srgb8(w, h, spp, max_bounce=6, seed=5)
        rgba = np.zeros((h, w, 4), dtype=np.uint8)
        for off in range(3):
            g.render_srgb8(w, h, spp, max_bounce=6, seed=5, out=rgba, rows=(off, 3))
        assert rgba.tobytes() == rgba_full.tobytes()
        with pytest.raises(api.RtpError):
            g.render(w, h, spp, rows=(3, 3))


def test_row_split_equals_oracle(gpu):
    sc = scenes.bunny_lambert()
    with api.Scene(sc) as g:
        o = oracle.Scene(sc)
        ig, fg, _ = g.render(64, 36, 2, max_bounce=8, seed=2, rows=(1, 3))
        io, fo, _ = o.render(64, 36, 2, max_bounce=8, seed=2, rows=(1, 3))
        assert np.sqrt(((ig - io) ** 2).mean()) <= 1e-6 and (fg == fo).all()
        assert (ig[0::3] == 0).all() and (ig[2::3] == 0).all()  # other rows untouched
        o.close()


def test_scene_on_one_device_through_create_multi(gpu):
    sc = scenes.bunny_lambert()
    cam = api.Camera(16 / 9, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    rays = np.concatenate([api.camera_rays(cam, 128, 72), scenes.incoherent_rays(5000)])
    with api.Scene(sc) as a, api.Scene(sc, device_mask=1) as b:
        assert b.devices() == 1
        assert a.hit(rays).tobytes() == b.hit(rays).tobytes()
        ia, fa, _ = a.render(80, 45, 2, seed=3)
        ib, fb, _ = b.render(80, 45, 2, seed=3, device_mask=1)
        assert ia.tobytes() == ib.tobytes() and fa.tobytes() == fb.tobytes()
        with pytest.raises(api.RtpError):
            b.render(80, 45, 2, seed=3, device_mask=1 << 5)  # names no device of this scene
    with pytest.raises(api.RtpError):
        api.Scene(sc, device_mask=1 << 31)


def test_one_call_two_devices(gpu, monkeypatch):
    two_gpus()
    monkeypatch.setenv("RTP_CHUNK_LOG2", "12")  # 4096-ray chunks: the batch below is dealt out over both devices
    sc = scenes.demo()
    cam = api.Camera(16 / 9, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    rays = np.concatenate([api.camera_rays(cam, 160, 90), scenes.incoherent_rays(20000)])
    with api.Scene(sc) as one, api.Scene(sc, device_mask=3) as two:
        assert two.devices() == 3
        h1, (h2, st2) = one.hit(rays), two.hit(rays, stats=True)
        assert h1.tobytes() == h2.tobytes() and st2.rays == len(rays)
        assert one.hit_full(rays).tobytes() == two.hit_full(rays).tobytes()
        w, h, spp = 160, 91, 4
        i1, f1, s1 = one.render(w, h, spp, max_bounce=8, seed=7)
        i2, f2, s2 = two.render(w, h, spp, max_bounce=8, seed=7)
        assert i1.tobytes() == i2.tobytes() and f1.tobytes() == f2.tobytes()  # bit-identical: no sum across devices
        assert s2.paths == s1.paths and s2.rays == s1.rays
        i3, _, s3 = two.render(w, h, spp, max_bounce=8, seed=7, device_mask=2)  # the second device alone
        assert i3.tobytes() == i1.tobytes() and s3.rays == s1.rays
        r1, _ = one.render_srgb8(w, h, spp, seed=7)
        r2, _ = two.render_srgb8(w, h, spp, seed=7)
        assert r1.tobytes() == r2.tobytes()
        o = oracle.Scene(sc)
        io, fo, _ = o.render(w, h, spp, max_bounce=8, seed=7)
        assert np.sqrt(((i2 - io) ** 2).mean()) <= 1e-6
        o.close()
