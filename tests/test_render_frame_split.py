"""The frame driver behind the four host-buffer render calls (rtp_render, rtp_render_srgb8, rtp_render_aov, rtp_render_adaptive): the
caller's tile and row split are dealt out over the devices taking part, and each device's rows are copied back plane by plane into
the caller's buffers. On one device a call with a row split writes exactly the rows it owns, with the bits of the same tile rendered
without the split, and leaves every other pixel as it was. On two devices every plane, the sample counts and the 8-bit pixels
included, is bit-identical to one device."""
import numpy as np
import pytest

from rtp_b200 import api, scenes

pytestmark = pytest.mark.gpu

W, H, SPP, DEPTH, SEED = 72, 45, 3, 6, 11
TILE = (5, 4, 50, 33)  # x, y, w, h
ROWS = (1, 3)          # row_offset, row_stride
OWNED = (slice(TILE[1] + ROWS[0], TILE[1] + TILE[3], ROWS[1]), slice(TILE[0], TILE[0] + TILE[2]))
SENTINEL = 0x7FF8_DEAD_BEEF_0003  # bits of a quiet NaN whose payload no computation produces
SENTINEL_N = 0xFFFFFFFF           # samples_out words nobody wrote
CALLS = ["render", "srgb8", "aov", "adaptive"]


def buffers(call, fill):
    """sentinel-filled caller buffers of one call; fill: the byte of the 8-bit frame"""
    def f64(*shape):
        return np.full(shape, SENTINEL, dtype=np.uint64).view(np.float64)

    if call == "render":
        return f64(H, W, 3), f64(H, W)
    if call == "srgb8":
        return (np.full((H, W, 4), fill, dtype=np.uint8),)
    if call == "aov":
        return f64(H, W, 3), f64(H, W), f64(H, W, 3), f64(H, W, 3)
    return f64(H, W, 3), f64(H, W), np.full((H, W), SENTINEL_N, dtype=np.uint32)


def run(g, call, fill=0xA5, **kw):
    """one call over TILE into fresh sentinel-filled buffers -> (buffers, stats)"""
    out = buffers(call, fill)
    kw = dict(max_bounce=DEPTH, seed=SEED, tile=TILE, **kw)
    if call == "render":
        st = g.render(W, H, SPP, out=out, **kw)[-1]
    elif call == "srgb8":
        st = g.render_srgb8(W, H, SPP, out=out[0], **kw)[-1]
    elif call == "aov":
        st = g.render_aov(W, H, SPP, out=out, **kw)[-1]
    else:
        st = g.render_adaptive(W, H, 2, 8, 2, rel_tol=0.05, out=out, **kw)[-1]
    return out, st


@pytest.fixture(scope="module")
def demo(gpu):
    with api.Scene(scenes.demo()) as g:
        yield g


@pytest.mark.parametrize("call", CALLS)
def test_one_device_writes_only_its_rows(demo, call):
    whole, _ = run(demo, call)
    for fill in ((0x00, 0xFF) if call == "srgb8" else (0xA5,)):  # an 8-bit pixel written with the fill's value would hide in one fill
        got, _ = run(demo, call, fill=fill, rows=ROWS)
        for g, w, blank in zip(got, whole, buffers(call, fill)):
            want = blank.copy()
            want[OWNED] = w[OWNED]
            assert g.tobytes() == want.tobytes()


@pytest.mark.parametrize("call", CALLS)
def test_two_devices_equal_one(gpu, call):
    if api.device_count() < 2:
        pytest.skip("needs two GPUs")
    with api.Scene(scenes.demo(), device_mask=0b11) as g:
        one, st1 = run(g, call, rows=ROWS, device_mask=0b01)
        two, st2 = run(g, call, rows=ROWS)
    for a, b in zip(one, two):
        assert a.tobytes() == b.tobytes()
    assert st2.paths == st1.paths and st2.rays == st1.rays
