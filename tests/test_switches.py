"""The library's RTP_* switches are read in one place and parsed one way (Switches, rtp_internal.h): a scene reads them when it is
created, the host-only build calls when they are called, and a 0/1 switch is on only when its value is a number other than 0."""
import pytest

from rtp_b200 import api, scenes


@pytest.mark.gpu
def test_chunk_size_is_read_per_scene(gpu, monkeypatch):
    sc = scenes.bunny_lambert()
    rays = scenes.incoherent_rays(5 * 4096 + 17)
    monkeypatch.delenv("RTP_CHUNK_LOG2", raising=False)
    with api.Scene(sc) as first:
        h1 = first.hit(rays)  # a host batch traced before the switch is set: the chunk size must not stick for the process
    monkeypatch.setenv("RTP_CHUNK_LOG2", "12")
    with api.Scene(sc) as second:
        h2, st = second.hit(rays, stats=True)
        per_chunk = 2 if second.info().any_order else 1  # the any-order walk is followed by the in-order pass over its defer list
        assert st.kernel_launches == 6 * per_chunk  # six chunks of at most 4096 rays
    assert h2.tobytes() == h1.tobytes()


def test_build_timing_zero_is_off(capfd, monkeypatch):
    sc = scenes.demo()
    monkeypatch.setenv("RTP_BUILD_TIMING", "0")
    api.bvh_build_order(sc)
    assert "[rtp build]" not in capfd.readouterr().err
    monkeypatch.setenv("RTP_BUILD_TIMING", "1")
    api.bvh_build_order(sc)
    assert any(line.startswith("[rtp build]") for line in capfd.readouterr().err.splitlines())
