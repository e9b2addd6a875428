"""Pins for the CPU oracle (CPU-only).

The reference has no tests or golden vectors for this path (SURVEY.md §4), so the oracle is pinned by:
published Philox known answers, analytic geometry, its own BVH-vs-brute-force differential, asset
invariants, committed golden hits, and an independent numpy restatement of the slab and triangle tests.
"""
import math
import os

import numpy as np
import pytest

import oracle
from rtp_b200 import _abi as A
from rtp_b200 import api, assets, scenes

MISS = 0xFFFFFFFF
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


# ----------------------------------------------------------------------------- random stream -----

def test_philox4x32_10_known_answers():
    """Random123 kat_vectors, philox4x32 10 rounds"""
    kat = [
        ([0, 0, 0, 0], [0, 0], [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
        ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
        ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0], [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]),
    ]
    for ctr, key, want in kat:
        assert list(oracle.philox(ctr, key)) == want


def test_stream_layout_and_f64_mapping():
    # draw k = word pair (k&1) of block k>>1 with counter (lo, hi, block, stream), key = seed
    seed, lo, hi, stream = 0x0123456789ABCDEF, 77, 5, A.RNG_STREAM_PATH
    d = oracle.rng_draws(seed, lo, hi, stream, 0, 6)
    for k in range(6):
        w = oracle.philox([lo, hi, k >> 1, stream], [seed & 0xFFFFFFFF, seed >> 32])
        u = (int(w[2 * (k & 1) + 1]) << 32) | int(w[2 * (k & 1)])
        assert d[k] == (u >> 11) * 2.0 ** -53
    assert ((d >= 0) & (d < 1)).all()
    # starting mid-stream gives the same values
    assert (oracle.rng_draws(seed, lo, hi, stream, 3, 3) == d[3:]).all()
    # the product's host copy and the vectorised numpy copy agree with the oracle
    assert (api.rng_draws(seed, lo, hi, stream, 0, 6) == d).all()
    v = scenes.philox_draws(seed, np.array([lo], dtype=np.uint32), np.array([hi], dtype=np.uint32), stream, 6)
    assert (v[0] == d).all()


def test_noise_integer_against_python_bigints():
    """randomness.rs:91-105 with Python integers as the independent arithmetic"""
    M = (1 << 64) - 1

    def ref(x, y, z, s):
        h = (0x369E6D3B899E43CF * x + 0x53F89E7FFDA3B07D * y + 0x3B13C1CA4937E629 * z + 0x577C2C6E4019D645 * s) & M
        sh = h - (1 << 64) if h >> 63 else h          # as isize
        h = ((sh >> 13) & M) ^ h                      # arithmetic shift
        h = (h * ((h * h * 60493 + 19990303) & M) + 1376312589) & M
        return h - (1 << 64) if h >> 63 else h

    rng = np.random.default_rng(0)
    for x, y, z, s in rng.integers(-10**6, 10**6, size=(200, 4)):
        assert oracle.lib().orc_noise_integer(int(x), int(y), int(z), int(s)) == ref(int(x), int(y), int(z), int(s))


# ----------------------------------------------------------------------------- assets -------------

def test_asset_invariants():
    b, f = assets.bunny(), assets.bunny_flat()
    assert (len(b.vertices), len(b.indices)) == (2503, 14904)
    assert (len(f.vertices), len(f.indices)) == (14902, 14904)
    assert b.indices.max() == 2502 and f.indices.max() == 14901
    # first-seen numbering (mesh.rs:151-166): the first face of bunny.obj is 1//1 2//2 3//3
    assert list(b.indices[:3]) == [0, 1, 2]
    e = assets.earthmap()
    assert e.shape == (512, 1024, 4) and (e[..., 3] == 255).all()


def test_fixture_bytes_are_pinned():
    """data/assets.npz holds the reference's bunny.obj, bunny_flat.obj and earthmap.tga as parsed by the oracle's loaders
    (tests/golden/make_fixtures.py). The asset files are not part of this repository, so the decoded arrays are pinned by digest:
    a regenerated or edited fixture shows up here."""
    import hashlib

    def sha(a):
        return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()

    b, f = assets.bunny(), assets.bunny_flat()
    assert sha(b.vertices) == "c2e0ae9c2eb0afebc8c06f8fbc28cf60e0ed2a8e9363fbb2dbbb8b627d8019fc"
    assert sha(b.indices.astype(np.uint32)) == "487804de833654c00a0942bf8414a4f2aef39996fb76a373bf10b23481fd6eb1"
    assert sha(f.vertices) == "23b3b02298c9475a30973e052edebda96564ad736d09c883392bc2f20a464fcb"
    assert sha(f.indices.astype(np.uint32)) == "21a7c11a84e8106b716ec70fbde2c056ef4812eea2e62723534ef7efc3a6bf5d"
    assert sha(assets.earthmap()) == "adbe9f16ab1c382f8fd913f55abc61e356a22766ae82d60a19c9294ff8910831"


def test_obj_parser_subset(tmp_path):
    text = "\n".join([
        "# comment", "o thing", "v 0 0 0", "v  1.5\t0 0", "v 0 1 0", "v 0 0 1e0", "vn 0 0 1", "vt 0.25 0.75", " v 9 9 9",
        "vx 1 2 3", "v 1 2", "f 1/1/1 2//1 3", "f 1 3 4 ", "s off", "f 2/1 3/1 4/1", "",
    ])
    p = tmp_path / "t.obj"
    p.write_text(text)
    for loader in (oracle.obj_load, api.obj.load):
        m = loader(str(p))
        # (p,t,n) triples: (0,0,0) (1,-,0) (2,-,-) | (0,-,-) (2,-,-)dup (3,-,-) | (1,0,-) (2,0,-) (3,0,-)
        assert len(m.vertices) == 8 and list(m.indices) == [0, 1, 2, 3, 2, 4, 5, 6, 7], loader
        assert list(m.vertices["position"][1]) == [1.5, 0, 0]
        assert list(m.vertices["normal"][0]) == [0, 0, 1] and list(m.vertices["normal"][2]) == [0, 0, 0]
        assert list(m.vertices["uv"][0]) == [0.25, 0.75] and list(m.vertices["uv"][1]) == [0, 0]
    p.write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nv 1 1 0\nf 1 2 3 4\n")
    with pytest.raises(oracle.OracleError) as e:
        oracle.obj_load(str(p))
    assert e.value.code == A.ERR_FORMAT
    with pytest.raises(api.RtpError) as e2:
        api.obj.load(str(p))
    assert e2.value.code == A.ERR_FORMAT
    with pytest.raises(api.RtpError) as e3:
        api.obj.load(str(tmp_path / "missing.obj"))
    assert e3.value.code == A.ERR_IO
    # OBJ indices are 1-based: the reference's `index - 1` (mesh.rs:64-69) underflows on a 0 and panics; the loader must not
    # quietly read it as "no normal / no uv"
    for face in ("f 1/0/0 2 3", "f 0 1 2", "f 1//0 2//1 3//1"):
        p.write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nvn 0 0 1\nvt 0 0\n" + face + "\n")
        with pytest.raises(api.RtpError) as e4:
            api.obj.load(str(p))
        assert e4.value.code == A.ERR_FORMAT, face


def test_bunny_obj_roundtrip_through_text(tmp_path):
    """write the fixture back as OBJ text (6 decimals, like the asset) and parse it with both loaders"""
    mesh = assets.bunny()
    lines = []
    # bunny.obj is smooth: vertex k uses position k and normal k
    for v in mesh.vertices:
        lines.append("v %.6f %.6f %.6f" % tuple(v["position"]))
    for v in mesh.vertices:
        lines.append("vn %.4f %.4f %.4f" % tuple(v["normal"]))
    ix = mesh.indices.reshape(-1, 3) + 1
    for a, b, c in ix:
        lines.append(f"f {a}//{a} {b}//{b} {c}//{c}")
    p = tmp_path / "bunny.obj"
    p.write_text("\n".join(lines) + "\n")
    mo, mp = oracle.obj_load(str(p)), api.obj.load(str(p))
    assert mo.vertices.tobytes() == mp.vertices.tobytes() and (mo.indices == mp.indices).all()
    assert mo.vertices["position"].tobytes() == mesh.vertices["position"].tobytes()
    assert (mo.indices == mesh.indices).all()


@pytest.mark.parametrize("bpp,flip", [(24, False), (24, True), (32, False), (32, True)])
def test_tga_decode(tmp_path, bpp, flip):
    w, h = 5, 3
    rng = np.random.default_rng(bpp + flip)
    px = rng.integers(0, 256, size=(h, w, bpp // 8), dtype=np.uint8)  # stored rows, BGR(A)
    hd = bytearray(18)
    hd[2], hd[12], hd[14], hd[16], hd[17] = 2, w, h, bpp, 0x20 if flip else 0
    p = tmp_path / "t.tga"
    p.write_bytes(bytes(hd) + px.tobytes())
    want = np.full((h, w, 4), 255, dtype=np.uint8)
    want[..., 0], want[..., 1], want[..., 2] = px[..., 2], px[..., 1], px[..., 0]
    if bpp == 32:
        want[..., 3] = px[..., 3]
    if flip:
        want = want[::-1]
    for loader in (oracle.tga_load, api.tga.load):
        assert (loader(str(p)) == want).all(), loader
    # save → load round trip (image.rs:116-137 writes 32 bpp, descriptor 0)
    for saver, loader in ((oracle.tga_save, api.tga.load), (api.tga.save, oracle.tga_load)):
        q = tmp_path / "s.tga"
        saver(want, str(q))
        raw = q.read_bytes()
        assert raw[2] == 2 and raw[16] == 32 and raw[17] == 0 and len(raw) == 18 + w * h * 4
        assert (loader(str(q)) == want).all()


def test_tga_rejects_unsupported_headers(tmp_path):
    hd = bytearray(18)
    hd[2], hd[12], hd[14], hd[16] = 10, 1, 1, 24  # RLE
    p = tmp_path / "rle.tga"
    p.write_bytes(bytes(hd) + b"\0\0\0")
    with pytest.raises(oracle.OracleError) as e:
        oracle.tga_load(str(p))
    assert e.value.code == A.ERR_FORMAT
    with pytest.raises(api.RtpError) as e2:
        api.tga.load(str(p))
    assert e2.value.code == A.ERR_FORMAT


def test_sky_panorama_is_deterministic():
    a = assets.sky_panorama(1)
    assert a.shape == (1024, 2048, 4) and (a[..., 3] == 255).all()
    import hashlib
    assert hashlib.sha256(a.tobytes()).hexdigest() == hashlib.sha256(assets.sky_panorama(1).tobytes()).hexdigest()
    assert (a[768, 1280, :3] == [255, 250, 225]).all()          # sun
    assert a[1000].mean() < a[520].mean()                        # zenith darker than horizon
    assert (assets.sky_panorama(2) != a).any()


# ----------------------------------------------------------------------------- host helpers -------

def test_lookat_unnormalised_basis():
    co = oracle.lookat([-1.5, 1.5, 2.5], [0.0, 0.5, 0.0], [0.0, 1.0, 0.0])
    t = api.Transformation.lookat([-1.5, 1.5, 2.5], [0.0, 0.5, 0.0], [0.0, 1.0, 0.0])
    m = np.array(list(co.orientation)).reshape(3, 3).T
    assert m.tobytes() == np.ascontiguousarray(t.orientation).tobytes()
    x, y, z = m[:, 0], m[:, 1], m[:, 2]
    assert abs(np.linalg.norm(z) - 1) < 1e-15
    assert abs(np.linalg.norm(x) - 0.9459) < 1e-4          # SURVEY §7.2(4): x = up × z is not normalised
    assert abs(x @ z) < 1e-15 and abs(y @ z) < 1e-15


def test_split_in_tiles():
    for (w, h), n in (((800, 600), 475), ((640, 360), 240), ((33, 1), 2), ((32, 32), 1)):
        to, tp = oracle.split_in_tiles(w, h, 32, 32), api.split_in_tiles(w, h, 32, 32)
        assert len(to) == n and (to == tp).all()
        cover = np.zeros((h, w), dtype=int)
        for oi, oj, tw, th in to:
            cover[oj:oj + th, oi:oi + tw] += 1
        assert (cover == 1).all()
    assert list(oracle.split_in_tiles(70, 40, 32, 32)[2]) == [64, 0, 6, 32]  # row-major, clipped at the edge


def test_to_srgb_u8():
    f = np.array([[[0.0, 1.0, 0.5], [-1.0, 2.0, np.nan], [0.2, 1e-9, 0.999999]]])
    a, b = oracle.to_srgb_u8(f), api.to_srgb_u8(f)
    assert (a == b).all()
    assert list(a[0, 0]) == [0, 255, int(255.0 * 0.5 ** (1 / 2.2)), 255]
    assert list(a[0, 1]) == [0, 255, 0, 255]  # clamp, NaN as u8 = 0


# ----------------------------------------------------------------------------- geometry -----------

def np_collide(bmin, bmax, o, d, tmin, tmax):
    """independent numpy restatement of utility.rs:137-154 (np.fmin/fmax are minNum/maxNum)"""
    with np.errstate(all="ignore"):
        inv = 1.0 / d
        t0 = (bmin - o) * inv
        t1 = (bmax - o) * inv
        lo = np.fmax(np.fmax(np.fmax(tmin, np.fmin(t0[0], t1[0])), np.fmin(t0[1], t1[1])), np.fmin(t0[2], t1[2]))
        hi = np.fmin(np.fmin(np.fmin(tmax, np.fmax(t0[0], t1[0])), np.fmax(t0[1], t1[1])), np.fmax(t0[2], t1[2]))
    return bool(hi >= lo)


def test_aabb_collide_against_numpy_and_nan_rules():
    rng = np.random.default_rng(1)
    n_true = 0
    for _ in range(3000):
        c = rng.normal(size=3)
        e = rng.uniform(0.01, 1.0, size=3)
        o = rng.normal(size=3) * 3
        d = (c + rng.normal(size=3) * 0.7) - o if rng.random() < 0.7 else rng.normal(size=3)
        if rng.random() < 0.3:
            d[rng.integers(3)] = 0.0
        if rng.random() < 0.1:
            o[rng.integers(3)] = (c - e)[rng.integers(3)]
        tmax = np.inf if rng.random() < 0.5 else rng.uniform(0, 6)
        got = oracle.aabb_collide(c - e, c + e, list(o) + list(d) + [1e-3, tmax])
        assert got == np_collide(c - e, c + e, o, d, 1e-3, tmax)
        n_true += got
    assert 100 < n_true < 2900
    # 0 * inf = NaN lanes are dropped by min/max: origin exactly on the min plane, direction parallel to it
    assert oracle.aabb_collide([0, 0, 0], [1, 1, 1], [0.0, 0.5, -1, 0, 0, 1, 1e-3, np.inf]) is False  # lane x: NaN/+inf → near=+inf
    assert oracle.aabb_collide([0, 0, 0], [1, 1, 1], [0.5, 0.5, -1, 0, 0, 1, 1e-3, np.inf]) is True
    # a NaN direction passes every box (all lanes dropped) …
    assert oracle.aabb_collide([0, 0, 0], [1, 1, 1], [5, 5, 5, np.nan, np.nan, np.nan, 1e-3, np.inf]) is True
    # … and >= is non-strict: a ray grazing a degenerate (flat) box still collides
    assert oracle.aabb_collide([0, 0, 0], [1, 0, 1], [0.5, 1, 0.5, 0, -1, 0, 1e-3, np.inf]) is True


def np_hit_triangle(a, b, c, o, d, tmin, tmax):
    """independent numpy restatement of hittable.rs:65-99 (scalar float64, same association)"""
    f = np.float64
    ba, ca, pa = a - b, a - c, a - o
    det = ba[0] * ca[1] * d[2] + ba[1] * ca[2] * d[0] + ba[2] * ca[0] * d[1] - ba[0] * ca[2] * d[1] - ba[1] * ca[0] * d[2] - ba[2] * ca[1] * d[0]
    if abs(det) < 1e-7:
        return None
    inv = f(1.0) / det
    t = (pa[0] * (ba[1] * ca[2] - ba[2] * ca[1]) + pa[1] * (ba[2] * ca[0] - ba[0] * ca[2]) + pa[2] * (ba[0] * ca[1] - ba[1] * ca[0])) * inv
    u = (pa[0] * (ca[1] * d[2] - ca[2] * d[1]) + pa[1] * (ca[2] * d[0] - ca[0] * d[2]) + pa[2] * (ca[0] * d[1] - ca[1] * d[0])) * inv
    v = (pa[0] * (ba[2] * d[1] - ba[1] * d[2]) + pa[1] * (ba[0] * d[2] - ba[2] * d[0]) + pa[2] * (ba[1] * d[0] - ba[0] * d[1])) * inv
    w = f(1.0) - u - v
    if t < tmin or t > tmax or u < 0 or v < 0 or w < 0:
        return None
    return t, u, v, w


def test_triangle_against_numpy_restatement():
    rng = np.random.default_rng(2)
    tri = rng.normal(size=(40, 3, 3))
    nrm = rng.normal(size=(40, 3, 3))
    uvs = rng.uniform(size=(40, 3, 2))
    mesh = api.Mesh.from_arrays(tri.reshape(-1, 3), normals=nrm.reshape(-1, 3), uvs=uvs.reshape(-1, 2))
    mats = [api.Material.new(api.Scatter.NONE, api.Absorb.BlackBody, api.Emit.DebugNormals)]
    sc = api.ExampleScene(scenes._bunny_camera(), api.SceneData(mats, [], [mesh]), "list", api.Hittable.triangles_of(mesh, 0), api.Emit.SkyGradient)
    o = oracle.Scene(sc)
    rays = np.zeros((400, 8))
    rays[:, 0:3] = rng.normal(size=(400, 3)) * 4
    target = tri[rng.integers(40, size=400)].mean(axis=1) + rng.normal(size=(400, 3)) * 0.2
    rays[:, 3:6] = target - rays[:, 0:3]
    rays[:, 6], rays[:, 7] = 1e-3, np.inf
    h = o.hit_full(rays)
    n_hit = 0
    for k in range(400):
        best, T = None, np.inf
        for j in range(40):                          # hittable.rs:110-120: later equal-or-closer hit replaces
            r = np_hit_triangle(tri[j, 0], tri[j, 1], tri[j, 2], rays[k, 0:3], rays[k, 3:6], 1e-3, T)
            if r is not None:
                best, T = (j, r), r[0]
        if best is None:
            assert h["leaf"][k] == MISS
            continue
        n_hit += 1
        j, (t, u, v, w) = best
        assert h["leaf"][k] == j and h["t"][k] == t
        d, org = rays[k, 3:6], rays[k, 0:3]
        assert (h["position"][k] == org + t * d).all()                     # utility.rs:67-69
        assert (h["normal"][k] == (w * nrm[j, 0] + u * nrm[j, 1]) + v * nrm[j, 2]).all()
        assert (h["uv"][k] == (w * uvs[j, 0] + u * uvs[j, 1]) + v * uvs[j, 2]).all()
    assert n_hit > 100


def test_sphere_roots_analytic():
    mats = [api.Material.new(api.Scatter.Lambert, api.Absorb.WhiteBody, api.Emit.NONE)]
    sc = api.ExampleScene(scenes._bunny_camera(), api.SceneData(mats, [], []), "bvh", api.Hittable.Sphere([0, 0, 0], 2.0, 0), api.Emit.SkyGradient)
    o = oracle.Scene(sc)
    rays = np.array([
        [0, 0, 5, 0, 0, -1, 1e-3, np.inf],      # near root t = 3
        [0, 0, 5, 0, 0, -2, 1e-3, np.inf],      # non-unit direction: t = 1.5
        [0, 0, 0, 0, 1, 0, 1e-3, np.inf],       # from inside: far root t = 2
        [0, 0, 5, 0, 0, -1, 1e-3, 2.5],         # t_max before the sphere
        [2, 0, 5, 0, 0, -1, 1e-3, np.inf],      # tangent: delta <= 0 rejects (hittable.rs:45)
        [0, 0, 5, 0, 0, -1, 4.0, np.inf],       # near root below t_min → far root t = 7
        [0, 0, 5, 0, 0, 1, 1e-3, np.inf],       # pointing away
    ], dtype=np.float64)
    h = o.hit_full(rays)
    assert list(h["leaf"]) == [0, 0, 0, MISS, MISS, 0, MISS]
    assert list(h["t"][[0, 1, 2, 5]]) == [3.0, 1.5, 2.0, 7.0]
    assert (h["normal"][0] == [0, 0, 1]).all() and (h["position"][0] == [0, 0, 2]).all()
    # uv = (0.5 - atan2(nz, nx)/TAU, asin(ny)/PI + 0.5)  (hittable.rs:61)
    assert h["uv"][0][0] == 0.5 - math.atan2(1.0, 0.0) / math.tau and h["uv"][0][1] == 0.5
    assert h["uv"][2][1] == math.asin(1.0) / math.pi + 0.5


def test_one_triangle_plane_and_debug_normals():
    """example_scenes.rs:222-262: hits on the lone triangle satisfy x+y+z = 1 and shade to (1,1,1)/sqrt(3)"""
    sc = scenes.one_triangle()
    o = oracle.Scene(sc)
    cam = api.Camera(1.0, sc.camera.fov, 1.0, 0.0, sc.camera.transformation)
    rays = oracle.camera_rays(cam, 96, 96)
    h = o.hit_full(rays)
    tri = h["leaf"] == 0
    assert 100 < tri.sum() < 96 * 96
    assert np.allclose(h["position"][tri].sum(axis=1), 1.0, atol=1e-12)
    img, fg, st = o.render(96, 96, 1, seed=5)
    # with jitter the hit set differs slightly from pixel centres; check every pixel that shows the debug colour
    k = 1.0 / math.sqrt(3.0)
    is_tri = np.isclose(img, k, atol=1e-12).all(axis=-1)
    assert abs(int(is_tri.sum()) - int(tri.sum())) < 0.1 * tri.sum()


def test_sky_gradient_closed_form():
    """material.rs:54-57 on rays that miss everything"""
    sc = scenes.three_balls()
    sc.hittables = sc.hittables[:0]
    o = oracle.Scene(sc)
    img, fg, st = o.render(32, 32, 1, seed=1)
    assert (fg == 0).all() and st.rays == 32 * 32
    assert (img[..., 2] == 1.0).all()                       # blue channel is (1-t)*1 + t*1
    t = (1.0 - img[..., 0]) / 0.5                           # red = (1-t) + 0.5 t
    assert (t >= 0).all() and (t <= 1).all()
    assert np.allclose(img[..., 1], (1 - t) + 0.7 * t, atol=1e-15)
    assert img[-1].mean() < img[0].mean()                   # j = 0 is the bottom row: top rows look up = bluer (less red)


# ----------------------------------------------------------------------------- BVH ----------------

@pytest.fixture(scope="module")
def bunny_oracle():
    sc = scenes.bunny_lambert()
    return sc, oracle.Scene(sc)


def test_bvh_shape(bunny_oracle):
    sc, o = bunny_oracle
    i = o.info()
    assert (i.n_leaves, i.n_nodes, i.depth) == (4969, 9937, 14)
    order = o.leaf_order()
    assert sorted(order) == list(range(4969))
    # post-order numbering: children before parent, root last (bvh.rs:43-52)
    assert o.root() == 9936
    box, lrl = o.node(o.root())
    assert lrl[2] == MISS and lrl[0] < 9936 and lrl[1] < 9936
    # root box = union of everything (ground sphere dominates)
    assert list(box[:3]) == [-1000.0, -2000.0, -1001.0] and list(box[3:]) == [1000.0, 1.53609, 999.0]
    # median split: left subtree holds floor(n/2) leaves
    _, l = o.node(lrl[0])
    def count(k):
        _, x = o.node(k)
        return 1 if x[2] != MISS else count(x[0]) + count(x[1])
    assert count(lrl[0]) == 4969 // 2


def test_bvh_vs_bruteforce_list(bunny_oracle):
    """the reference's own differential: Hittable::Bvh vs Hittable::List over the same primitives"""
    sc, o = bunny_oracle
    cam = api.Camera(16 / 9, sc.camera.fov, 1.0, 0.0, sc.camera.transformation)
    rays = np.concatenate([oracle.camera_rays(cam, 160, 90)[::3], scenes.incoherent_rays(4000, seed=3)])
    hb, hl = o.hit_full(rays, mode=0), o.hit_full(rays, mode=1)
    assert (hb["leaf"] == hl["leaf"]).all()
    assert hb["t"].tobytes() == hl["t"].tobytes()
    assert hb["normal"].tobytes() == hl["normal"].tobytes()


def test_bvh_vs_list_axis_aligned_and_boundary_rays(bunny_oracle):
    """rays with zero direction components / origins on box planes exercise the 0*inf = NaN lanes (SURVEY §8 a-note-1 caveat)"""
    sc, o = bunny_oracle
    rng = np.random.default_rng(4)
    pos = assets.bunny().vertices["position"]
    rays = []
    for k in range(1500):
        p = pos[rng.integers(len(pos))].copy()
        axis = rng.integers(3)
        d = np.zeros(3)
        d[axis] = rng.choice([-1.0, 1.0])
        if rng.random() < 0.5:
            d[(axis + 1) % 3] = rng.normal()
        org = p - 3 * d
        org[(axis + 2) % 3] = p[(axis + 2) % 3]   # shares an exact coordinate with a vertex → lands on box planes
        rays.append(list(org) + list(d) + [1e-3, np.inf])
    rays = np.array(rays)
    hb, hl = o.hit_full(rays, mode=0), o.hit_full(rays, mode=1)
    same = (hb["leaf"] == hl["leaf"]) & (hb["t"].view(np.uint64) == hl["t"].view(np.uint64))
    # the leaf's own slab gate can reject a primitive the brute-force scan accepts (ray exactly in a box plane);
    # everything else must agree
    diff = np.nonzero(~same)[0]
    for k in diff:
        assert hb["leaf"][k] == MISS or hb["t"][k] >= hl["t"][k]
    # (this degenerate family is exactly where Bvh and List legitimately differ in the reference: a 0*inf lane makes
    # the box gate reject, utility.rs:140-153 — the GPU path must follow the Bvh behaviour, tests/test_gpu_parity.py)
    assert 0 < len(diff) < 0.5 * len(rays)


def test_golden_hits_regression(bunny_oracle):
    """committed golden vector: oracle hits for every 97th ray of the C2 batch (made by tests/golden/make_golden_hits.py)"""
    sc, o = bunny_oracle
    z = np.load(os.path.join(GOLDEN, "c2_hits_every97.npz"))
    cam = api.Camera(1920 / 1080, sc.camera.fov, 1.0, 0.0, sc.camera.transformation)
    rays = oracle.camera_rays(cam, 1920, 1080)[::97]
    h = o.hit(rays)
    assert (h["leaf"] == z["leaf"]).all() and (h["t"].view(np.uint64) == z["t_bits"]).all()


# ----------------------------------------------------------------------------- integrator ---------

def test_render_is_independent_of_thread_count_and_tiling(bunny_oracle):
    sc, o = bunny_oracle
    a, fa, sa = o.render(64, 36, 3, seed=9, threads=1)
    b, fb, sb = o.render(64, 36, 3, seed=9, threads=5)
    assert a.tobytes() == b.tobytes() and fa.tobytes() == fb.tobytes() and sa.rays == sb.rays
    # tile rectangles reproduce the same pixels
    t, _, _ = o.render(64, 36, 3, seed=9, tile=(32, 4, 20, 17))
    assert t[4:21, 32:52].tobytes() == a[4:21, 32:52].tobytes()
    assert (t[:4] == 0).all() and (t[:, :32] == 0).all()
    # different seed → different image; ≤ max_bounce rays per path
    c, _, sc2 = o.render(64, 36, 3, seed=10)
    assert (c != a).any()
    assert sa.paths == 64 * 36 * 3 and sa.paths <= sa.rays <= 8 * sa.paths


def test_sample_ranges_sum_to_full_frame(bunny_oracle):
    sc, o = bunny_oracle
    full, ffg, _ = o.render(48, 27, 5, seed=2)
    a, fa, _ = o.render(48, 27, 5, seed=2, sample_range=(0, 3), flags=A.RENDER_RAW_SUMS)
    b, fb, _ = o.render(48, 27, 5, seed=2, sample_range=(3, 5), flags=A.RENDER_RAW_SUMS)
    assert np.allclose((a + b) / 5, full, rtol=1e-14, atol=1e-16)
    assert ((fa + fb) / 5 == ffg).all()


def test_depth_limit_and_first_hit_flag():
    sc = scenes.bunny_lambert()
    o = oracle.Scene(sc)
    _, _, s1 = o.render(40, 24, 2, max_bounce=1, seed=1)
    assert s1.rays == s1.paths                      # depth 1: exactly the primary ray (render.rs:128-131)
    rgb1, hit1, n1 = o.trace_one(40, 24, 20, 2, 0, max_bounce=1)
    assert n1 == 1 and hit1 and (rgb1 == 0).all()   # ground hit, bounce budget exhausted → black
    with pytest.raises(oracle.OracleError):
        o.render(8, 8, 1, max_bounce=0)             # assert!(depth >= 1), render.rs:97


def test_materials_smoke_values():
    """every scatter / absorb / emit / texture variant evaluates to finite, plausible colours"""
    for name in ("three_balls", "two_balls", "earth", "one_triangle", "glass_bunny", "demo"):
        o = oracle.Scene(getattr(scenes, name)())
        img, fg, st = o.render(48, 48, 2, seed=1)
        assert np.isfinite(img).all() and (img >= 0).all() and img.max() <= 6.0 + 1e-9, name
        assert 0 < fg.mean() <= 1, name


def test_texture_sampling_rules():
    sc = scenes.two_balls()
    sc.scene_data.texture_table += [api.Texture.Image(assets.earthmap()), api.Texture.Noise(3), api.Texture.DebugUVs, api.Texture.Missing]
    o = oracle.Scene(sc)
    e = assets.earthmap()
    # texture.rs:40-49: i = (u*w).clamp(0,w-1) as u32, texel (i,j) at i + j*w, /255, no filtering
    for (u, v), (i, j) in (((0.0, 0.0), (0, 0)), ((0.999999, 0.999999), (1023, 511)), ((1.5, -2.0), (1023, 0)), ((0.5, 0.25), (512, 128)),
                           ((float("nan"), 0.5), (0, 256))):
        assert (o.texture_sample(4, [0, 0, 0], [u, v]) == e[j, i, :3] / 255.0).all(), (u, v)
    assert list(o.texture_sample(6, [0, 0, 0], [0.3, 0.7])) == [0.3, 0.7, 0.0]
    assert list(o.texture_sample(7, [0, 0, 0], [0.3, 0.7])) == [0.0, 0.0, 0.0]
    # checker (texture.rs:51-60): even cells → `even` texture (id 1), odd → id 0
    assert list(o.texture_sample(2, [0.5, 0.5, 0.5], [0, 0])) == [0.9, 0.0, 0.5]
    assert list(o.texture_sample(2, [1.5, 0.5, 0.5], [0, 0])) == [0.2, 0.2, 0.2]
    assert list(o.texture_sample(2, [-0.5, 0.5, 0.5], [0, 0])) == [0.2, 0.2, 0.2]   # floor(-0.5) = -1 → odd
    # noise / perlin stay in [0,1] and are lattice-continuous
    n = o.texture_sample(5, [1.2, 3.4, -5.6], [0, 0])
    assert 0 <= n[0] <= 1 and n[0] == n[1] == n[2]
    assert (o.texture_sample(5, [1.9, 3.1, -5.01], [0, 0]) == n).all()
    p0 = o.texture_sample(3, [2.0, 3.0, 4.0], [0, 0])
    assert p0[0] == 0.5                                                              # perlin is 0 on lattice points
    p1, p2 = o.texture_sample(3, [2.3, 3.3, 4.3], [0, 0]), o.texture_sample(3, [2.3000001, 3.3, 4.3], [0, 0])
    assert 0 <= p1[0] <= 1 and abs(p1[0] - p2[0]) < 1e-5


def test_stdrng_stream_and_more_balls_scene():
    """`StdRng::from_seed([249; 32])` (example_scenes.rs:98) restated as ChaCha12 (scenes.StdRngStream): the block function is pinned by
    the published zero-key known answers for 8, 12 and 20 rounds; the scene generator (example_scenes.rs:63-138) by its invariants"""
    kat = {20: "76b8e0ada0f13d90405d6ae55386bd28bdd219b8a08ded1aa836efcc8b770dc7da41597c5157488d7724e03fb8d84a376a43b8f41518a11cc387b669b2ee6586",
           12: "9bf49a6a0755f953811fce125f2683d50429c3bb49e074147e0089a52eae155f0564f879d27ae3c02ce82834acfa8c793a629f2ca0de6919610be82f411326be",
           8: "3e00ef2f895f40d67f5bb8e81f09a5a12c840ec3ce9a7f3b181be188ef711a1e984ce172b9216f419f445367456d5619314a42a3da86b001387bfdb80e0cfe42"}
    for rounds, want in kat.items():
        r = scenes.StdRngStream(bytes(32), rounds)
        assert b"".join(w.to_bytes(4, "little") for w in r.block(0)).hex() == want
    r = scenes.StdRngStream(bytes(32))
    words = [r.next_u32() for _ in range(40)]  # the keystream in order, block after block (64-bit counter in words 12-13)
    assert words[:16] == r.block(0) and words[16:32] == r.block(1) and words[32:] == r.block(2)[:8]
    r = scenes.StdRngStream(bytes(32))
    lo, hi = r.block(0)[0], r.block(0)[1]
    assert r.next_u64() == (hi << 32) | lo  # rand_core BlockRng::next_u64: low word first
    r = scenes.StdRngStream(bytes([249] * 32))
    assert all(0.0 <= r.gen() < 1.0 for _ in range(1000))

    sc = scenes.more_balls()
    h = sc.hittables
    assert len(h) == 4 + 62 * 61 and len(sc.scene_data.material_table) == len(h) and sc.root_kind == "list"
    small = h[4:]
    assert (small["radius"] >= 0.1).all() and (small["radius"] <= 0.3).all() and (small["center"][:, 1] == small["radius"]).all()
    cell = np.array([(x, z) for x in range(-31, 31) for z in range(-31, 31) if z != 0], dtype=np.float64)
    assert (np.abs(small["center"][:, [0, 2]] - cell) <= 0.5 - small["radius"][:, None] + 1e-12).all()  # each ball stays inside its cell
    assert (small["material"] == np.arange(4, len(h))).all()
    kinds = np.array([m.scatter.kind for m in sc.scene_data.material_table[4:]])
    frac = [(kinds == k).mean() for k in (A.SCATTER_LAMBERT, A.SCATTER_METAL, A.SCATTER_DIELECTRIC)]
    assert abs(frac[0] - 0.7) < 0.03 and abs(frac[1] - 0.21) < 0.03 and abs(frac[2] - 0.09) < 0.02, frac
    # more_balls_optimized: the same list under Bvh::new; closest hits agree with the linear scan
    ob, ol = oracle.Scene(scenes.more_balls_optimized()), oracle.Scene(sc)
    assert ob.info().n_nodes == 2 * len(h) - 1
    cam = api.Camera(1.0, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    rays = oracle.camera_rays(cam, 96, 96)
    hb, hl = ob.hit(rays), ol.hit(rays)
    assert (hb["leaf"] == hl["leaf"]).all() and hb["t"].tobytes() == hl["t"].tobytes() and (hb["leaf"] != 0xFFFFFFFF).mean() > 0.5
    ob.close(); ol.close()
