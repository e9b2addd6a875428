"""CPU-only checks of the drop-in boundary: the C-ABI library loads, exports every symbol include/rtp.h
declares, its struct layouts match the ctypes mirror, host-side logic (BVH order, validation, errors) agrees
with the oracle, and compute entry points fail loudly without a GPU (no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import oracle
from rtp_b200 import _abi as A
from rtp_b200 import api, scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "rtp.h")


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rtp_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = A.load()
    names = declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/rtp.h but not exported by librtp_b200.so"
    # and the ctypes prototype table covers exactly the header
    assert sorted(A.PROTOTYPES) == names
    assert lib.rtp_abi_version() == A.ABI_VERSION


def test_struct_layouts_match_the_header(tmp_path):
    """compile include/rtp.h as plain C and compare sizeof/offsetof with the ctypes/numpy mirrors"""
    structs = {
        "rtp_ray": A.RAY_DTYPE.itemsize, "rtp_hit": A.HIT_DTYPE.itemsize, "rtp_hit_full": A.HIT_FULL_DTYPE.itemsize,
        "rtp_vertex": A.VERTEX_DTYPE.itemsize, "rtp_hittable": A.HITTABLE_DTYPE.itemsize, "rtp_mesh": C.sizeof(A.Mesh),
        "rtp_emit": C.sizeof(A.Emit), "rtp_material": C.sizeof(A.Material), "rtp_texture": C.sizeof(A.Texture),
        "rtp_scene_desc": C.sizeof(A.SceneDesc), "rtp_camera": C.sizeof(A.Camera), "rtp_render_params": C.sizeof(A.RenderParams),
        "rtp_stats": C.sizeof(A.Stats), "rtp_scene_info": C.sizeof(A.SceneInfo), "rtp_image": C.sizeof(A.Image),
        "rtp_any_tables": C.sizeof(A.AnyTables),
    }
    offsets = {
        ("rtp_material", "emit"): A.Material.emit.offset, ("rtp_texture", "rgba"): A.Texture.rgba.offset,
        ("rtp_scene_desc", "background"): A.SceneDesc.background.offset, ("rtp_camera", "position"): A.Camera.position.offset,
        ("rtp_render_params", "seed"): A.RenderParams.seed.offset, ("rtp_render_params", "flags"): A.RenderParams.flags.offset,
        ("rtp_render_params", "device_mask"): A.RenderParams.device_mask.offset, ("rtp_render_params", "row_stride"): A.RenderParams.row_stride.offset,
        ("rtp_scene_desc", "nested"): A.SceneDesc.nested.offset, ("rtp_scene_desc", "n_nested"): A.SceneDesc.n_nested.offset,
        ("rtp_stats", "device_ms"): A.Stats.device_ms.offset, ("rtp_stats", "trace_ms"): A.Stats.trace_ms.offset, ("rtp_hit_full", "uv"): A.HIT_FULL_DTYPE.fields["uv"][1],
        ("rtp_hittable", "center"): A.HITTABLE_DTYPE.fields["center"][1],
        ("rtp_any_tables", "any_E"): A.AnyTables.any_E.offset, ("rtp_any_tables", "cull"): A.AnyTables.cull.offset,
    }
    src = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){"]
    for s in structs:
        src.append(f'printf("{s} %zu\\n", sizeof({s}));')
    for (s, f) in offsets:
        src.append(f'printf("{s}.{f} %zu\\n", offsetof({s}, {f}));')
    src.append("return 0;}")
    c = tmp_path / "layout.c"
    c.write_text("\n".join(src))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(c)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for s, size in structs.items():
        assert int(got[s]) == size, s
    for (s, f), off in offsets.items():
        assert int(got[f"{s}.{f}"]) == off, (s, f)


@pytest.mark.parametrize("name", ["bunny_lambert", "glass_bunny", "demo", "two_balls", "one_triangle", "earth"])
def test_host_bvh_order_equals_oracle(name):
    """the product's Bvh::new (rtp_host.cpp) and the oracle's (rtp_oracle.c) are separate implementations"""
    sc = getattr(scenes, name)()
    order, info = api.bvh_build_order(sc)
    o = oracle.Scene(sc)
    oi = o.info()
    assert (info.n_leaves, info.n_nodes, info.depth) == (oi.n_leaves, oi.n_nodes, oi.depth)
    assert (order == o.leaf_order()).all()


def test_bvh_order_with_many_centroid_ties():
    """a grid of identical spheres has massive centroid ties on every axis: order must be (key, LeafId) in both builds"""
    parts = [api.Hittable.Sphere([x, y, z], 0.25, 0) for z in range(4) for y in range(5) for x in range(7)]
    rng = np.random.default_rng(0)
    perm = rng.permutation(len(parts))
    hit = api.Hittable.concat([parts[k] for k in perm])
    mats = [api.Material.new(api.Scatter.Lambert, api.Absorb.WhiteBody, api.Emit.NONE)]
    sc = api.ExampleScene(scenes._bunny_camera(), api.SceneData(mats, [], []), "bvh", hit, api.Emit.SkyGradient)
    order, info = api.bvh_build_order(sc)
    o = oracle.Scene(sc)
    assert (order == o.leaf_order()).all()
    assert info.n_nodes == 2 * len(parts) - 1 and info.depth == o.info().depth
    # first split is on x at the median: the left half holds the 70 smallest (x, id) keys
    xs = hit["center"][:, 0]
    want_left = sorted(range(len(parts)), key=lambda k: (xs[k], k))[: len(parts) // 2]
    assert sorted(order[: len(parts) // 2]) == sorted(want_left)


def test_list_root_keeps_caller_order():
    sc = scenes.three_balls()
    order, info = api.bvh_build_order(sc)
    assert list(order) == [0, 1, 2, 3] and info.n_nodes == 0 and info.root_kind == A.ROOT_LIST


def _bad(sc_mutator, code=A.ERR_INVALID):
    sc = scenes.one_triangle()
    sc_mutator(sc)
    with pytest.raises(api.RtpError) as e:
        api.bvh_build_order(sc)
    assert e.value.code == code and e.value.message
    with pytest.raises(api.RtpError) as e2:  # rtp_scene_create validates before it touches the device
        api.Scene(sc)
    assert e2.value.code == code
    with pytest.raises(oracle.OracleError) as e3:
        oracle.Scene(sc)
    assert e3.value.code == code


def test_scene_validation_errors():
    _bad(lambda s: setattr(s.scene_data.mesh_table[0], "material", 7))
    _bad(lambda s: s.scene_data.mesh_table[0].indices.__setitem__(1, 99))
    _bad(lambda s: s.hittables["material"].__setitem__(1, 5))
    _bad(lambda s: s.hittables["triangle"].__setitem__(0, 3))
    _bad(lambda s: s.hittables["mesh"].__setitem__(0, 2))
    _bad(lambda s: setattr(s, "background", api.Emit.SkySphere(0)))           # no textures in this scene
    _bad(lambda s: s.scene_data.material_table.__setitem__(1, api.Material.new(api.Scatter.Lambert, api.Absorb.AlbedoMap(3), api.Emit.NONE)))
    _bad(lambda s: setattr(s, "hittables", s.hittables[:0]))                  # Bvh::new(vec![]) is unreachable!() (bvh.rs:40)
    _bad(lambda s: s.hittables["center"].__setitem__(1, [np.nan, 0, 0]))      # partial_cmp().unwrap() (bvh.rs:63)

    _bad(lambda s: s.hittables["kind"].__setitem__(0, 9))                      # not a Hittable variant
    # nested containers are accepted (tests/test_nested_hittables.py), their runs are validated
    sc = scenes.one_triangle()
    sc.hittables["kind"][0], sc.hittables["mesh"][0], sc.hittables["triangle"][0] = A.HITTABLE_LIST, 0, 4
    with pytest.raises(api.RtpError) as e:
        api.bvh_build_order(sc)
    assert e.value.code == A.ERR_INVALID and "nested run" in str(e.value)


def test_abi_version_is_checked():
    sc = scenes.one_triangle()
    desc, keep = api.build_desc(sc)
    desc.abi_version = 99
    lib = A.load()
    assert lib.rtp_bvh_build_order(C.byref(desc), None, 0, None) == A.ERR_INVALID
    assert b"abi_version" in lib.rtp_last_error()
    h = C.c_void_p()
    assert lib.rtp_scene_create(C.byref(desc), C.byref(h)) == A.ERR_INVALID and not h.value
    assert lib.rtp_scene_create(None, C.byref(h)) == A.ERR_INVALID
    assert lib.rtp_scene_create(C.byref(desc), None) == A.ERR_INVALID


def _has_gpu():
    return api.device_count() > 0


@pytest.mark.skipif(_has_gpu(), reason="checks the behaviour WITHOUT a device")
def test_compute_entry_points_fail_loudly_without_a_gpu():
    """no CPU fallback: a valid scene cannot be created, and rtp_init reports why"""
    with pytest.raises(api.RtpError) as e:
        api.init(0)
    assert e.value.code == A.ERR_CUDA and "no CPU fallback" in e.value.message
    with pytest.raises(api.RtpError) as e2:
        api.Scene(scenes.one_triangle())
    assert e2.value.code == A.ERR_CUDA
    with pytest.raises(api.RtpError) as e3:
        api.camera_rays(scenes.one_triangle().camera, 4, 4)
    assert e3.value.code == A.ERR_CUDA
    lib = A.load()
    p = C.c_void_p()
    assert lib.rtp_host_alloc(64, C.byref(p)) == A.ERR_CUDA


def test_null_arguments_return_invalid():
    lib = A.load()
    assert lib.rtp_obj_load(None, None) == A.ERR_INVALID
    assert lib.rtp_tga_load(None, None) == A.ERR_INVALID
    assert lib.rtp_camera_lookat(None, None, None, None) == A.ERR_INVALID
    assert lib.rtp_trace_closest(None, None, 0, None, None) == A.ERR_INVALID
    assert lib.rtp_render(None, None, None, None, None, None) == A.ERR_INVALID
    assert lib.rtp_scene_get_info(None, None) == A.ERR_INVALID
    lib.rtp_scene_destroy(None)  # no-op
    lib.rtp_mesh_free(None)
    lib.rtp_image_free(None)
    lib.rtp_host_free(None)


def test_product_does_not_reference_the_oracle():
    """the product path must never route through oracle/ (or any CPU fallback)"""
    pkg = os.path.join(ROOT, "raytracing-potato_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cpp", ".h", ".hpp", "Makefile")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "rtp_oracle" not in text and "liboracle" not in text and "import oracle" not in text, os.path.join(dirpath, f)
    out = subprocess.run(["ldd", A.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in out


def test_traversal_plan_of_scenes():
    """host half of the any-order walk (prepare_any_order, rtp_host.cpp; DESIGN.md §4b), no device needed: which primitives are
    exempt from distance culling, which scenes are eligible at all, and that small scenes get the order-free tree"""
    _, info = api.bvh_build_order(scenes.bunny_lambert())
    assert (info.any_order, info.n_big) == (1, 1)  # the ground sphere
    assert 0 < info.culling_depth <= 16 and 0 < info.free_tree_depth <= 16
    _, info = api.bvh_build_order(scenes.demo())
    assert (info.any_order, info.n_big) == (1, 2)  # the ground and earth spheres dwarf the triangles; the small light sphere does not
    _, info = api.bvh_build_order(scenes.two_balls())
    assert (info.any_order, info.n_big) == (1, 0)  # two equal spheres: neither is outsized, the sphere term of the slack covers them
    _, info = api.bvh_build_order(scenes.more_balls_optimized())
    assert (info.any_order, info.n_big, info.n_leaves) == (1, 1, 3786)  # only the r = 1000 ground
    _, info = api.bvh_build_order(scenes.three_balls())  # a List root has no culling tree
    assert (info.any_order, info.culling_depth, info.free_tree_depth) == (0, 0, 0)

    mats = [api.Material.new(api.Scatter.Lambert, api.Absorb.WhiteBody, api.Emit.NONE)]

    def scene_of(hittables, meshes=()):
        return api.ExampleScene(scenes._bunny_camera(), api.SceneData(mats, [], list(meshes)), "bvh", hittables, api.Emit.SkyGradient)

    many = api.Hittable.concat([api.Hittable.Sphere([x, 0.0, 0.0], 0.4, 0) for x in range(40)] +
                               [api.Hittable.Sphere([3.0 * x, 50.0, 0.0], 20.0 + x, 0) for x in range(12)])
    _, info = api.bvh_build_order(scene_of(many))  # twelve outsized spheres: the eight largest are exempt, the others widen the slack
    assert (info.any_order, info.n_big) == (1, 8)
    inverted = api.Hittable.concat([api.Hittable.Sphere([0.0, 0.0, 0.0], -0.5, 0), api.Hittable.Sphere([2.0, 0.0, 0.0], 0.5, 0)])
    _, info = api.bvh_build_order(scene_of(inverted))  # an inverted leaf box: reference topology, literal slab test, in-order walk
    assert info.any_order == 0

    # a fine grid of small triangles on a ground made of two huge ones: only the two huge triangles are exempt
    pos, idx = [], []
    for x in range(12):
        for y in range(12):
            b = len(pos)
            pos += [[0.1 * x, 0.1 * y, 0.0], [0.1 * x + 0.1, 0.1 * y, 0.0], [0.1 * x, 0.1 * y + 0.1, 0.05]]
            idx += [b, b + 1, b + 2]
    b = len(pos)
    pos += [[-500.0, -500.0, -1.0], [500.0, -500.0, -1.0], [500.0, 500.0, -1.0], [-500.0, 500.0, -1.0]]
    idx += [b, b + 1, b + 2, b, b + 2, b + 3]
    mesh = api.Mesh.from_arrays(pos, indices=idx, material=0)
    _, info = api.bvh_build_order(scene_of(api.Hittable.triangles_of(mesh, 0), [mesh]))
    assert (info.any_order, info.n_big, info.n_leaves) == (1, 2, 146)


def build_c_driver(tmp_path):
    """tests/c_driver.c: a plain-C host of the boundary, compiled against include/rtp.h and linked with -lrtp_b200"""
    lib_dir = os.path.dirname(A.LIB_PATH)
    exe = tmp_path / "c_driver"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c_driver.c"), "-o", str(exe),
                    "-L", lib_dir, "-lrtp_b200", f"-Wl,-rpath,{lib_dir}", "-lm"], check=True)
    return exe


def test_plain_c_driver_host_side(tmp_path):
    """host-only entry points work from C; validation precedes the device; without a GPU the compute call is RTP_ERR_CUDA"""
    exe = build_c_driver(tmp_path)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr + r.stdout
    assert "host checks passed" in r.stdout


@pytest.mark.gpu
def test_plain_c_driver_on_the_gpu(tmp_path):
    exe = build_c_driver(tmp_path)
    r = subprocess.run([str(exe), "gpu"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr + r.stdout
    assert "GPU checks passed" in r.stdout
