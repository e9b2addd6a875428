"""Nested containers (SURVEY.md 8f-3): `Hittable::List` as a BVH leaf or list item and `Hittable::Bvh` as a list item
(hittable.rs:13-14, 22-23, 110-120, 142-147; bvh.rs:70-124). Three implementations must agree bit for bit:
  * a LITERAL pure-Python recursion written from the Rust sources (this file, on top of test_bvh_restatement.LiteralBvh's
    primitives): `Hittable::hit` dispatch, `hit_list` with its cloned, shrinking ray, nested `Bvh::new` / `hit_node`,
    `bounding_box_list` (AABB::default() for an empty list, a left fold of unions otherwise), a panic for the box of a Bvh;
  * the C oracle, which recurses the same way (oracle/rtp_oracle.c hittable_hit);
  * the product, which FLATTENS the nesting into one gated sequence (rtp_host.cpp NestedFlattener) and walks its culling tree.
"""
import numpy as np
import pytest

import oracle
from rtp_b200 import _abi as A
from rtp_b200 import api
from test_bvh_restatement import MISS, Box, LiteralBvh, div, soup_rays, soup_scene
from test_gpu_parity import assert_images_equal


class Node:
    """python mirror of a nested Hittable: kind 'prim' (record), 'list' (items), 'bvh' (items)"""

    def __init__(self, kind, record=None, items=None):
        self.kind, self.record, self.items = kind, record, items or []


class LiteralNested(LiteralBvh):
    def __init__(self, sc, root_kind, tree):
        self.sc, self.mesh = sc, sc.scene_data.mesh_table
        self.root_kind, self.tree = root_kind, tree
        self.bvhs = {}
        if root_kind == "bvh":
            self.root_bvh = self.new_bvh(tree)

    def bbox(self, node):  # hittable.rs:27-34
        if node.kind == "prim":
            return self.bounding_box(node.record)
        if node.kind == "list":  # hittable.rs:142-147
            if not node.items:
                return Box([0.0, 0.0, 0.0], [0.0, 0.0, 0.0])
            box = self.bbox(node.items[0])
            for x in node.items[1:]:
                box = box.union(self.bbox(x))
            return box
        raise RuntimeError("Do not take the bounding box of a Bvh")  # hittable.rs:32

    def new_bvh(self, items):  # bvh.rs:70-91
        self.nodes = []
        root = self.make([(i, self.bbox(x)) for i, x in enumerate(items)], 0)
        return self.nodes, root, items

    def hit_any(self, node, o, d, t_min, t_max):  # hittable.rs:18-25
        if node.kind == "prim":
            return self.hit_leaf(node.record, o, d, t_min, t_max)
        if node.kind == "list":
            return self.hit_items(node.items, o, d, t_min, t_max)
        key = id(node)
        if key not in self.bvhs:
            self.bvhs[key] = self.new_bvh(node.items)
        r = self.hit_bvh(self.bvhs[key], o, d, t_min, t_max)
        return None if r is None else r[0]

    def hit_items(self, items, o, d, t_min, t_max, want_index=False):  # hittable.rs:110-120
        hit, index = None, None
        for i, x in enumerate(items):
            new = self.hit_any(x, o, d, t_min, t_max)
            if new is not None:
                t_max = new[0]
                hit, index = new, i
        return (hit, index) if want_index else hit

    def hit_bvh(self, bvh, o, d, t_min, t_max):  # bvh.rs:121-124
        nodes, root, items = bvh
        inv = [div(1.0, d[k]) for k in range(3)]
        return self.node_hit(nodes, items, root, o, d, inv, t_min, t_max)

    def node_hit(self, nodes, items, node, o, d, inv, t_min, t_max):  # bvh.rs:93-119
        nd = nodes[node]
        if nd[0] == "leaf":
            if nd[1].collide(o, inv, t_min, t_max):
                r = self.hit_any(items[nd[2]], o, d, t_min, t_max)
                return None if r is None else (r, nd[2])
            return None
        if not nd[1].collide(o, inv, t_min, t_max):
            return None
        hit = None
        new = self.node_hit(nodes, items, nd[2], o, d, inv, t_min, t_max)
        if new is not None:
            t_max = new[0][0]
            hit = new
        new = self.node_hit(nodes, items, nd[3], o, d, inv, t_min, t_max)
        if new is not None:
            hit = new
        return hit

    def hit(self, ray):
        o = [float(x) for x in ray["origin"]]
        d = [float(x) for x in ray["direction"]]
        if self.root_kind == "bvh":
            return self.hit_bvh(self.root_bvh, o, d, float(ray["t_min"]), float(ray["t_max"]))
        r, index = self.hit_items(self.tree, o, d, float(ray["t_min"]), float(ray["t_max"]), want_index=True)
        return None if r is None else (r, index)


def marshal(tree, pool):
    """python tree (list of Node) -> top-level rtp_hittable array, nested items go to `pool` (inner containers first)"""
    out = []
    for node in tree:
        if node.kind == "prim":
            out.append(np.asarray(node.record).reshape(1))
        else:
            items = marshal(node.items, pool)
            out.append(pool.List(items) if node.kind == "list" else pool.Bvh(items))
    return api.Hittable.concat(out)


def nested_scene(seed, root_kind):
    """a triangle soup + spheres regrouped into nested containers; every primitive appears exactly once"""
    base = soup_scene(seed, 90, True)
    prims = [Node("prim", record=base.hittables[i]) for i in range(len(base.hittables))]
    rng = np.random.default_rng(seed)
    rng.shuffle(prims)
    p = iter(prims)

    def take(k):
        return [next(p) for _ in range(k)]

    if root_kind == "bvh":
        tree = take(20)
        tree.append(Node("list", items=take(7)))                                        # a List as a BVH leaf
        tree.append(Node("list", items=[Node("list", items=take(3)), *take(2), Node("list", items=[])]))  # lists in a list; an empty one adds the origin to the box
        tree.append(Node("list", items=[]))                                             # an empty leaf: AABB::default(), never hit, still sorted
        tree.append(Node("list", items=take(1)))
        tree += list(p)
    else:
        tree = take(5)
        tree.append(Node("bvh", items=[*take(25), Node("list", items=take(6))]))         # a Bvh in the root list, one of its leaves a List
        tree.append(Node("list", items=[Node("bvh", items=take(12)), *take(3)]))         # a List holding a Bvh
        tree.append(Node("bvh", items=take(1)))                                         # a one-leaf Bvh
        tree += list(p)
    pool = api.NestedPool()
    top = marshal(tree, pool)
    sc = api.ExampleScene(base.camera, base.scene_data, root_kind, top, base.background, pool.array())
    return sc, tree


def check_against_literal(hits, lit, rays):
    n_hit = 0
    for k, ray in enumerate(rays):
        want = lit.hit(ray)
        g = hits[k]
        if want is None:
            assert g["leaf"] == MISS, (k, g)
            continue
        (t, pos, nrm, uv, material), top = want
        n_hit += 1
        assert (int(g["leaf"]), int(g["material"])) == (top, material), (k, g, want)
        assert np.float64(t).tobytes() == g["t"].tobytes(), (k, t, g["t"])
        if "position" in g.dtype.names:
            assert np.array(pos).tobytes() == g["position"].tobytes() and np.array(nrm).tobytes() == g["normal"].tobytes(), (k, g)
    assert n_hit > len(rays) // 3


@pytest.mark.parametrize("seed,root_kind", [(1, "bvh"), (2, "list"), (3, "bvh"), (4, "list")])
def test_oracle_recursion_equals_the_literal_recursion(seed, root_kind):
    sc, tree = nested_scene(seed, root_kind)
    lit = LiteralNested(sc, root_kind, tree)
    o = oracle.Scene(sc)
    rays = soup_rays(seed + 20, 700)
    check_against_literal(o.hit_full(rays), lit, rays)
    o.close()


def evaluation_order(tree, root_kind, lit):
    """ids of the root container's items in the order the reference's sequential process meets their primitives"""
    order = []

    def prims_of(node, top):
        if node.kind == "prim":
            order.append(top)
        elif node.kind == "list":
            for x in node.items:
                prims_of(x, top)
        else:
            nodes, root, items = lit.new_bvh(node.items)
            walk(nodes, items, root, lambda i: top)

    def walk(nodes, items, n, top_of):
        nd = nodes[n]
        if nd[0] == "leaf":
            prims_of(items[nd[2]], top_of(nd[2]))
        else:
            walk(nodes, items, nd[2], top_of)
            walk(nodes, items, nd[3], top_of)

    if root_kind == "bvh":
        nodes, root, items = lit.new_bvh(tree)
        walk(nodes, items, root, lambda i: i)
    else:
        for i, x in enumerate(tree):
            prims_of(x, i)
    return order


@pytest.mark.parametrize("seed,root_kind", [(1, "bvh"), (2, "list")])
def test_flattened_sequence_is_the_reference_evaluation_order(seed, root_kind):
    """host half of rtp_scene_create (no device): the flattened primitive sequence, reported as root-item ids per slot"""
    sc, tree = nested_scene(seed, root_kind)
    lit = LiteralNested(sc, root_kind, tree)
    order, info = api.bvh_build_order(sc)
    assert list(order) == evaluation_order(tree, root_kind, lit)
    assert info.n_leaves == len(order)


def test_nesting_errors_are_the_reference_panics():
    base = soup_scene(5, 12, False)
    h = base.hittables
    pool = api.NestedPool()
    inner = pool.Bvh(h[0:4])
    for kind, top, msg in [
        ("bvh", api.Hittable.concat([inner, h[4:6]]), "bounding box of a Bvh"),                      # a Bvh as a BVH leaf (hittable.rs:32)
        ("bvh", api.Hittable.concat([pool.List(api.Hittable.concat([inner])), h[4:6]]), "bounding box of a Bvh"),  # ... or inside a List leaf
    ]:
        sc = api.ExampleScene(base.camera, base.scene_data, kind, top, base.background, pool.array())
        with pytest.raises(api.RtpError, match=msg):
            api.bvh_build_order(sc)
        with pytest.raises(oracle.OracleError, match=msg):
            oracle.Scene(sc)
    # an empty nested Bvh: unreachable!() (bvh.rs:40)
    pool = api.NestedPool()
    sc = api.ExampleScene(base.camera, base.scene_data, "list", api.Hittable.concat([h[0:2], pool.Bvh(h[0:0])]), base.background, pool.array())
    with pytest.raises(api.RtpError, match="empty list"):
        api.bvh_build_order(sc)
    # a run outside the nested table / a container that names itself
    bad = np.zeros(1, dtype=A.HITTABLE_DTYPE)
    bad["kind"], bad["mesh"], bad["triangle"] = A.HITTABLE_LIST, 0, 5
    sc = api.ExampleScene(base.camera, base.scene_data, "list", api.Hittable.concat([h[0:2], bad]), base.background, h[0:2])
    with pytest.raises(api.RtpError, match="nested run out of range"):
        api.bvh_build_order(sc)
    cyc = np.zeros(1, dtype=A.HITTABLE_DTYPE)
    cyc["kind"], cyc["mesh"], cyc["triangle"] = A.HITTABLE_LIST, 0, 1
    sc = api.ExampleScene(base.camera, base.scene_data, "list", api.Hittable.concat([cyc]), base.background, cyc)
    with pytest.raises(api.RtpError, match="nested run out of range"):
        api.bvh_build_order(sc)


@pytest.mark.gpu
@pytest.mark.parametrize("seed,root_kind", [(1, "bvh"), (2, "list"), (3, "bvh"), (4, "list")])
def test_gpu_nested_scene_equals_oracle_and_literal(seed, root_kind, monkeypatch):
    sc, tree = nested_scene(seed, root_kind)
    lit = LiteralNested(sc, root_kind, tree)
    o = oracle.Scene(sc, libm="device")
    rays = soup_rays(seed + 20, 6000)
    want = o.hit_full(rays)
    for env in ({}, {"RTP_TRAVERSAL": "inorder"}, {"RTP_TRACE_KERNEL": "simple"}, {"RTP_F32_CULLING": "0"}):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        with api.Scene(sc) as g:
            got = g.hit_full(rays)
            assert (got["leaf"] == want["leaf"]).all() and (got["material"] == want["material"]).all(), env
            assert got["t"].tobytes() == want["t"].tobytes(), env
            assert got["position"].tobytes() == want["position"].tobytes() and got["normal"].tobytes() == want["normal"].tobytes(), env
            assert got["uv"].tobytes() == want["uv"].tobytes(), env
            if not env:
                check_against_literal(got[:400], lit, rays[:400])
        for k in env:
            monkeypatch.delenv(k)
    # and through the integrator
    with api.Scene(sc) as g:
        ig, fg, sg = g.render(48, 32, 2, max_bounce=4, seed=3)
        io, fo, so = o.render(48, 32, 2, max_bounce=4, seed=3)
        assert_images_equal(ig, io, f"nested {seed} {root_kind}")
        assert (fg == fo).all() and sg.rays == so.rays, (sg.rays, so.rays)
    o.close()
