"""RT_ACCEL_BVH's tree built on the device (rt_bvh_build.cuh, option bvh_build): the tree equals a numpy restatement of the
Karras LBVH node for node, carries the host builder's leaf boxes bit for bit, and every answer through it (closest hits,
whole paths) is the host tree's and brute force's.  The depth guard hands a tree deeper than the traversal's stack to the
host builder before any ray is traced."""
import random

import numpy as np
import pytest

import raytrace_clj_b200 as rt
from raytrace_clj_b200 import hitable as hit
from raytrace_clj_b200 import shader as shad
from raytrace_clj_b200 import texture as tex
from raytrace_clj_b200.util import vec3

pytestmark = pytest.mark.gpu

FMAX = float(np.finfo(np.float32).max)
BRUTE, BVH = rt.native.RT_ACCEL_BRUTE_FORCE, rt.native.RT_ACCEL_BVH
HOST, DEVICE = 0, 2
MAX_DEPTH = 48          # entries of bvh_closest's stack
NX, NY = 320, 200


# ---- numpy restatement of the device build -------------------------------------------------------------------------
def _children(nodes):
    return nodes[:, 12:14].copy().view(np.int32)


def _child_boxes(nodes):
    """[count, 2, 6]: (lo.xyz, hi.xyz) of each node's left and right child as stored."""
    return nodes[:, :12].reshape(-1, 2, 6)


def leaf_boxes(nodes, n):
    """[n, 6] float32: the box every leaf ~k is stored with (each leaf must appear exactly once, or twice in the n == 1 root)."""
    ch, cb = _children(nodes), _child_boxes(nodes)
    out = np.full((n, 6), np.nan, np.float32)
    seen = np.zeros(n, np.int64)
    for side in range(2):
        leaf = ch[:, side] < 0
        k = ~ch[leaf, side]
        out[k] = cb[leaf, side]
        np.add.at(seen, k, 1)
    return out, seen


def _bitlen32(v):
    return np.frexp(v.astype(np.float64))[1].astype(np.int64)       # exact for v < 2^53; 0 -> 0


def _clz64(x):
    hi, lo = (x >> np.uint64(32)).astype(np.uint64), (x & np.uint64(0xFFFFFFFF)).astype(np.uint64)
    return np.where(hi > 0, 32 - _bitlen32(hi), 64 - _bitlen32(lo))


def _spread3(v):
    x = v.astype(np.uint64) & np.uint64(0x1FFFFF)
    for sh, m in ((32, 0x1F00000000FFFF), (16, 0x1F0000FF0000FF), (8, 0x100F00F00F00F00F), (4, 0x10C30C30C30C30C3),
                  (2, 0x1249249249249249)):
        x = (x | (x << np.uint64(sh))) & np.uint64(m)
    return x


def morton_codes(boxes):
    c = np.float32(0.5) * (boxes[:, :3] + boxes[:, 3:])
    lo, hi = c.min(axis=0), c.max(axis=0)
    ext = hi - lo
    code = np.zeros(len(boxes), np.uint64)
    for a in range(3):
        q = np.zeros(len(boxes), np.uint32)
        if ext[a] > 0:
            f = ((c[:, a] - lo[a]) / ext[a]) * np.float32(2 ** 21)
            q = np.minimum(f.astype(np.uint32), np.uint32(2 ** 21 - 1))
        code |= _spread3(q) << np.uint64(2 - a)
    return code


def karras_tree(boxes):
    """Karras 2012 over the leaves' Morton codes (stable order for equal codes, index prefix as the tie-breaker), boxes
    fitted bottom up.  Returns (nodes [n-1, 16] f32 in the library's layout, depth of the deepest leaf)."""
    n = len(boxes)
    code = morton_codes(boxes)
    order = np.argsort(code, kind="stable").astype(np.int64)
    sc = code[order]

    def delta(i, j):
        ok = (j >= 0) & (j < n)
        jj = np.clip(j, 0, n - 1)
        a, b = sc[i], sc[jj]
        d = np.where(a != b, _clz64(a ^ b), 64 + 32 - _bitlen32((i ^ jj).astype(np.uint64)))
        return np.where(ok, d, -1)

    i = np.arange(n - 1, dtype=np.int64)
    d = np.where(delta(i, i + 1) > delta(i, i - 1), 1, -1)
    dmin = delta(i, i - d)
    lmax = np.full(n - 1, 2, np.int64)
    while True:
        grow = delta(i, i + lmax * d) > dmin
        if not grow.any():
            break
        lmax = np.where(grow, lmax * 2, lmax)
    l = np.zeros(n - 1, np.int64)
    t = lmax // 2
    while (t >= 1).any():
        take = (t >= 1) & (delta(i, i + (l + t) * d) > dmin)
        l += np.where(take, t, 0)
        t //= 2
    j = i + l * d
    dnode = delta(i, j)
    s = np.zeros(n - 1, np.int64)
    t = l.copy()
    active = np.ones(n - 1, bool)
    while active.any():
        t = np.where(active, (t + 1) // 2, t)
        take = active & (delta(i, i + (s + t) * d) > dnode)
        s += np.where(take, t, 0)
        active &= t > 1
    gamma = i + s * d + np.minimum(d, 0)
    left = np.where(np.minimum(i, j) == gamma, ~order[gamma], gamma)
    right = np.where(np.maximum(i, j) == gamma + 1, ~order[np.minimum(gamma + 1, n - 1)], gamma + 1)
    ch = np.stack([left, right], axis=1)
    # bottom up: a node is fitted once both children are
    node_box = np.zeros((n - 1, 6), np.float32)
    height = np.full(n - 1, -1, np.int64)
    child_box = np.zeros((n - 1, 2, 6), np.float32)
    while (height < 0).any():
        todo = height < 0
        ready = todo.copy()
        hs = []
        for side in range(2):
            c = ch[:, side]
            is_leaf = c < 0
            ready &= is_leaf | (height[np.where(is_leaf, 0, c)] >= 0)
        for side in range(2):
            c = ch[ready, side]
            is_leaf = c < 0
            b = np.where(is_leaf[:, None], boxes[np.where(is_leaf, ~c, 0)], node_box[np.where(is_leaf, 0, c)])
            child_box[ready, side] = b
            hs.append(np.where(is_leaf, 0, height[np.where(is_leaf, 0, c)]))
        assert ready.any(), "no node can be fitted: the children do not form a tree"
        node_box[ready, :3] = np.minimum(child_box[ready, 0, :3], child_box[ready, 1, :3])
        node_box[ready, 3:] = np.maximum(child_box[ready, 0, 3:], child_box[ready, 1, 3:])
        height[ready] = 1 + np.maximum(hs[0], hs[1])
    nodes = np.zeros((n - 1, 16), np.float32)
    nodes[:, :12] = child_box.reshape(n - 1, 12)
    nodes[:, 12:14] = ch.astype(np.int32).view(np.float32)
    return nodes, int(height[0])


def tree_depth(nodes):
    ch = _children(nodes)
    depth, frontier, dmax = 0, np.array([0]), 0
    while len(frontier):
        depth += 1
        c = ch[frontier].ravel()
        if (c < 0).any():
            dmax = depth
        frontier = np.unique(c[c >= 0])
    return dmax


# ---- scenes ----------------------------------------------------------------------------------------------------------
def _lambert(rgb=(0.5, 0.5, 0.5)):
    return shad.lambertian(albedo=tex.constant(color=vec3(*rgb)))


def _spheres(centres, radii):
    return {"camera": rt.scene._random_scene_camera(NX, NY),
            "world": hit.hitlist(items=[hit.sphere(center=vec3(*c), radius=float(r), material=_lambert()) for c, r in zip(centres, radii)])}


def _caterpillar():
    """Leaves whose Morton codes are 0, then one bit each from bit 0 to bit 62, then all ones: successive leaves share one
    more leading bit, so the Karras tree is a caterpillar about 63 deep.  Centroids sit mid-cell (units s = 2^-16, every
    coordinate exact in float32), so the float rounding of the leaf boxes cannot move a leaf to another cell."""
    s, b = 2.0 ** -16, 4.0 * 2.0 ** -16
    cs = [(b, b, b), (b + 2 ** 21 * s,) * 3]
    for j in range(21):
        for a in range(3):
            p = [b, b, b]
            p[a] = b + (2 ** j + 0.5) * s
            cs.append(tuple(p))
    return _spheres(cs, [s / 4] * len(cs))


SCENES = {
    "random": lambda: rt.scene.make_random_scene(NX, NY, 11, True, random.Random(1)),
    "sweep10k": lambda: rt.scene.make_scale_sweep_scene(NX, NY, 10_000, random.Random(5)),
    "sweep100k": lambda: rt.scene.make_scale_sweep_scene(NX, NY, 100_000, random.Random(5)),
    "cornell": lambda: rt.scene.make_cornell_box(NX, NY, True, random.Random(2)),
    "final": lambda: rt.scene.make_final(NX, NY, random.Random(2)),
    "one": lambda: _spheres([(0, 0, -1)], [0.5]),
    "two": lambda: _spheres([(0, 0, -1), (0.3, 0.2, -2)], [0.5, 0.7]),
    "same_centre": lambda: _spheres([(0.0, 0.0, 0.0)] * 64, np.linspace(0.05, 0.9, 64)),   # symmetric boxes: equal centroids
    "caterpillar": _caterpillar,
}
_cache = {}


def scene(name):
    if name not in _cache:
        sc = SCENES[name]()
        flat = rt.native.marshal_world(sc["world"])
        cam_type, cam = rt.native.marshal_camera(sc["camera"])
        _cache[name] = (flat, cam_type, cam)
    return _cache[name]


@pytest.fixture(scope="module")
def renderer():
    r = rt.native.Renderer([0])
    yield r
    r.close()


def build(renderer, name, mode):
    """The tree of `name` built with bvh_build = mode (set_scene marks it out of date; rt_get_bvh builds it)."""
    flat, cam_type, cam = scene(name)
    renderer.set_option("bvh_build", mode)
    renderer.set_scene(flat)
    renderer.set_camera(cam_type, cam)
    nodes, info = renderer.bvh()
    return flat, nodes, info


def n_list(nodes):
    ch = _children(nodes)
    return int((~ch[ch < 0]).max()) + 1


def check_structure(nodes, info, n):
    """Every listed leaf once, n - 1 internal nodes reached from node 0, boxes that contain everything below them, and
    the reported depth the true one."""
    ch = _children(nodes)
    assert info["nodes"] == len(nodes) == max(1, n - 1)
    assert np.all(nodes[:, 14:16].view(np.uint32) == 0)
    boxes, seen = leaf_boxes(nodes, n)
    assert np.all(seen == (2 if n == 1 else 1))
    if n > 1:
        internal = ch[ch >= 0]
        assert len(internal) == n - 2 and len(np.unique(internal)) == n - 2 and not (internal == 0).any()
        cb = _child_boxes(nodes)
        for side in range(2):
            c = ch[:, side]
            sub = c >= 0
            own_lo = np.minimum(cb[c[sub], 0, :3], cb[c[sub], 1, :3])
            own_hi = np.maximum(cb[c[sub], 0, 3:], cb[c[sub], 1, 3:])
            assert np.all(cb[sub, side, :3] <= own_lo) and np.all(cb[sub, side, 3:] >= own_hi)
    assert info["depth"] == tree_depth(nodes)
    return boxes


# ---- tests -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["random", "sweep10k", "sweep100k", "cornell", "final", "two", "same_centre"])
def test_device_tree_equals_the_numpy_restatement(renderer, name):
    flat, nodes, info = build(renderer, name, DEVICE)
    assert info["builder"] == "device" and info["build_ns"] > 0
    n = n_list(nodes)
    boxes, _ = leaf_boxes(nodes, n)
    want, depth = karras_tree(boxes)
    print(f"[bvh-build] {name}: {n} leaves, depth {info['depth']}, device build {info['build_ns'] / 1e3:.1f} us")
    assert np.array_equal(nodes.view(np.uint32), want.view(np.uint32))
    assert info["depth"] == depth


@pytest.mark.parametrize("name", ["random", "sweep10k", "sweep100k", "cornell", "final", "one", "two", "same_centre"])
def test_device_tree_has_the_host_leaf_boxes_and_a_valid_structure(renderer, name):
    _, host, hinfo = build(renderer, name, HOST)
    _, dev, dinfo = build(renderer, name, DEVICE)
    assert hinfo["builder"] == "host" and hinfo["build_ns"] == 0 and dinfo["builder"] == "device"
    n = n_list(host)
    assert n_list(dev) == n
    hb = check_structure(host, hinfo, n)
    db = check_structure(dev, dinfo, n)
    assert np.array_equal(hb.view(np.uint32), db.view(np.uint32))
    if n == 1:
        assert np.array_equal(host.view(np.uint32), dev.view(np.uint32))


def _camera_and_secondary_rays(renderer, flat, cam, g, n=120_000):
    camd = np.asarray(cam, np.float64)
    o = np.tile(camd[0:3], (n, 1)).astype(np.float32)
    d = (camd[3:6] + g.random((n, 1)) * camd[6:9] + g.random((n, 1)) * camd[9:12] - camd[0:3]).astype(np.float32)
    tm = g.random(n).astype(np.float32)
    renderer.set_accel(BRUTE)
    t0, id0 = renderer.trace_primary(o, d, tm)
    h = id0 >= 0
    p = (o[h].astype(np.float64) + t0[h][:, None] * d[h].astype(np.float64)).astype(np.float32)
    nd = g.normal(size=p.shape).astype(np.float32)
    return (o, d, tm), (p, nd, tm[h])


def _answers(renderer, rays, pix, smp):
    out = [renderer.trace_primary(*r) for r in rays]
    renderer.reset_counters()
    paths = renderer.trace_paths(NX, NY, pix, smp, 50, seed=3)
    return out, paths, renderer.counters()


@pytest.mark.parametrize("name", ["random", "sweep10k", "sweep100k", "cornell", "final"])
def test_device_tree_answers_equal_the_host_tree_and_brute_force(renderer, name):
    flat, cam_type, cam = scene(name)
    renderer.set_scene(flat)
    renderer.set_camera(cam_type, cam)
    g = np.random.default_rng(9)
    rays = _camera_and_secondary_rays(renderer, flat, cam, g)
    m = 150_000
    pix = g.integers(0, NX * NY, m).astype(np.int32)
    smp = g.integers(0, 64, m).astype(np.int32)
    try:
        renderer.set_accel(BRUTE)
        res = {"brute": _answers(renderer, rays, pix, smp)}
        for label, mode in (("host", HOST), ("device", DEVICE)):
            renderer.set_option("bvh_build", mode)
            renderer.set_scene(flat)
            renderer.set_accel(BVH)
            assert renderer.bvh()[1]["builder"] == label
            res[label] = _answers(renderer, rays, pix, smp)
        b = res["brute"]
        for label in ("host", "device"):
            x = res[label]
            for (tb, ib), (tx, ix) in zip(b[0], x[0]):
                assert np.array_equal(ib, ix) and np.array_equal(tb, tx), (label, int((ib != ix).sum()))
            same = np.array_equal(b[1][0], x[1][0]) and np.array_equal(b[1][1], x[1][1]) and np.array_equal(b[1][2], x[1][2])
            if not same:                                                   # diagnostics before failing
                bad = np.nonzero((b[1][1] != x[1][1]) | np.any(b[1][0] != x[1][0], axis=1))[0]
                print(f"[bvh-build] {name} {label}: {len(bad)} of {m} paths differ; first {bad[:6]}, nrays "
                      f"{b[1][1][bad[:6]]} vs {x[1][1][bad[:6]]}")
            assert same, label
            assert x[2]["rays"] == int(x[1][1].sum()) and x[2]["bvh_node_tests"] > 0
        # tree quality: box tests and exact leaf tests per ray of the device tree within 2x of the host tree's
        h, dv = res["host"][2], res["device"][2]
        box = dv["bvh_node_tests"] / h["bvh_node_tests"]
        leaf = dv["sphere_tests"] / h["sphere_tests"]
        print(f"[bvh-build] {name}: per ray, host tree {h['bvh_node_tests'] / h['rays']:.2f} box / {h['sphere_tests'] / h['rays']:.2f} "
              f"exact tests, device tree {dv['bvh_node_tests'] / dv['rays']:.2f} / {dv['sphere_tests'] / dv['rays']:.2f}; "
              f"ratios {box:.3f} / {leaf:.3f}")
        if name in ("random", "sweep100k"):
            assert box <= 2.0 and leaf <= 2.0, (box, leaf)
    finally:
        renderer.set_accel(BRUTE)
        renderer.set_option("bvh_build", 1)


def test_device_builds_are_deterministic(renderer):
    _, a, ia = build(renderer, "sweep10k", DEVICE)
    _, b, ib = build(renderer, "sweep10k", DEVICE)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and ia["depth"] == ib["depth"]


def test_multi_device_context_holds_one_tree_on_every_device():
    import torch

    n_dev = torch.cuda.device_count()
    if n_dev < 2:
        pytest.skip("one device visible")
    flat, cam_type, cam = scene("sweep10k")
    ids = list(range(min(n_dev, 8)))
    with rt.native.Renderer(ids) as r:
        r.set_option("bvh_build", DEVICE)
        r.set_scene(flat)
        r.set_camera(cam_type, cam)
        r.set_accel(BVH)
        trees = [r.bvh(k) for k in range(len(ids))]
        for nodes, info in trees:
            assert info["builder"] == "device"
            assert np.array_equal(nodes.view(np.uint32), trees[0][0].view(np.uint32))
        lin, _ = r.render(NX, NY, 4 * len(ids), 50, seed=5)
    with rt.native.Renderer([0]) as r1:
        r1.set_option("bvh_build", DEVICE)
        r1.set_scene(flat)
        r1.set_camera(cam_type, cam)
        r1.set_accel(BVH)
        lin1, _ = r1.render(NX, NY, 4 * len(ids), 50, seed=5)
    assert np.allclose(lin, lin1, rtol=1e-5, atol=1e-6)


def test_window_growth_rebuilds_on_the_device(renderer):
    """Moving spheres: a new thin-lens camera whose shutter is wider than the scene's [0, 1] grows the movers' window; the
    tree is rebuilt on the device with the host builder's leaf boxes for the new window, and rays timed across the whole
    window still get brute force's answers."""
    flat, cam_type, cam = scene("random")
    assert (np.asarray(flat.sphere_flags) & rt.native.RT_SPHERE_MOVING).any()
    wide = rt.camera.thin_lens_camera(lookfrom=vec3(13, 2, 3), lookat=vec3(0, 0, 0), vup=vec3(0, 1, 0), vfov=20,
                                      aspect=NX / NY, aperture=0.1, focus_dist=10.0, t0=-1.5, t1=2.5)
    wide_type, wide_cam = rt.native.marshal_camera(wide)
    trees = {}
    try:
        for label, mode in (("host", HOST), ("device", DEVICE)):
            renderer.set_option("bvh_build", mode)
            renderer.set_camera(cam_type, cam)                       # rt_set_scene covers the shutter of the camera already set
            renderer.set_scene(flat)
            renderer.set_accel(BVH)
            before = renderer.bvh()
            renderer.set_camera(wide_type, wide_cam)
            renderer.render(16, 16, 1, 5, seed=1)                    # the render grows the window and rebuilds the tree
            after = renderer.bvh()
            assert before[1]["builder"] == after[1]["builder"] == label
            n = n_list(after[0])
            b0, _ = leaf_boxes(before[0], n)
            b1, _ = leaf_boxes(after[0], n)
            assert not np.array_equal(b0, b1)                        # the movers' boxes grew
            trees[label] = b1
        assert np.array_equal(trees["host"].view(np.uint32), trees["device"].view(np.uint32))
        g = np.random.default_rng(3)
        n = 120_000
        (o, d, _), _ = _camera_and_secondary_rays(renderer, flat, cam, g, n)
        tm = g.uniform(-1.5, 2.5, n).astype(np.float32)
        renderer.set_accel(BRUTE)
        tb, ib = renderer.trace_primary(o, d, tm)
        renderer.set_accel(BVH)
        assert renderer.bvh()[1]["builder"] == "device"
        tx, ix = renderer.trace_primary(o, d, tm)
        assert np.array_equal(ib, ix) and np.array_equal(tb, tx)
    finally:
        renderer.set_accel(BRUTE)
        renderer.set_option("bvh_build", 1)


def _compare_random_rays(renderer, flat, g, n=50_000):
    """Rays from up to 50 radii away aimed within half a radius of a random sphere's centre (the direction taken from the
    float32 origin, so that even the caterpillar's tiny spheres are hit)."""
    c = np.asarray(flat.center0_r, np.float64)
    k = g.integers(0, flat.n_spheres, n)
    r = np.abs(c[k, 3:4])
    o = (c[k, :3] + g.normal(size=(n, 3)) * 50 * r).astype(np.float32)
    d = (c[k, :3] + g.normal(size=(n, 3)) * 0.5 * r - o.astype(np.float64)).astype(np.float32)
    renderer.set_accel(BRUTE)
    tb, ib = renderer.trace_primary(o, d, None, 0.001, FMAX)
    renderer.set_accel(BVH)
    tx, ix = renderer.trace_primary(o, d, None, 0.001, FMAX)
    renderer.set_accel(BRUTE)
    assert (ib >= 0).sum() > n // 10
    assert np.array_equal(ib, ix) and np.array_equal(tb, tx)


@pytest.mark.parametrize("name", ["one", "two", "same_centre"])
def test_edge_sizes_answer_as_brute_force(renderer, name):
    flat, _, info = build(renderer, name, DEVICE)
    assert info["builder"] == "device"
    try:
        _compare_random_rays(renderer, flat, np.random.default_rng(5))
    finally:
        renderer.set_option("bvh_build", 1)


def test_a_million_leaves(renderer):
    """1 M listed spheres (the sweep's r = 0.2 grid, marshalled with numpy): the device tree equals the restatement, has the
    host builder's leaf boxes, and answers as brute force."""
    base = scene("two")[0]
    n = 1_000_000
    side = 1000
    g = np.random.default_rng(11)
    a, b = np.meshgrid(np.arange(side) - side // 2, np.arange(side) - side // 2, indexing="ij")
    c0r = np.zeros((n, 4), np.float32)
    c0r[:, 0] = a.ravel() + 0.9 * g.random(n)
    c0r[:, 1] = 0.2
    c0r[:, 2] = b.ravel() + 0.9 * g.random(n)
    c0r[:, 3] = 0.2
    flat = rt.native.FlatScene(center0_r=c0r, center1=c0r.copy(), t0t1=np.tile(np.float32([0, 1]), (n, 1)),
                               sphere_flags=np.zeros(n, np.uint32), material_id=np.zeros(n, np.int32),
                               mat_type=base.mat_type, mat_param=base.mat_param, mat_tex=base.mat_tex, tex_type=base.tex_type,
                               tex_params=base.tex_params, tex_children=base.tex_children)
    _cache["million"] = (flat,) + scene("random")[1:]
    try:
        _, host, hinfo = build(renderer, "million", HOST)
        _, dev, dinfo = build(renderer, "million", DEVICE)
        assert hinfo["builder"] == "host" and dinfo["builder"] == "device"
        nl = n_list(dev)
        db = check_structure(dev, dinfo, nl)
        hb, _ = leaf_boxes(host, nl)
        assert np.array_equal(hb.view(np.uint32), db.view(np.uint32))
        want, depth = karras_tree(db)
        assert np.array_equal(dev.view(np.uint32), want.view(np.uint32)) and dinfo["depth"] == depth
        print(f"[bvh-build] 1 M leaves: depth {depth}, device build {dinfo['build_ns'] / 1e6:.2f} ms")
        _compare_random_rays(renderer, flat, np.random.default_rng(6), 20_000)
    finally:
        _cache.pop("million", None)
        renderer.set_option("bvh_build", 1)


def test_depth_guard_takes_the_host_build_before_any_traversal(renderer):
    """A caterpillar Morton tree deeper than the traversal's stack: the device build reports it, the host tree is published
    instead, and only then is a single ray traced."""
    flat, nodes, info = build(renderer, "caterpillar", DEVICE)      # rt_get_bvh only: no ray has been traced
    assert info["builder"] == "host" and info["depth"] <= MAX_DEPTH
    n = n_list(nodes)
    boxes = check_structure(nodes, info, n)
    _, morton_depth = karras_tree(boxes)
    print(f"[bvh-build] caterpillar: {n} leaves, Morton tree depth {morton_depth}, published host tree depth {info['depth']}")
    assert morton_depth > MAX_DEPTH                                  # the scene does produce an over-deep device tree
    try:
        _compare_random_rays(renderer, flat, np.random.default_rng(8))
    finally:
        renderer.set_option("bvh_build", 1)
