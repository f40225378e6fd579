"""rt_set_scene_device (csrc/rt_scene_build.cuh): a sphere scene whose per-primitive arrays are torch CUDA tensors is built on
the GPU into the very blob rt_set_scene uploads for the same values, byte for byte; everything downstream (window growth,
the BVH builders, whole paths) then sees the same scene, rejections match the host path's, and the build is ordered after
the caller's stream."""
import ctypes as C
import functools
import random

import numpy as np
import pytest

import raytrace_clj_b200 as rt

gpu = pytest.mark.gpu
N = rt.native
BRUTE, BVH = N.RT_ACCEL_BRUTE_FORCE, N.RT_ACCEL_BVH
DEV = "cuda:0"


# ---- scenes ---------------------------------------------------------------------------------------------------------
def _flat(sc):
    """The marshalled scene with rt_set_scene's values.  A bvh-node world marshals with the tie rule RT_TIE_BVH, a field of
    rt_scene_ext that takes the host path through rt_set_scene_ex; the device path, like rt_set_scene, resolves exact ties
    by RT_TIE_HITLIST, so the reference here is the same arrays under that rule."""
    flat = N.marshal_world(sc["world"])
    flat.tie_rule = N.RT_TIE_HITLIST
    assert not flat.has_ext
    return flat, *N.marshal_camera(sc["camera"])


@functools.lru_cache(None)
def scene(name):
    """(flat, cam_type, cam) of a named scene."""
    if name == "random":
        return _flat(rt.scene.make_random_scene(1200, 800, 11, True, random.Random(1)))
    if name == "random-static":
        return _flat(rt.scene.make_random_scene(1200, 800, 11, False, random.Random(1)))
    if name == "stress":
        return _flat(rt.scene.make_material_stress_scene(1200, 800, 11, random.Random(4)))
    if name == "two-spheres":
        return _flat(rt.scene.make_two_spheres(1200, 800))
    if name.startswith("sweep:"):
        return _flat(rt.scene.make_scale_sweep_scene(1920, 1080, int(name.split(":")[1]), random.Random(5)))
    if name == "grid-1m":
        from scripts.bvh_build_bench import million
        return million()
    raise ValueError(name)


def synth(n, seed=0, radius=None, negative=False, movers=False, reversed_times=False, ground=False):
    """n spheres with the random scene's tables: optional equal radii, negative radii (hollow glass), movers, t0 > t1, and
    a ground sphere (direct when n > 16)."""
    base = scene("random")[0]
    g = np.random.default_rng(seed)
    c0r = np.zeros((n, 4), np.float32)
    c0r[:, :3] = g.uniform(-10, 10, (n, 3))
    c0r[:, 3] = radius if radius is not None else g.uniform(0.1, 1.0, n)
    if negative:
        c0r[::3, 3] *= -1
    if ground:
        c0r[0] = (0, -1000, 0, 1000)
    c1 = c0r.copy()
    c1[:, :3] += g.uniform(-1, 1, (n, 3)).astype(np.float32)
    tt = np.tile(np.float32([0, 1]), (n, 1))
    if reversed_times:
        tt = np.ascontiguousarray(tt[:, ::-1])
    fl = np.zeros(n, np.uint32)
    if movers:
        fl[1::2] |= N.RT_SPHERE_MOVING
    fl[::5] |= N.RT_SPHERE_UV
    mat = g.integers(0, len(base.mat_type), n).astype(np.int32)
    return N.FlatScene(center0_r=c0r, center1=c1, t0t1=tt, sphere_flags=fl, material_id=mat, mat_type=base.mat_type,
                       mat_param=base.mat_param, mat_tex=base.mat_tex, tex_type=base.tex_type, tex_params=base.tex_params,
                       tex_children=base.tex_children)


def set_device(r, flat, stream=None):
    r.set_scene_device(**flat.sphere_tensors(DEV), **flat.tables(), stream=stream)


def blobs(r, flat):
    r.set_scene(flat)
    host = r.scene_blob()
    set_device(r, flat)
    dev = r.scene_blob()
    return host, dev


def assert_same(host, dev):
    assert host.shape == dev.shape
    diff = np.flatnonzero(host != dev)
    assert diff.size == 0, f"{diff.size} bytes differ, first at {diff[:8]}"


@pytest.fixture(scope="module")
def renderer():
    with N.Renderer([0]) as r:
        yield r


# ---- 0. the symbols (no device needed) ------------------------------------------------------------------------------
def test_library_exports_and_binds_device_scene():
    L = N.load_library()
    for name in ("rt_set_scene_device", "rt_get_scene_blob"):
        assert name in N.ABI_SYMBOLS
        assert getattr(L, name).argtypes is not None
    assert callable(N.Renderer.set_scene_device) and callable(N.Renderer.scene_blob)
    assert callable(N.FlatScene.sphere_tensors)


# ---- 1. blob equality -----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["random", "random-static", "stress", "two-spheres", "sweep:1000", "sweep:10000", "sweep:100000",
                                  "grid-1m"])
@pytest.mark.parametrize("direct", [1, 0])
def test_blob_equals_host(renderer, name, direct):
    renderer.set_option("direct_spheres", direct)
    try:
        assert_same(*blobs(renderer, scene(name)[0]))
    finally:
        renderer.set_option("direct_spheres", 1)


@gpu
@pytest.mark.parametrize("kw", [dict(n=1), dict(n=16), dict(n=17), dict(n=17, ground=True), dict(n=500, radius=0.5),
                                dict(n=500, radius=0.5, ground=True), dict(n=300, negative=True, ground=True),
                                dict(n=300, movers=True, ground=True), dict(n=300, movers=True, reversed_times=True),
                                dict(n=3000, movers=True, negative=True, ground=True)],
                         ids=lambda kw: "-".join(f"{k}{v}" for k, v in kw.items()))
@pytest.mark.parametrize("direct", [1, 0])
def test_blob_equals_host_edge_cases(renderer, kw, direct):
    renderer.set_option("direct_spheres", direct)
    try:
        assert_same(*blobs(renderer, synth(**kw)))
    finally:
        renderer.set_option("direct_spheres", 1)


# ---- 2. window growth -----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["random", "synth-2000-movers"])
def test_window_growth_rebuilds_the_same_records(renderer, name):
    flat, cam_type, cam = scene("random")
    if name != "random":      # 2000 listed leaves: 8 tensor-core tiles
        flat = synth(2000, movers=True, ground=True)
    narrow, wide = np.array(cam, np.float32), np.array(cam, np.float32)
    narrow[22], narrow[23] = 0.25, 0.5
    wide[22], wide[23] = -0.5, 1.5
    pix, smp = np.arange(64, dtype=np.int32), np.zeros(64, np.int32)
    out = []
    for setter in (renderer.set_scene, lambda f: set_device(renderer, f)):
        renderer.set_camera(N.RT_CAM_THIN_LENS, narrow)
        setter(flat)
        before = renderer.scene_blob()
        renderer.set_camera(N.RT_CAM_THIN_LENS, wide)
        renderer.trace_paths(120, 80, pix, smp, 4, seed=1)    # widens the window: the records are rebuilt
        out.append((before, renderer.scene_blob()))
    assert_same(out[0][0], out[1][0])
    assert_same(out[0][1], out[1][1])
    assert (out[0][0] != out[0][1]).any(), "the wider shutter must change the movers' records"


# ---- 3. same answers ------------------------------------------------------------------------------------------------
def _paths(r, cam_type, cam, accel):
    r.set_camera(cam_type, cam)
    r.set_accel(accel)
    g = np.random.default_rng(3)
    pix = g.integers(0, 320 * 200, 20_000).astype(np.int32)
    smp = g.integers(0, 64, 20_000).astype(np.int32)
    rad, nr, term, log = r.trace_paths(320, 200, pix, smp, 50, seed=9, log_bounces=6)
    return rad, nr, term, log["hit_id"], log["t"].view(np.uint64)


@gpu
@pytest.mark.parametrize("name", ["random", "sweep:100000"])
@pytest.mark.parametrize("accel", [BRUTE, BVH])
def test_paths_identical(renderer, name, accel):
    flat, cam_type, cam = scene(name)
    renderer.set_scene(flat)
    ref = _paths(renderer, cam_type, cam, accel)
    set_device(renderer, flat)
    got = _paths(renderer, cam_type, cam, accel)
    renderer.set_accel(BRUTE)
    for a, b in zip(ref, got):
        np.testing.assert_array_equal(a, b)


@gpu
@pytest.mark.parametrize("name", ["random", "sweep:10000"])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_bvh_nodes_identical(renderer, name, mode):
    flat, cam_type, cam = scene(name)
    renderer.set_option("bvh_build", mode)
    try:
        renderer.set_camera(cam_type, cam)
        renderer.set_scene(flat)
        ref, ref_info = renderer.bvh()
        set_device(renderer, flat)
        got, got_info = renderer.bvh()
    finally:
        renderer.set_option("bvh_build", 1)
    assert ref_info["builder"] == got_info["builder"] and ref_info["depth"] == got_info["depth"]
    np.testing.assert_array_equal(ref.view(np.uint32), got.view(np.uint32))


# ---- 4. validation --------------------------------------------------------------------------------------------------
def _error(fn):
    with pytest.raises(N.NativeError) as e:
        fn()
    msg = str(e.value)
    return msg[msg.index("("):]     # "(status): message", without the entry point's name


def _bad_scenes():
    f = synth(40, movers=True)
    bad_mat = f.copy(); bad_mat.material_id[-1] = len(f.mat_type)
    bad_flag = f.copy(); bad_flag.sphere_flags[7] |= 8
    same_t = f.copy(); same_t.t0t1[5] = (0.5, 0.5)
    two = f.copy(); two.sphere_flags[30] |= 16; two.material_id[12] = -1          # the material error comes first
    iso = f.copy(); iso.mat_type = iso.mat_type.copy(); iso.mat_type[0] = N.RT_MAT_ISOTROPIC
    perlin = f.copy(); perlin.tex_type = perlin.tex_type.copy(); perlin.tex_type[0] = N.RT_TEX_PERLIN_NOISE
    return dict(bad_mat=bad_mat, bad_flag=bad_flag, same_t=same_t, two=two, iso=iso, perlin=perlin)


@gpu
@pytest.mark.parametrize("case", ["bad_mat", "bad_flag", "same_t", "two", "iso", "perlin"])
def test_rejections_match_host(renderer, case):
    good, cam_type, cam = scene("random")
    bad = _bad_scenes()[case]
    renderer.set_scene(good)
    ref = _paths(renderer, cam_type, cam, BRUTE)
    host = _error(lambda: renderer.set_scene(bad))
    set_device(renderer, good)
    dev = _error(lambda: set_device(renderer, bad))
    assert host == dev
    for a, b in zip(ref, _paths(renderer, cam_type, cam, BRUTE)):   # the previous scene is still in place
        np.testing.assert_array_equal(a, b)


@gpu
def test_host_pointer_rejected(renderer):
    import torch
    good, cam_type, cam = scene("random")
    set_device(renderer, good)
    ref = _paths(renderer, cam_type, cam, BRUTE)
    t = good.sphere_tensors(DEV)
    host_c0 = np.ascontiguousarray(good.center0_r, np.float32)
    dtypes = dict(mat_type=np.int32, mat_param=np.float32, mat_tex=np.int32, tex_type=np.int32, tex_params=np.float32,
                  tex_children=np.int32)
    k = {a: np.ascontiguousarray(v, dtypes[a]) for a, v in good.tables().items()}   # held until the call has returned
    p = lambda x, ty: C.cast(C.c_void_p(x.data_ptr()), ty)
    d = N._SceneDesc(good.n_spheres, host_c0.ctypes.data_as(N._f32p), p(t["center1"], N._f32p), p(t["t0t1"], N._f32p),
                     p(t["sphere_flags"], N._u32p), p(t["material_id"], N._i32p), len(k["mat_type"]),
                     k["mat_type"].ctypes.data_as(N._i32p), k["mat_param"].ctypes.data_as(N._f32p),
                     k["mat_tex"].ctypes.data_as(N._i32p), len(k["tex_type"]), k["tex_type"].ctypes.data_as(N._i32p),
                     k["tex_params"].ctypes.data_as(N._f32p), k["tex_children"].ctypes.data_as(N._i32p))
    torch.cuda.synchronize()
    rc = renderer.L.rt_set_scene_device(renderer.h, C.byref(d), None)
    assert rc == -1 and b"not device memory" in renderer.L.rt_last_error(renderer.h)
    with pytest.raises(ValueError):
        renderer.set_scene_device(torch.from_numpy(host_c0), t["material_id"], **good.tables())
    for a, b in zip(ref, _paths(renderer, cam_type, cam, BRUTE)):
        np.testing.assert_array_equal(a, b)


# ---- 5. stream ordering ---------------------------------------------------------------------------------------------
@gpu
def test_reads_after_the_callers_stream(renderer):
    import torch
    flat = scene("sweep:10000")[0]
    moved = flat.copy()
    moved.center0_r[:, 0] += np.float32(0.125)
    renderer.set_scene(moved)
    want = renderer.scene_blob()
    t = flat.sphere_tensors(DEV)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(50_000_000)              # the write below lands long after the call is made
        t["center0_r"][:, 0] += 0.125
        renderer.set_scene_device(**t, **flat.tables())   # stream = torch's current stream: s
    assert_same(want, renderer.scene_blob())


# ---- 6. animation ---------------------------------------------------------------------------------------------------
@gpu
def test_animation_frames(renderer):
    import torch
    flat = scene("random")[0]
    t = flat.sphere_tensors(DEV)
    step = torch.linspace(-0.01, 0.01, flat.n_spheres, device=DEV)
    for frame in range(20):
        t["center0_r"][:, 1] += step * (1 + frame % 3)
        renderer.set_scene_device(**t, **flat.tables())
        dev = renderer.scene_blob()
        host = flat.copy()
        host.center0_r = t["center0_r"].cpu().numpy()
        renderer.set_scene(host)
        assert_same(renderer.scene_blob(), dev)


# ---- 7. multiple devices --------------------------------------------------------------------------------------------
@gpu
def test_every_device_holds_the_same_blob():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    flat = scene("random")[0]
    with N.Renderer([0, 1]) as r:
        r.set_scene(flat)
        host = r.scene_blob(0)
        set_device(r, flat)
        assert_same(host, r.scene_blob(0))
        assert_same(host, r.scene_blob(1))
