"""rt_render_views: K cameras of one scene rendered in one call.  View v must render exactly the paths that
rt_set_camera(camera v) + rt_render renders, so every test compares a batch with the K single renders: the float sums
agree to summation order (1e-5 relative) and rgb8 to 1."""
import random

import numpy as np
import pytest

import raytrace_clj_b200 as rt
from raytrace_clj_b200 import camera as camm
from raytrace_clj_b200.native import (RT_ACCEL_BVH, RT_ACCEL_BRUTE_FORCE, RT_VARIANT_MEGAKERNEL, RT_VARIANT_WAVEFRONT,
                                      NativeError)

pytestmark = pytest.mark.gpu

VARIANTS = [RT_VARIANT_WAVEFRONT, RT_VARIANT_MEGAKERNEL]
NX, NY = 37, 23      # nx * ny = 851: not a multiple of 32, so warps straddle views


SCENES = {
    "random": lambda: rt.scene.make_random_scene(NX, NY, 11, True, random.Random(1)),        # >= 160 leaves: tensor-core cull
    "small": lambda: rt.scene.make_random_scene(NX, NY, 3, True, random.Random(3)),          # < 160 leaves: FP32 cull
    "cornell": lambda: rt.scene.make_cornell_box(NX, NY, True, random.Random(2)),            # generic leaves
    "final": lambda: rt.scene.make_final(NX, NY, random.Random(2), nb=4, ns=100),            # media, Perlin, image
    "sweep10k": lambda: rt.scene.make_scale_sweep_scene(NX, NY, 10_000, random.Random(5)),  # with RT_ACCEL_BVH
}
_cache = {}


def scene(name):
    if name not in _cache:
        sc = SCENES[name]()
        _cache[name] = (rt.native.marshal_world(sc["world"]), sc["camera"])
    return _cache[name]


def mixed_views(base):
    """The scene's own camera, a pinhole, a thin lens with aperture > 0, and two shutter windows of an animation."""
    o = np.asarray(base.origin, np.float64)
    look = o + (-np.asarray(base.w, np.float64) if hasattr(base, "w") else np.array([0.0, 0.0, -1.0]))
    up = np.array([0.0, 1.0, 0.0])
    aspect = NX / NY
    side = np.cross(look - o, up)
    side = side / max(np.linalg.norm(side), 1e-9)
    dist = float(np.linalg.norm(look - o))
    return [
        base,
        camm.pinhole_camera(lookfrom=o + 0.3 * side, lookat=look, vup=up, vfov=35.0, aspect=aspect),
        camm.thin_lens_camera(lookfrom=o - 0.2 * side, lookat=look, vup=up, vfov=25.0, aspect=aspect, aperture=0.2,
                              focus_dist=max(dist, 1.0), t0=0.0, t1=1.0),
        camm.thin_lens_camera(lookfrom=o, lookat=look, vup=up, vfov=30.0, aspect=aspect, aperture=0.0, focus_dist=1.0,
                              t0=0.0, t1=0.5),
        camm.thin_lens_camera(lookfrom=o, lookat=look, vup=up, vfov=30.0, aspect=aspect, aperture=0.0, focus_dist=1.0,
                              t0=0.5, t1=1.0),
    ]


@pytest.fixture(scope="module")
def renderer():
    r = rt.native.Renderer([0])
    yield r
    r.close()


def singles(r, cams, nx, ny, ns, depth, seed, variant):
    lins, imgs = [], []
    for c in cams:
        r.set_camera(*rt.native.marshal_camera(c) if not isinstance(c, tuple) else c)
        lin, img = r.render(nx, ny, ns, depth, seed=seed, variant=variant)
        lins.append(lin)
        imgs.append(img)
    return np.stack(lins), np.stack(imgs)


def assert_same(batch, single):
    (bl, bi), (sl, si) = batch, single
    assert bl.shape == sl.shape and bi.shape == si.shape
    bad = np.abs(bl - sl) > 1e-5 * np.abs(sl) + 1e-7
    assert not bad.any(), f"{bad.sum()} linear values differ beyond summation order; max {np.abs(bl - sl).max()}"
    assert np.abs(bi.astype(int) - si.astype(int)).max() <= 1


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("name", list(SCENES))
def test_views_equal_single_renders(renderer, name, variant):
    flat, base = scene(name)
    renderer.set_accel(RT_ACCEL_BVH if name == "sweep10k" else RT_ACCEL_BRUTE_FORCE)
    try:
        renderer.set_scene(flat)
        cams = mixed_views(base)
        batch = renderer.render_views(cams, NX, NY, 4, 50, seed=9, variant=variant)
        assert_same(batch, singles(renderer, cams, NX, NY, 4, 50, 9, variant))
        one = renderer.render_views(cams[2:3], NX, NY, 4, 50, seed=9, variant=variant)   # K = 1 is rt_render
        assert_same(one, singles(renderer, cams[2:3], NX, NY, 4, 50, 9, variant))
    finally:
        renderer.set_accel(RT_ACCEL_BRUTE_FORCE)


@pytest.mark.parametrize("variant", VARIANTS)
def test_many_views_with_queue_refills(renderer, variant):
    """12 views of 37 x 23 x 16 spp (163 k paths) through queues of 32 k paths: the stacked frame takes several refills."""
    flat, base = scene("random")
    cams = (mixed_views(base) * 3)[:12]
    with rt.native.Renderer([0]) as r:
        r.set_option("wave_capacity", 1 << 15)
        r.set_scene(flat)
        batch = r.render_views(cams, NX, NY, 16, 50, seed=4, variant=variant)
        assert_same(batch, singles(r, cams, NX, NY, 16, 50, 4, variant))


def _cube_map(origin, nx):
    dirs = [(1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)]
    ups = [(0, 1, 0), (0, 1, 0), (0, 0, -1), (0, 0, 1), (0, 1, 0), (0, 1, 0)]
    o = np.asarray(origin, np.float64)
    return [camm.pinhole_camera(lookfrom=o, lookat=o + np.array(d, np.float64), vup=np.array(u, np.float64), vfov=90.0,
                                aspect=1.0) for d, u in zip(dirs, ups)]


@pytest.mark.parametrize("name", ["random", "small"])   # tensor-core cull / FP32 cull, whose camera rays take the common form
@pytest.mark.parametrize("variant", VARIANTS)
def test_cube_map_and_distinct_origins(renderer, variant, name):
    flat, _ = scene(name)
    renderer.set_scene(flat)
    wave = variant == RT_VARIANT_WAVEFRONT
    cube = _cube_map((0.5, 1.5, 3.0), 24)     # one origin bit for bit: the common-origin cull is on for the batch
    renderer.reset_counters()
    batch = renderer.render_views(cube, 24, 24, 8, 50, seed=2, variant=variant)
    assert renderer.counters()["common_origin_rays"] == (6 * 24 * 24 * 8 if wave else 0)
    assert_same(batch, singles(renderer, cube, 24, 24, 8, 50, 2, variant))
    moved = _cube_map((0.5, 1.5, 3.0), 24)[:3] + _cube_map((0.5, 1.5, 3.5), 24)[3:]   # distinct origins: off
    renderer.reset_counters()
    batch = renderer.render_views(moved, 24, 24, 8, 50, seed=2, variant=variant)
    assert renderer.counters()["common_origin_rays"] == 0
    assert_same(batch, singles(renderer, moved, 24, 24, 8, 50, 2, variant))
    o = np.array([0.5, 1.5, 3.0])
    lens = [camm.thin_lens_camera(lookfrom=o, lookat=o + np.array([1.0, 0.0, 0.0]), vup=np.array([0.0, 1.0, 0.0]), vfov=90.0,
                                  aspect=1.0, aperture=0.2, focus_dist=1.0, t0=0.0, t1=1.0)] + cube[1:]   # aperture > 0: off
    renderer.reset_counters()
    renderer.render_views(lens, 24, 24, 2, 50, seed=2, variant=variant)
    assert renderer.counters()["common_origin_rays"] == 0


def test_context_camera_survives_and_rejections_change_nothing():
    flat, base = scene("random")
    cams = mixed_views(base)
    with rt.native.Renderer([0]) as r:
        r.set_scene(flat)
        lin, _ = r.render_views(cams[:2], NX, NY, 2, 20, seed=1)        # no rt_set_camera needed
        assert lin.shape == (2, NY, NX, 3)
        with pytest.raises(NativeError):
            r.render(NX, NY, 2, 20)                                    # the batch set no camera: RT_ERR_STATE
        ct, cf = rt.native.marshal_camera(cams[3])
        r.set_camera(ct, cf)
        ref = r.render(NX, NY, 2, 20, seed=5)
        r.render_views(cams, NX, NY, 2, 20, seed=1)
        assert_same(r.render(NX, NY, 2, 20, seed=5), ref)              # the camera set before the batch is back

        L = r.L
        types, camf = rt.native.marshal_views(cams)
        out = np.empty((len(cams), NY, NX, 3), np.float32)
        fp = rt.native._p(camf, rt.native._f32p)
        ip = rt.native._p(types, rt.native._i32p)
        lp = rt.native._p(out, rt.native._f32p)

        def call(n=len(cams), ip=ip, fp=fp, nx=NX, ny=NY, ns=2, depth=20, variant=RT_VARIANT_WAVEFRONT):
            return L.rt_render_views(r.h, n, ip, fp, nx, ny, ns, depth, 1, variant, lp, None)

        assert call(n=0) == -1
        assert call(ip=None) == -1
        assert call(fp=None) == -1
        assert call(nx=40000, ny=40000) == -1                          # one image over (2^31 - 1) / 3 pixels
        assert call(nx=12000, ny=12000) == -1                          # each image fits, the 5 stacked do not
        assert "n_views * nx * ny" in L.rt_last_error(r.h).decode()
        assert call(depth=256) == -1
        assert call(ns=1 << 24) == -1
        bad = types.copy()
        bad[3] = 7
        assert call(ip=rt.native._p(bad, rt.native._i32p)) == -2
        assert "view 3" in L.rt_last_error(r.h).decode()
        assert call(depth=256, variant=RT_VARIANT_MEGAKERNEL) == 0     # the megakernel takes any depth
        assert_same(r.render(NX, NY, 2, 20, seed=5), ref)


@pytest.mark.parametrize("variant", VARIANTS)
def test_device_leg_equals_the_host_call(renderer, variant):
    import torch

    flat, base = scene("random")
    renderer.set_scene(flat)
    cams = mixed_views(base)
    k, ns = len(cams), 8
    _, img = renderer.render_views(cams, NX, NY, ns, 50, seed=6, variant=variant)
    dev = torch.device("cuda:0")
    s = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(s):
        d_sum = torch.full((k, NY, NX, 3), float("nan"), device=dev)
        d_sum.zero_()            # queued on s before the render: the render must run after it
        renderer.render_views_accumulate_device(cams, NX, NY, 0, 3, d_sum.data_ptr(), seed=6, variant=variant,
                                                stream=s.cuda_stream, sync=False)
        renderer.render_views_accumulate_device(cams, NX, NY, 3, ns - 3, d_sum.data_ptr(), seed=6, variant=variant,
                                                stream=s.cuda_stream, sync=False)
        rgb = torch.zeros((k, NY, NX, 3), dtype=torch.uint8, device=dev)
        renderer.resolve_views_device(k, NX, NY, ns, d_sum.data_ptr(), rgb.data_ptr(), stream=s.cuda_stream, sync=False)
    s.synchronize()
    assert np.abs(rgb.cpu().numpy().astype(int) - img.astype(int)).max() <= 1


@pytest.mark.parametrize("variant", VARIANTS)
def test_counters_add_up(renderer, variant):
    flat, base = scene("small")
    renderer.set_scene(flat)
    cams = mixed_views(base)
    renderer.reset_counters()
    renderer.render_views(cams, NX, NY, 4, 50, seed=3, variant=variant)
    b = renderer.counters()
    renderer.reset_counters()
    singles(renderer, cams, NX, NY, 4, 50, 3, variant)
    s = renderer.counters()
    assert b["samples"] == len(cams) * NX * NY * 4 == s["samples"]
    for key in ("rays", "term_light", "term_absorb", "term_depth", "term_miss"):
        assert b[key] == s[key], key


def test_multi_device_batch_matches_single_device():
    import torch

    n_dev = torch.cuda.device_count()
    if n_dev < 2:
        pytest.skip("needs 2 GPUs")
    flat, base = scene("random")
    cams = mixed_views(base)
    with rt.native.Renderer([0]) as r1:
        r1.set_scene(flat)
        ref = r1.render_views(cams, NX, NY, 8, 50, seed=11)
    for rows in (0, 1):
        with rt.native.Renderer(list(range(n_dev))) as r2:
            r2.set_option("rows", rows)
            r2.set_scene(flat)
            got = r2.render_views(cams, NX, NY, 8, 50, seed=11)
        assert np.allclose(got[0], ref[0], rtol=1e-4, atol=1e-4), rows
        assert np.abs(got[1].astype(int) - ref[1].astype(int)).max() <= 1
