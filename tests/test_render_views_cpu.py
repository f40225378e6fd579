"""The camera list of Renderer.render_views, marshalled on the host (no GPU needed)."""
import numpy as np
import pytest

import raytrace_clj_b200 as rt
from raytrace_clj_b200 import camera as camm
from raytrace_clj_b200.native import RT_CAM_PINHOLE, RT_CAM_THIN_LENS, marshal_camera, marshal_views


def _cams():
    o, at, up = np.array([13.0, 2.0, 3.0]), np.zeros(3), np.array([0.0, 1.0, 0.0])
    return [camm.pinhole_camera(lookfrom=o, lookat=at, vup=up, vfov=20.0, aspect=2.0),
            camm.thin_lens_camera(lookfrom=o, lookat=at, vup=up, vfov=20.0, aspect=2.0, aperture=0.1, focus_dist=10.0,
                                  t0=0.25, t1=0.75)]


def test_marshal_views_accepts_cameras_and_marshalled_pairs():
    cams = _cams()
    types, recs = marshal_views(cams + [marshal_camera(cams[1])])
    assert types.dtype == np.int32 and recs.dtype == np.float32 and recs.shape == (3, 24)
    assert types.tolist() == [RT_CAM_PINHOLE, RT_CAM_THIN_LENS, RT_CAM_THIN_LENS]
    for v, c in enumerate(cams):
        t, f = marshal_camera(c)
        assert types[v] == t and np.array_equal(recs[v], f)
    assert np.array_equal(recs[2], recs[1])
    assert recs.flags.c_contiguous     # 24 * K floats, view v at 24 v, as rt_render_views reads them


def test_marshal_views_keeps_unknown_types_for_the_library():
    types, _ = marshal_views([(7, np.zeros(24, np.float32))])   # rt_render_views rejects it, naming the view
    assert types.tolist() == [7]


@pytest.mark.parametrize("bad, err", [
    ([], ValueError),
    ("cameras", TypeError),
    (None, TypeError),
    ([(0, np.zeros(23, np.float32))], ValueError),
    ([(0, np.zeros((4, 6), np.float32))], ValueError),
    ([(0, np.zeros(24, np.int32))], TypeError),
    ([(0.5, np.zeros(24, np.float32))], TypeError),
    ([(True, np.zeros(24, np.float32))], TypeError),
    ([np.zeros(24, np.float32)], TypeError),
    ([(0, np.zeros(24, np.float32), 1)], TypeError),
])
def test_marshal_views_rejects_malformed_lists(bad, err):
    with pytest.raises(err):
        marshal_views(bad)


def test_marshal_views_names_the_view():
    with pytest.raises(ValueError, match="view 1"):
        marshal_views([marshal_camera(_cams()[0]), (0, np.zeros(5, np.float32))])


def test_render_views_is_exported():
    assert {"rt_render_views", "rt_render_views_accumulate_device", "rt_resolve_views_device"} <= set(rt.native.ABI_SYMBOLS)
