"""CPU-side tests: host mirror, marshaller, Philox reference vectors, C-ABI surface."""
import ctypes
import os
import random
import re

import numpy as np
import pytest

import raytrace_clj_b200 as rt
from raytrace_clj_b200.util import vec3

from helpers import philox4x32_10

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_philox_known_answers():
    """Random123 kat_vectors for philox4x32-10."""
    out = philox4x32_10([[0, 0, 0, 0]], [[0, 0]])[0]
    assert [hex(int(x)) for x in out] == ["0x6627e8d5", "0xe169c58d", "0xbc57ac4c", "0x9b00dbd8"]
    out = philox4x32_10([[0xFFFFFFFF] * 4], [[0xFFFFFFFF] * 2])[0]
    assert [hex(int(x)) for x in out] == ["0x408f276d", "0x41c83b0e", "0xa20bc7c6", "0x6d5451fd"]
    out = philox4x32_10([[0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344]], [[0xA4093822, 0x299F31D0]])[0]
    assert [hex(int(x)) for x in out] == ["0xd16cfe09", "0x94fdcceb", "0x5001e420", "0x24126ea1"]


def test_random_scene_statistics_scene_318_412():
    ns = []
    for seed in range(30):
        sc = rt.scene.make_random_scene(200, 100, 11, True, random.Random(seed))
        ns.append(rt.native.marshal_world(sc["world"]).n_spheres)
    assert 485 <= min(ns) and max(ns) <= 489 and 485.8 < np.mean(ns) < 487.0   # SURVEY §8: 485-489, mean 486.3
    flat = rt.native.marshal_world(rt.scene.make_random_scene(200, 100, 11, True, random.Random(1))["world"])
    n_small = flat.n_spheres - 5
    movers = int((flat.sphere_flags & 2).astype(bool).sum())
    assert 0.72 < movers / n_small < 0.88                                        # 80 % diffuse movers
    types = flat.mat_type[flat.material_id]
    assert (types == 3).sum() == 1 and (flat.sphere_flags & 1).sum() == 1        # one sky dome, a UVSphere light
    assert 0.08 < (types == 1).sum() / n_small < 0.22 and 0.01 < (types == 2).sum() / n_small < 0.10
    small = flat.center0_r[flat.center0_r[:, 3] == np.float32(0.2)]
    assert len(small) == n_small and np.all(small[:, 1] == np.float32(0.2))
    assert np.all(np.linalg.norm(small[:, :3] - np.array([4, 0.2, 0]), axis=1) > 0.9)
    mv = (flat.sphere_flags & 2).astype(bool)
    dy = flat.center1[mv, 1] - flat.center0_r[mv, 1]
    assert np.all(dy >= 0) and np.all(dy < 0.5) and np.all(flat.center1[mv, 0] == flat.center0_r[mv, 0])
    static = rt.native.marshal_world(rt.scene.make_random_scene(200, 100, 11, False, random.Random(1))["world"])
    assert not (static.sphere_flags & 2).any()


def test_flatten_bvh_dedup_and_order():
    m = rt.shader.lambertian(albedo=rt.texture.constant(color=vec3(.5, .5, .5)))
    spheres = [rt.hitable.sphere(center=vec3(i, 0, 0), radius=0.4, material=m) for i in range(7)]
    world = rt.hitable.make_bvh(spheres, 0.0, 1.0, random.Random(3))
    leaves = rt.native.flatten_world(world)
    assert len(leaves) == 7 and {id(x) for x in leaves} == {id(x) for x in spheres}
    # a 1-element bvh node holds the same object as both children (hitable.clj:113-114)
    one = rt.hitable.make_bvh(spheres[:1], 0.0, 1.0, random.Random(0))
    assert one.left is one.right and len(rt.native.flatten_world(one)) == 1
    flat = rt.native.marshal_world(world)
    assert flat.n_spheres == 7 and len(flat.mat_type) == 1 and len(flat.tex_type) == 1   # shared records de-duplicated


def test_marshaller_rejects_out_of_scope_records():
    class RectXY:   # hitable.clj:269 — outside the accelerated path
        pass

    with pytest.raises(rt.native.UnsupportedSceneError):
        rt.native.marshal_world(rt.hitable.hitlist(items=[RectXY()]))

    class Marble:   # texture.clj:88
        pass

    s = rt.hitable.sphere(center=vec3(0, 0, 0), radius=1, material=rt.shader.lambertian(albedo=Marble()))
    with pytest.raises(rt.native.UnsupportedSceneError):
        rt.native.marshal_world(rt.hitable.hitlist(items=[s]))
    with pytest.raises(rt.native.UnsupportedSceneError):
        rt.native.marshal_world(rt.hitable.hitlist(items=[]))


def test_checker_children_precede_parent():
    flat = rt.native.marshal_world(rt.scene.make_two_spheres(200, 100)["world"])
    for t in np.nonzero(flat.tex_type == 2)[0]:
        assert np.all(flat.tex_children[t] >= 0) and np.all(flat.tex_children[t] < t)


def test_ppm_roundtrip(tmp_path):
    img = (np.arange(5 * 7 * 3) % 256).astype(np.uint8).reshape(5, 7, 3)
    p = tmp_path / "x.ppm"
    rt.ppm.save(str(p), img)
    assert p.read_bytes().startswith(b"P6\n7 5\n255\n")
    assert np.array_equal(rt.ppm.read_ppm(str(p)), img)


def test_abi_library_exports_every_declared_symbol():
    """The C-ABI library loads without a GPU and exports exactly what include/raytrace_b200.h declares."""
    from raytrace_clj_b200 import build

    path = build.build_library()
    lib = ctypes.CDLL(path)
    header = open(os.path.join(ROOT, "include", "raytrace_b200.h")).read()
    declared = set(re.findall(r"^(?:int|void|const char\*)\s+(rt_\w+)\s*\(", header, flags=re.M))
    assert declared == set(rt.native.ABI_SYMBOLS), declared ^ set(rt.native.ABI_SYMBOLS)
    for sym in declared:
        assert getattr(lib, sym) is not None
    lib.rt_abi_version.restype = ctypes.c_int
    assert lib.rt_abi_version() == 2


_NO_DEVICE_CHECK = """
import pytest
import raytrace_clj_b200 as rt
with pytest.raises(rt.native.NativeError) as e:
    rt.native.Renderer([0])
assert "-5" in str(e.value) or "no usable CUDA device" in str(e.value)
with pytest.raises(rt.native.NativeError):
    sc = rt.scene.make_two_spheres(8, 8)
    rt.core.render(sc["camera"], sc["world"], 8, 8, 1)
"""


def test_no_cpu_fallback_without_gpu():
    """Without a CUDA device the product path fails loudly (RT_ERR_NODEVICE), it never renders on the CPU.  The check runs
    in a child process that sees no device (CUDA_VISIBLE_DEVICES empty), so a machine with GPUs runs it too."""
    import subprocess
    import sys

    res = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHECK], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]


def test_product_never_imports_oracle():
    """oracle/ is test infrastructure: nothing under the product package may reference it."""
    pkg = os.path.join(ROOT, "raytrace_clj_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                src = open(os.path.join(dirpath, f), errors="ignore").read()
                assert not re.search(r"^\s*(import|from)\s+oracle", src, flags=re.M), f
                assert "liboracle" not in src, f


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU restatement on the host cores) prints ONE JSON line with the keys the
    driver reads, and needs no GPU."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "c1",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "samples_per_sec" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("c1")


def test_no_kernel_spills_registers():
    """ptxas -v of the in-tree build: no kernel spills (spills are pure overhead in issue-bound kernels).  The one
    exception is deliberate: the register-capped megakernel (launch bound 2 CTAs / SM), kept only as the A/B build
    of the reproducibility check (option "mega_regcap")."""
    import subprocess

    from raytrace_clj_b200 import build as rtbuild

    rtbuild.build_library()
    log = open(os.path.join(os.path.dirname(rtbuild.OUT), "csrc", "build.log")).read()
    kernels = {}
    cur = None
    for line in log.splitlines():
        m = re.search(r"Compiling entry function '([^']+)'", line)
        if m:
            cur = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            kernels[cur] = (int(m.group(1)), int(m.group(2)))
            cur = None
    assert len(kernels) >= 20                      # every kernel reported
    spilling = {k: v for k, v in kernels.items() if v != (0, 0)}
    assert all("mega_kernel<4, 256, 2, false>" in k for k in spilling), spilling


def test_documented_options_are_the_implemented_ones():
    """Every knob rt_set_option accepts (rt_api.cu) is named in the header's comment, and nothing else is."""
    import re

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    api = open(os.path.join(root, "raytrace_clj_b200", "csrc", "rt_api.cu")).read()
    body = api[api.index("int rt_set_option("):]
    body = body[:body.index("\n}\n")]
    implemented = set(re.findall(r'k == "([a-z_0-9]+)"', body))
    header = open(os.path.join(root, "include", "raytrace_b200.h")).read()
    doc = header[header.index("Per-context tuning knob"):header.index("int rt_set_option(")]
    documented = set(re.findall(r'"([a-z_0-9]+)"', doc))
    assert implemented and implemented == documented, implemented ^ documented
