"""RT_ACCEL_BVH tree built on the host (bvh_build 0) against the device (bvh_build 2), alternating, per workload:
build time (wall of the call that builds — rt_get_bvh right after rt_set_scene — and the device build's CUDA-event time,
both including the bounding-sphere upload), box / exact tests per ray of each tree, the device frame time through each
tree (the C5 shape: 1920x1080, 64 spp, depth 50), and the time to image split into rt_set_scene (host marshalling),
tree build, and rt_set_camera + rt_render.  Prints a text table (profiles/r03_bvh_build.txt)."""
import ctypes as C
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import bench
import raytrace_clj_b200 as rt

BVH = rt.native.RT_ACCEL_BVH
REPS = 5


def gpu_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "nvidia-smi unavailable"


def million():
    """The sweep's grid of r = 0.2 spheres at 1 M leaves, marshalled with numpy (the Python scene builder is too slow)."""
    base, cam_type, cam = bench.build_scene("sweep:1000", 1920, 1080, 5)
    n, side = 1_000_000, 1000
    g = np.random.default_rng(11)
    a, b = np.meshgrid(np.arange(side) - side // 2, np.arange(side) - side // 2, indexing="ij")
    c0r = np.zeros((n, 4), np.float32)
    c0r[:, 0], c0r[:, 1], c0r[:, 2], c0r[:, 3] = a.ravel() + 0.9 * g.random(n), 0.2, b.ravel() + 0.9 * g.random(n), 0.2
    flat = rt.native.FlatScene(center0_r=c0r, center1=c0r.copy(), t0t1=np.tile(np.float32([0, 1]), (n, 1)),
                               sphere_flags=np.zeros(n, np.uint32), material_id=np.zeros(n, np.int32), mat_type=base.mat_type,
                               mat_param=base.mat_param, mat_tex=base.mat_tex, tex_type=base.tex_type, tex_params=base.tex_params,
                               tex_children=base.tex_children)
    return flat, cam_type, cam


def build_only(r):
    info = np.zeros(4, np.int64)
    t0 = time.perf_counter()
    rc = r.L.rt_get_bvh(r.h, 0, None, 0, info.ctypes.data_as(C.POINTER(C.c_int64)))
    dt = time.perf_counter() - t0
    r._check(rc, "rt_get_bvh")
    return dt, info


def measure(label, flat, cam_type, cam, nx, ny, spp, frames=True, reps=REPS):
    n_list = None
    rows = {0: {"build": [], "ev": [], "scene": [], "image": [], "render": [], "frame": [], "depth": 0}, 2: None}
    rows[2] = {k: ([] if isinstance(v, list) else v) for k, v in rows[0].items()}
    img = np.empty((ny, nx, 3), np.uint8)
    g = np.random.default_rng(1)
    pix = g.integers(0, nx * ny, 200_000).astype(np.int32)
    smp = g.integers(0, spp, 200_000).astype(np.int32)
    per_ray = {}
    with rt.native.Renderer([0]) as r:
        r.set_accel(BVH)
        for rep in range(reps + 1):                 # the first round warms allocations and modules up
            for mode in (0, 2):
                R = rows[mode]
                r.set_option("bvh_build", mode)
                t0 = time.perf_counter()
                r.set_scene(flat)
                t1 = time.perf_counter()
                tb, info = build_only(r)
                t2 = time.perf_counter()
                if frames:
                    r.set_camera(cam_type, cam)
                    r.reset_counters()
                    r.render(nx, ny, spp, 50, seed=7, linear=False, rgb8=True, out_rgb8=img)
                    frame_ns = r.counters()["kernel_ns"]
                t3 = time.perf_counter()
                if rep == 0:
                    continue
                R["scene"].append(t1 - t0); R["build"].append(tb); R["ev"].append(info[3] * 1e-9); R["depth"] = int(info[1])
                R["builder"] = int(info[2])
                if frames:
                    R["render"].append(t3 - t2); R["frame"].append(frame_ns * 1e-9); R["image"].append(t3 - t0)
            n_list = int(info[0]) + 1
        for mode in (0, 2):
            r.set_option("bvh_build", mode)
            r.set_scene(flat)
            r.set_camera(cam_type, cam)
            r.set_accel(BVH)
            r.reset_counters()
            r.trace_paths(nx, ny, pix, smp, 50, seed=3)
            c = r.counters()
            per_ray[mode] = (c["bvh_node_tests"] / c["rays"], c["sphere_tests"] / c["rays"])
    med = lambda v: float(np.median(v)) * 1e3 if v else float("nan")
    print(f"\n== {label}: {flat.n_spheres} primitives, {n_list} listed leaves, frame {nx}x{ny} {spp} spp depth 50 "
          f"(medians of {reps}, ms)")
    print(f"{'tree':7s} {'depth':>5s} {'build wall':>10s} {'build ev':>9s} {'box/ray':>8s} {'exact/ray':>9s} {'frame dev':>9s} "
          f"{'set_scene':>9s} {'cam+render':>10s} {'to image':>9s}")
    for mode, name in ((0, "host"), (2, "device")):
        R = rows[mode]
        print(f"{name:7s} {R['depth']:5d} {med(R['build']):10.2f} {med(R['ev']) if mode else 0.0:9.2f} {per_ray[mode][0]:8.2f} "
              f"{per_ray[mode][1]:9.2f} {med(R['frame']):9.2f} {med(R['scene']):9.2f} {med(R['render']):10.2f} {med(R['image']):9.2f}")
    sys.stdout.flush()


def main():
    print("GPU:", gpu_line())
    print("host:", os.cpu_count(), "logical CPUs")
    for w in ("c5-1k", "c5-10k", "c5-100k", "c2"):
        nx, ny, spp, _, scene_name, seed = bench.WORKLOADS[w]
        flat, cam_type, cam = bench.build_scene(scene_name, nx, ny, seed)
        measure(w, flat, cam_type, cam, nx, ny, spp)
    for n in (2000, 4000):
        flat, cam_type, cam = bench.build_scene(f"sweep:{n}", 1920, 1080, 5)
        measure(f"sweep:{n} (C5 shape)", flat, cam_type, cam, 1920, 1080, 64)
    flat, cam_type, cam = million()
    measure("1 M leaves (build only)", flat, cam_type, cam, 1920, 1080, 64, frames=False, reps=2)


if __name__ == "__main__":
    main()
