"""Scene upload from host arrays (rt_set_scene: host marshalling + upload) against device arrays (rt_set_scene_device: the
blob built on the GPU from torch CUDA tensors), alternating in one process, per workload: the wall time of the scene call
with a device synchronise, and the time to image with RT_ACCEL_BVH (scene call, tree build, rt_set_camera + rt_render of the
C5 frame).  Then an animation loop at 100 k spheres (1920x1080, 64 spp, BVH): every frame moves every centre with a torch
op and renders; the device path hands the tensors over, the host path copies them to the host first.  Prints a text table
(profiles/r04_scene_device.txt)."""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
import raytrace_clj_b200 as rt
from scripts.bvh_build_bench import million

BVH = rt.native.RT_ACCEL_BVH
REPS = 7
DEV = "cuda:0"


def gpu_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "nvidia-smi unavailable"


def med(v):
    return float(np.median(v)) * 1e3 if v else float("nan")


def plain(flat):
    """rt_set_scene's values: a bvh-node world (C2) marshals with the tie rule RT_TIE_BVH, an rt_scene_ext field that would
    take the host path through rt_set_scene_ex; both paths here resolve exact ties by RT_TIE_HITLIST."""
    flat = flat.copy()
    flat.tie_rule = rt.native.RT_TIE_HITLIST
    assert not flat.has_ext
    return flat


def measure(label, flat, cam_type, cam, nx, ny, spp, frames=True, reps=REPS):
    flat = plain(flat)
    tensors = flat.sphere_tensors(DEV)
    tables = flat.tables()
    paths = {"host": lambda r: r.set_scene(flat), "device": lambda r: r.set_scene_device(**tensors, **tables)}
    rows = {p: {"scene": [], "image": []} for p in paths}
    img = np.empty((ny, nx, 3), np.uint8)
    with rt.native.Renderer([0]) as r:
        r.set_accel(BVH)
        for rep in range(reps + 1):                       # the first round warms allocations and modules up
            for name, set_scene in paths.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                set_scene(r)
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                if frames:
                    r.set_camera(cam_type, cam)
                    r.render(nx, ny, spp, 50, seed=7, linear=False, rgb8=True, out_rgb8=img)
                else:
                    r.bvh()                                # the tree build, as the first render would do it
                torch.cuda.synchronize()
                t2 = time.perf_counter()
                if rep:
                    rows[name]["scene"].append(t1 - t0)
                    rows[name]["image"].append(t2 - t0)
        n_list = r.bvh()[1]["nodes"] + 1
    what = "scene + tree" if not frames else "to image"
    print(f"\n== {label}: {flat.n_spheres} spheres, {n_list} listed leaves"
          + (f", frame {nx}x{ny} {spp} spp depth 50, BVH" if frames else " (build only)") + f" (medians of {reps}, ms)")
    print(f"{'path':7s} {'scene call':>10s} {what:>12s}")
    for name in paths:
        print(f"{name:7s} {med(rows[name]['scene']):10.2f} {med(rows[name]['image']):12.2f}")
    sys.stdout.flush()


def animation(frames=20):
    nx, ny, spp, _, scene_name, seed = bench.WORKLOADS["c5-100k"]
    flat, cam_type, cam = bench.build_scene(scene_name, nx, ny, seed)
    tables = flat.tables()
    img = np.empty((ny, nx, 3), np.uint8)
    out = {}
    with rt.native.Renderer([0]) as r:
        r.set_accel(BVH)
        r.set_camera(cam_type, cam)
        for rep in range(2):                               # round 0: warm-up
            for name in ("host", "device"):
                t = flat.sphere_tensors(DEV)
                host = flat.copy()
                step = torch.linspace(-1e-3, 1e-3, flat.n_spheres, device=DEV)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for f in range(frames):
                    t["center0_r"][:, 0] += step               # the simulation step
                    if name == "device":
                        r.set_scene_device(**t, **tables)
                    else:
                        host.center0_r = t["center0_r"].cpu().numpy()
                        r.set_scene(host)
                    r.render(nx, ny, spp, 50, seed=f, linear=False, rgb8=True, out_rgb8=img)
                torch.cuda.synchronize()
                if rep:
                    out[name] = (time.perf_counter() - t0) / frames
    print(f"\n== animation: {flat.n_spheres} spheres moved by a torch op every frame, {nx}x{ny} {spp} spp depth 50, BVH, "
          f"{frames} frames (ms per frame)")
    for name, what in (("host", ".cpu() -> set_scene -> render"), ("device", "set_scene_device -> render")):
        print(f"{name:7s} {out[name] * 1e3:8.2f}   {what}")


def main():
    print("GPU:", gpu_line())
    print("host:", os.cpu_count(), "logical CPUs")
    for w in ("c2", "c5-1k", "c5-10k", "c5-100k"):
        nx, ny, spp, _, scene_name, seed = bench.WORKLOADS[w]
        flat, cam_type, cam = bench.build_scene(scene_name, nx, ny, seed)
        measure(w, flat, cam_type, cam, nx, ny, spp)
    flat, cam_type, cam = million()
    measure("1 M leaves", flat, cam_type, cam, 1920, 1080, 64, frames=False, reps=3)
    animation()
    print("\nGPU (after):", gpu_line())


if __name__ == "__main__":
    main()
