"""One rt_render_views call against K back-to-back rt_render calls (rt_set_camera + rt_render per view) for K in
{1, 2, 4, 8, 16, 32}: a turntable of K thin-lens views around the scene.  The two are alternated, warm-up excluded,
medians over the repeats.  Per view: wall time of the call(s) (they return after the images are on the host) and device
time (RT_CTR_KERNEL_NS of every call), plus samples/s.  Workloads: the C1 shape, the C2 shape and 100 k sweep leaves
with RT_ACCEL_BVH at 480x270x16 spp.  Prints a text table (profiles/r05_render_views.txt)."""
import argparse
import math
import os
import random
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import raytrace_clj_b200 as rt
from raytrace_clj_b200 import camera as camm

KS = [1, 2, 4, 8, 16, 32]
WORKLOADS = {   # name: (nx, ny, spp, depth, scene, accel)
    "c1": (200, 100, 100, 50, "random", rt.native.RT_ACCEL_BRUTE_FORCE),
    "c2": (1200, 800, 10, 50, "random", rt.native.RT_ACCEL_BRUTE_FORCE),
    "sweep100k-bvh": (480, 270, 16, 50, "sweep100k", rt.native.RT_ACCEL_BVH),
}


def gpu_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "nvidia-smi unavailable"


def make_scene(name, nx, ny):
    if name == "random":
        return rt.scene.make_random_scene(nx, ny, 11, True, random.Random(1))
    return rt.scene.make_scale_sweep_scene(nx, ny, 100_000, random.Random(5))


def turntable(base, k, nx, ny):
    """k thin-lens views on a circle around the vertical axis through the point the scene's camera looks at."""
    o = np.asarray(base.origin, np.float64)
    w = np.asarray(getattr(base, "w", (0.0, 0.0, 1.0)), np.float64)
    dist = 10.0
    look = o - dist * w
    r = o - look
    out = []
    for v in range(k):
        a = 2.0 * math.pi * v / k
        rr = np.array([math.cos(a) * r[0] + math.sin(a) * r[2], r[1], -math.sin(a) * r[0] + math.cos(a) * r[2]])
        out.append(camm.thin_lens_camera(lookfrom=look + rr, lookat=look, vup=np.array([0.0, 1.0, 0.0]), vfov=20.0,
                                         aspect=nx / ny, aperture=0.1, focus_dist=dist, t0=0.0, t1=1.0))
    return out


def timed(r, fn):
    r.reset_counters()
    t0 = time.perf_counter()
    dev_ns = fn()
    return time.perf_counter() - t0, dev_ns


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--ks", default=",".join(map(str, KS)))
    ap.add_argument("--no-linear", action="store_true", help="return the rgb8 images only (both arms)")
    ap.add_argument("--pinned", action="store_true",
                    help="both arms write into page-locked output buffers from rt_host_alloc, allocated once per K")
    args = ap.parse_args()
    print(f"# command: python {' '.join(sys.argv)}")
    print(f"# GPU: {gpu_line()}")
    print(f"# rt_render_views (one call, K views) vs K x (rt_set_camera + rt_render); medians of {args.reps} alternated repeats after one warm-up each")
    print(f"{'workload':>14} {'K':>3} | {'batch wall/view ms':>18} {'singles wall/view ms':>20} {'wall speedup':>12} | "
          f"{'batch dev/view ms':>17} {'singles dev/view ms':>19} | {'batch Msamples/s':>16} {'singles Msamples/s':>18}")
    for wl in args.workloads.split(","):
        nx, ny, spp, depth, sname, accel = WORKLOADS[wl]
        sc = make_scene(sname, nx, ny)
        flat = rt.native.marshal_world(sc["world"])
        with rt.native.Renderer([0]) as r:
            r.set_accel(accel)
            r.set_scene(flat)
            for k in map(int, args.ks.split(",")):
                cams = turntable(sc["camera"], k, nx, ny)
                marsh = [rt.native.marshal_camera(c) for c in cams]
                lin_b = img_b = None
                if args.pinned:   # page-locked outputs: the device writes the caller's buffers directly
                    img_b = r.host_empty((k, ny, nx, 3), np.uint8)
                    lin_b = None if args.no_linear else r.host_empty((k, ny, nx, 3), np.float32)
                types, recs = rt.native.marshal_views(marsh)

                def batch():
                    if args.pinned:
                        r._check(r.L.rt_render_views(r.h, k, rt.native._p(types, rt.native._i32p), rt.native._p(recs, rt.native._f32p),
                                                     nx, ny, spp, depth, 1, rt.native.RT_VARIANT_WAVEFRONT,
                                                     rt.native._p(lin_b, rt.native._f32p), rt.native._p(img_b, rt.native._u8p)),
                                 "rt_render_views")
                    else:
                        r.render_views(marsh, nx, ny, spp, depth, seed=1, linear=not args.no_linear)
                    return r.counters()["kernel_ns"]

                def singles():
                    ns = 0
                    for v, c in enumerate(marsh):
                        r.set_camera(*c)
                        if args.pinned:
                            r.render(nx, ny, spp, depth, seed=1, linear=not args.no_linear, out_rgb8=img_b[v],
                                     out_linear=None if lin_b is None else lin_b[v])
                        else:
                            r.render(nx, ny, spp, depth, seed=1, linear=not args.no_linear)
                        ns += r.counters()["kernel_ns"]
                    return ns

                batch(); singles()   # warm-up: modules, buffers, the tree
                bw, bd, sw, sd = [], [], [], []
                for _ in range(args.reps):
                    w, d = timed(r, batch); bw.append(w); bd.append(d)
                    w, d = timed(r, singles); sw.append(w); sd.append(d)
                mb, ms = float(np.median(bw)), float(np.median(sw))
                db, ds = float(np.median(bd)) * 1e-9, float(np.median(sd)) * 1e-9
                samples = k * nx * ny * spp
                print(f"{wl:>14} {k:>3} | {mb / k * 1e3:>18.3f} {ms / k * 1e3:>20.3f} {ms / mb:>12.2f} | "
                      f"{db / k * 1e3:>17.3f} {ds / k * 1e3:>19.3f} | {samples / mb / 1e6:>16.1f} {samples / ms / 1e6:>18.1f}",
                      flush=True)


if __name__ == "__main__":
    main()
