#!/usr/bin/env python
"""bench.py — samples/sec of the path-tracing hot path on BASELINE.json's quoted configuration.

A "step" is one full pass of the hot path over the workload: every pixel of the 1200x800 random-
spheres scene (make-random-scene n=11 moving=true, scene seed 1, ~486 spheres), 10 samples per
pixel, depth 50 (BASELINE.json configs[1]).  `value` = samples/s with the scene resident in HBM
(kernels + reduce + resolve timed with CUDA events on the launching stream); `e2e` = the same
metric through the C-ABI calls a front end makes (rt_set_scene + rt_set_camera + rt_render with
HOST buffers: the scene arrays are ordinary numpy memory, the 8-bit frame lands in a page-locked
buffer from rt_host_alloc), host<->device copies inside the timed region.

N > 1 (torchrun, one rank per GPU): every rank renders its own 10-spp sample slice of the same
frame (weak scaling: global spp = 10 N), the float sums are combined with one NCCL reduce over
NVLink and rank 0 resolves; time = max over ranks.  `e2e` at N > 1 is what the drop-in's caller —
ONE process, core.clj:99-108 — would get: rank 0 alone drives an N-device context
(rt_create(ids, N) + rt_render with host buffers; sample slices on every device, cross-device
reduce inside the library) while the other ranks idle.  The `strong_c3` block adds BASELINE
config 3 (3840x2160, 1024 spp) through that same in-library path: total work fixed, split over
the N devices by sample slices and by interleaved rows, reduce time reported separately.

`--impl reference` times the CPU restatement of the reference (oracle/, double precision C++ with
OpenMP on all host threads) — the Clojure original cannot run here (no JVM in the image).
"""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

FLOP_PER_TEST = 17.0            # SURVEY §8(d): oc (3) + oc.d (5) + oc.oc - r^2 (6) + b'^2 - a c' (3)
TF32_PEAK_MEASURED_TFLOPS = 2043.3 * 2 * 148 * 1.965e9 / 1e12   # csrc/tcprobe.cu, profiles/r02_tcprobe.txt
FLOP_COMMON_ORIGIN_TEST = 10.0  # what the common-origin form EXECUTES per test (5 FFMA): the rest is hoisted per sphere
NOMINAL_FP32_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12   # 74.45: SMs x lanes x 2 flop x max SM clock

WORKLOADS = {
    # name: (nx, ny, spp, depth, scene builder name, scene seed)
    "c2": (1200, 800, 10, 50, "random", 1),
    "c1": (200, 100, 100, 50, "random", 1),
    "c3": (3840, 2160, 1024, 50, "random", 1),          # use with --scaling strong at N GPUs (sample slices)
    "c3-slice": (3840, 2160, 16, 50, "random", 1),
    "c4": (1200, 800, 64, 50, "stress", 4),
    # config 5: brute-force scale sweep, 1920x1080, 64 spp
    "c5-100": (1920, 1080, 64, 50, "sweep:100", 5),
    "c5-1k": (1920, 1080, 64, 50, "sweep:1000", 5),
    "c5-10k": (1920, 1080, 64, 50, "sweep:10000", 5),
    "c5-100k": (1920, 1080, 64, 50, "sweep:100000", 5),
    # beyond spheres (SURVEY §8 f-2 / f-4), for the record
    "cornell": (600, 600, 64, 50, "cornell", 2),
    "final": (600, 600, 64, 50, "final", 2),
}
SCENE_DESC = {"random": "make-random-scene n=11 moving=true", "stress": "make-random-scene n=11, 10/45/45 % Lambert/metal/glass",
              "cornell": "make-cornell-box classic", "final": "make-final (book 2), synthetic earth map"}


def build_scene(name, nx, ny, seed):
    import raytrace_clj_b200 as rt

    rng = random.Random(seed)
    if name == "random":
        sc = rt.scene.make_random_scene(nx, ny, 11, True, rng)
    elif name == "stress":
        sc = rt.scene.make_material_stress_scene(nx, ny, 11, rng)
    elif name.startswith("sweep:"):
        sc = rt.scene.make_scale_sweep_scene(nx, ny, int(name.split(":")[1]), rng)
    elif name == "cornell":
        sc = rt.scene.make_cornell_box(nx, ny, True, rng)
    elif name == "final":
        sc = rt.scene.make_final(nx, ny, rng)
    else:
        raise ValueError(name)
    flat = rt.native.marshal_world(sc["world"])
    cam_type, cam = rt.native.marshal_camera(sc["camera"])
    return flat, cam_type, cam


def workload_string(name, flat):
    """ONE description of the workload, used verbatim by both arms (the driver compares them)."""
    nx, ny, spp, depth, scene_name, scene_seed = WORKLOADS[name]
    desc = SCENE_DESC.get(scene_name, "5 hero objects + static r=0.2 spheres on a grid, scene.clj:369-375 placement rule")
    return (f"{name}: {nx}x{ny}, {spp} spp, depth {depth}, {flat.n_spheres} primitives ({desc}, scene seed {scene_seed}), "
            f"brute force over every primitive")


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(out_dir, images):
    """Writes each [ny, nx, c] image as out_dir/<name>.npy, keeping its dtype (float32 or float64).  When all of them
    together pass 64 MB, every image keeps the same fixed, seeded sample of pixels instead: [k, c] in increasing pixel
    order (row-major over [ny, nx]), and pixel_index.npy (float64) holds those k flat pixel indices.  The device adds
    float samples in a varying order, so two runs agree to the last bits of the sums (and 1 of 255 in rgb8), not exactly."""
    os.makedirs(out_dir, exist_ok=True)
    ny, nx = next(iter(images.values())).shape[:2]
    n_pix = ny * nx
    bytes_per_pix = sum(a.shape[2] * a.itemsize for a in images.values())
    if n_pix * bytes_per_pix > DUMP_LIMIT_BYTES:
        k = (DUMP_LIMIT_BYTES - 4096) // (bytes_per_pix + 8)       # 4 KiB left for the .npy headers
        idx = np.sort(np.random.default_rng(0).choice(n_pix, k, replace=False))
        images = {name: a.reshape(n_pix, a.shape[2])[idx] for name, a in images.items()}
        np.save(os.path.join(out_dir, "pixel_index.npy"), idx.astype(np.float64))
    for name, a in images.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); power.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "power_w_max": float(max(power)), "samples": len(sm)}


def run_reference(args, world, rank):
    """The reference's own CPU implementation of the path — here its C++ restatement (oracle/), all host
    threads; each step = one full pass over the workload when that stays bounded (C2: ~3 s per step on 16
    threads), else a bounded sample of its spp, stated in `cpu_baseline.sample`."""
    if rank != 0:
        return 0
    import oracle

    nx, ny, spp, depth, scene_name, scene_seed = WORKLOADS[args.workload]
    flat, cam_type, cam = build_scene(scene_name, nx, ny, scene_seed)
    S = oracle.Scene(flat)
    cores = host_cores()            # torchrun exports OMP_NUM_THREADS=1: ask for every core explicitly
    # bounded: at most ~6 s of CPU work per step at ~0.25 G tests/s per core
    budget = 6.0 * 0.25e9 * cores / (nx * ny * 2.6 * flat.n_spheres)
    step_spp = int(max(1, min(spp, budget)))
    for w in range(args.warmup):
        S.render_accumulate(cam_type, cam, nx, ny, 0, 1, depth, seed=w, n_threads=cores)
    t0 = time.perf_counter()
    samples = tests = 0
    for k in range(args.steps):
        sum_rgb, c = S.render_accumulate(cam_type, cam, nx, ny, (k * step_spp) % max(1, spp), step_spp, depth, seed=1 + k, n_threads=cores)
        samples += c["samples"]
        tests += c["sphere_tests"]
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        # the last step's float sums over its samples (row 0 = bottom) and the 8-bit frame they resolve to (row 0 = top)
        dump_outputs(args.dump_outputs, {"linear_sum": sum_rgb, "rgb8": oracle.resolve(sum_rgb, step_spp).astype(np.float64)})
    v = samples / dt
    sample = f"{nx}x{ny}, {step_spp} of {spp} spp per step, depth {depth}, brute force over {flat.n_spheres} primitives, double precision"
    line = {
        "impl": "reference", "metric": "samples_per_sec", "value": v, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_string(args.workload, flat)},
        "tests_per_sec": tests / dt,
        "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample,
                         "note": "C++ double-precision restatement of raytrace-clj (oracle/); the Clojure original "
                                 "cannot run here (no JVM)"},
        "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


CULL_TC = 1   # set by main() from --cull


def in_library_run(rt, device_ids, flat, cam_type, cam, nx, ny, spp, depth, variant, steps, warmup, reduce_mode, rows, seed0=600, accel=0):
    """ONE process driving len(device_ids) GPUs through the C ABI with host buffers — what the JVM caller would do
    (core.clj:99-108): rt_set_scene + rt_set_camera + rt_render per step, wall clock.  Returns a record."""
    with rt.native.Renderer(device_ids) as r:
        out_img = r.host_empty((ny, nx, 3), np.uint8)   # page-locked result buffer (rt_host_alloc): the D2H read lands in it directly
        r.set_option("reduce", reduce_mode)
        r.set_option("rows", rows)
        r.set_option("cull_tc", CULL_TC)
        if accel:
            r.set_accel(accel)        # per context; every rt_set_scene below rebuilds the tree (inside the timed region)

        def one(seed, n_spp):
            r.set_scene(flat)
            r.set_camera(cam_type, cam)
            r.render(nx, ny, n_spp, depth, seed=seed, variant=variant, linear=False, rgb8=True, out_rgb8=out_img)

        for w in range(warmup):
            one(500 + w, spp)
        if warmup == 0:
            # allocations and module load only — but with enough samples per device (4) that the wavefront queues
            # get their full size here, not inside the timed frame
            one(499, min(spp, 4 * max(1, len(device_ids))))
        r.reset_counters()
        t0 = time.perf_counter()
        for k in range(steps):
            one(seed0 + k, spp)
        dt = time.perf_counter() - t0
        c = r.counters()
    return {"value": nx * ny * spp * steps / dt, "unit": "samples/s", "ms_per_step": dt / steps * 1e3, "steps": steps,
            "devices": len(device_ids), "partition": "interleaved rows" if rows else "sample slices",
            "reduce": "ncclReduce (single process, ncclCommInitAll)" if reduce_mode else "NVLink peer loads fused into the resolve kernel",
            "reduce_ms_per_step": c["reduce_ns"] * 1e-6 / steps, "device_ms_last_step": c["kernel_ns"] * 1e-6,
            "tests_per_sec": c["sphere_tests"] / dt, "samples_check": c["samples"] == nx * ny * spp * steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--variant", type=int, default=int(os.environ.get("RT_VARIANT", "1")), help="1 wavefront (default), 0 megakernel")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every GPU renders the workload's spp (global spp = spp x N); strong: the spp are divided")
    ap.add_argument("--accel", default="brute", choices=["brute", "bvh"], help="closest-hit search: brute force (the roofline path) or the GPU BVH")
    ap.add_argument("--cull", default="tc", choices=["tc", "fp32"],
                    help="brute-force cull: tc = tcgen05 tensor cores where the list fits (the library's default), fp32 = FP32 pipe only")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong-c3", action="store_true", help="skip the BASELINE config 3 strong-scaling block")
    ap.add_argument("--e2e-steps", type=int, default=0, help="default: min(steps, 10)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy: linear_sum (the float "
                         "sums over its samples) and rgb8 (the resolved frame, as floats); inputs depend only on the arguments. "
                         "bench_outputs/ in the repository is git-ignored for this")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        return run_reference(args, world, rank)

    import torch
    import torch.distributed as dist

    import raytrace_clj_b200 as rt
    from raytrace_clj_b200 import build as rtbuild

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the render path has no CPU fallback")
    rtbuild.build_library()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    cpu_group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        cpu_group = dist.new_group(backend="gloo")   # host-side barriers that keep the GPUs free (the in-library legs)

    nx, ny, spp, depth, scene_name, scene_seed = WORKLOADS[args.workload]
    if args.scaling == "strong":
        if spp % world:
            raise SystemExit(f"--scaling strong: {spp} spp do not divide over {world} GPUs")
        spp //= world                                # per-GPU sample slice
    flat, cam_type, cam = build_scene(scene_name, nx, ny, scene_seed)
    r = rt.native.Renderer([local_rank])
    r.set_scene(flat)
    r.set_camera(cam_type, cam)
    accel_id = rt.native.RT_ACCEL_BVH if args.accel == "bvh" else 0
    if accel_id:
        r.set_accel(accel_id)
    global CULL_TC
    cull_tc = CULL_TC = 1 if args.cull == "tc" else 0
    r.set_option("cull_tc", cull_tc)
    # the tensor-core cull keeps 1024 leaves' features in shared memory per launch; longer lists take several launches per iteration
    # (and lists below 160 leaves, where a 256-column feature tile would be mostly padding; up to 8 "direct" spheres are not listed)
    tc_active = bool(cull_tc) and accel_id == 0 and args.variant == 1 and 160 + 8 <= flat.n_spheres and not flat.generic
    info = r.device_info()

    d_sum = torch.zeros(ny, nx, 3, device=dev, dtype=torch.float32)
    d_rgb = torch.zeros(ny, nx, 3, device=dev, dtype=torch.uint8)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev, dtype=torch.float32)   # > 126 MB L2
    stream = torch.cuda.current_stream(dev)
    total_spp = spp * world

    def step(seed):
        d_sum.zero_()
        r.render_accumulate_device(nx, ny, rank * spp, spp, d_sum.data_ptr(), max_depth=depth, seed=seed,
                                   variant=args.variant, stream=stream.cuda_stream, sync=False)
        if world > 1:
            dist.reduce(d_sum, dst=0, op=dist.ReduceOp.SUM)
        if rank == 0:
            r.resolve_device(nx, ny, total_spp, d_sum.data_ptr(), d_rgb.data_ptr(), stream=stream.cuda_stream, sync=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    fp32_peak = r.measure_fp32_peak() if rank == 0 else (0.0, 0.0)

    for w in range(args.warmup):
        step(1000 + w)
    barrier()
    r.reset_counters()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for k in range(args.steps):
        flush.fill_(float(k))                       # L2 flush between timed iterations (untimed)
        ev[k][0].record(stream)
        d_sum.zero_()
        kev[k][0].record(stream)
        r.render_accumulate_device(nx, ny, rank * spp, spp, d_sum.data_ptr(), max_depth=depth, seed=1 + k,
                                   variant=args.variant, stream=stream.cuda_stream, sync=False)
        kev[k][1].record(stream)
        if world > 1:
            dist.reduce(d_sum, dst=0, op=dist.ReduceOp.SUM)
        if rank == 0:
            r.resolve_device(nx, ny, total_spp, d_sum.data_ptr(), d_rgb.data_ptr(), stream=stream.cuda_stream, sync=False)
        ev[k][1].record(stream)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the last timed step's float sums over all its samples (row 0 = bottom) and the 8-bit frame (row 0 = top)
        dump_outputs(args.dump_outputs, {"linear_sum": d_sum.cpu().numpy(), "rgb8": d_rgb.cpu().numpy().astype(np.float32)})
    my_ms = sum(a.elapsed_time(b) for a, b in ev)
    my_kernel_ms = sum(a.elapsed_time(b) for a, b in kev)
    ctr = r.counters()
    launches = ctr["kernel_launches"]
    t = torch.tensor([my_ms, my_kernel_ms], device=dev, dtype=torch.float64)
    cnt = torch.tensor([ctr["samples"], ctr["rays"], ctr["sphere_tests"], ctr["candidates"], ctr["direct_tests"]], device=dev,
                       dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    total_ms, kernel_ms = float(t[0]), float(t[1])
    samples, rays, tests, cands, direct = (float(x) for x in cnt)
    value = samples / (total_ms * 1e-3)

    # ---- end to end through the C ABI with host buffers ------------------------------------
    e2e_steps = args.e2e_steps or min(args.steps, 10)
    e2e_rec = None
    strong = None
    if world == 1:
        e2e_rec = in_library_run(rt, [local_rank], flat, cam_type, cam, nx, ny, spp, depth, args.variant, e2e_steps, 1, 0, 0, accel=accel_id)
    else:
        # the drop-in's caller is ONE process: rank 0 drives all N devices through rt_create(ids, N) + rt_render with
        # host buffers while the other ranks sit on a HOST barrier (their GPUs stay free); both reduce flavours
        r.close()
        r = None
        del d_sum, d_rgb, flush
        torch.cuda.empty_cache()
        dist.barrier(group=cpu_group)
        if rank == 0:
            ids = list(range(world))
            e2e_rec = in_library_run(rt, ids, flat, cam_type, cam, nx, ny, spp * world, depth, args.variant, e2e_steps, 2, 0, 0, accel=accel_id)
            e2e_rec["nccl"] = in_library_run(rt, ids, flat, cam_type, cam, nx, ny, spp * world, depth, args.variant, e2e_steps, 2, 1, 0, accel=accel_id)
        dist.barrier(group=cpu_group)

    # ---- BASELINE config 3, strong scaling: 3840x2160, 1024 spp split over the N devices of ONE context -----------
    if not args.no_strong_c3 and args.workload == "c2":
        if world > 1:
            dist.barrier(group=cpu_group)
        if rank == 0:
            cnx, cny, cspp, cdepth, cscene, cseed = WORKLOADS["c3"]
            cflat, ccam_type, ccam = build_scene(cscene, cnx, cny, cseed)
            ids = list(range(world))
            strong = {"workload": workload_string("c3", cflat), "n_gpus": world, "scaling": "strong",
                      "path": "in-library: one process, rt_create(ids, N) + rt_set_scene + rt_set_camera + rt_render with host buffers, "
                              "1 frame per leg, wall clock"}
            legs = [("sample_slices", 0, 0)] + ([("sample_slices_nccl", 1, 0), ("interleaved_rows", 0, 1)] if world > 1 else [])
            for name, red, rows in legs:
                strong[name] = in_library_run(rt, ids, cflat, ccam_type, ccam, cnx, cny, cspp, cdepth, args.variant, 1, 0, red, rows)
        if world > 1:
            dist.barrier(group=cpu_group)

    # ---- stage shares: one extra (untimed) step with per-stage CUDA events (rank 0, wavefront only) ------
    stage = None
    if rank == 0 and args.variant == 1 and args.accel == "brute":
        with rt.native.Renderer([local_rank]) as rp:
            rp.set_option("cull_tc", cull_tc)
            rp.set_scene(flat)
            rp.set_camera(cam_type, cam)
            ps = torch.zeros(ny, nx, 3, device=dev, dtype=torch.float32)
            rp.render_accumulate_device(nx, ny, 0, spp, ps.data_ptr(), max_depth=depth, seed=1, variant=args.variant, sync=True)   # warm
            rp.reset_counters()
            rp.set_profile(True)
            ps.zero_()
            rp.render_accumulate_device(nx, ny, 0, spp, ps.data_ptr(), max_depth=depth, seed=1, variant=args.variant, sync=True)
            pc = rp.counters()
        stage = {k: pc[k + "_ns"] * 1e-6 for k in ("cull", "refine", "tiebreak", "shade")}
        stage["tests"] = pc["sphere_tests"]

    if rank == 0:
        step_s = total_ms / args.steps * 1e-3
        tests_gpu = tests / world / args.steps                  # per GPU per step
        achieved_tflops = FLOP_PER_TEST * tests_gpu / step_s / 1e12            # per GPU, whole render step incl. reduce + resolve
        # what the cull EXECUTES: the camera rays (one per sample when they share an origin) run the 10-flop common-origin form
        n_prims = flat.n_spheres
        cam_tests = (samples / world / args.steps) * n_prims if ((cam[21] == 0.0 or cam_type == 0) and not tc_active) else 0.0
        executed_tflops = (FLOP_COMMON_ORIGIN_TEST * cam_tests + FLOP_PER_TEST * (tests_gpu - cam_tests)) / step_s / 1e12
        peak_measured = max(fp32_peak)
        line = {
            "metric": "samples_per_sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": workload_string(args.workload, flat),
                "variant": "megakernel" if args.variant == 0 else "wavefront",
                "accel": "GPU BVH (RT_ACCEL_BVH): tests_per_sec counts the exact leaf tests actually made" if args.accel == "bvh" else "brute force",
                "parallelism": (f"sample slices x{world}: every GPU renders {spp} spp of the frame, one NCCL reduce"
                                if world > 1 else "single GPU"),
                "l2": "flushed between timed iterations (256 MiB fill); the scene itself is staged in shared memory",
                "cull": ("tcgen05 tensor cores: the line-sphere discriminant of every (ray, primitive) pair as a 3xTF32 GEMM (32 K-slots) into TMEM, "
                         "sign-bit epilogue, FP32 confirm of the ~0.5 % candidates" if tc_active else "FP32 pipe (17-flop conservative test, 10.4 instructions per pair)"),
                "precision": "conservative cull over all primitives (never loses an exact hit), FP64 refine of survivors, FP32 shading",
            },
            "tests_per_sec": tests / (total_ms * 1e-3),
            "rays_per_sample": rays / samples,
            "cull_survivors_per_ray": cands / rays,
            "direct_tests_per_ray": direct / rays,
            "kernel_ms_per_step": kernel_ms / args.steps,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {
                "bound": "fp32", "achieved": achieved_tflops, "peak": peak_measured, "unit": "TFLOP/s",
                "frac": achieved_tflops / peak_measured if peak_measured else None,
                "frac_executed_flop": executed_tflops / peak_measured if peak_measured else None,
                "peak_source": "measured on this box: FFMA-chain microbenchmark (rt_measure_fp32_peak), max of scalar "
                               "FFMA and packed FFMA2",
                "peak_ffma_tflops": fp32_peak[0], "peak_ffma2_tflops": fp32_peak[1],
                "peak_nominal": NOMINAL_FP32_TFLOPS, "frac_of_nominal": achieved_tflops / NOMINAL_FP32_TFLOPS,
                "flop_per_test": FLOP_PER_TEST,
                "tensor": None if not tc_active else {
                    "executed_tf32_flop_per_test": 64, "achieved": 64.0 * tests_gpu / step_s / 1e12, "peak": TF32_PEAK_MEASURED_TFLOPS,
                    "unit": "TFLOP/s", "frac": 64.0 * tests_gpu / step_s / 1e12 / TF32_PEAK_MEASURED_TFLOPS,
                    "note": "what the tensor pipe executes for the cull: 32 TF32 multiply-adds per pair (hi/lo split of 11 feature products), "
                            "whole step; peak = tcgen05 kind::tf32 M128 N256 K8 issue rate measured by csrc/tcprobe.cu on this pool's B200 "
                            "(2043 MAC/clk/SM x 148 SMs x 1.965 GHz; profiles/r02_tcprobe.txt). The kernel's own bound is the epilogue: one "
                            "ALU-pipe funnel shift (half rate) and 4 bytes of TMEM read per pair, 64 pairs/clk/SM at best",
                },
                "traffic": None,
                "traffic_note": "not measured inside this run; the committed `ncu --set full` captures under profiles/ hold the "
                                "dram__bytes of a wf_cull launch (ray record in, pairs out: the kernel is FP32-issue bound, not HBM bound)",
                "note": "denominator = the non-tensor FP32 pipe (what the 17-flop test costs without tensor cores); with the tensor-core cull "
                        "the dot products leave that pipe, so `frac` can pass what the FP32 pipe alone could reach (see `tensor`). "
                        "HBM is not the bound (scene in shared memory). `achieved` = 17 algorithmic flop x "
                        "(rays x primitives) / ms_per_step (the whole step: cull + refine + tie-break + shade + reduce + resolve); "
                        "`frac_executed_flop` counts the camera rays' tests at the 10 flop their common-origin form executes",
                "dominant_kernel": None if not stage else {
                    "name": "wf_cull_tc" if tc_active else "wf_cull", "ms_per_step": stage["cull"],
                    "achieved": FLOP_PER_TEST * stage["tests"] / (stage["cull"] * 1e-3) / 1e12,
                    "frac": FLOP_PER_TEST * stage["tests"] / (stage["cull"] * 1e-3) / 1e12 / peak_measured,
                    "share_of_step": stage["cull"] / max(1e-9, sum(stage[k] for k in ("cull", "refine", "tiebreak", "shade"))),
                    "other_stages_ms": {k: stage[k] for k in ("refine", "tiebreak", "shade")},
                    "note": "one lane, stages serialised with CUDA events (rt_set_profile): shares, not the overlapped step",
                },
            },
            "e2e": {"value": e2e_rec["value"], "unit": "samples/s", "h2d_bytes_per_step": flat.nbytes() + 24 * 4,
                    "d2h_bytes_per_step": nx * ny * 3, "steps": e2e_steps, "ms_per_step": e2e_rec["ms_per_step"],
                    "path": ("rt_set_scene + rt_set_camera + rt_render, host buffers (8-bit frame into a page-locked rt_host_alloc buffer)" if world == 1 else
                             f"ONE process, rt_create over {world} devices + rt_set_scene + rt_set_camera + rt_render, host buffers; "
                             f"{e2e_rec['partition']}, {e2e_rec['reduce']}"),
                    "reduce_ms_per_step": e2e_rec["reduce_ms_per_step"],
                    **({"nccl_reduce": e2e_rec["nccl"]} if "nccl" in e2e_rec else {})},
            "device": info,
        }
        if strong:
            line["strong_c3"] = strong
        if world == 1 and not args.no_cpu_baseline:
            import oracle

            S = oracle.Scene(flat)
            cores = host_cores()
            # bounded sample: about 15 s of CPU work at ~0.25 G tests/s per core (2.6 rays per sample)
            budget = 15.0 * 0.25e9 * cores / (nx * ny * 2.6 * flat.n_spheres)
            cpu_spp = int(max(1, min(spp, budget)))
            S.render_accumulate(cam_type, cam, nx, ny, 0, 1, depth, seed=9, n_threads=cores)          # warm-up
            t0 = time.perf_counter()
            _, c = S.render_accumulate(cam_type, cam, nx, ny, 0, cpu_spp, depth, seed=1, n_threads=cores)
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {
                "value": c["samples"] / dt, "unit": "samples/s", "cores": cores, "kind": "port",
                "tests_per_sec": c["sphere_tests"] / dt, "seconds": dt,
                "sample": f"{nx}x{ny}, {cpu_spp} of {spp} spp, depth {depth}, brute force, double precision",
                "note": "C++ restatement of raytrace-clj (oracle/), OpenMP; the Clojure original cannot run here (no JVM)",
            }
            # the reference itself does NOT brute-force: every scene is wrapped in make-bvh (hitable.clj:108-123).  The same
            # restatement traversing its own reference-style BVH states the reference's real algorithmic complexity.
            S.build_bvh(0.0, 1.0, seed=1)
            t0 = time.perf_counter()
            _, cb = S.render_accumulate(cam_type, cam, nx, ny, 0, cpu_spp, depth, seed=1, n_threads=cores, use_bvh=True)
            dtb = time.perf_counter() - t0
            line["cpu_baseline"]["bvh"] = {"value": cb["samples"] / dtb, "unit": "samples/s", "seconds": dtb,
                                           "leaf_tests_per_ray": cb["sphere_tests"] / cb["rays"], "aabb_tests_per_ray": cb["aabb_tests"] / cb["rays"],
                                           "note": "same restatement through bvh-node.hit? / AABB.hit? (hitable.clj:36-48, 97-106)"}
        print(json.dumps(line))
    if r is not None:
        r.close()
    if world > 1:
        dist.barrier(group=cpu_group)
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
