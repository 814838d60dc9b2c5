#!/usr/bin/env python
"""bench.py — Mrays/s of the B200-native voxel raytracer on BASELINE.json's workload.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload c2|c0|c1|c3|c4] [--dump-outputs DIR]

Default workload (the one BASELINE.json's metric is quoted on): a "step" is one full frame (1920x1080 primary
rays) of the 256^3 mixed-transparent Space (BASELINE.json configs[2], SURVEY.md §8(d) C2) traced through the C ABI
of libaicb200.so.  N > 1: one process per GPU (torchrun), the frame is sharded by interleaved 16-row strips (strong
scaling, total work fixed) and delivered to rank 0 (P2P stores over NVLink, or an NCCL gather).
The other BASELINE configs are bench lines too: c0 (32^3, 256x256, the reference's CPU case), c1 (128^3 res-16,
1080p), c3 (256^3 res-16, 3840x2160 — the 8-GPU config), and c4 (256^3 light propagation: converge, then per step
10 000 random block edits + propagation to epsilon 1 + a re-render; metric cube-updates/s).

Prints ONE JSON line (rank 0).  `value` = rays / device time with inputs resident in HBM;
`e2e` = the same through the host-buffer call (cube-delta H2D + frame D2H inside the timed
region); `roofline` = algorithmic bytes / kernel time vs the measured HBM peak;
`cpu_baseline` = the oracle (CPU restatement of the reference, all host threads) on a bounded
sample of the same frame.  `--impl reference` times only that CPU path.

`--dump-outputs DIR` writes what the last timed step computed, as the caller of the GPU path receives it, to
DIR/<name>.npy (see dump_outputs), so that two builds can be compared output for output on identical inputs.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "all-is-cubes_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

STRIP_ROWS = 16


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=100)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--workload", default="c2", choices=["c0", "c1", "c2", "c3", "c4"])
    p.add_argument("--light-n", type=int, default=256, help="c4: edge of the Space")
    p.add_argument("--pageable", action="store_true", help="e2e: the caller's output buffer is pageable host memory")
    p.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample")
    p.add_argument("--gather", default="p2p", choices=["p2p", "p2p-barrier", "nccl"],
                   help="N>1: 'p2p' = the encode kernel stores its strips straight into rank 0's frame over NVLink "
                        "(CUDA IPC mapped peer memory) and an arrival counter in that memory replaces the collective; "
                        "'p2p-barrier' = the same stores + an NCCL barrier; 'nccl' = packed strips + NCCL gather + reassembly")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (float32/float64)")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        # the CPU arm renders a row sample sized by its own timing, so its output is not the same from run to run
        p.error("--dump-outputs applies to the GPU path, not to --impl reference")
    return args


DUMP_BYTES = 63_000_000   # array data; with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy: float64 for 64-bit inputs, float32 otherwise (exact for the uint8
    pixels and light texels).  If they would come to more than DUMP_BYTES, each multi-dimensional array is cut to the
    same fraction of its records (entries along the last axis, e.g. the RGBA of a pixel), chosen with a fixed seed so that
    every run keeps the same records: <name>.npy then has shape [k, channels] and <name>_index.npy (float64) holds the
    flat record indices."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: a.astype(np.float64 if a.dtype.itemsize == 8 else np.float32) for k, a in arrays.items()}
    whole = sum(a.nbytes for a in arrays.values())
    fraction = 1.0
    if whole > DUMP_BYTES:
        fixed = sum(a.nbytes for a in arrays.values() if a.ndim < 2)
        per_record = sum(a.nbytes + 8 * (a.size // a.shape[-1]) for a in arrays.values() if a.ndim >= 2)
        fraction = (DUMP_BYTES - fixed) / per_record
    for name, a in arrays.items():
        if fraction < 1.0 and a.ndim >= 2:
            records = a.reshape(-1, a.shape[-1])
            k = int(records.shape[0] * fraction)
            index = np.sort(np.random.default_rng(0).choice(records.shape[0], k, replace=False))
            np.save(os.path.join(out_dir, f"{name}_index.npy"), index.astype(np.float64))
            a = records[index]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def make_workload(name):
    """Returns (space, options, width, height, description)."""
    import aicb200
    from aicb200 import scenes
    if name == "c0":
        space = scenes.config_c0()
        opts = aicb200.GraphicsOptions.unaltered_colors()
        w, h = 256, 256
        desc = "C0: 32^3 solid/empty res-1, 256x256, UNALTERED_COLORS"
    elif name == "c1":
        space = scenes.config_c1(n=128)
        opts = aicb200.GraphicsOptions.unaltered_colors()
        opts.view_distance = 512.0
        w, h = 1920, 1080
        desc = "C1: 128^3, 256 res-16 recursive blocks, opaque, 1920x1080, UNALTERED_COLORS"
    elif name == "c3":
        space = scenes.config_c1(n=256)
        opts = aicb200.GraphicsOptions.unaltered_colors()
        opts.view_distance = 1024.0
        w, h = 3840, 2160
        desc = "C3: 256^3, res-16 recursive blocks, 3840x2160, UNALTERED_COLORS"
    else:
        space = scenes.config_c2(n=256, with_light=True)
        opts = aicb200.GraphicsOptions(view_distance=1024.0)  # GraphicsOptions::default(): fog Abrupt, Linear light, Volumetric
        w, h = 1920, 1080
        desc = ("C2: 256^3 mixed transparent (alpha .125/.25/.5, res-1 + res-16), light volume, 1920x1080, "
                "GraphicsOptions::default() with view_distance 1024")
    return space, opts, w, h, desc


# ------------------------------------------------------------------------------------------------
# CPU baseline (the oracle; the Rust reference cannot be built in this image)
# ------------------------------------------------------------------------------------------------
def effective_cpus():
    """Host threads this process can actually run concurrently: the affinity mask capped by the cgroup
    CPU quota (the GPU boxes expose 128 logical CPUs behind a 16-CPU quota; oversubscribing a quota
    only adds throttling)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(round(int(quota) / int(period)))))
    except (OSError, ValueError):
        pass
    return max(1, n)


def cpu_sample(space, cam, opts, height, target_seconds):
    """Times the oracle (all usable host threads, dynamic 64-pixel work items) on rows spread evenly over
    the frame, repeated until ~target_seconds; returns (Mrays/s, cores, description, rows)."""
    import orc
    oscene = orc.OracleScene(space)
    threads = effective_cpus()
    width = cam.data.fb_width
    # calibrate on 16 rows spread over the frame
    probe = [int((i + 0.5) * height / 16) for i in range(16)]
    t0 = time.perf_counter()
    orc.render_rowlist(oscene, cam, opts, probe, n_threads=threads)
    per_row = max((time.perf_counter() - t0) / len(probe), 1e-5)
    n_rows = int(max(16, min(height, target_seconds / per_row)))
    rows = sorted(set(int((i + 0.5) * height / n_rows) for i in range(n_rows)))
    passes = int(max(1, min(50, target_seconds / max(per_row * len(rows), 1e-3))))
    t0 = time.perf_counter()
    for _ in range(passes):
        orc.render_rowlist(oscene, cam, opts, rows, n_threads=threads)
    dt = time.perf_counter() - t0
    rays = width * len(rows) * passes
    return (rays / dt / 1e6, threads,
            f"{len(rows)} rows spread evenly over the frame x {passes} passes ({rays} rays, {dt:.1f} s, {threads} threads; "
            f"{os.cpu_count()} logical CPUs visible)", rows)


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; kind 'port') on this box's host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import __graft_entry__ as g
    g.build_oracle()
    import aicb200
    import orc
    # This arm never loads libaicb200.so: the scene is numpy, and the camera matrices come from the oracle library
    # (the same host source compiled under orc_* names, oracle/Makefile).
    aicb200.use_camera_library(orc.lib(), "orc_")
    if args.workload == "c4":
        return run_reference_light(args)
    space, opts, w, h, desc = make_workload(args.workload)
    from aicb200 import scenes
    cam = scenes.standard_camera(space, opts, w, h)
    threads = effective_cpus()
    # each step = one bounded sample of the frame, sized so the whole run stays within minutes
    per_step = max(1.0, min(args.cpu_seconds, 150.0 / max(1, args.steps + args.warmup)))
    mr, _, sample, rows = cpu_sample(space, cam, opts, h, per_step)
    oscene = orc.OracleScene(space)

    def one_step():
        t0 = time.perf_counter()
        orc.render_rowlist(oscene, cam, opts, rows, n_threads=threads)
        return w * len(rows), time.perf_counter() - t0

    for _ in range(args.warmup):
        one_step()
    tot_rays, tot_t = 0, 0.0
    for _ in range(args.steps):
        r, t = one_step()
        tot_rays += r
        tot_t += t
    value = tot_rays / tot_t / 1e6
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(1, args.steps),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64 geometry / f32 colour",
        "data": "synthetic",
        "config": {"workload": desc, "sample": sample, "threads": threads,
                   "note": "CPU port of the Rust reference (no rustc in this image); libaicb200.so is not loaded by this arm"},
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))

# ------------------------------------------------------------------------------------------------
# C4: light propagation (BASELINE configs[4])
# ------------------------------------------------------------------------------------------------
C4_EDITS = 10000


def c4_description(n):
    return (f"C4: {n}^3 res-1 Space, LightPhysics::Rays{{30}}, octant sky; converged (fast_evaluate_light + "
            f"evaluate_light(1)) before timing; step = {C4_EDITS} random block edits + propagation to epsilon 1 + "
            f"re-render 1920x1080 (Linear lighting)")


def light_bytes(updates, node_visits):
    """SURVEY 8(d): nodes_visited x (48 + 2) + 4 per update (chart node record + sky term = 48 B, cell 2 B, the stored
    texel 4 B).  The per-hit term (4 + 140 B per visible block met) is not counted by the kernel and left out: a
    lower bound of the algorithmic bytes."""
    return 50 * node_visits + 4 * updates


def run_reference_light(args):
    """--impl reference --workload c4: the oracle's update_light_from_queue as the reference runs it with its
    `auto-threads` feature (batches of 32 cubes computed in parallel, applied in order) on a bounded Space."""
    import orc
    from aicb200 import scenes
    n = 40   # bounded sample: 256^3 would take tens of minutes on the host
    threads = min(32, effective_cpus())   # (a batch is 32 cubes)
    space = scenes.config_c4(n)
    ol = orc.OracleLight(space)
    ol.fast_evaluate()
    ol.evaluate_threaded(1, threads)
    n_edits = max(1, C4_EDITS * n ** 3 // args.light_n ** 3)
    tot_u, tot_t, tot_v = 0, 0.0, 0
    for step in range(args.warmup + args.steps):
        cubes, ids = scenes.c4_edits(space, n_edits, step)
        v0 = int(orc.lib().orc_light_node_visits(ol.handle))
        t0 = time.perf_counter()
        ol.set_cubes(cubes, ids)
        u, _ = ol.evaluate_threaded(1, threads)
        dt = time.perf_counter() - t0
        if step >= args.warmup:
            tot_u += u
            tot_t += dt
            tot_v += int(orc.lib().orc_light_node_visits(ol.handle)) - v0
    value = tot_u / max(tot_t, 1e-9)
    sample = (f"{n}^3 Space of the same recipe, {n_edits} edits per step (the same edit density), {args.steps} steps, "
              f"{tot_u} cube updates in {tot_t:.1f} s, {threads} threads (the reference's threaded update_light_from_queue: "
              f"batches of 32 computed in parallel, applied serially)")
    line = {
        "impl": "reference", "metric": "cube-updates/s", "value": value, "unit": "cube-updates/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(1, args.steps),
        "higher_is_better": True, "scaling": "replicas", "vs_baseline": None, "dtype": "f32 light / u8 packed",
        "data": "synthetic",
        "config": {"workload": c4_description(args.light_n), "sample": sample, "threads": threads,
                   "chart_node_visits_per_s": tot_v / max(tot_t, 1e-9),
                   "note": "CPU port of the Rust reference (no rustc in this image); libaicb200.so is not loaded by this arm"},
        "cpu_baseline": {"value": value, "unit": "cube-updates/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "cube-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def run_light(args):
    """--workload c4: light propagation is not sharded (SURVEY 8(e): replicas only) — rank 0 runs it, the line says so."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — libaicb200 has no CPU fallback (use --impl reference for the CPU path)")
    import __graft_entry__ as g
    g.build_library()
    g.build_oracle()
    import aicb200
    from aicb200 import scenes
    n = args.light_n
    space = scenes.config_c4(n)
    opts = aicb200.GraphicsOptions(view_distance=4.0 * n)   # default options: Linear lighting, fog Abrupt, Volumetric
    cam = scenes.standard_camera(space, opts, 1920, 1080)
    rt = aicb200.SpaceRaytracer(space, opts)
    # ---- setup (untimed, reported): the flood that converges the whole volume ---------------------------
    t0 = time.perf_counter()
    rt.light_fast_evaluate()
    upd0, md0, nv0 = rt.light_evaluate(1)
    conv_s = time.perf_counter() - t0
    conv = rt.light_stats()
    r = aicb200.RtRenderer(cam)
    r.rt = rt
    sampler = ClockSampler(0)
    host_frame = np.zeros((1080, 1920, 4), dtype=np.uint8)

    def step(k, render):
        cubes, ids = scenes.c4_edits(space, C4_EDITS, k)
        t0 = time.perf_counter()
        u, md = rt.light_edit_and_propagate(cubes, ids, 1)   # H2D: the edit list; blocks until the propagation is done
        st = rt.light_stats()
        img = r.draw() if render else None                   # D2H: the frame
        return u, md, st, time.perf_counter() - t0, img

    for k in range(max(3, args.warmup)):
        step(k, True)
    sampler.start()
    tot_u = tot_v = 0
    dev_s = e2e_s = 0.0
    render_ms = []
    launches = 0
    for k in range(args.steps):
        u, md, st, wall, img = step(max(3, args.warmup) + k, True)
        tot_u += u
        tot_v += st["chart_node_visits"]
        dev_s += st["device_seconds"]
        e2e_s += wall
        render_ms.append(img.info.kernel_ms)
        launches += 2 + 7 * st["rounds"] + 4   # edits + tile rebuild; 7 kernels per relaxation round; the 4 kernels of the re-render
    clocks = sampler.stop()
    if args.dump_outputs:   # the last step's (updates, max difference), the light it left in the Space, its re-render
        dump_outputs(args.dump_outputs, {"light_update": np.array([u, md], dtype=np.int64),
                                         "light": rt.light_download(), "frame": img.data})
    value = tot_u / dev_s
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = light_bytes(tot_u, tot_v) / dev_s / 1e9
    line = {
        "metric": "cube-updates/s", "value": value, "unit": "cube-updates/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": 1e3 * dev_s / args.steps, "higher_is_better": True,
        "scaling": "replicas", "vs_baseline": None, "dtype": "f32 light / u8 packed", "data": "synthetic",
        "config": {"workload": c4_description(n), "edits_per_step": C4_EDITS, "cube_updates_per_step": tot_u / args.steps,
                   "chart_node_visits_per_s": tot_v / dev_s, "rerender_frame_ms": float(np.mean(render_ms)),
                   "initial_convergence": {"cube_updates": upd0, "wall_seconds": conv_s, "device_seconds": conv["device_seconds"],
                                           "cube_updates_per_s": upd0 / max(conv["device_seconds"], 1e-9),
                                           "chart_node_visits": nv0, "rounds": conv["rounds"]},
                   "l2": "every step edits and relaxes different cubes of a 256^3 volume (scene + light + queue: 0.2 GB > L2)",
                   "sharding": "none (light propagation runs on one GPU; SURVEY 8(e) replicas only)"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)",
                     "kernel": "k_walk_chains<compute> + k_walk_chains<mark> (chart walk, one warp per cube)", "kernel_ms": 1e3 * dev_s / args.steps,
                     "algorithmic_bytes_per_step": int(light_bytes(tot_u, tot_v) / args.steps),
                     "formula": "50 B per chart node visited + 4 B per cube update (SURVEY 8(d), per-hit term not counted)"},
        "e2e": {"value": tot_u / e2e_s, "unit": "cube-updates/s", "h2d_bytes_per_step": C4_EDITS * 14,
                "d2h_bytes_per_step": 1920 * 1080 * 4, "includes": "edit list H2D, propagation, re-render, frame D2H"},
        "gpu_launches": launches,
        "clocks": clocks,
    }
    # CPU baseline: the oracle on a bounded Space of the same recipe
    import orc
    nb = 48
    threads = min(32, effective_cpus())
    sp2 = scenes.config_c4(nb)
    ol = orc.OracleLight(sp2)
    t0 = time.perf_counter()
    ol.fast_evaluate()
    nup, _ = ol.evaluate_threaded(1, threads)
    dt = time.perf_counter() - t0
    line["cpu_baseline"] = {"value": nup / dt, "unit": "cube-updates/s", "cores": threads, "kind": "port",
                            "sample": f"initial convergence of a {nb}^3 Space of the same recipe: {nup} cube updates in {dt:.1f} s, "
                                      f"{threads} threads (the reference's threaded update_light_from_queue: batches of 32 "
                                      f"computed in parallel, applied serially)"}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# clocks sampling
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.samples = []
        self.proc = None
        self.device_index = device_index
        self.first = 0

    def mark(self):
        """The timed region begins: samples taken before this point (nvidia-smi needs ~0.1 s to start streaming, so it
        is started before the warm-up) are not reported."""
        self.first = len(self.samples)

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.device_index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples[self.first:]:
            parts = [p.strip() for p in s.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — libaicb200 has no CPU fallback (use --impl reference for the CPU path)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import __graft_entry__ as g
    if rank == 0:
        g.build_library()
        g.build_oracle()
    if world > 1:
        dist.barrier()
    import aicb200
    from aicb200 import abi, scenes
    lib = aicb200.load_library()

    space, opts, w, h, desc = make_workload(args.workload)
    cam = scenes.standard_camera(space, opts, w, h)
    ctx = aicb200.Context(local_rank)
    rt = aicb200.SpaceRaytracer(space, opts, ctx)
    o_abi = opts.to_abi(True)
    shard = abi.Shard(STRIP_ROWS, rank, world)
    n_local = lib.aicb_shard_pixel_count(C.byref(cam.data), C.byref(shard))
    n_max = max(lib.aicb_shard_pixel_count(C.byref(cam.data), C.byref(abi.Shard(STRIP_ROWS, r, world))) for r in range(world))
    from aicb200 import multi
    d_out = torch.empty((n_max, 4), dtype=torch.uint8, device="cuda")
    gather_scratch = [torch.empty_like(d_out) for _ in range(world)] if (world > 1 and rank == 0) else None
    frame = torch.empty((h, w, 4), dtype=torch.uint8, device="cuda") if rank == 0 else None
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    # a dedicated (non-default) stream: its handle is what the library launches on, and what the
    # CUDA events below are recorded on
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    info = abi.RenderInfo()

    def check(st):
        if st != 0:
            raise RuntimeError(lib.aicb_last_error().decode())

    gather_mode = args.gather if world > 1 else "none"
    use_counter = gather_mode == "p2p"
    if gather_mode == "p2p-barrier":
        gather_mode = "p2p"
    peer = None
    peers = []
    if gather_mode == "p2p":
        try:
            # Two shared frames when the counters are used: frame k + 1 is stored into the other buffer while rank 0 is
            # still through with frame k, so a step does not contain a round trip of the consumed counter (every frame
            # is still rendered by all ranks and delivered to rank 0; two frames are in flight).
            for _ in range(2 if use_counter else 1):
                pf = multi.PeerFrame(ctx, h, w, rank, world)
                peers.append(pf)
                # touch the mapping once from every rank
                check(lib.aicb_render_srgb8_device_frame(rt.handle, C.byref(cam.data), C.byref(o_abi), C.byref(shard),
                                                         pf.ptr, w * h, C.c_void_p(stream.cuda_stream)))
            peer = peers[0]
            torch.cuda.synchronize()
            ok = torch.tensor([1], device="cuda")
        except Exception as e:  # noqa: BLE001 — any failure falls back to the NCCL gather
            sys.stderr.write(f"[rank {rank}] p2p frame unavailable ({e}); falling back to NCCL gather\n")
            ok = torch.tensor([0], device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            gather_mode, peer, peers = "nccl", None, []

    release_on_device = True   # e2e: rank 0 releases the frame after its device -> host copy instead
    frame_no = [0]

    def device_step():
        """One frame with everything resident in HBM: trace kernel + delivery of the strips to rank 0."""
        nonlocal peer
        if gather_mode == "p2p":
            peer = peers[frame_no[0] % len(peers)]
            frame_no[0] += 1
            if use_counter:   # no collective: counters behind the frame's pixels, all in stream order
                peer.begin_frame(stream.cuda_stream)
            check(lib.aicb_render_srgb8_device_frame(rt.handle, C.byref(cam.data), C.byref(o_abi), C.byref(shard),
                                                     peer.ptr, w * h, C.c_void_p(stream.cuda_stream)))
            if use_counter:
                peer.end_frame(stream.cuda_stream, release=release_on_device)
            else:
                dist.barrier()  # NCCL barrier on the current stream: rank 0's frame is complete after it
        else:
            check(lib.aicb_render_srgb8_device(rt.handle, C.byref(cam.data), C.byref(o_abi), C.byref(shard),
                                               d_out.data_ptr(), n_local, C.c_void_p(stream.cuda_stream)))
            if world > 1:
                multi.gather_frame(d_out, h, w, rank, world, frame=frame, scratch=gather_scratch)

    def timed(fn, steps):
        """K steps; per-step CUDA events on the launch stream, L2 flushed between steps (outside the
        events); returns total ms = sum over steps, MAX over ranks."""
        evs = []
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        for _ in range(steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            evs.append((e0, e1))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up, then the timed region ------------------------------------------------------------
    # one blocking render first: it sizes the hit stream for this workload (the blocking call re-issues the frame when
    # the stream overflows; the asynchronous calls below would report AICB_ERR_RETRY instead)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()   # (streams a sample every 20 ms from here on; the ones of the timed region are reported)
    sizing = torch.empty((n_local, 4), dtype=torch.uint8).pin_memory()
    check(lib.aicb_render_srgb8(rt.handle, C.byref(cam.data), C.byref(o_abi), C.byref(shard), sizing.data_ptr(), n_local, None))
    del sizing
    for _ in range(max(3, args.warmup)):
        device_step()
    torch.cuda.synchronize()
    check(lib.aicb_render_finish(rt.handle, C.byref(info)))

    sampler.mark()
    check(lib.aicb_ctx_stage_timing(ctx.handle, 0))   # the timed frames carry no per-kernel event records
    total_ms = timed(device_step, args.steps)
    if args.dump_outputs and rank == 0:   # the frame the last timed step delivered to rank 0
        if world == 1:
            last = d_out[:n_local].cpu()
        elif gather_mode == "p2p":
            last = torch.empty((h * w, 4), dtype=torch.uint8).pin_memory()
            peer.read(last, stream.cuda_stream)
        else:
            last = frame.cpu()
        dump_outputs(args.dump_outputs, {"frame": last.numpy().reshape(h, w, 4)})
    # kernel-only duration of the last frame from the library's own events (same stream); a frame that overflowed its
    # hit stream inside the timed region would make this call fail (AICB_ERR_RETRY) and with it the run
    check(lib.aicb_render_finish(rt.handle, C.byref(info)))
    kernel_ms_last = float(info.kernel_ms)
    check(lib.aicb_ctx_stage_timing(ctx.handle, 1))   # ... the launches below do (stage_ms)
    rays_per_frame = w * h
    value = rays_per_frame * args.steps / (total_ms * 1e-3) / 1e6

    # ---- dominant-kernel time, averaged over the timed region's launches ---------------------------
    kernel_ms, stage_ms = [], []
    for _ in range(max(3, min(args.steps, 10))):
        flush.zero_()
        check(lib.aicb_render_srgb8_device(rt.handle, C.byref(cam.data), C.byref(o_abi), C.byref(shard),
                                           d_out.data_ptr(), n_local, C.c_void_p(stream.cuda_stream)))
        torch.cuda.synchronize()
        check(lib.aicb_render_finish(rt.handle, C.byref(info)))
        kernel_ms.append(float(info.kernel_ms))
        stage_ms.append([float(v) for v in info.stage_ms])
    kernel_avg_ms = float(np.mean(kernel_ms))
    stage_avg_ms = [float(v) for v in np.mean(np.array(stage_ms), axis=0)]   # gen, march, shade, encode
    clocks = sampler.stop() if rank == 0 else None  # sampled over the timed region and the kernel-time launches

    if peers and use_counter and rank == 0 and any(pf.timed_out() for pf in peers):
        raise SystemExit("bench.py: a wait on the frame's arrival counter gave up (a rank did not deliver its strips)")
    # ---- N > 1: the delivered frame must equal the frame one GPU renders alone -----------------------
    frame_check = None
    if world > 1:
        device_step()
        torch.cuda.synchronize()
        dist.barrier()
        if rank == 0:
            got = torch.empty((h * w, 4), dtype=torch.uint8).pin_memory()
            if gather_mode == "p2p":
                peer.read(got, stream.cuda_stream)
            else:
                got.copy_(frame.view(h * w, 4))
            alone = torch.empty((h * w, 4), dtype=torch.uint8).pin_memory()
            check(lib.aicb_render_srgb8(rt.handle, C.byref(cam.data), C.byref(o_abi), None, alone.data_ptr(), h * w, None))
            frame_check = bool(torch.equal(got, alone))
            if not frame_check:
                raise SystemExit("bench.py: N-rank frame differs from the 1-rank frame")
        dist.barrier()

    # ---- algorithmic bytes of this launch from device counters (one untimed AUX pass) ---------------
    r = aicb200.RtRenderer(cam, ctx)
    r.rt = rt
    aux = r.draw_colorbuf(shard=(STRIP_ROWS, rank, world), want_depth=False, want_hit=False, want_steps=False)
    ai = aux["info"]
    alg_bytes = ai.algorithmic_bytes - 16 * ai.counters[5] + 4 * ai.counters[5]  # sRGB8 output instead of ColorBuf
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    # the dominant kernel is the marching kernel: cells / voxels it steps over (2 B each), the palette entry of each
    # surface whose transmittance it applies (32 B) and the descriptor of each block it enters (32 B); the light
    # texels belong to the shading kernel and the pixels to the encode kernel (SURVEY 8(d) counts them per frame)
    march_bytes = 2 * ai.counters[0] + 2 * ai.counters[1] + 32 * ai.counters[2] + 32 * ai.counters[4]
    march_ms = stage_avg_ms[1]
    achieved = march_bytes / (march_ms * 1e-3) / 1e9
    traffic = None   # DRAM bytes of the marching kernel per launch from the committed ncu --set full capture
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        if tr.get("workload") == args.workload and world == 1:
            traffic = int(tr["traffic_bytes_per_launch"])
    except (OSError, ValueError, KeyError):
        pass
    frame_achieved = alg_bytes / (kernel_avg_ms * 1e-3) / 1e9

    # ---- e2e: host buffers through the public API ------------------------------------------------------
    n_delta = 1024
    rng = np.random.default_rng(0)
    cubes = np.stack([rng.integers(0, space.size[a], n_delta) + space.lower[a] for a in range(3)], axis=1).astype(np.int32)
    delta_ids = space.block_ids[cubes[:, 0] - space.lower[0], cubes[:, 1] - space.lower[1], cubes[:, 2] - space.lower[2]].copy()
    delta_light = space.light[cubes[:, 0] - space.lower[0], cubes[:, 1] - space.lower[1], cubes[:, 2] - space.lower[2]].copy() \
        if space.light is not None else None
    host_out = torch.empty((n_local, 4), dtype=torch.uint8).pin_memory()
    host_frame = torch.empty((h, w, 4), dtype=torch.uint8).pin_memory() if rank == 0 else None
    h2d_bytes = cubes.nbytes + delta_ids.nbytes + (delta_light.nbytes if delta_light is not None else 0)

    def e2e_step():
        """update(): a batch of cube deltas H2D (same values: the image is unchanged); draw(): frame D2H."""
        rt.update_cubes(cubes[:64], delta_ids[:64], None if delta_light is None else delta_light[:64])
        if world == 1:
            check(lib.aicb_render_srgb8(rt.handle, C.byref(cam.data), C.byref(o_abi), C.byref(shard),
                                        host_out.data_ptr(), n_local, None))
        else:
            nonlocal release_on_device
            release_on_device = False     # the frame is released after rank 0 has copied it out
            device_step()
            release_on_device = True
            if rank == 0:
                if gather_mode == "p2p":
                    peer.read(host_frame, stream.cuda_stream)
                    if use_counter:
                        peer.release(stream.cuda_stream)
                else:
                    host_frame.copy_(frame, non_blocking=False)

    for _ in range(2):
        e2e_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    k_e2e = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(k_e2e):
        e2e_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = rays_per_frame * k_e2e / float(t.item()) / 1e6
    h2d_step = 64 * (12 + 2 + (4 if delta_light is not None else 0))
    d2h_step = w * h * 4
    # the same call with a PAGEABLE destination (what a Rust Vec<[u8; 4]> or a numpy array is): the library stages the
    # frame in its own pinned buffer and copies it out on the host
    e2e_pageable = None
    if world == 1:
        page_out = np.zeros((n_local, 4), dtype=np.uint8)

        def pageable_step():
            rt.update_cubes(cubes[:64], delta_ids[:64], None if delta_light is None else delta_light[:64])
            check(lib.aicb_render_srgb8(rt.handle, C.byref(cam.data), C.byref(o_abi), C.byref(shard),
                                        page_out.ctypes.data, n_local, None))

        for _ in range(2):
            pageable_step()
        t0 = time.perf_counter()
        for _ in range(k_e2e):
            pageable_step()
        e2e_pageable = rays_per_frame * k_e2e / (time.perf_counter() - t0) / 1e6
        assert np.array_equal(page_out, host_out.numpy()), "pageable and pinned destinations differ"

    if rank == 0:
        cpu = None
        if world == 1:
            import orc  # the checker, used here only as the reported CPU baseline
            mr, cores, sample, _ = cpu_sample(space, cam, opts, h, args.cpu_seconds)
            cpu = {"value": mr, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample}
        line = {
            "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64 geometry / f32 colour", "data": "synthetic",
            "config": {"workload": desc, "rays_per_step": rays_per_frame, "sharding": f"{world} x interleaved {STRIP_ROWS}-row strips",
                       "gather": ("p2p stores + arrival counter (no collective), two frames in flight" if (gather_mode == "p2p" and use_counter) else
                                  "p2p stores + NCCL barrier" if gather_mode == "p2p" else gather_mode),
                       "n_rank_frame_equals_1_rank_frame": frame_check,
                       "l2": "256 MiB buffer rewritten between timed steps", "scene_device_bytes": rt.device_bytes,
                       "cubes_traced_per_frame_this_rank": int(ai.cubes_traced)},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)",
                         "kernel": "trace_kernel (marching)", "kernel_ms": march_ms,
                         "algorithmic_bytes_per_launch": int(march_bytes),
                         "frame": {"kernels": ["gen_kernel", "trace_kernel", "shade_kernel", "encode_kernel"],
                                   "stage_ms": stage_avg_ms, "frame_ms": kernel_avg_ms,
                                   "algorithmic_bytes_per_frame": int(alg_bytes), "achieved": frame_achieved,
                                   "frac": frame_achieved / peak},
                         "counters": {"outer_steps": ai.counters[0], "inner_steps": ai.counters[1], "surface_hits": ai.counters[2],
                                      "light_texels": ai.counters[3], "blocks_entered": ai.counters[4], "pixels": ai.counters[5]}},
            "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": h2d_step, "d2h_bytes_per_step": d2h_step,
                    "destination": "pinned host buffer", "pageable_destination_value": e2e_pageable},
            "gpu_launches": 4 * args.steps,
            "clocks": clocks,
        }
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "c4":
        run_light(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
