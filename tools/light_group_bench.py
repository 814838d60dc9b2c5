"""C4 light propagation on a device group: the relaxation sharded by slabs (aicb_group_light_*).

    python tools/light_group_bench.py --devices 0,1,2,3 [--steps K] [--warmup W] [--n 256] [--trace-dir DIR]

bench.py --workload c4's recipe on a DeviceGroup: scenes.config_c4, converge (fast_evaluate + propagate to epsilon 1),
then steps of scenes.c4_edits (10 000 edits) + propagate to epsilon 1 + a group re-render at 1920x1080.  Prints one JSON
line shaped like bench c4's, with "scaling": "slabs", the per-member share of the cube updates and, per round and
member stream, the time in the exchange kernels (k_group_*) and the time outside the stream's own kernels (on distinct
devices: waiting at barriers, i.e. load imbalance plus barrier latency), from one extra step traced with torch.profiler
(a run of its own, not timed).  The same device may be named several times: the exchanges then run on one GPU, and the
time outside a stream's kernels also holds the other members' kernels sharing that GPU."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "all-is-cubes_b200"))

C4_EDITS = 10_000


def card(device):
    """Name and power limit of the card, read in the same run as the measurement."""
    try:
        out = subprocess.run(["nvidia-smi", f"--id={device}", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [v.strip() for v in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:   # noqa: BLE001 - reported, not hidden
        return {"name": None, "error": str(e)}


def trace_breakdown(trace_path, rounds):
    """Per (device, stream) of the traced step: work-kernel time, exchange-kernel time and the rest of the stream's
    span, per round."""
    events = json.load(open(trace_path)).get("traceEvents", [])
    streams = defaultdict(list)
    for e in events:
        if e.get("cat") == "kernel":
            a = e.get("args", {})
            streams[(a.get("device"), a.get("stream"))].append((e["ts"], e["dur"], e["name"]))
    out = []
    for key in sorted(streams, key=lambda k: (k[0] or 0, k[1] or 0)):
        ks = streams[key]
        span = max(t + d for t, d, _ in ks) - min(t for t, _, _ in ks)
        busy = sum(d for _, d, _ in ks)
        exchange = sum(d for _, d, n in ks if "k_group_" in n)
        out.append({"device": key[0], "stream": key[1], "kernels": len(ks), "span_ms": span / 1e3,
                    "outside_own_kernels_ms_per_round": (span - busy) / 1e3 / max(rounds, 1),
                    "exchange_kernels_ms_per_round": exchange / 1e3 / max(rounds, 1),
                    "work_kernels_ms_per_round": (busy - exchange) / 1e3 / max(rounds, 1)})
    return out


def main():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--devices", required=True, help="comma-separated device ids, one per member (repeats allowed)")
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=2)
    p.add_argument("--n", type=int, default=256, help="edge of the Space")
    p.add_argument("--trace-dir", default=None, help="where the profiled step's trace goes (default: a temporary directory)")
    args = p.parse_args()
    devices = [int(d) for d in args.devices.split(",")]

    import numpy as np
    import torch
    import aicb200
    from aicb200 import scenes

    if not torch.cuda.is_available():
        raise SystemExit("light_group_bench.py: no CUDA device (there is no CPU fallback)")
    space = scenes.config_c4(args.n)
    opts = aicb200.GraphicsOptions(view_distance=4.0 * args.n)
    cam = scenes.standard_camera(space, opts, 1920, 1080)
    g = aicb200.DeviceGroup(devices)
    g.update(space)
    t0 = time.perf_counter()
    g.light_fast_evaluate()
    upd0, _, nv0 = g.light_evaluate(1)
    conv_wall = time.perf_counter() - t0
    conv = g.light_stats()

    def step(k):
        cubes, ids = scenes.c4_edits(space, C4_EDITS, k)
        t = time.perf_counter()
        u, md = g.light_edit_and_propagate(cubes, ids, 1)
        st = g.light_stats()
        members = [g.light_stats(m)["cube_updates"] for m in range(len(devices))]
        img = g.draw(cam, opts)
        return u, st, members, time.perf_counter() - t, img

    warm = max(1, args.warmup)
    for k in range(warm):
        step(k)
    tot_u = tot_rounds = 0
    dev_s = e2e_s = 0.0
    per_member = np.zeros(len(devices))
    render_ms = []
    for k in range(args.steps):
        u, st, members, wall, img = step(warm + k)
        tot_u += u
        tot_rounds += st["rounds"]
        dev_s += st["device_seconds"]
        e2e_s += wall
        per_member += members
        render_ms.append(img.info.kernel_ms)

    # one more step under the profiler, for the time spent in barriers and exchanges
    from torch.profiler import ProfilerActivity, profile
    trace_dir = args.trace_dir or tempfile.mkdtemp(prefix="light_group_bench_")
    os.makedirs(trace_dir, exist_ok=True)
    cubes, ids = scenes.c4_edits(space, C4_EDITS, warm + args.steps)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        g.light_edit_and_propagate(cubes, ids, 1)
    traced_rounds = g.light_stats()["rounds"]
    trace_path = os.path.join(trace_dir, f"light_group_{len(devices)}.pt.trace.json")
    prof.export_chrome_trace(trace_path)
    breakdown = trace_breakdown(trace_path, traced_rounds)

    line = {
        "metric": "cube-updates/s", "value": tot_u / dev_s, "unit": "cube-updates/s", "n_gpus": len(set(devices)),
        "members": devices, "steps": args.steps, "warmup": warm, "ms_per_step": 1e3 * dev_s / args.steps,
        "higher_is_better": True, "scaling": "slabs",
        "config": {"workload": f"C4 {args.n}^3 light propagation (scenes.config_c4, Rays{{30}}): {C4_EDITS} edits + "
                               f"propagate to epsilon 1 + group re-render 1920x1080 per step",
                   "cube_updates_per_step": tot_u / args.steps, "rounds_per_step": tot_rounds / args.steps,
                   "rerender_frame_ms": float(np.mean(render_ms)),
                   "member_share_of_updates": [float(v) for v in per_member / max(per_member.sum(), 1)],
                   "initial_convergence": {"cube_updates": upd0, "wall_seconds": conv_wall,
                                           "device_seconds": conv["device_seconds"], "chart_node_visits": nv0,
                                           "rounds": conv["rounds"]},
                   "device_time": "the slowest member's, CUDA events on its stream around the propagation"},
        "per_round_breakdown": {"rounds": traced_rounds, "streams": breakdown,
                                "source": "one extra step traced with torch.profiler (kernel spans per stream)"},
        "e2e": {"value": tot_u / e2e_s, "unit": "cube-updates/s", "includes": "edit list, propagation, re-render, frame D2H"},
        "card": card(devices[0]),
    }
    print(json.dumps(line))


if __name__ == "__main__":
    main()
