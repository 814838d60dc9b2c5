"""C4 light propagation driven in budgeted steps (aicb_light_step), as a host drives light once per tick.

    python tools/light_step_bench.py [--budget-us 1000,4000,16000] [--max-updates N,...] [--ticks 3] [--n 256]
                                     [--devices 0,1]

bench.py --workload c4's recipe: scenes.config_c4, converge (fast_evaluate + propagate to epsilon 1), then ticks of
scenes.c4_edits (10 000 edits).  For every budget, each tick submits its edits with the first step and steps with that
budget until nothing above epsilon 1 is queued, taking the changed cubes (aicb_light_take_changes) after each step.
Beside it, a second scene in the same state runs one unbudgeted edit_and_propagate of the same edits: the reference
update rate of the same run.  Prints one JSON line per budget with the per-step device time against the budget
(median / p90 / max), the updates per step, the update rate over the drain against the unbudgeted rate, the changed
cubes per take and the take time, with the card name and power limit.  --devices runs both on a DeviceGroup."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "all-is-cubes_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from light_group_bench import C4_EDITS, card  # noqa: E402

EPS = 1
EPS_PRIORITY = EPS // 2 + 1   # Priority::from_difference(epsilon)


def quantiles(v):
    v = np.asarray(v, dtype=np.float64)
    if v.size == 0:
        return None
    return {"median": float(np.median(v)), "p90": float(np.percentile(v, 90)), "max": float(v.max()), "n": int(v.size)}


def main():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--budget-us", default="1000,4000,16000", help="comma-separated time budgets per step (microseconds)")
    p.add_argument("--max-updates", default="", help="comma-separated update caps per step (instead of / besides time)")
    p.add_argument("--ticks", type=int, default=3, help="ticks of 10 000 edits per budget")
    p.add_argument("--n", type=int, default=256, help="edge of the Space")
    p.add_argument("--devices", default=None, help="comma-separated device ids of a DeviceGroup (default: one scene)")
    args = p.parse_args()
    budgets = [("budget_us", float(v)) for v in args.budget_us.split(",") if v] + \
              [("max_updates", int(v)) for v in args.max_updates.split(",") if v]

    import torch
    import aicb200
    from aicb200 import scenes

    if not torch.cuda.is_available():
        raise SystemExit("light_step_bench.py: no CUDA device (there is no CPU fallback)")
    space = scenes.config_c4(args.n)
    devices = [int(d) for d in args.devices.split(",")] if args.devices else None

    def make():
        if devices:
            t = aicb200.DeviceGroup(devices)
            t.update(space)
        else:
            t = aicb200.SpaceRaytracer(space, aicb200.GraphicsOptions())
        t.light_fast_evaluate()
        t.light_evaluate(EPS)
        return t

    ref, stp = make(), make()
    stp.light_track_changes(True)
    stp.light_take_changes()
    batch = 0
    for kind, value in budgets:
        step_ms, step_updates, take_ms, take_n = [], [], [], []
        drain_updates = drain_s = ref_updates = ref_s = 0.0
        steps_per_drain = []
        for _ in range(args.ticks):
            cubes, ids = scenes.c4_edits(space, C4_EDITS, batch)
            batch += 1
            ref.light_edit_and_propagate(cubes, ids, EPS)
            st = ref.light_stats()
            ref_updates += st["cube_updates"]
            ref_s += st["device_seconds"]
            limit = {kind: value}
            info = stp.light_step(cubes, ids, epsilon=EPS, **limit)
            steps = 0
            while True:
                steps += 1
                step_ms.append(info["device_ms"])
                step_updates.append(info["update_count"])
                drain_updates += info["update_count"]
                drain_s += info["device_ms"] * 1e-3
                t = time.perf_counter()
                changed, _ = stp.light_take_changes()
                take_ms.append(1e3 * (time.perf_counter() - t))
                take_n.append(len(changed))
                if info["max_queue_priority"] <= EPS_PRIORITY or steps >= 100_000:
                    break
                info = stp.light_step(epsilon=EPS, **limit)
            steps_per_drain.append(steps)
        line = {
            "metric": "budgeted light steps", kind: value, "ticks": args.ticks, "edits_per_tick": C4_EDITS,
            "members": devices or [0],
            "step_device_ms": quantiles(step_ms),
            "budget_ms": value * 1e-3 if kind == "budget_us" else None,
            "steps_over_budget": int(sum(1 for v in step_ms if kind == "budget_us" and v * 1e3 > value)),
            "updates_per_step": quantiles(step_updates),
            "steps_per_drain": steps_per_drain,
            "drain_updates_per_s": drain_updates / drain_s if drain_s else None,
            "unbudgeted_updates_per_s": ref_updates / ref_s if ref_s else None,
            "drain_updates_per_tick": drain_updates / args.ticks,
            "unbudgeted_updates_per_tick": ref_updates / args.ticks,
            "changed_cubes_per_take": quantiles(take_n),
            "take_ms": quantiles(take_ms),
            "config": {"workload": f"C4 {args.n}^3 (scenes.config_c4, Rays{{30}}), {C4_EDITS} edits per tick, epsilon {EPS}",
                       "device_time": "CUDA events on the stream around each step (group: the slowest member's)",
                       "take_time": "host clock around aicb_light_take_changes (count, take, copy to the host)"},
            "card": card((devices or [0])[0]),
        }
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
