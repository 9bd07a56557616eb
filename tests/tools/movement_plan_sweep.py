"""Movement-plan sweep (GPU): ka_plan_last device time and the full against the changed-rows-only device JSON, end to end.

Scenarios (BASELINE shapes, synth seeds): "balanced" = the current assignment is this solver's own output for the full broker
set, then a fraction of every rack is removed (0 = a re-run); "as synthesised" = the generator's current lists.

  python tests/tools/movement_plan_sweep.py [--steps 20] [--out DIR]

Per scenario it prints one JSON line: the plan totals, the plan kernel's device time (torch.profiler, CUDA activities; a
separate pass from the end-to-end timing) with the bytes it must read, Q * (RF + S + 1) * 4, over that time, the wall time of
a whole ka_plan_last call, and the median wall time of solve_dense_json with and without changed_only (pinned host buffers,
warmed, --steps timed calls each, interleaved) with the bytes of each text. The card's name and power limit come first."""
import argparse
import dataclasses
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import kafka_assigner_b200 as kab  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def scenarios():
    for key in ("c3", "c5"):
        base = kab.synth.make_config(key, "mixed")
        out, _, _ = kab.Solver(0).solve_cluster(base)
        fracs = (0.05,) if key == "c3" else (0.0, 0.01, 0.05, 0.2)
        for f in fracs:
            cl = kab.synth.make_config(key, "mixed", remove_frac=f) if f else base
            yield "%s balanced %s" % (key, "re-run" if not f else "-%d%%" % round(100 * f)), dataclasses.replace(cl, cur=out.copy())
    yield "c5 as synthesised -1%", kab.synth.make_config("c5", "mixed", remove_frac=0.01)


def plan_kernel_ms(s, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            s.last_plan()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if "ka_plan_kernel" in e.name]
    return sum(e.device_time for e in ev) / max(len(ev), 1) / 1000.0, len(ev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    rows = [{"card": card()}]
    print(json.dumps(rows[0]), flush=True)
    for name, cl in scenarios():
        s = kab.Solver(0)
        s.set_brokers(cl.broker_id, cl.rack_index)
        names = s.marshal_names(cl.topic_names)
        cap = 64 + cl.T * cl.P * (50 + 12 * cl.RF) + int(cl.P * names[1][-1])
        buf = torch.empty(cap, dtype=torch.uint8).pin_memory().numpy()
        h_hash = torch.from_numpy(cl.topic_hash).pin_memory().numpy()
        h_cur = torch.from_numpy(np.ascontiguousarray(cl.cur)).pin_memory().numpy()
        times = {False: [], True: []}
        size = {}
        for step in range(3 + a.steps):   # 3 warm-up pairs, then timed pairs; the two forms alternate
            for changed in (False, True):
                t0 = time.perf_counter()
                text, st = s.solve_dense_json(cl.topic_names, h_hash, h_cur, json_buf=buf, names_slab=names, changed_only=changed)
                dt = time.perf_counter() - t0
                size[changed] = len(text)
                if step >= 3:
                    times[changed].append(dt * 1e3)
        totals, _, _, _ = s.last_plan()          # the plan of the last (changed-only) solve
        t0 = time.perf_counter()
        for _ in range(a.steps):
            s.last_plan()
        call_ms = (time.perf_counter() - t0) * 1e3 / a.steps
        kern_ms, nk = plan_kernel_ms(s, a.steps)
        Q = cl.T * cl.P
        nbytes = Q * (cl.RF + cl.RF + 1) * 4
        r = dict(scenario=name, Q=Q, totals=totals,
                 pct=dict(changed=100.0 * (totals["rows_moved"] + totals["rows_reordered"]) / Q,
                          moved=100.0 * totals["rows_moved"] / Q,
                          replicas_added=100.0 * totals["replicas_added"] / (Q * cl.RF),
                          leaders_changed=100.0 * totals["leaders_changed"] / Q),
                 plan_kernel_ms=round(kern_ms, 4), plan_kernels_profiled=nk, plan_bytes=nbytes,
                 plan_GBps=round(nbytes / (kern_ms * 1e-3) / 1e9, 1) if kern_ms > 0 else None,
                 plan_call_ms=round(call_ms, 3),
                 json_full_ms=round(float(np.median(times[False])), 3), json_changed_ms=round(float(np.median(times[True])), 3),
                 json_full_spread_ms=[round(min(times[False]), 3), round(max(times[False]), 3)],
                 json_changed_spread_ms=[round(min(times[True]), 3), round(max(times[True]), 3)],
                 json_full_MB=round(size[False] / 1e6, 2), json_changed_MB=round(size[True] / 1e6, 2), steps=a.steps)
        rows.append(r)
        print(json.dumps(r), flush=True)
        s.close()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "movement_plan_sweep.json"), "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
