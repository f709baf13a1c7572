#!/usr/bin/env python
"""The whole two-step solve driven from the host (povar_bundle_adjust) against the same solve as one graph launch
on the caller's stream (povar_bundle_adjust_async).

    python tools/time_async_solve.py --out profiles/async_solve_b200.json [--reps 5] [--shapes ...]

Problems: the synthetic ladybug-49, trafalgar-257 and venice-1778 shapes (synthetic.generate_named), all with the
benchmark's flags (alpha 0.1, 20 power-series terms, 50 + 50 iterations).  One handle per route, both restarted from
the same initial state before every solve; the routes alternate, --reps solves each.  Recorded per route:
  wall     host clock from the call to the end of a synchronise of the stream (median)
  blocked  how long the calling thread is held: the whole solve for the host route, until the call returns for the
           async route (median)
and the async route's first call, which builds and instantiates the graph, and the final cost and a digest of the
non-timing log columns of each route.  Device name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from povar_b200 import capi, synthetic  # noqa: E402

SHAPES = {"ladybug-49": "ladybug49", "trafalgar-257": "trafalgar257", "venice-1778": "venice1778"}
COLUMNS = ("step", "iteration", "step_is_valid", "step_is_successful", "cost", "cost_valid", "trial_cost",
           "num_obs_valid", "relative_decrease", "trust_region_radius", "linear_solver_iterations")


def device_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def digest(its):
    h = hashlib.sha256()
    for e in its:
        for f in COLUMNS:
            h.update(np.asarray(getattr(e, f)).tobytes())
    return h.hexdigest()[:16]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/async_solve_b200.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--shapes", nargs="*", default=list(SHAPES))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing is measured")
    result = {"device": device_info(), "reps": args.reps, "shapes": {}}
    opt = capi.default_options(alpha=0.1, power_sc_iterations=20, verbosity_level=0,
                               max_num_iterations_step_1=50, max_num_iterations_step_2=50)
    for label in args.shapes:
        sp = synthetic.generate_named(SHAPES[label])
        hp = capi.HostProblem.from_unordered(sp.num_cams, sp.num_lms, sp.obs_cam, sp.obs_lm, sp.obs_xy, sp.cam_params)
        solvers = {r: capi.Solver(hp, opt) for r in ("host", "async")}
        P0, X0 = solvers["host"].get_state(capi.STATE_POSE)
        stream = torch.cuda.current_stream()
        rec = {"cameras": hp.num_cams, "landmarks": hp.num_lms, "observations": hp.num_obs}
        times = {r: {"wall": [], "blocked": []} for r in solvers}
        last = {}
        for rep in range(args.reps + 1):   # rep 0: warm-up (the async route builds its graph)
            for route, s in solvers.items():
                s.set_state(capi.STATE_POSE, P0, X0)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if route == "host":
                    its, summary = s.bundle_adjust(opt)
                    t_ret = time.perf_counter()
                else:
                    job = s.bundle_adjust_async(opt)
                    t_ret = time.perf_counter()
                    stream.synchronize()
                t_end = time.perf_counter()
                if route == "async":
                    its, summary = job.result()
                if rep == 0:
                    if route == "async":
                        rec["async_first_call_s"] = t_ret - t0
                    continue
                times[route]["wall"].append(t_end - t0)
                times[route]["blocked"].append(t_ret - t0)
                last[route] = (its, summary)
        for route in solvers:
            its, summary = last[route]
            rec[route] = {"wall_median_s": float(np.median(times[route]["wall"])),
                          "blocked_median_s": float(np.median(times[route]["blocked"])),
                          "wall_s": times[route]["wall"], "blocked_s": times[route]["blocked"],
                          "trials": len(its), "final_cost": summary.final_cost, "digest": digest(its)}
        result["shapes"][label] = rec
        print(label, json.dumps({k: v for k, v in rec.items() if k not in ("host", "async")}),
              {r: (round(rec[r]["wall_median_s"] * 1e3, 2), round(rec[r]["blocked_median_s"] * 1e3, 3),
                   rec[r]["trials"], rec[r]["final_cost"], rec[r]["digest"]) for r in ("host", "async")}, flush=True)
        for s in solvers.values():
            s.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("device:", result["device"])


if __name__ == "__main__":
    main()
