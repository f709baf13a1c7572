#!/usr/bin/env python
"""Handle creation from an unordered observation list that lives on the GPU: the host route against
povar_create_device.

    python tools/time_device_create.py --out profiles/device_create_b200.json [--reps 5]

Input: the venice-1778 shape (synthetic.generate_named, seed 1005) with its observations shuffled by a fixed seed,
as torch CUDA tensors.  Routes, alternated, median of --reps each (host clock, every route ends synchronised):
  host     the lists copied to the host, povar_canonical_order, the gather of cameras and image coordinates, then
           povar_create (which uploads them again)
  device   povar_create_device on the tensors (canonical order and index made on the GPU)
and the state read back: get_state into host memory against get_state_device into CUDA tensors (plus a synchronise).
Then one capped two-step solve on a handle of each route; the final cost and a digest of the trace must agree.
Device name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
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

SHUFFLE_SEED = 17


def device_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def host_route(dp, prob, opt):
    """lists down, canonical order on the host, povar_create"""
    import torch
    cam = dp.obs_cam.cpu().numpy()
    lm = dp.obs_lm.cpu().numpy()
    uv = dp.obs_uv.cpu().numpy()
    P = dp.cam_P.cpu().numpy()
    n = cam.shape[0]
    perm = np.empty(n, dtype=np.int64)
    lm_ptr = np.empty(prob.num_lms + 1, dtype=np.int64)
    rc = capi.load().povar_canonical_order(prob.num_cams, prob.num_lms, n, cam.ctypes.data_as(C.POINTER(C.c_int32)),
                                           lm.ctypes.data_as(C.POINTER(C.c_int32)),
                                           perm.ctypes.data_as(C.POINTER(C.c_int64)),
                                           lm_ptr.ctypes.data_as(C.POINTER(C.c_int64)))
    assert rc == capi.OK
    hp = capi.HostProblem(prob.num_cams, prob.num_lms, lm_ptr, cam[perm], uv[perm], P)
    torch.cuda.synchronize()
    return capi.Solver(hp, opt)


def digest(its):
    h = hashlib.sha256()
    for e in its:
        h.update(np.array([e.cost], dtype=np.float64).tobytes())
        h.update(np.array([e.step_is_successful, e.linear_solver_iterations], dtype=np.int64).tobytes())
    return h.hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/device_create_b200.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--shape", default="venice1778")
    ap.add_argument("--iterations", type=int, default=3, help="LM trials per step of the closing solve")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("time_device_create: needs a CUDA device")
    dev_info = device_info()
    prob = synthetic.generate_named(a.shape)
    order = np.random.default_rng(SHUFFLE_SEED).permutation(prob.num_obs)
    uv = prob.obs_xy[order].copy()
    uv[:, 1] = -uv[:, 1]
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    dp = capi.DeviceProblem(t(prob.cam_params[:, :12]), t(prob.obs_cam[order]), t(prob.obs_lm[order]), t(uv),
                            num_lms=prob.num_lms)
    opt = capi.default_options(verbosity_level=0, max_num_iterations_step_1=a.iterations,
                               max_num_iterations_step_2=a.iterations)
    torch.cuda.synchronize()

    def time_create(route):
        t0 = time.perf_counter()
        s = host_route(dp, prob, opt) if route == "host" else capi.Solver(dp, opt)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        s.close()
        return dt

    for route in ("host", "device"):   # warm-up: module loading, pools, cub's first launches
        time_create(route)
    create = {"host": [], "device": []}
    for _ in range(a.reps):
        for route in ("host", "device"):
            create[route].append(time_create(route))

    s = capi.Solver(dp, opt)
    state = {"host": [], "device": []}
    P_h = np.empty((prob.num_cams, 3, 4))
    X_h = np.empty((prob.num_lms, 3))
    for _ in range(a.reps + 1):
        t0 = time.perf_counter()
        s.get_state(capi.STATE_POSE, out=(P_h, X_h))
        state["host"].append(time.perf_counter() - t0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        P_d, X_d = s.get_state_device(capi.STATE_POSE)
        torch.cuda.synchronize()
        state["device"].append(time.perf_counter() - t0)
    for k in state:
        state[k] = state[k][1:]   # the first pair warms up
    assert np.array_equal(P_d.cpu().numpy(), P_h) and np.array_equal(X_d.cpu().numpy(), X_h)
    s.close()

    runs = {}
    for route in ("host", "device"):
        s = host_route(dp, prob, opt) if route == "host" else capi.Solver(dp, opt)
        its, summary = s.bundle_adjust()
        runs[route] = {"final_cost": summary.final_cost, "trials": len(its), "digest": digest(its)}
        s.close()
    assert runs["host"] == runs["device"], runs

    med = lambda v: float(np.median(v))
    res = {
        "device": dev_info,
        "shape": {"name": a.shape, "cameras": prob.num_cams, "landmarks": prob.num_lms, "observations": prob.num_obs,
                  "shuffle_seed": SHUFFLE_SEED},
        "reps": a.reps,
        "create_ms": {k: {"median": 1e3 * med(v), "all": [1e3 * x for x in v]} for k, v in create.items()},
        "get_state_pose_ms": {k: {"median": 1e3 * med(v), "all": [1e3 * x for x in v]} for k, v in state.items()},
        "solve_check": runs,
    }
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("device", "create_ms", "get_state_pose_ms")}, indent=1))


if __name__ == "__main__":
    main()
