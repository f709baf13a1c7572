#!/usr/bin/env python
"""Per-trial time of the CHOLESKY step-1 solve, dense against tile-sparse storage of the reduced camera system.

    python tools/time_cholesky.py --out profiles/cholesky_tiles.json [--reps 3] [--scaled10k]

  venice1778   dense (automatic) and tile-sparse (forced) handles, solves alternating between them
  scene10k     generate(10000, 200000, 1_000_000, seed=77, window_frac=0.005): 115 GB dense, so tile-sparse only
  scaled10k    (--scaled10k) one tile-sparse solve of bench.py's 10,000-camera shape (25 % window)

Per solve, from povar_get_timings: prepare (Hll^-1, B, b and the assembly of S; the first tile-sparse solve of a
handle also builds the co-visibility bitmap, the order and the symbolic factorisation) and reduced solve (LL^T and
both substitutions); kernel launches from povar_launch_count.  Memory: bytes of S / L (dense matrix or stored tiles)
plus the inverted diagonal tiles.  FP64 tensor-core FLOPs of the factorisation are counted off the tile pattern (the
symbolic factorisation is redone here in numpy from the library's camera order): 2 * 64^3 per panel tile and per
update tile.  The host time of the ordering and symbolic step is timed through povar_debug_cholesky_symbolic (which
also builds the bitmap on the host).  Device name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from povar_b200 import capi, synthetic  # noqa: E402

TILE = 64
LAM = 1e-2


def device_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def column_counts(hp, perm):
    """stored tiles below the diagonal of every tile column, from the camera order (the library's rule)"""
    T = -(-12 * hp.num_cams // TILE)
    P = np.eye(T, dtype=bool)
    pos = perm.astype(np.int64)[hp.obs_cam.astype(np.int64)]
    deg = np.diff(hp.lm_ptr)
    d_obs = np.repeat(deg, deg)                      # degree of the landmark of every observation
    start_obs = np.repeat(hp.lm_ptr[:-1], deg)
    step = 1 << 22
    for o0 in range(0, hp.num_obs, step):            # every ordered pair of observations of one landmark
        o1 = min(hp.num_obs, o0 + step)
        d = d_obs[o0:o1]
        i = np.repeat(np.arange(o0, o1), d)
        j = np.repeat(start_obs[o0:o1], d) + np.arange(i.size) - np.repeat(np.cumsum(d) - d, d)
        for ea in (0, 11):
            for eb in (0, 11):
                I = (12 * pos[i] + ea) // TILE
                J = (12 * pos[j] + eb) // TILE
                P[np.maximum(I, J), np.minimum(I, J)] = True
    for c in range(hp.num_cams):
        t0, t1 = 12 * int(perm[c]) // TILE, (12 * int(perm[c]) + 11) // TILE
        P[t1, t0] = True
    for k in range(T):
        rows = np.nonzero(P[k + 1:, k])[0] + k + 1
        if rows.size:
            P[np.ix_(rows, rows)] |= np.tril(np.ones((rows.size, rows.size), dtype=bool))
    return P.sum(axis=0) - 1


def factor_flops(m):
    m = m.astype(np.float64)
    return float(np.sum(2.0 * TILE ** 3 * (m + m * (m + 1) / 2)))


def make_solver(hp, storage):
    s = capi.Solver(hp, capi.default_options(alpha=0.1, solver_type_step_1=capi.CHOLESKY, verbosity_level=0))
    s.debug_set_cholesky_storage(storage)
    s.initialize_varproj_lm_pOSE(0.1)
    assert s.linearize_pOSE(0.1) == capi.OK
    return s


def timed_solve(s):
    s.reset_timings()
    l0 = s.launch_count()
    inc, _, rc = s.solve(LAM)
    t = s.timings()
    assert rc == capi.OK and np.all(np.isfinite(inc))
    return {"prepare_s": t.prepare_time, "reduced_solve_s": t.solve_reduced_system_time,
            "launches": s.launch_count() - l0}, inc


def summarize(runs):
    return {k: float(np.median([r[k] for r in runs])) for k in runs[0]}


def storage_bytes(hp, s, dense):
    n_pad = -(-12 * hp.num_cams // TILE) * TILE
    linv = n_pad * TILE * 8
    if dense:
        return {"S_L_bytes": n_pad * n_pad * 8, "linv_bytes": linv}
    return {"S_L_bytes": int(s.debug_read("chol_tiles")[0]) * TILE * TILE * 8, "linv_bytes": linv}


def scene(name, hp, reps, with_dense, out):
    print(f"[{name}] {hp.num_cams} cameras, {hp.num_obs} observations", flush=True)
    t0 = time.perf_counter()
    perm, tiles = capi.cholesky_symbolic(hp)
    symbolic_host_s = time.perf_counter() - t0
    T = -(-12 * hp.num_cams // TILE)
    m = column_counts(hp, perm)
    assert int(m.sum() + T) == tiles, (int(m.sum() + T), tiles)
    flops = factor_flops(m)
    res = {"cameras": hp.num_cams, "observations": hp.num_obs, "tiles_T": T, "stored_tiles": int(tiles),
           "lower_tiles": T * (T + 1) // 2, "symbolic_host_s_incl_host_bitmap": symbolic_host_s,
           "factor_flops_tiles": flops}
    handles = {}
    if with_dense:
        handles["dense"] = make_solver(hp, 0)
        res["factor_flops_dense"] = factor_flops(np.arange(T - 1, -1, -1))
    handles["tiles"] = make_solver(hp, 1)
    first = {}
    incs = {}
    for k, s in handles.items():
        first[k], incs[k] = timed_solve(s)   # warm-up; the tile-sparse one builds its pattern here
    res["first_solve"] = first
    runs = {k: [] for k in handles}
    for _ in range(reps):
        for k, s in handles.items():
            r, incs[k] = timed_solve(s)
            runs[k].append(r)
    for k, s in handles.items():
        res[k] = dict(summarize(runs[k]), **storage_bytes(hp, s, k == "dense"), runs=runs[k])
        res[k]["factor_tflops_per_s_incl_substitution"] = (res["factor_flops_dense" if k == "dense" else "factor_flops_tiles"] /
                                               res[k]["reduced_solve_s"] / 1e12)
    if with_dense:
        res["rel_diff_tiles_vs_dense"] = float(np.linalg.norm(incs["tiles"] - incs["dense"]) /
                                               np.linalg.norm(incs["dense"]))
    res["one_time_setup_s"] = first["tiles"]["prepare_s"] - res["tiles"]["prepare_s"]
    for s in handles.values():
        s.close()
    out[name] = res
    print(json.dumps({k: v for k, v in res.items() if k not in ("dense", "tiles")}, indent=1), flush=True)
    for k in handles:
        print(k, json.dumps({a: b for a, b in res[k].items() if a != "runs"}), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scaled10k", action="store_true")
    ap.add_argument("--skip", default="", help="comma-separated scenes to leave out")
    a = ap.parse_args()
    out = {"device": device_info(), "lambda": LAM, "alpha": 0.1}
    print(out["device"], flush=True)
    skip = set(a.skip.split(","))

    def hp_of(sp):
        return capi.HostProblem.from_unordered(sp.num_cams, sp.num_lms, sp.obs_cam, sp.obs_lm, sp.obs_xy,
                                               sp.cam_params)

    if "venice1778" not in skip:
        scene("venice1778", hp_of(synthetic.generate_named("venice1778")), a.reps, True, out)
    if "scene10k" not in skip:
        scene("scene10k", hp_of(synthetic.generate(10000, 200000, 1_000_000, seed=77, window_frac=0.005)), a.reps,
              False, out)
    if a.scaled10k:
        scene("scaled10k", hp_of(synthetic.generate_named("scaled10k")), 1, False, out)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
