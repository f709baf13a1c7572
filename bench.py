#!/usr/bin/env python
"""Benchmark of the PoVar hot path on B200: stratified two-step solve of a synthetic
venice-1778-shaped BAL problem (BASELINE.json, configs[3]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One "step" = one full stratified solve (step 1 pOSE PoVar + step 2 RIPOBA) of the workload.
  value  LM iterations/s of the whole job with the problem resident in HBM (state reset between steps)
  e2e    the same through the C ABI from HOST buffers: povar_create (index build + H2D upload),
         povar_bundle_adjust, povar_get_state (D2H), povar_destroy inside the timed region
  roofline      the dominant kernel of a power-series term, timed with CUDA events on the handle's stream
  cpu_baseline  the reference program compiled from its own sources (oracle/_ref/bal_ref), all host
                threads, on a bounded sample of the same workload (a few LM iterations per step)

--impl reference runs only that CPU arm and prints the same line shape with "impl": "reference".
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALPHA = 0.1
POWER_ITERS = 20
BAL_REF = os.path.join(ROOT, "oracle", "_ref", "bal_ref")

# reference-layout byte model of one power-series term (SURVEY.md 8d): dense [Jp|Jl] blocks
# streamed once + Hll^-1 + B^-1 + vectors


def ref_layout_bytes(nnz, L, C, joint=False):
    return (228 * nnz + 76 * L + 1232 * C) if joint else (484 * nnz + 76 * L + 1440 * C)


# bytes the matrix-free kernels have to move per launch (DESIGN.md "kernels"): index + observation
# streams, per-landmark records, per-camera vectors, each counted once
def own_bytes_landmark_pass(slots, slices, L, C):
    # sliced-ELL landmark half (k_sell_walk<E0LandmarkOp<pose>>), 32 landmarks per slice: camera index + uv per slot
    # (padding included: it is streamed), slice header (32 landmark ids + row pointer), per landmark the packed X
    # (32 B) and fold (6 x 8 B in step 1) read and H written (32 B), camera records once (176 B each; the blocks
    # stage them from L2)
    return 20 * slots + 132 * slices + (32 + 48 + 32) * L + 176 * C


def own_bytes_camera_pass(nnz, L, C, items):
    return 20 * nnz + 64 * L + 96 * C + 96 * items


def make_problem(workload):
    from povar_b200 import synthetic
    t = time.time()
    sp = synthetic.generate_named(workload)
    return sp, time.time() - t


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip().split(",")
                sm, smax = float(out[0]), float(out[1])
                self.samples.append((sm, smax))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                   out[2:6]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        return {"sm_mhz": statistics.median(s[0] for s in self.samples),
                "sm_max_mhz": max(s[1] for s in self.samples), "reasons": sorted(self.reasons)}


# ---------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own program on the host cores
# ---------------------------------------------------------------------------------------------
def run_reference_sample(path, threads, it1, it2, robust, workdir):
    log = os.path.join(workdir, "ba_log_ref.json")
    cmd = [BAL_REF, "--input", path, "--num-threads", str(threads), "--alpha", str(ALPHA),
           "--power-sc-iterations", str(POWER_ITERS), "--solver-type-step-1", "POWER_VARPROJ",
           "--solver-type-step-2", "RIPOBA", "--residual-robust-norm", robust,
           "--max-num-iterations-step-1", str(it1), "--max-num-iterations-step-2", str(it2),
           "--log-log-path", log]
    t = time.time()
    res = subprocess.run(cmd, capture_output=True, text=True, cwd=workdir)
    wall = time.time() - t
    if res.returncode != 0:
        raise RuntimeError("bal_ref failed: " + res.stderr[-1000:])
    with open(log) as f:
        data = json.load(f)
    optimize = data["_static"]["timing"]["optimize"]
    trials = len(data["iteration"])
    terms = sum(data["linear_solver_iterations"])
    t_series = sum(data["solve_reduced_system_time"])
    return {"optimize_s": optimize, "trials": trials, "power_terms": terms, "power_series_s": t_series,
            "wall_s": wall, "final_cost": data["cost"][-1], "load_s": data["_static"]["timing"]["load"]}


def reference_arm(args, sp, path, workdir):
    threads = os.cpu_count() or 1
    it1, it2 = args.ref_iters
    # warm-up runs would cost minutes on the CPU; one untimed tiny run checks the binary, then K samples
    steps = args.steps
    runs = [run_reference_sample(path, threads, it1, it2, args.robust, workdir) for _ in range(steps)]
    trials = sum(r["trials"] for r in runs)
    t = sum(r["optimize_s"] for r in runs)
    terms = sum(r["power_terms"] for r in runs)
    t_series = sum(r["power_series_s"] for r in runs)
    nnz, L, C = sp.num_obs, sp.num_lms, sp.num_cams
    value = trials / t
    sample = (f"bal_ref --num-threads {threads}, {it1}+{it2} LM iterations of the {args.workload} solve per step "
              f"(same data_custom file, same flags), {steps} step(s)")
    return {
        "value": value, "ms_per_step": 1e3 * t / steps, "cores": threads, "sample": sample,
        "sample_lm_iterations": [it1, it2], "sample_trials_logged": trials / steps,
        "sample_final_cost": runs[-1]["final_cost"],
        "spmv_ref_layout_gbs": (ref_layout_bytes(nnz, L, C) * terms / t_series / 1e9) if t_series > 0 else None,
        "s_per_power_term": (t_series / terms) if terms else None, "trials_per_step": trials / steps,
        "load_s": runs[0]["load_s"],
    }


DUMP_BYTES = 60_000_000      # payload of --dump-outputs: with the .npy headers, below 64 MB


def dump_outputs(out_dir, its, summ, P, X):
    """Write what a caller of the timed solve receives, one float64 .npy per output, so that two builds can be
    compared output for output on the same seeded problem: every field of the per-trial records (trial_<field>) and
    of the summary (summary_<field>) except the timings and the message, the final cameras [C, 3, 4] and landmarks
    [L, 4].  Landmarks beyond what fits in DUMP_BYTES are a fixed seeded sample of rows, listed in landmark_rows."""
    from povar_b200 import capi

    def fields(struct):
        return [f for f, _ in struct._fields_ if not f.endswith("_time") and f != "message"]

    out = {f"trial_{f}": np.array([getattr(e, f) for e in its], dtype=np.float64) for f in fields(capi.Iteration)}
    out.update({f"summary_{f}": np.float64(getattr(summ, f)) for f in fields(capi.SolveSummary)})
    out["cameras"] = np.asarray(P, dtype=np.float64)
    room = DUMP_BYTES - sum(np.asarray(a).nbytes for a in out.values())
    X = np.asarray(X, dtype=np.float64)
    if X.nbytes > room:
        rows = np.sort(np.random.default_rng(0).choice(X.shape[0], room // (X[0].nbytes + 8), replace=False))
        out["landmark_rows"] = rows.astype(np.float64)
        X = X[rows]
    out["landmarks"] = X
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="venice1778")
    ap.add_argument("--robust", default="CAUCHY")
    ap.add_argument("--ref-iters", type=int, nargs=2, default=[2, 2],
                    help="LM iterations of step 1 / step 2 in each CPU reference sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--max-iters", type=int, nargs=2, default=[50, 50])
    ap.add_argument("--trace-out", default=None,
                    help="write the logged trace of the last timed solve (cost, accept/reject, term counts) as json: "
                         "what runs at different GPU counts are compared by (tools/compare_traces.py)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last timed solve returned (per-trial records, summary, "
                         "final cameras and landmarks) as DIR/<name>.npy in float64, below 64 MB in all (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU solve returned: it needs --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")

    config = {"workload": f"synthetic {args.workload} shape, POWER_VARPROJ + RIPOBA, power-sc-iterations {POWER_ITERS}, "
                          f"alpha {ALPHA}, robust norm {args.robust}",
              "parallelism": f"landmark-sharded x{world}", "l2": "inputs larger than L2 (no flush needed)"}

    # ---------------- reference arm: rank 0 only, CPU only
    if args.impl == "reference":
        if rank != 0:
            return
        sp, _ = make_problem(args.workload)
        from povar_b200 import synthetic
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, f"{args.workload}.txt")
            synthetic.write_bal(sp, path)
            if not os.path.exists(BAL_REF):
                print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/bal_ref missing (run make -C oracle ref)"}))
                return
            r = reference_arm(args, sp, path, tmp)
        config.update({"cameras": sp.num_cams, "landmarks": sp.num_lms, "observations": sp.num_obs})
        line = {
            "impl": "reference", "metric": "lm_iterations_per_s", "value": r["value"], "unit": "LM iterations/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config,
            "cpu_baseline": {"value": r["value"], "unit": "LM iterations/s", "cores": r["cores"], "kind": "reference",
                             "sample": r["sample"], "sample_lm_iterations": r["sample_lm_iterations"],
                             "sample_trials_logged": r["sample_trials_logged"],
                             "full_workload": False, "spmv_ref_layout_gbs": r["spmv_ref_layout_gbs"],
                             "s_per_power_term": r["s_per_power_term"]},
            "e2e": {"value": r["value"], "unit": "LM iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return

    # ---------------- our arm
    import torch
    import torch.distributed as dist
    from povar_b200 import capi, synthetic

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    sp, t_gen = make_problem(args.workload)      # every rank generates the same seeded problem
    hp_full = capi.HostProblem.from_unordered(sp.num_cams, sp.num_lms, sp.obs_cam, sp.obs_lm, sp.obs_xy, sp.cam_params)
    hp = hp_full.shard(rank, world) if world > 1 else hp_full
    nnz, L, C = hp_full.num_obs, hp_full.num_lms, hp_full.num_cams
    config.update({"cameras": C, "landmarks": L, "observations": nnz})

    comm = None
    if world > 1:
        ids = [capi.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        comm = capi.make_comm(rank, world, local_rank, ids[0])

    opt = capi.default_options(alpha=ALPHA, power_sc_iterations=POWER_ITERS, verbosity_level=0,
                               robust_norm=capi.NORM_NAMES[args.robust],
                               max_num_iterations_step_1=args.max_iters[0],
                               max_num_iterations_step_2=args.max_iters[1])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- resident: one handle, state reset between steps
    solver = capi.Solver(hp, opt, comm)
    P0 = hp.cam_P.copy()
    series_exchange = ("none (1 GPU)" if world == 1 else
                       "peer-memory stores fused into the term kernel (CUDA IPC over NVLink)"
                       if solver.peer_exchange_active() else "ncclAllReduce per term")

    def resident_step():
        solver.set_state(capi.STATE_POSE, P0, None)
        return solver.bundle_adjust()

    for _ in range(args.warmup):
        its, summ = resident_step()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = solver.launch_count()
    # device clock: CUDA events on the stream the handle launches on (torch's current stream sees
    # none of it); the host LM loop between the launches is inside the bracket, as it must be
    hstream = torch.cuda.ExternalStream(solver.cuda_stream(), device=torch.device("cuda", local_rank))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.perf_counter()
    ev0.record(hstream)
    trials = 0
    terms = 0
    series_t = 0.0
    phase_keys = ("residual_evaluation_time", "jacobian_evaluation_time", "prepare_time",
                  "solve_reduced_system_time", "back_substitution_time", "iteration_time")
    phases = dict.fromkeys(phase_keys, 0.0)
    for _ in range(args.steps):
        its, summ = resident_step()
        trials += len(its)
        terms += summ.power_terms
        series_t += summ.power_series_time
        for e in its:
            for k in phase_keys:
                phases[k] += getattr(e, k)
    ev1.record(hstream)
    barrier()
    t_res_host = time.perf_counter() - t0
    t_res = reduce_max(ev0.elapsed_time(ev1) * 1e-3)
    launches = solver.launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs:
        # read now: the roofline runs below overwrite the handle's state
        P_out, X_out = solver.get_state(capi.STATE_JOINT)
        if world > 1:       # cameras are replicated, landmarks come back per shard in rank order
            shards = [None] * world
            dist.all_gather_object(shards, X_out)
            X_out = np.concatenate(shards)
    final_cost = its[-1].cost
    step1_trials = sum(1 for e in its if e.step == 1)
    # what the solve produced, so that runs at different GPU counts can be compared from their bench lines: the
    # sharded result may differ from the 1-GPU one by summation order only (SURVEY 8e)
    import hashlib
    solve_result = {
        "final_cost": summ.final_cost, "initial_cost": summ.initial_cost,
        "accepted_steps": int(summ.num_successful_steps), "rejected_steps": int(summ.num_unsuccessful_steps),
        "lm_trials": len(its), "step1_trials": step1_trials, "power_terms": int(summ.power_terms),
        "cost_first5": [e.cost for e in its[:5]],
        "cost_step2_first": next((e.cost for e in its if e.step == 2), None),
        # sha256 over the logged costs printed with 7 significant digits and the accept/reject and term-count
        # columns: equal across GPU counts unless a cost sits within ~1e-9 of a rounding boundary
        "trace_digest_7digits": hashlib.sha256(";".join(
            f"{e.cost:.6e},{int(e.step_is_successful)},{e.linear_solver_iterations}" for e in its).encode()).hexdigest()[:16],
    }

    # ---- roofline of the dominant kernel (CUDA events on the handle's stream)
    solver.set_state(capi.STATE_POSE, P0, None)
    solver.initialize_varproj_lm_pOSE(ALPHA)
    solver.linearize_pOSE(ALPHA)
    solver.solve(1e-4)
    ksec = solver.bench_power_kernels(capi.STATE_POSE, 20)
    ksec = solver.bench_power_kernels(capi.STATE_POSE, 50)
    term_s = solver.bench_power_terms(capi.STATE_POSE, 100)
    items = solver.debug_count("item_cam")
    slots, slices = solver.debug_count("sell_cam"), solver.debug_count("slice_ptr") - 1
    lnnz, lL = hp.num_obs, hp.num_lms
    own_a, own_b = own_bytes_landmark_pass(slots, slices, lL, C), own_bytes_camera_pass(lnnz, lL, C, items)
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    dom = 0 if ksec[0] >= ksec[1] else 1
    dom_bytes = own_a if dom == 0 else own_b
    dom_name = "k_sell_walk<E0LandmarkOp<pose>>" if dom == 0 else "k_passB_e0_v2<pose>"
    traffic = None
    tj = {}
    try:   # measured DRAM bytes per launch of that kernel (one ncu --set full capture, committed)
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f).get(args.workload, {})
        if tj.get("n_gpus") == world:
            traffic = tj.get(dom_name)
    except Exception:
        pass
    achieved = dom_bytes / ksec[dom] / 1e9
    roofline = {
        "bound": "hbm", "kernel": dom_name,
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650 GB/s",
        "traffic": traffic,
        "traffic_source": ("profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full "
                           "--cache-control none capture of this kernel on this workload (static, not re-measured in "
                           "this run; L2 as the previous launch left it -- with ncu's default flush before every "
                           "pass: traffic_cold_l2)"
                           if traffic is not None else None),
        "traffic_cold_l2": tj.get(dom_name + "_cold_l2") if traffic is not None else None,
        "series_exchange": series_exchange,
        "solve_result": solve_result,
        "bytes_per_launch": dom_bytes, "kernel_us": 1e6 * ksec[dom],
        "term_kernels_us": {"landmark_pass": 1e6 * ksec[0], "camera_pass": 1e6 * ksec[1],
                            "item_reduce_multi_gpu_only": 1e6 * ksec[2], "binv_norms_test": 1e6 * ksec[3]},
        "sell_slots": slots, "sell_slots_per_observation": slots / max(lnnz, 1),   # < 1: long landmarks stay in CSR

        "term_us": 1e6 * term_s,
        "term_own_bytes": own_a + own_b,
        "term_own_gbs": (own_a + own_b) / term_s / 1e9,
        # the reference streams dense blocks: same work expressed in its byte model (SURVEY 8d), per rank
        "term_ref_layout_bytes": ref_layout_bytes(lnnz, lL, C),
        "term_ref_layout_equiv_gbs": ref_layout_bytes(lnnz, lL, C) / term_s / 1e9,
        "note": "matrix-free kernels: Jacobian blocks are recomputed in registers, so a term moves ~6x fewer "
                "bytes than the reference layout; frac is against the bytes THIS layout must move",
    }
    solver.close()
    if args.trace_out and rank == 0:
        with open(args.trace_out, "w") as f:
            json.dump({"workload": args.workload, "n_gpus": world, "max_iters": args.max_iters,
                       "step": [e.step for e in its], "iteration": [e.iteration for e in its],
                       "cost": [e.cost for e in its], "step_is_successful": [int(e.step_is_successful) for e in its],
                       "linear_solver_iterations": [e.linear_solver_iterations for e in its],
                       "trust_region_radius": [e.trust_region_radius for e in its]}, f)

    # ---- end to end from host buffers: create (H2D) + solve + read back (D2H) + destroy
    # inputs are page-locked once, outside the timed region (the contract: H2D from pinned host memory);
    # every per-observation index array is built on the device from the canonical list, so the upload
    # is that list plus the small host-built tables
    pinned = []
    rt = torch.cuda.cudart()
    # the result is read back into the caller's own (page-locked) buffers, as a host application would keep them
    out_P, out_X = np.zeros((hp.num_cams, 3, 4)), np.zeros((hp.num_lms, 4))
    for arr in (hp.lm_ptr, hp.obs_cam, hp.obs_uv, hp.cam_P, out_P, out_X):
        if int(rt.cudaHostRegister(arr.ctypes.data, arr.nbytes, 0)) == 0:
            pinned.append(arr)
    h2d = (hp.lm_ptr.nbytes // 2 + hp.obs_cam.nbytes + hp.obs_uv.nbytes + hp.cam_P.nbytes)
    d2h = hp.cam_P.nbytes + hp.num_lms * 4 * 8

    # host phases of a step and the link it crosses, for the record: end-to-end differs from the resident number by
    # povar_create (H2D + index build), the read-back and the destruction of the handle, which depend on the host
    # (one build measured 118 to 420 ms per step on different boxes; cudaHostAlloc / cudaFreeHost of the handle's
    # scratch, 130 ms in one trace, were a cause and are gone: DESIGN.md 6)
    e2e_phases = {"create": 0.0, "solve": 0.0, "read_back": 0.0, "destroy": 0.0}

    def e2e_step(timed=True):
        t_a = time.perf_counter()
        s = capi.Solver(hp, opt, comm)
        t_b = time.perf_counter()
        its_, summ_ = s.bundle_adjust()
        t_c = time.perf_counter()
        s.get_state(capi.STATE_JOINT, out=(out_P, out_X))
        t_d = time.perf_counter()
        s.close()
        t_e = time.perf_counter()
        if timed:
            for k, v in zip(e2e_phases, (t_b - t_a, t_c - t_b, t_d - t_c, t_e - t_d)):
                e2e_phases[k] += v
        return len(its_)

    def link_gbs():
        n = 64 << 20
        hbuf = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        dbuf = torch.empty(n, dtype=torch.uint8, device="cuda")
        a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        dbuf.copy_(hbuf, non_blocking=True)
        a.record()
        dbuf.copy_(hbuf, non_blocking=True)
        b.record()
        hbuf.copy_(dbuf, non_blocking=True)
        c.record()
        torch.cuda.synchronize()
        return {"h2d": n / (a.elapsed_time(b) * 1e-3) / 1e9, "d2h": n / (b.elapsed_time(c) * 1e-3) / 1e9}

    link = link_gbs()
    e2e_step(timed=False)
    # every step makes (and destroys) its own handle and stream and ends with a blocking read-back, so
    # the bracket is two events on torch's stream: device timestamps taken while nothing is in flight
    ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.perf_counter()
    ee0.record()
    e2e_trials = 0
    for _ in range(args.steps):
        e2e_trials += e2e_step()
    ee1.record()
    barrier()
    t_e2e_host = time.perf_counter() - t0
    t_e2e = reduce_max(ee0.elapsed_time(ee1) * 1e-3)
    for arr in pinned:
        rt.cudaHostUnregister(arr.ctypes.data)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, its, summ, P_out, X_out)

    # ---- CPU baseline on a bounded sample (rank 0, N == 1 only)
    cpu = None
    if world == 1 and not args.no_cpu_baseline and os.path.exists(BAL_REF):
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, f"{args.workload}.txt")
            synthetic.write_bal(sp, path)
            sub = argparse.Namespace(**vars(args))
            sub.steps = 1
            r = reference_arm(sub, sp, path, tmp)
        cpu = {"value": r["value"], "unit": "LM iterations/s", "cores": r["cores"], "kind": "reference",
               "sample": r["sample"], "sample_lm_iterations": r["sample_lm_iterations"],
               "sample_trials_logged": r["sample_trials_logged"], "full_workload": False,
               "ms_per_lm_iteration": 1e3 / r["value"],
               "spmv_ref_layout_gbs": r["spmv_ref_layout_gbs"], "s_per_power_term": r["s_per_power_term"],
               "load_s": r["load_s"]}

    line = {
        "metric": "lm_iterations_per_s", "value": trials / t_res, "unit": "LM iterations/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_res / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config,
        "solve_s": t_res / args.steps, "lm_iterations_per_solve": trials / args.steps,
        "step1_lm_iterations": step1_trials, "final_cost": final_cost,
        "power_terms_per_solve": terms / args.steps,
        "power_series_ms_per_term": 1e3 * series_t / max(terms, 1),
        # device time of the phases of a solve (CUDA events inside the library, rank 0), like the reference's log
        "phase_ms_per_solve": {k.replace("_time", ""): 1e3 * v / args.steps for k, v in phases.items()},
        "e2e": {"value": e2e_trials / t_e2e, "unit": "LM iterations/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h), "solve_s": t_e2e / args.steps,
                "host_phase_ms_per_step": {k: 1e3 * v / args.steps for k, v in e2e_phases.items()},
                "pinned_copy_gbs_measured": link},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "timing": "CUDA events on the handle's stream (value) / on torch's stream around blocking calls (e2e), "
                  "max over ranks; host perf_counter beside them",
        "host_clock_s": {"resident": t_res_host, "e2e": t_e2e_host},
        "setup_s": {"generate": t_gen},
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    # stdout carries ONE JSON line: libraries that print there while they initialise (NCCL's version banner) go to
    # stderr -- at the file-descriptor level, their writes do not pass through sys.stdout
    sys.stdout.flush()
    _real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(_real_stdout, "w")
    main()
    sys.stdout.flush()
