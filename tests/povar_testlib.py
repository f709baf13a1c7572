"""Shared helpers of the test-suite: golden fixtures, problem construction for both sides."""
from __future__ import annotations

import atexit
import hashlib
import json
import os
import shutil
import tempfile

import numpy as np

from oracle import povar_oracle as O
from povar_b200 import capi, synthetic

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

_traces = None
_files = {}
_regen_dir = None


def _private_tmp() -> str:
    """Directory of this test process for regenerated problem files: a fixed name in the shared temp directory
    can belong to another user (or to a concurrent run) and then cannot be rewritten."""
    global _regen_dir
    if _regen_dir is None:
        _regen_dir = tempfile.mkdtemp(prefix="povar_golden_")
        atexit.register(shutil.rmtree, _regen_dir, True)
    return _regen_dir


def traces():
    global _traces
    if _traces is None:
        with open(os.path.join(GOLD, "traces.json")) as f:
            _traces = json.load(f)
    return _traces


_traces_large = None


def traces_large():
    """Traces of the reference on BASELINE.json's larger configurations (tools/make_golden_large.py)."""
    global _traces_large
    if _traces_large is None:
        with open(os.path.join(GOLD, "traces_large.json")) as f:
            _traces_large = json.load(f)
    return _traces_large


def golden_file(shape: str) -> str:
    """Path of the data_custom file of a golden shape.  Small ones are committed; larger ones are
    regenerated from the seeded generator and checked against the recorded sha256."""
    if shape in _files:
        return _files[shape]
    files = traces()["files"]
    meta = files[shape] if shape in files else traces_large()["files"][shape]
    if meta["committed"]:
        path = os.path.join(GOLD, f"{shape}.txt")
    else:
        path = os.path.join(_private_tmp(), f"{shape}.txt")
        synthetic.write_bal(synthetic.generate_named(shape), path)
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 20), b""):
            h.update(blk)
    assert h.hexdigest() == meta["sha256"], f"{shape}: regenerated file differs from the golden one"
    _files[shape] = path
    return path


def write_bal9(path, sp, rng):
    """A BAL file (9 parameters per camera) of a synthetic problem, the input of --create-dataset; returns the cameras."""
    with open(path, "w") as f:
        f.write(f"{sp.num_cams} {sp.num_lms} {sp.num_obs}\n")
        for c, l, (x, y) in zip(sp.obs_cam, sp.obs_lm, sp.obs_xy):
            f.write(f"{c} {l}     {x:.10e} {y:.10e}\n")
        cams = rng.normal(size=(sp.num_cams, 9))
        cams[:, 6] = 1000.0 + rng.normal(size=sp.num_cams)
        cams[:, 7:] *= 1e-7
        for v in cams.reshape(-1):
            f.write(f"{v:.16e}\n")
        for v in sp.points.reshape(-1):
            f.write(f"{v:.16e}\n")
    return cams


def create_dataset_lines(text, num_obs, num_cams):
    """Lines of a --create-dataset output without a trailing empty one, the random camera-matrix entries (the first 8
    of each camera's 15 lines) as None: what two programs writing the same input must agree on."""
    lines = text.split("\n")
    if lines and lines[-1] == "":
        lines.pop()
    first_cam = 1 + num_obs
    return [None if 0 <= i - first_cam < 15 * num_cams and (i - first_cam) % 15 < 8 else s
            for i, s in enumerate(lines)]


def flags_to_options(flags):
    """reference CLI flags of a golden config -> keyword options shared by both sides"""
    kw = dict(alpha=0.1, power_sc_iterations=20)
    it = iter(flags)
    for k in it:
        v = next(it)
        if k == "--solver-type-step-1":
            kw["solver_type_step_1"] = capi.STEP1_NAMES[v]
        elif k == "--solver-type-step-2":
            kw["solver_type_step_2"] = capi.STEP2_NAMES[v]
        elif k == "--residual-robust-norm":
            kw["robust_norm"] = capi.NORM_NAMES[v]
        elif k == "--residual-huber-parameter":
            kw["huber_parameter"] = float(v)
        elif k == "--power-sc-iterations":
            kw["power_sc_iterations"] = int(v)
        elif k == "--alpha":
            kw["alpha"] = float(v)
        elif k == "--optimized-cost":
            kw["optimized_cost"] = {"ERROR": 0, "ERROR_VALID": 1, "ERROR_VALID_AVG": 2}[v]
        elif k == "--max-num-iterations-step-1":
            kw["max_num_iterations_step_1"] = int(v)
        elif k == "--max-num-iterations-step-2":
            kw["max_num_iterations_step_2"] = int(v)
        else:
            raise KeyError(k)
    return kw


def oracle_options(kw):
    return O.Options(**kw)


def step2_start(iteration):
    for i in range(1, len(iteration)):
        if iteration[i] == 0:
            return i
    return len(iteration)


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    den = max(float(np.max(np.abs(b))), 1e-300)
    return float(np.max(np.abs(a - b))) / den


def assert_trace_close(meta, costs, successful, lin_its, label=""):
    """Compare a two-step trace with the reference's golden one (`bal_ref --num-threads 1`).

    Tolerances follow BASELINE.json's north_star -- 1e-9 relative on the cost of every step-1
    trial and of the first trials of step 2, 1e-6 afterwards, identical accept/reject decisions
    and linear-solver iteration counts -- EXCEPT where the reference does not agree with itself:
    its 8-thread run (different scatter order, SURVEY F10) is stored next to the 1-thread run,
    and once the two have drifted apart by d the comparison allows 50*d (late in step 2 the
    iteration is chaotic: 1e-16 perturbations grow to 1e-6 and even change the trial count).
    Returns the worst relative cost deviation seen.
    """
    ref, ref8 = meta["threads1"], meta["threads8"]
    k2 = step2_start(ref["iteration"])
    n8 = len(ref8["cost"])
    drift = 0.0
    worst = 0.0
    stable = True
    n = min(len(costs), len(ref["cost"]))
    for i in range(n):
        if i < n8:
            drift = max(drift, abs(ref["cost"][i] - ref8["cost"][i]) / abs(ref["cost"][i]))
            if ref8["step_is_successful"][i] != ref["step_is_successful"][i]:
                drift = max(drift, 1.0)
        else:
            drift = max(drift, 1.0)
        if drift > 1e-10:
            stable = False
        base = 1e-9 if i < k2 + 6 else 1e-6
        tol = max(base, 50.0 * drift)
        dev = abs(costs[i] - ref["cost"][i]) / abs(ref["cost"][i])
        worst = max(worst, dev if tol < 1.0 else 0.0)
        assert dev <= tol, f"{label} trial {i}: cost {costs[i]!r} vs reference {ref['cost'][i]!r} (rel {dev:.2e} > {tol:.1e})"
        if stable:
            assert bool(successful[i]) == bool(ref["step_is_successful"][i]), f"{label} trial {i}: accept/reject differs"
            assert int(lin_its[i]) == int(ref["linear_solver_iterations"][i]), \
                f"{label} trial {i}: linear solver iterations {lin_its[i]} vs {ref['linear_solver_iterations'][i]}"
    if stable:
        assert len(costs) == len(ref["cost"]), f"{label}: {len(costs)} trials vs {len(ref['cost'])}"
    return worst
