"""Generate the golden fixtures under tests/golden/ from the reference itself.

Runs HERE (needs /root/reference compiled by `make -C oracle ref`); the fixtures are committed so
that the GPU box, which has no /root/reference, can check against them.

  tests/golden/kernel_cod.npz      row vectors and the kernels returned by the reference's own
                                   BalBundleAdjustmentHelper::kernel_COD (oracle/cod_probe.cpp)
  tests/golden/index.npz           what the reference itself holds after loading a data_custom file: pose_idx_
                                   of every LandmarkBlockSC (sc/landmark_block.hpp:104-108), the observation
                                   stored for each (landmark, camera) pair and the camera matrices
                                   (oracle/index_probe.cpp), for tiny / small and shuffled copies of them
  tests/golden/<shape>.txt         data_custom-format problem files (povar_b200.synthetic), small ones only
  tests/golden/traces.json         per-configuration ba_log.json columns of `bal_ref --num-threads 1`
                                   (cost, step_is_successful, trust_region_radius,
                                   linear_solver_iterations, iteration) plus the same run with 8 threads:
                                   the reference is not bit-reproducible across thread counts (SURVEY
                                   F10), and its own 1-vs-8-thread deviation is the yardstick for how
                                   far a re-implementation can be expected to agree late in step 2.
  tests/golden/create_dataset_small.json   what `--create-dataset` writes for the seeded BAL file of
                                   tests/test_host_abi.py, the random camera-matrix entries masked
  tests/golden/dump_config.json    what `--dump-config --input x` prints (every default)
                                   These two come from the reference program where it is built, otherwise from this
                                   project's bal; their "source" says which.
"""
from __future__ import annotations

import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from povar_b200 import synthetic  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
BAL_REF = os.path.join(ROOT, "oracle", "_ref", "bal_ref")
COD_PROBE = os.path.join(ROOT, "oracle", "_ref", "cod_probe")
INDEX_PROBE = os.path.join(ROOT, "oracle", "_ref", "index_probe")
BAL_OURS = os.path.join(ROOT, "povar_b200", "bin", "bal")

# (name, shape, extra reference flags).  --alpha / --power-sc-iterations are always explicit (SURVEY F3).
CONFIGS = [
    ("tiny_povar", "tiny", []),
    ("small_povar", "small", []),
    ("small_poba", "small", ["--solver-type-step-1", "POWER_SCHUR_COMPLEMENT"]),
    ("small_pcg_ripcg", "small", ["--solver-type-step-1", "PCG", "--solver-type-step-2", "RIPCG"]),
    ("small_cholesky", "small", ["--solver-type-step-1", "CHOLESKY"]),
    ("small_cauchy", "small", ["--residual-robust-norm", "CAUCHY"]),
    ("small_huber", "small", ["--residual-robust-norm", "HUBER", "--residual-huber-parameter", "30"]),
    ("small_m5", "small", ["--power-sc-iterations", "5"]),
    ("ladybug49_povar", "ladybug49", []),
    ("ladybug49_poba", "ladybug49", ["--solver-type-step-1", "POWER_SCHUR_COMPLEMENT"]),
    ("ladybug49_pcg_ripcg", "ladybug49", ["--solver-type-step-1", "PCG", "--solver-type-step-2", "RIPCG"]),
    ("ladybug49_cauchy", "ladybug49", ["--residual-robust-norm", "CAUCHY"]),
    # --optimized-cost (bal/solver_options.hpp:48-57, solver/bal_bundle_adjustment.cpp:163-205): the accept test,
    # rho (ERROR_VALID_AVG divides l_diff by the valid count) and the function-tolerance test use the valid sums
    ("small_error_valid", "small", ["--optimized-cost", "ERROR_VALID"]),
    ("small_error_valid_avg", "small", ["--optimized-cost", "ERROR_VALID_AVG"]),
    ("ladybug49_error_valid_avg", "ladybug49", ["--optimized-cost", "ERROR_VALID_AVG"]),
]
COMMITTED_FILES = {"tiny", "small"}
KEYS = ["iteration", "cost", "cost_valid", "num_obs_valid", "step_is_valid", "step_is_successful",
        "trust_region_radius", "linear_solver_iterations", "relative_decrease"]


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 20), b""):
            h.update(blk)
    return h.hexdigest()


def run_ref(path, flags, threads, workdir):
    log = os.path.join(workdir, "ba_log.json")
    # the reference's CLI rejects a repeated flag, so per-config flags replace the base ones
    merged = {"--alpha": "0.1", "--power-sc-iterations": "20"}
    merged.update(dict(zip(flags[0::2], flags[1::2])))
    cmd = [BAL_REF, "--input", path, "--num-threads", str(threads)]
    for k, v in merged.items():
        cmd += [k, v]
    cmd += ["--log-log-path", log]
    res = subprocess.run(cmd, capture_output=True, text=True, cwd=workdir)
    if res.returncode != 0:
        raise RuntimeError(f"bal_ref failed: {' '.join(cmd)}\n{res.stderr[-2000:]}")
    with open(log) as f:
        data = json.load(f)
    out = {k: data[k] for k in KEYS}
    out["termination_type"] = data["_static"]["solver"]["termination_type"]
    out["num_successful_steps"] = data["_static"]["solver"]["num_successful_steps"]
    return out


def make_kernel_cod():
    rng = np.random.default_rng(42)
    out = {}
    for n in (4, 12):
        vecs = rng.normal(size=(200, n))
        vecs[0] = 0.0
        vecs[0, n - 1] = 1.0                       # axis-aligned: zero tail after pivoting
        vecs[1] = 1.0                              # ties: first maximum wins
        vecs[2] = -np.arange(1, n + 1)             # negative pivot
        vecs[3, :] = 0.0
        vecs[3, 0] = -2.0
        vecs[4] = np.abs(vecs[4])
        vecs[5, 1], vecs[5, 2] = 7.0, -7.0        # |tie| with opposite signs
        text = f"{n} {vecs.shape[0]}\n" + "\n".join(" ".join("%.17g" % v for v in row) for row in vecs) + "\n"
        res = subprocess.run([COD_PROBE], input=text, capture_output=True, text=True, check=True)
        tok = res.stdout.split()
        kern = np.empty((vecs.shape[0], n, n - 1))
        p = 0
        for t in range(vecs.shape[0]):
            r, c = int(tok[p]), int(tok[p + 1])
            assert (r, c) == (n, n - 1), (r, c)
            p += 2
            kern[t] = np.array(tok[p:p + r * c], dtype=np.float64).reshape(r, c)
            p += r * c
        out[f"vec{n}"] = vecs
        out[f"kernel{n}"] = kern
    np.savez_compressed(os.path.join(GOLD, "kernel_cod.npz"), **out)
    print("kernel_cod.npz written")


def run_index_probe(path):
    """degrees [L], cameras [N], uv [N, 2], P [C, 12] exactly as the reference's own structures hold them"""
    res = subprocess.run([INDEX_PROBE, path], capture_output=True, text=True, check=True)
    lines = res.stdout.split("\n")
    C, L, N = (int(v) for v in lines[0].split())
    deg = np.empty(L, dtype=np.int32)
    cams = np.empty(N, dtype=np.int32)
    p = 0
    for l in range(L):
        tok = lines[1 + l].split()
        deg[l] = int(tok[0])
        cams[p:p + deg[l]] = [int(t) for t in tok[1:]]
        p += deg[l]
    assert p == N
    uv = np.array([[float(t) for t in lines[1 + L + i].split()] for i in range(N)], dtype=np.float64).reshape(N, 2)
    P = np.array([[float(t) for t in lines[1 + L + N + c].split()] for c in range(C)], dtype=np.float64)
    return deg, cams, uv, P


def make_index_fixture():
    """tests/golden/index.npz: the reference's own pose_idx_ / Landmark::obs for committed and shuffled files."""
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for shape, shuffle in (("tiny", None), ("tiny", 3), ("small", None), ("small", 11), ("ladybug49", 5)):
            prob = synthetic.generate_named(shape)
            path = os.path.join(tmp, "p.txt")
            synthetic.write_bal(prob, path, shuffle_seed=shuffle)
            if shuffle is None:
                assert sha256(path) == sha256(os.path.join(GOLD, f"{shape}.txt"))
            deg, cams, uv, P = run_index_probe(path)
            key = shape if shuffle is None else f"{shape}_shuffle{shuffle}"
            out[key + "/deg"], out[key + "/cam"], out[key + "/uv"], out[key + "/P"] = deg, cams, uv, P
    np.savez_compressed(os.path.join(GOLD, "index.npz"), **out)
    print("index.npz written:", sorted({k.split("/")[0] for k in out}))


def make_ba_log_keys():
    """Key set of the reference's own ba_log.json (tests/test_host_abi.py checks povar_write_ba_log against it)."""
    def keys(x, p=""):
        out = []
        for k, v in x.items():
            out.append(p + k)
            if isinstance(v, dict):
                out += keys(v, p + k + ".")
        return out
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run([BAL_REF, "--input", os.path.join(GOLD, "tiny.txt"), "--alpha", "0.1", "--power-sc-iterations", "20",
                        "--num-threads", "1", "--max-num-iterations-step-1", "3", "--max-num-iterations-step-2", "2"],
                       cwd=tmp, capture_output=True, check=True)
        with open(os.path.join(tmp, "ba_log.json")) as f:
            data = json.load(f)
    with open(os.path.join(GOLD, "ba_log_keys.json"), "w") as f:
        json.dump({"_comment": "every key of the ba_log.json the reference program (oracle/_ref/bal_ref) writes; "
                               "made by tools/make_golden.py", "keys": sorted(keys(data))}, f, indent=1)
    print("ba_log_keys.json written")


def make_bal_cli_fixtures():
    """tests/golden/create_dataset_small.json and dump_config.json (tests/test_host_abi.py compares this project's
    bal with them, and with the reference program where it is built)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import povar_testlib as common
    if os.path.exists(BAL_REF):
        prog, source = BAL_REF, "the reference program (oracle/_ref/bal_ref)"
    else:
        prog, source = BAL_OURS, "this project's bal; the reference program was not built where this file was made"
    sp = synthetic.generate_named("small")
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, "problem-16-400-pre.txt")
        common.write_bal9(src, sp, np.random.default_rng(7))
        subprocess.run([prog, "--input", src, "--create-dataset"], cwd=tmp, capture_output=True, check=True)
        with open(os.path.join(tmp, "data_custom", os.path.basename(src))) as f:
            lines = common.create_dataset_lines(f.read(), sp.num_obs, sp.num_cams)
        dump = subprocess.run([prog, "--dump-config", "--input", "x"], cwd=tmp, capture_output=True, text=True).stdout
    with open(os.path.join(GOLD, "create_dataset_small.json"), "w") as f:
        json.dump({"_comment": "--create-dataset output for common.write_bal9(synthetic 'small', default_rng(7)), one "
                               "entry per line, null where the program draws a random camera-matrix entry; made by "
                               "tools/make_golden.py", "source": source, "lines": lines}, f, indent=0)
    with open(os.path.join(GOLD, "dump_config.json"), "w") as f:
        json.dump({"_comment": "--dump-config --input x print-out; made by tools/make_golden.py", "source": source,
                   "dump": dump}, f, indent=1)
    print("create_dataset_small.json and dump_config.json written from", prog)


def main():
    """python tools/make_golden.py            everything (kernel_COD vectors, index fixture, all traces)
    python tools/make_golden.py NAME ...   only these configurations / "index" / "cod" / "keys" / "cli", merged into the
                                           existing traces.json"""
    os.makedirs(GOLD, exist_ok=True)
    want = set(sys.argv[1:])
    out_path = os.path.join(GOLD, "traces.json")
    doc = {"files": {}, "traces": {}, "reference_flags": "--alpha 0.1 --power-sc-iterations 20 (+ per-config flags)"}
    if want and os.path.exists(out_path):
        with open(out_path) as f:
            doc = json.load(f)
    if not want or "cod" in want:
        make_kernel_cod()
    if not want or "index" in want:
        make_index_fixture()
    if not want or "keys" in want:
        make_ba_log_keys()
    if not want or "cli" in want:
        make_bal_cli_fixtures()
    configs = [c for c in CONFIGS if not want or c[0] in want]
    paths = {}
    with tempfile.TemporaryDirectory() as tmp:
        for shape in sorted({c[1] for c in configs}):
            prob = synthetic.generate_named(shape)
            path = os.path.join(GOLD if shape in COMMITTED_FILES else tmp, f"{shape}.txt")
            if not (shape in COMMITTED_FILES and os.path.exists(path)):
                synthetic.write_bal(prob, path)
            paths[shape] = path
            doc["files"][shape] = {"sha256": sha256(path), "num_cams": prob.num_cams,
                                   "num_lms": prob.num_lms, "num_obs": prob.num_obs,
                                   "committed": shape in COMMITTED_FILES}
        for name, shape, flags in configs:
            one = run_ref(paths[shape], flags, 1, tmp)
            many = run_ref(paths[shape], flags, 8, tmp)
            doc["traces"][name] = {"shape": shape, "flags": flags, "threads1": one,
                                   "threads8": {"cost": many["cost"], "step_is_successful": many["step_is_successful"],
                                                "iteration": many["iteration"]}}
            k2 = [i for i in range(1, len(one["iteration"])) if one["iteration"][i] == 0]
            print(f"{name}: {len(one['cost'])} trials, step 2 starts at {k2[0] if k2 else None}, "
                  f"final cost {one['cost'][-1]:.6e}")
    with open(out_path, "w") as f:
        json.dump(doc, f, indent=1)
    print("traces.json written")


if __name__ == "__main__":
    main()
