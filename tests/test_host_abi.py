"""CPU-side checks of the C ABI: the library loads, exports every declared symbol, host-side
entry points (reader, canonical order, sharding) agree with the oracle, and compute entry points
refuse to run without a GPU instead of falling back to anything."""
import ctypes
import os
import re

import numpy as np
import pytest

import povar_testlib as common
from oracle import povar_oracle as O
from povar_b200 import capi, synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "povar_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(povar_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = capi.load()
    names = _declared_symbols()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/povar_b200.h but not exported"
    assert set(names) == set(capi.SIGNATURES), set(names) ^ set(capi.SIGNATURES)
    assert lib.povar_abi_version() == 3


def test_option_defaults_are_the_reference_code_defaults():
    o = capi.default_options()
    ref = O.Options()       # bal/solver_options.hpp:88-307
    for f in ("solver_type_step_1", "solver_type_step_2", "robust_norm", "huber_parameter", "alpha",
              "max_num_iterations_step_1", "max_num_iterations_step_2", "min_relative_decrease",
              "initial_trust_region_radius", "min_trust_region_radius", "max_trust_region_radius",
              "min_linear_solver_iterations", "max_linear_solver_iterations", "eta", "r_tolerance",
              "jacobi_scaling_epsilon", "function_tolerance", "power_sc_iterations", "initial_vee",
              "vee_factor"):
        assert getattr(o, f) == getattr(ref, f), f
    assert o.alpha == 0.01 and o.power_sc_iterations == 10      # not the README's 0.1 / 20 (SURVEY F3)


@pytest.mark.parametrize("shape", ["tiny", "small"])
def test_bal_reader_matches_oracle_loader_bit_exactly(shape, tmp_path):
    path = common.golden_file(shape)
    hp = capi.HostProblem.read(path)
    op = O.load_bal(path)
    assert (hp.num_cams, hp.num_lms, hp.num_obs) == (op.C, op.L, op.nnz)
    assert np.array_equal(hp.lm_ptr, op.lm_ptr)
    assert np.array_equal(hp.obs_cam, op.obs_cam)
    assert np.array_equal(hp.obs_uv, op.uv)                      # y already flipped
    assert np.array_equal(hp.cam_P.reshape(-1, 3, 4), op.P)
    # canonical order does not depend on the order of the observation lines
    prob = synthetic.generate_named(shape)
    shuffled = tmp_path / "shuffled.txt"
    synthetic.write_bal(prob, str(shuffled), shuffle_seed=11)
    hs = capi.HostProblem.read(str(shuffled))
    assert np.array_equal(hs.lm_ptr, hp.lm_ptr) and np.array_equal(hs.obs_cam, hp.obs_cam)
    assert np.array_equal(hs.obs_uv, hp.obs_uv)


@pytest.mark.parametrize("key", ["tiny", "tiny_shuffle3", "small", "small_shuffle11", "ladybug49_shuffle5"])
def test_reader_indexing_matches_the_reference_structures_bit_exactly(key, tmp_path):
    """tests/golden/index.npz holds what the reference ITSELF keeps after loading the file: `pose_idx_` of every
    LandmarkBlockSC (sc/landmark_block.hpp:104-108), the observation stored per (landmark, camera) pair
    (Landmark::obs, bal/bal_problem.hpp:226, after the loader's y flip) and the camera matrices -- dumped by
    oracle/index_probe.cpp from the compiled reference (tools/make_golden.py).  povar_bal_read, the numpy oracle's
    loader and povar_canonical_order must reproduce them bit for bit, whatever the order of the file's lines."""
    g = np.load(os.path.join(common.GOLD, "index.npz"))
    deg, cam, uv, P = g[key + "/deg"], g[key + "/cam"], g[key + "/uv"], g[key + "/P"]
    shape, _, shuffle = key.partition("_shuffle")
    prob = synthetic.generate_named(shape)
    path = tmp_path / "p.txt"
    synthetic.write_bal(prob, str(path), shuffle_seed=int(shuffle) if shuffle else None)
    lm_ptr = np.concatenate([[0], np.cumsum(deg)])
    hp = capi.HostProblem.read(str(path))
    assert (hp.num_cams, hp.num_lms, hp.num_obs) == (P.shape[0], deg.shape[0], cam.shape[0])
    assert np.array_equal(hp.lm_ptr, lm_ptr) and np.array_equal(hp.obs_cam, cam)
    assert np.array_equal(hp.obs_uv.reshape(-1, 2), uv)
    assert np.array_equal(hp.cam_P.reshape(-1, 12), P)
    op = O.load_bal(str(path))
    assert np.array_equal(op.lm_ptr, lm_ptr) and np.array_equal(op.obs_cam, cam) and np.array_equal(op.uv, uv)
    assert np.array_equal(op.P.reshape(-1, 12), P)
    rng = np.random.default_rng(1)
    perm = rng.permutation(prob.num_obs)
    hu = capi.HostProblem.from_unordered(prob.num_cams, prob.num_lms, prob.obs_cam[perm], prob.obs_lm[perm],
                                         prob.obs_xy[perm], prob.cam_params)
    assert np.array_equal(hu.lm_ptr, lm_ptr) and np.array_equal(hu.obs_cam, cam)
    assert np.array_equal(hu.obs_uv.reshape(-1, 2), uv)


def test_bal_reader_errors(tmp_path):
    with pytest.raises(capi.PovarError) as e:
        capi.HostProblem.read(str(tmp_path / "missing.txt"))
    assert e.value.code == capi.ERR_IO
    dup = tmp_path / "dup.txt"                                   # duplicate (cam, lm): bal_problem.cpp:227
    dup.write_text("2 1 2\n0 0 1.0 2.0\n0 0 1.5 2.5\n" + "\n".join(["0"] * 30) + "\n0 0 0\n")
    with pytest.raises(capi.PovarError) as e:
        capi.HostProblem.read(str(dup))
    assert e.value.code == capi.ERR_INVALID
    short = tmp_path / "short.txt"
    short.write_text("2 1 2\n0 0 1.0 2.0\n")
    with pytest.raises(capi.PovarError):
        capi.HostProblem.read(str(short))
    oob = tmp_path / "oob.txt"
    oob.write_text("2 1 1\n5 0 1.0 2.0\n" + "\n".join(["0"] * 30) + "\n0 0 0\n")
    with pytest.raises(capi.PovarError):
        capi.HostProblem.read(str(oob))
    # hostile headers: sizes the file cannot hold are refused before anything is allocated from them
    for k, header in enumerate(["2000000000 2000000000 2000000000", "3000000000 1 1", "1 1 9223372036854775807"]):
        bad = tmp_path / f"hostile{k}.txt"
        bad.write_text(header + "\n0 0 1.0 2.0\n")
        with pytest.raises(capi.PovarError) as e:
            capi.HostProblem.read(str(bad))
        assert e.value.code == capi.ERR_IO
    with pytest.raises(capi.PovarError) as e:                    # a directory: fopen works, ftell / fread do not
        capi.HostProblem.read(str(tmp_path))
    assert e.value.code == capi.ERR_IO


def test_canonical_order_from_generator_arrays():
    sp = synthetic.generate_named("small")
    rng = np.random.default_rng(0)
    perm = rng.permutation(sp.num_obs)
    hp = capi.HostProblem.from_unordered(sp.num_cams, sp.num_lms, sp.obs_cam[perm], sp.obs_lm[perm],
                                         sp.obs_xy[perm], sp.cam_params)
    op = O.build_problem(sp.num_cams, sp.num_lms, sp.obs_cam, sp.obs_lm, sp.obs_xy, sp.cam_params)
    assert np.array_equal(hp.lm_ptr, op.lm_ptr)
    assert np.array_equal(hp.obs_cam, op.obs_cam)
    assert np.array_equal(hp.obs_uv, op.uv)
    with pytest.raises(capi.PovarError):
        capi.HostProblem.from_unordered(3, 3, np.array([0, 1, 0]), np.array([2, 2, 2]),
                                        np.zeros((3, 2)), np.zeros((3, 15)))


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_partition_is_contiguous_and_balanced(world):
    hp = capi.HostProblem.read(common.golden_file("small"))
    shards = [hp.shard(r, world) for r in range(world)]
    assert shards[0].lm_begin == 0 and shards[-1].lm_end == hp.num_lms
    for a, b in zip(shards[:-1], shards[1:]):
        assert a.lm_end == b.lm_begin
    assert sum(s.num_obs for s in shards) == hp.num_obs
    assert np.array_equal(np.concatenate([s.obs_cam for s in shards]), hp.obs_cam)
    ideal = hp.num_obs / world
    max_deg = int(np.max(np.diff(hp.lm_ptr)))
    for s in shards:
        assert abs(s.num_obs - ideal) <= max_deg + 1
        assert s.lm_ptr[0] == 0 and s.lm_ptr[-1] == s.num_obs


def test_partition_edge_cases():
    lib = capi.load()
    lm_ptr = np.array([0, 2, 4], dtype=np.int64)
    bounds = np.empty(5, dtype=np.int32)
    assert lib.povar_partition_landmarks(2, lm_ptr.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), 4,
                                         bounds.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))) == 0
    assert bounds[0] == 0 and bounds[4] == 2 and np.all(np.diff(bounds) >= 0)   # empty shards allowed
    assert lib.povar_partition_landmarks(2, lm_ptr.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), 0,
                                         bounds.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))) == capi.ERR_INVALID


def test_no_cpu_fallback_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    hp = capi.HostProblem.read(common.golden_file("tiny"))
    with pytest.raises(capi.PovarError) as e:
        capi.Solver(hp)
    assert e.value.code == capi.ERR_NO_DEVICE
    # the package itself never imports the oracle
    import povar_b200
    pkg = os.path.dirname(povar_b200.__file__)
    for root, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cpp", ".h", ".cuh")):
                text = open(os.path.join(root, fn), errors="ignore").read()
                assert "povar_oracle" not in text and "import oracle" not in text, fn


def test_bal_binary_refuses_to_run_without_a_gpu():
    import subprocess
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from povar_b200 import build
    res = subprocess.run([build.BAL, "--input", common.golden_file("tiny"), "--verbosity-level", "0"],
                         capture_output=True, text=True)
    assert res.returncode != 0
    assert "no CUDA device" in res.stderr


# ---------------------------------------------------------------------------------------------
# --create-dataset: BAL file (9 parameters per camera) -> the 15-parameter file the solver loads
# (bal/bal_problem.cpp:306-471), compared with the output stored in tests/golden/ (its "source" names the program that
# wrote it) and, where the reference program is built, with that program's own output
# ---------------------------------------------------------------------------------------------
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "bal_ref")


def test_create_dataset_writes_the_reference_format(tmp_path):
    import json
    import subprocess
    from povar_b200 import build, synthetic
    rng = np.random.default_rng(7)
    sp = synthetic.generate_named("small")
    src = tmp_path / "problem-16-400-pre.txt"
    cams9 = common.write_bal9(src, sp, rng)
    ours = tmp_path / "ours"
    ours.mkdir()
    res = subprocess.run([build.BAL, "--input", str(src), "--create-dataset", "--create-dataset-seed", "11"],
                         cwd=ours, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    out = ours / "data_custom" / src.name
    tok = out.read_text().split()
    C, L, N = sp.num_cams, sp.num_lms, sp.num_obs
    assert [int(t) for t in tok[:3]] == [C, L, N]
    assert len(tok) == 3 + 4 * N + 15 * C + 3 * L
    obs = np.array(tok[3:3 + 4 * N], dtype=np.float64).reshape(N, 4)
    assert np.array_equal(obs[:, 0], sp.obs_cam) and np.array_equal(obs[:, 1], sp.obs_lm)
    assert np.allclose(obs[:, 2:], sp.obs_xy, rtol=0, atol=5.1e-7)          # %lf: six decimals
    cam = np.array(tok[3 + 4 * N:3 + 4 * N + 15 * C], dtype=np.float64).reshape(C, 15)
    assert np.array_equal(cam[:, 8:12], np.tile([0.0, 0.0, 0.0, 1.0], (C, 1)))
    assert np.allclose(cam[:, 12:], cams9[:, 6:], rtol=0, atol=5.1e-7)
    draws = cam[:, :8].reshape(-1)
    assert abs(draws.mean()) < 0.2 and 0.8 < draws.std() < 1.2              # N(0, 1)
    # reproducible with a seed, and loadable by the solver's reader
    again = tmp_path / "again.txt"
    capi.create_dataset(str(src), str(again), seed=11)
    assert again.read_bytes() == out.read_bytes()
    hp = capi.HostProblem.read(str(out))
    assert (hp.num_cams, hp.num_lms, hp.num_obs) == (C, L, N)
    # the stored output for the same input (and the reference program's, where it is built): identical text except for
    # the random draws
    mine = common.create_dataset_lines(out.read_text(), N, C)
    with open(os.path.join(common.GOLD, "create_dataset_small.json")) as f:
        recorded = json.load(f)["lines"]
    if os.path.exists(REF_BIN):
        theirs = tmp_path / "theirs"
        theirs.mkdir()
        res = subprocess.run([REF_BIN, "--input", str(src), "--create-dataset"], cwd=theirs, capture_output=True,
                             text=True)
        assert res.returncode == 0, res.stderr[-500:]
        assert common.create_dataset_lines((theirs / "data_custom" / src.name).read_text(), N, C) == recorded
    assert len(mine) == len(recorded), (len(mine), len(recorded))
    for i, (a, b) in enumerate(zip(mine, recorded)):
        assert a == b, (i, a, b)


def _sell_key(cams, span=896):
    """Centre of the first stretch of `span` cameras that holds most of the landmark's observations."""
    best = (0, 0)
    j = 0
    for i in range(len(cams)):
        j = max(j, i)
        while j + 1 < len(cams) and cams[j + 1] - cams[i] < span:
            j += 1
        if j - i > best[1] - best[0]:
            best = (i, j)
    return (int(cams[best[0]]) + int(cams[best[1]])) // 2


def _sell_reference(hp, max_window=4096, width=32, max_deg=32):
    """The sliced-ELL rule restated with numpy sorts (engine.cu build_sell): landmarks with 1..32 observations
    in the order of their key camera (stable), windows of `window`, inside a window stable by descending
    degree, 32 landmarks (one per lane) per slice, slice length = the largest degree in it."""
    deg = np.diff(hp.lm_ptr)
    ok = np.nonzero((deg > 0) & (deg <= max_deg))[0]
    key = np.array([_sell_key(hp.obs_cam[hp.lm_ptr[l]:hp.lm_ptr[l + 1]]) for l in ok], dtype=np.int64)
    by_cam = ok[np.argsort(key, kind="stable")]
    window = max_window
    while window > 512 and window * 128 > len(ok):
        window //= 2
    slice_ptr, sell_lm = [0], []
    for w0 in range(0, len(by_cam), window):
        win = by_cam[w0:w0 + window]
        order = win[np.argsort(-deg[win], kind="stable")]
        for i in range(0, len(order), width):
            grp = list(order[i:i + width])
            sell_lm += grp + [-1] * (width - len(grp))
            slice_ptr.append(slice_ptr[-1] + int(deg[order[i]]))
    return np.array(slice_ptr), np.array(sell_lm), np.nonzero(deg > max_deg)[0]


def test_sell_key_centres_the_cameras_it_can_cover():
    assert _sell_key(np.array([10, 11, 12, 13, 1500])) == 11      # an outlier does not move the key
    assert _sell_key(np.array([100, 400, 700])) == 400            # everything fits: the middle of first and last
    assert _sell_key(np.array([5])) == 5
    assert _sell_key(np.array([0, 1000, 1001, 1002])) == 1001


@pytest.mark.parametrize("shape", ["small", "ladybug49", "trafalgar257"])
def test_sliced_ell_order_matches_its_rule_for_any_thread_count(shape):
    sp = synthetic.generate_named(shape)
    hp = capi.HostProblem.from_unordered(sp.num_cams, sp.num_lms, sp.obs_cam, sp.obs_lm, sp.obs_xy, sp.cam_params)
    ref = _sell_reference(hp)
    for threads in (1, 3, 8):
        got = capi.sell_layout(hp, threads)
        for a, b in zip(got, ref):
            assert np.array_equal(a, b), (shape, threads)
    # small shards keep only the landmarks with few observations in the set (sell_max_degree)
    for a, b in zip(capi.sell_layout(hp, 2, 12), _sell_reference(hp, max_deg=12)):
        assert np.array_equal(a, b), shape


def test_sell_max_degree_shrinks_on_small_shards():
    assert capi.sell_max_degree(4_999_019) == 32          # venice-1778 on one GPU: 33 rows per resident warp
    assert capi.sell_max_degree(2_500_000) == 32
    assert capi.sell_max_degree(1_250_000) == 16          # on four
    assert capi.sell_max_degree(625_000) == 8             # on eight: one slice of ~5 rows per warp
    assert capi.sell_max_degree(30_000) == 8
    assert capi.sell_max_degree(50_000_000) == 32


@pytest.mark.parametrize("shape,world", [("small", 1), ("trafalgar257", 1), ("venice89", 1), ("venice1778", 1),
                                         ("venice1778", 8)])
def test_landmark_half_plan_covers_the_slices_and_their_cameras(shape, world):
    """plan_landmark_half (engine.cu): contiguous slice ranges with (nearly) equal rows, one per warp; per block a
    window of the camera table that holds every camera its slices observe (on these shapes), inside what an SM
    has of shared memory."""
    sp = synthetic.generate_named(shape)
    hp = capi.HostProblem.from_unordered(sp.num_cams, sp.num_lms, sp.obs_cam, sp.obs_lm, sp.obs_xy, sp.cam_params)
    if world > 1:
        hp = hp.shard(world - 1, world)
    T = capi.sell_max_degree(hp.num_obs)
    slice_ptr, sell_lm, _ = capi.sell_layout(hp, 0, T)
    S = len(slice_ptr) - 1
    deg = np.diff(hp.lm_ptr)
    for model, rec, stage in ((0, 176, 640), (1, 208, 896), (2, 176, 896)):
        info, rs, lo = capi.landmark_plan(hp, model, sms=148, max_deg=T)
        W, D, bps = info["warps"], info["stages"], info["blocks_per_sm"]
        assert (W, D, bps) in ((8, 3, 4), (16, 3, 2), (32, 3, 1), (32, 2, 1), (24, 2, 1), (16, 2, 1))
        assert info["smem_bytes"] == ((1 + W * D) * 8 + 127) // 128 * 128 + W * D * stage + info["win_cams"] * rec
        assert bps * (info["smem_bytes"] + 1024) <= 228 * 1024
        assert info["ranges"] == min(148 * bps * W, S) and info["blocks"] >= -(-info["ranges"] // W)
        assert rs[0] == 0 and rs[-1] == S and np.all(np.diff(rs) >= 0)
        cost = np.diff(slice_ptr[rs] + 2 * rs)                       # rows + 2 per slice
        longest = int(np.diff(slice_ptr).max()) + 2
        assert cost.max() <= (slice_ptr[-1] + 2 * S) / info["ranges"] + longest + 1   # equal cost up to one slice
        assert info["covered"] == 1
        for b in range(-(-info["ranges"] // W)):
            s0, s1 = rs[b * W], rs[min((b + 1) * W, info["ranges"])]
            lms = sell_lm[32 * s0:32 * s1]
            lms = lms[lms >= 0]
            if len(lms) == 0:
                continue
            first, last = hp.obs_cam[hp.lm_ptr[lms]], hp.obs_cam[hp.lm_ptr[lms + 1] - 1]
            assert lo[b] <= first.min() and last.max() < lo[b] + info["win_cams"] <= hp.num_cams, (shape, model, b)


def test_ba_log_has_every_key_of_the_reference_log(tmp_path):
    """povar_write_ba_log (what `bal --log-log-path` writes) against the key set of the reference program's own
    ba_log.json, plus the derived columns of bal/ba_log_utils.cpp:100-175 on a hand-made trace."""
    import json
    hp = capi.HostProblem.read(common.golden_file("tiny"))
    opt = capi.default_options(solver_type_step_1=capi.POWER_VARPROJ)
    rows = [  # step, iteration, valid, successful, cost, cost_valid, trial_cost, n_valid
        (1, 0, 1, 1, 100.0, 100.0, 100.0, 131),
        (1, 1, 1, 1, 60.0, 60.0, 60.0, 131),
        (1, 2, 1, 0, 60.0, 60.0, 75.0, 131),      # rejected: the log repeats the previous cost
        (1, 3, 1, 1, 50.0, 50.0, 50.0, 131),
        (2, 0, 1, 1, 40.0, 39.0, 40.0, 130),      # step 2 starts again at iteration 0
        (2, 1, 1, 1, 30.0, 29.0, 30.0, 129),
    ]
    its = []
    for k, (step, it, valid, succ, cost, cv, trial, nv) in enumerate(rows):
        e = capi.Iteration()
        e.step, e.iteration, e.step_is_valid, e.step_is_successful = step, it, valid, succ
        e.cost, e.cost_valid, e.trial_cost, e.num_obs_valid = cost, cv, trial, nv
        e.residual_mean, e.residual_valid_mean = 2.0 + k, 1.0 + k
        e.relative_decrease, e.trust_region_radius, e.linear_solver_iterations = 0.5, 1e4 / (k + 1), (7 if it else 0)
        e.iteration_time, e.cumulative_time = 0.01, 0.01 * (k + 1)
        e.residual_evaluation_time, e.jacobian_evaluation_time = 1e-3, (2e-3 if it else 0.0)
        e.prepare_time, e.solve_reduced_system_time, e.back_substitution_time = 3e-3, 4e-3, 5e-3
        its.append(e)
    summ = capi.SolveSummary()
    summ.num_iterations, summ.num_successful_steps, summ.num_unsuccessful_steps = len(its), 4, 1
    summ.initial_cost, summ.final_cost, summ.total_time = 100.0, 30.0, 0.06
    summ.message = b'Solver did not converge after maximum number of 2 iterations "quoted"'
    path = tmp_path / "ba_log.json"
    capi.write_ba_log(str(path), hp, opt, its, summ, input_path="data_custom/tiny.txt", load_time=0.5)
    data = json.loads(path.read_text())

    def keys(x, p=""):
        out = []
        for k, v in x.items():
            out.append(p + k)
            if isinstance(v, dict):
                out += keys(v, p + k + ".")
        return out
    with open(os.path.join(common.GOLD, "ba_log_keys.json")) as f:
        want = json.load(f)["keys"]
    have = set(keys(data))
    assert [k for k in want if k not in have] == []
    n = len(its)
    for k, v in data.items():
        if not k.startswith("_"):
            assert isinstance(v, list) and len(v) == n, k
    assert data["_type"] == "rootba_povar"
    assert data["cost"] == [100.0, 60.0, 60.0, 50.0, 40.0, 30.0]
    # previous - current, only for successful trials with iteration > 0; after a rejected trial the previous
    # summary's own cost is its trial cost (bal_bundle_adjustment.cpp:74-78)
    assert data["cost_change"] == [0.0, 40.0, 0.0, 25.0, 0.0, 10.0]
    assert data["num_obs_valid_change"] == [0, 0, 0, 0, 0, 1]
    assert data["linear_solver_type"] == ["", "bal_power_sc", "bal_power_sc", "bal_power_sc", "", "bal_power_sc"]
    assert data["num_obs"] == [131] * n and data["step_is_nonmonotonic"] == [False] * n
    assert abs(data["cost_avg_valid"][4] - 39.0 / 130) < 1e-15
    assert data["residual_block_mean"] == [2.0 + k for k in range(n)]
    assert data["residual_block_valid_mean"] == [1.0 + k for k in range(n)]
    st = data["_static"]
    assert st["problem_info"]["num_observations"] == hp.num_obs and st["problem_info"]["input_path"] == "data_custom/tiny.txt"
    deg = np.diff(hp.lm_ptr)
    assert st["problem_info"]["per_lm_obs"]["max"] == deg.max() and abs(st["problem_info"]["per_lm_obs"]["mean"] - deg.mean()) < 1e-12
    assert st["solver"]["solver_type"] == "power_variable_projection"
    assert st["solver"]["message"].endswith('"quoted"')
    assert st["solver"]["num_linear_solves"] == 4 and st["solver"]["num_jacobian_evaluations"] == 4
    assert abs(st["solver"]["linear_solver_time_in_seconds"] - n * 12e-3) < 1e-12
    assert abs(st["timing"]["total"] - 0.56) < 1e-12


def _parse_dump(text):
    """{section.key: value} of a --dump-config print-out (the subset of TOML both programs write)."""
    out, section = {}, ""
    for line in text.splitlines():
        line = line.strip()
        if line.startswith("[") and line.endswith("]") and "=" not in line:
            section = line[1:-1]
        elif "=" in line and section:
            k, v = [t.strip() for t in line.split("=", 1)]
            out[f"{section}.{k}"] = v
    return out


def _assert_dump_agrees(ours, theirs):
    """Every key we print is printed by the other program too, with the same value."""
    assert set(ours) <= set(theirs), sorted(set(ours) - set(theirs))
    for k, v in ours.items():
        a, b = v.strip('"'), theirs[k].strip('"')
        try:
            assert float(a) == float(b), (k, a, b)
        except ValueError:
            assert a == b, (k, a, b)


_CONFIG_TOML = (
    '# comment\n[dataset]\ninput = "data_custom/p.txt"   # trailing comment\n\n[solver]\nalpha = 0.1\n'
    'solver_type_step_1 = "PCG"\nsolver_type_step_2 = "RIPCG"\npower_sc_iterations = 20\nnum_threads = 4\n'
    'max_num_iterations_step_2 = 7\n\n[solver.residual]\nrobust_norm = "CAUCHY"\nhuber_parameter = 3.5\n\n'
    '[solver.log]\nlog_path = "out/ba_log.json"\nsave_log_flags = [\n"JSON",\n]\n\n[batch_run]\nsomething = 1\n')
_CONFIG_OVERRIDES = ["--alpha", "0.25", "--residual-huber-parameter", "2"]


def test_config_file_and_dump_config_follow_the_reference(tmp_path):
    """rootba_config.toml is read first, the command line overrides it, --dump-config prints the effective
    options in the reference's layout (cli/bal_cli_utils.cpp:96-122); defaults equal the reference's own."""
    import json
    import subprocess
    from povar_b200 import build
    # defaults: every key we print has the reference's default value -- as the stored print-out of --dump-config
    # has it (tests/golden/dump_config.json, its "source" names the program that wrote it), as the reference program
    # prints it where that program is built, and, for the numeric solver options, as the oracle restates the
    # reference's code defaults (bal/solver_options.hpp:88-307)
    ours = _parse_dump(subprocess.run([build.BAL, "--dump-config", "--input", "x"], cwd=tmp_path, capture_output=True,
                                      text=True).stdout)
    assert ours["solver.alpha"] == "0.01" and ours["solver.power_sc_iterations"] == "10"
    with open(os.path.join(common.GOLD, "dump_config.json")) as f:
        recorded = _parse_dump(json.load(f)["dump"])
    _assert_dump_agrees(ours, recorded)
    ref_defaults = O.Options()
    checked = 0
    for k, v in ours.items():
        section, _, name = k.rpartition(".")
        if section.startswith("solver") and hasattr(ref_defaults, name) and not v.startswith('"'):
            assert float(v) == float(getattr(ref_defaults, name)), (k, v, getattr(ref_defaults, name))
            checked += 1
    assert checked >= 15
    if os.path.exists(REF_BIN):
        theirs = _parse_dump(subprocess.run([REF_BIN, "--dump-config", "--input", "x"], cwd=tmp_path,
                                            capture_output=True, text=True).stdout)
        _assert_dump_agrees(recorded, theirs)
        _assert_dump_agrees(ours, theirs)
    # a config file, partly overridden on the command line
    (tmp_path / "rootba_config.toml").write_text(_CONFIG_TOML)
    res = subprocess.run([build.BAL, "--dump-config"] + _CONFIG_OVERRIDES, cwd=tmp_path, capture_output=True, text=True)
    got = _parse_dump(res.stdout)
    assert got["dataset.input"] == '"data_custom/p.txt"'
    assert got["solver.alpha"] == "0.25"                        # command line wins
    assert got["solver.solver_type_step_1"] == '"PCG"' and got["solver.solver_type_step_2"] == '"RIPCG"'
    assert got["solver.power_sc_iterations"] == "20" and got["solver.max_num_iterations_step_2"] == "7"
    assert got["solver.residual.robust_norm"] == '"CAUCHY"' and float(got["solver.residual.huber_parameter"]) == 2.0
    assert got["solver.log.log_path"] == '"out/ba_log.json"'
    # --config names another file; -C changes the directory first; a missing file means defaults
    other = tmp_path / "sub"
    other.mkdir()
    (other / "alt.toml").write_text("[solver]\neta = 0.5\n")
    got = _parse_dump(subprocess.run([build.BAL, "-C", str(other), "--config", "alt.toml", "--dump-config", "--input", "x"],
                                     capture_output=True, text=True).stdout)
    assert float(got["solver.eta"]) == 0.5 and got["solver.alpha"] == "0.01"


def test_reference_reads_back_our_dump_config(tmp_path):
    """The reference program reads the config file our --dump-config prints.  This needs the reference program
    itself (oracle/_ref/bal_ref, built from the reference's own sources by `make -C oracle ref`)."""
    import subprocess
    from povar_b200 import build
    if not os.path.exists(REF_BIN):
        pytest.skip("oracle/_ref/bal_ref not built (needs the reference's sources: make -C oracle ref)")
    (tmp_path / "rootba_config.toml").write_text(_CONFIG_TOML)
    res = subprocess.run([build.BAL, "--dump-config"] + _CONFIG_OVERRIDES, cwd=tmp_path, capture_output=True, text=True)
    other = tmp_path / "sub"
    other.mkdir()
    (other / "rootba_config.toml").write_text(res.stdout)
    back = _parse_dump(subprocess.run([REF_BIN, "--dump-config"], cwd=other, capture_output=True, text=True).stdout)
    assert float(back["solver.alpha"]) == 0.25 and back["solver.solver_type_step_1"] == '"PCG"'
    assert back["solver.residual.robust_norm"] == '"CAUCHY"' and back["solver.log.log_path"] == '"out/ba_log.json"'


def test_ctypes_structs_have_the_library_s_layout():
    """capi.py mirrors the public structs by hand; a size mismatch would corrupt memory in povar_bundle_adjust."""
    lib = capi.load()
    mirrors = [capi.Options, capi.ProblemDesc, capi.CommDesc, capi.ResidualInfo, capi.Iteration, capi.SolveSummary,
               capi.BalData, capi.BaLogInfo, capi.PhaseTimes]
    for which, cls in enumerate(mirrors):
        assert lib.povar_abi_sizeof(which) == ctypes.sizeof(cls), cls.__name__
    assert lib.povar_abi_sizeof(99) == -1


def test_bal_reader_parses_numbers_like_strtod_on_many_threads(tmp_path):
    """The reader converts tokens with std::from_chars on several threads: every value must be the correctly
    rounded double (what the reference's fscanf("%lf") and Python's float() give), whatever the notation, and the
    multi-threaded path (files above 1 MB) must agree with a token-by-token Python parse."""
    rng = np.random.default_rng(3)
    C, L = 7, 60000
    deg = rng.integers(2, 5, L)
    cams = np.concatenate([np.sort(rng.choice(C, d, replace=False)) for d in deg])
    lms = np.repeat(np.arange(L), deg)
    N = len(cams)
    order = rng.permutation(N)
    fmts = ["%.6f", "%.17g", "%.3e", "%+.10e", "%.1f", "%d"]
    toks = []
    for k in order:
        x, y = rng.normal(0, 300, 2)
        f = fmts[k % len(fmts)]
        toks.append(f"{cams[k]} {lms[k]}   {f % (x if f != '%d' else int(x))}\t{fmts[(k + 1) % len(fmts)] % (y if fmts[(k + 1) % len(fmts)] != '%d' else int(y))}")
    camtok = ["%.17g" % v for v in rng.normal(size=15 * C)]
    camtok[3] = "1e-320"          # subnormal
    camtok[4] = "0.1"
    camtok[5] = "123456789012345678901234567890"
    camtok[6] = "-0.0"
    lmtok = ["%.6e" % v for v in rng.normal(size=3 * L)]
    path = tmp_path / "numbers.txt"
    path.write_text(f"{C} {L} {N}\n" + "\n".join(toks) + "\n" + " ".join(camtok) + "\n" + "\n".join(lmtok) + "\n")
    assert path.stat().st_size > (1 << 20)
    hp = capi.HostProblem.read(str(path))
    assert (hp.num_cams, hp.num_lms, hp.num_obs) == (C, L, N)
    # Python parse of the same tokens
    flat = path.read_text().split()
    obs = flat[3:3 + 4 * N]
    pc = np.array([int(t) for t in obs[0::4]])
    pl = np.array([int(t) for t in obs[1::4]])
    px = np.array([float(t) for t in obs[2::4]])
    py = -np.array([float(t) for t in obs[3::4]])
    perm = np.lexsort((pc, pl))
    assert np.array_equal(hp.obs_cam, pc[perm])
    assert np.array_equal(hp.obs_uv[:, 0], px[perm]) and np.array_equal(hp.obs_uv[:, 1], py[perm])
    want = np.array([float(t) for t in camtok]).reshape(C, 15)
    assert np.array_equal(hp.cam_params.view(np.uint64), want.view(np.uint64))      # bit for bit, -0.0 and subnormals too
    # a malformed token anywhere is an error, not a silently shifted parse
    bad = tmp_path / "bad.txt"
    bad.write_text(path.read_text().replace(lmtok[-5], "abc", 1))
    with pytest.raises(capi.PovarError):
        capi.HostProblem.read(str(bad))


def test_reference_driver_with_the_plugin_links_and_fails_loudly_without_a_gpu(tmp_path):
    """oracle/_ref/bal_ref_b200 = the reference's own driver with LinearizorB200 (integration/) behind its Linearizor
    interface: it must exist after build(), load libpovar_b200.so, get as far as povar_create and stop there."""
    import subprocess
    import torch
    plugin = os.path.join(ROOT, "oracle", "_ref", "bal_ref_b200")
    if not os.path.exists(plugin):
        pytest.skip("oracle/_ref/bal_ref_b200 not built (needs /root/reference: make -C oracle plugin)")
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    res = subprocess.run([plugin, "--input", common.golden_file("tiny"), "--alpha", "0.1", "--power-sc-iterations", "20"],
                         cwd=tmp_path, capture_output=True, text=True)
    assert res.returncode != 0
    assert "no CUDA device (this library has no CPU fallback)" in res.stderr
    assert "linearizor_b200.hpp" in res.stderr          # the CHECK in the plug-in's constructor, not a crash elsewhere
