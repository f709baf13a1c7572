"""povar_create_device and the device-memory state calls on the B200: the canonical order made on the GPU gives the
host route's index arrays and therefore its traces bit for bit, alone and sharded; bad input is rejected without
spoiling the next create; the calls are ordered against the caller's torch stream."""
import ctypes
import os

import numpy as np
import pytest
import torch

import povar_testlib as common
from povar_b200 import capi, synthetic

pytestmark = pytest.mark.gpu

INDEX_ARRAYS = ("lm_ptr", "obs_cam", "obs_lm", "cam_ptr", "csc_lm", "sell_lm")


def _lists(hp):
    """the canonical list of a HostProblem as (obs_cam, obs_lm, obs_uv) numpy arrays"""
    lm = np.repeat(np.arange(hp.num_lms, dtype=np.int32), np.diff(hp.lm_ptr))
    return hp.obs_cam.copy(), lm, hp.obs_uv.reshape(-1, 2).copy()


def _orders(n):
    """three seeded shuffles and the reversed list"""
    return [np.random.default_rng(s).permutation(n) for s in (1, 2, 3)] + [np.arange(n)[::-1].copy()]


def _device_problem(hp, order, dev="cuda:0", **kw):
    cam, lm, uv = _lists(hp)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return capi.DeviceProblem(t(hp.cam_P.reshape(-1, 12)), t(cam[order]), t(lm[order]), t(uv[order]),
                              num_lms=hp.num_lms, **kw)


def _index(s):
    return {k: s.debug_read(k) for k in INDEX_ARRAYS}


def _assert_same_index(a, b, label):
    for k in INDEX_ARRAYS:
        assert np.array_equal(a[k], b[k]), f"{label}: {k} differs"


@pytest.mark.parametrize("shape", ["tiny", "small", "ladybug49"])
def test_device_order_gives_the_host_index(shape):
    hp = capi.HostProblem.read(common.golden_file(shape))
    opt = capi.default_options(verbosity_level=0)
    s = capi.Solver(hp, opt)
    ref = _index(s)
    s.close()
    for i, order in enumerate(_orders(hp.num_obs)):
        s = capi.Solver(_device_problem(hp, order), opt)
        _assert_same_index(_index(s), ref, f"{shape} order {i}")
        s.close()


@pytest.mark.parametrize("key", ["tiny_shuffle3", "small_shuffle11", "ladybug49_shuffle5"])
def test_device_order_matches_the_reference_structures(key):
    """tests/golden/index.npz: the reference's own per-landmark degrees and camera order (see test_host_abi)"""
    g = np.load(os.path.join(common.GOLD, "index.npz"))
    shape, _, shuffle = key.partition("_shuffle")
    prob = synthetic.generate_named(shape)
    order = np.random.default_rng(int(shuffle)).permutation(prob.num_obs)
    uv = prob.obs_xy[order].copy()
    uv[:, 1] = -uv[:, 1]
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    dp = capi.DeviceProblem(t(prob.cam_params[:, :12]), t(prob.obs_cam[order]), t(prob.obs_lm[order]), t(uv),
                            num_lms=prob.num_lms)
    s = capi.Solver(dp, capi.default_options(verbosity_level=0))
    assert np.array_equal(np.diff(s.debug_read("lm_ptr")), g[key + "/deg"])
    assert np.array_equal(s.debug_read("obs_cam"), g[key + "/cam"])
    s.close()


def _solve(solver):
    its, summary = solver.bundle_adjust()
    P, X = solver.get_state(capi.STATE_JOINT)
    return dict(cost=[e.cost for e in its], succ=[e.step_is_successful for e in its],
                lin=[e.linear_solver_iterations for e in its], P=P, X=X, final=summary.final_cost)


def _assert_same_run(a, b, label):
    for k in ("cost", "succ", "lin"):
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), f"{label}: {k} differs"
    assert np.array_equal(a["P"], b["P"]) and np.array_equal(a["X"], b["X"]), f"{label}: final state differs"
    assert a["final"] == b["final"]


SOLVERS = {"povar": [], "poba": ["--solver-type-step-1", "POWER_SCHUR_COMPLEMENT"],
           "pcg_ripcg": ["--solver-type-step-1", "PCG", "--solver-type-step-2", "RIPCG"],
           "cholesky": ["--solver-type-step-1", "CHOLESKY"],
           "huber": ["--residual-robust-norm", "HUBER", "--residual-huber-parameter", "30"],
           "error_valid": ["--optimized-cost", "ERROR_VALID"]}
CASES = [(shape, name) for shape in ("tiny", "small") for name in SOLVERS] + [("ladybug49", "povar")]


@pytest.mark.parametrize("shape,name", CASES)
def test_device_created_handle_runs_the_host_trace(shape, name):
    traces = {**common.traces()["traces"]}
    meta = traces.get(f"{shape}_{name}")
    flags = meta["flags"] if meta else SOLVERS[name]
    kw = common.flags_to_options(flags)
    hp = capi.HostProblem.read(common.golden_file(shape))
    s = capi.Solver(hp, capi.default_options(verbosity_level=0, **kw))
    ref = _solve(s)
    s.close()
    s = capi.Solver(_device_problem(hp, _orders(hp.num_obs)[0]), capi.default_options(verbosity_level=0, **kw))
    got = _solve(s)
    s.close()
    _assert_same_run(got, ref, f"{shape}_{name}")
    if meta:
        common.assert_trace_close(meta, got["cost"], got["succ"], got["lin"], label=f"{shape}_{name} (device)")


def _worker_shards(rank, world, hid, path, kw, out_dir):
    import torch as _torch  # noqa: F401  (initialises CUDA in the spawned process)
    hp_all = capi.HostProblem.read(path)
    runs = {}
    for route in ("host", "device"):
        if route == "host":
            prob = hp_all.shard(rank, world)
        else:
            prob = _device_problem(hp_all, np.random.default_rng(7).permutation(hp_all.num_obs)).shard(rank, world)
        s = capi.Solver(prob, capi.default_options(verbosity_level=0, **kw), capi.make_comm(rank, world, 0, hid))
        runs[route] = _solve(s)
        runs[route]["range"] = (prob.lm_begin, prob.lm_end)
        s.close()
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"),
             **{f"{r}_{k}": np.asarray(v) for r, d in runs.items() for k, v in d.items()})
    capi.load().povar_comm_finalize()


@pytest.mark.parametrize("name,world", [("small_povar", 2), ("small_poba", 3)])
def test_device_created_shards_run_the_host_sharded_trace(name, world, tmp_path):
    import torch.multiprocessing as mp
    meta = common.traces()["traces"][name]
    kw = common.flags_to_options(meta["flags"])
    path = common.golden_file(meta["shape"])
    mp.spawn(_worker_shards, args=(world, capi.host_id(), path, kw, str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        z = np.load(tmp_path / f"rank{r}.npz")
        assert np.array_equal(z["host_range"], z["device_range"])
        for k in ("cost", "succ", "lin", "P", "X", "final"):
            assert np.array_equal(z[f"host_{k}"], z[f"device_{k}"]), f"{name} x{world} rank {r}: {k} differs"


def _raw_create(desc):
    lib = capi.load()
    h = capi._H()
    rc = lib.povar_create_device(ctypes.byref(desc), ctypes.byref(capi.default_options(verbosity_level=0)), None,
                                 ctypes.byref(h))
    if rc == capi.OK:
        lib.povar_destroy(h)
    return rc


def _raw_desc(dp, **kw):
    d = capi.DeviceProblemDesc(dp.num_cams, dp.num_lms_total, dp.num_obs, dp.lm_begin, dp.lm_end,
                               dp.obs_cam.data_ptr(), dp.obs_lm.data_ptr(), dp.obs_uv.data_ptr(), dp.cam_P.data_ptr(),
                               torch.cuda.current_stream().cuda_stream)
    for k, v in kw.items():
        setattr(d, k, v)
    return d


def test_bad_input_is_rejected_and_the_next_create_works():
    hp = capi.HostProblem.read(common.golden_file("small"))
    good = _device_problem(hp, _orders(hp.num_obs)[0])
    host_uv = np.zeros((hp.num_obs, 2))
    cases = {}
    for label, col, i, val in (("duplicate", None, None, None), ("cam = C", "obs_cam", 3, hp.num_cams),
                               ("cam = -1", "obs_cam", 5, -1), ("lm = num_lms", "obs_lm", 7, hp.num_lms)):
        cam, lm = good.obs_cam.clone(), good.obs_lm.clone()
        if col is None:
            cam[1], lm[1] = cam[0], lm[0]
        else:
            (cam if col == "obs_cam" else lm)[i] = val
        cases[label] = (capi.DeviceProblem(good.cam_P, cam, lm, good.obs_uv, num_lms=hp.num_lms), {})
    cases["host pointer"] = (good, {"obs_uv": host_uv.ctypes.data})
    cases["bad range"] = (good, {"lm_begin": 5, "lm_end": 4})
    if torch.cuda.device_count() > 1:
        other = good.obs_uv.to("cuda:1")
        cases["other GPU"] = (good, {"obs_uv": other.data_ptr()})
    for label, (dp, kw) in cases.items():
        assert _raw_create(_raw_desc(dp, **kw)) == capi.ERR_INVALID, label
        assert capi.load().povar_last_error(None), label
        assert _raw_create(_raw_desc(good)) == capi.OK, f"create after {label}"
    torch.cuda.synchronize()


def test_inputs_from_a_side_stream_are_waited_for():
    hp = capi.HostProblem.read(common.golden_file("small"))
    s = capi.Solver(hp, capi.default_options(verbosity_level=0))
    ref = _index(s)
    s.close()
    src = _device_problem(hp, _orders(hp.num_obs)[1])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)   # the copies below land long after create was called
        dst = [torch.full_like(t, -1) for t in (src.cam_P, src.obs_cam, src.obs_lm, src.obs_uv)]
        for d, t in zip(dst, (src.cam_P, src.obs_cam, src.obs_lm, src.obs_uv)):
            d.copy_(t)
        dp = capi.DeviceProblem(*dst, num_lms=hp.num_lms)
        s = capi.Solver(dp, capi.default_options(verbosity_level=0))
    _assert_same_index(_index(s), ref, "side stream")
    s.close()
    torch.cuda.synchronize()


def test_inputs_are_neither_written_nor_needed_after_create():
    meta = common.traces()["traces"]["small_povar"]
    kw = common.flags_to_options(meta["flags"])
    hp = capi.HostProblem.read(common.golden_file("small"))
    s = capi.Solver(hp, capi.default_options(verbosity_level=0, **kw))
    ref = _solve(s)
    s.close()
    dp = _device_problem(hp, _orders(hp.num_obs)[2])
    before = [t.clone() for t in (dp.cam_P, dp.obs_cam, dp.obs_lm, dp.obs_uv)]
    s = capi.Solver(dp, capi.default_options(verbosity_level=0, **kw))
    for b, t in zip(before, (dp.cam_P, dp.obs_cam, dp.obs_lm, dp.obs_uv)):
        assert torch.equal(b, t)
        t.fill_(7)   # right after create returns, before the solve
    _assert_same_run(_solve(s), ref, "inputs overwritten after create")
    s.close()


@pytest.mark.parametrize("which", [capi.STATE_POSE, capi.STATE_JOINT])
def test_device_state_calls_are_stream_ordered_and_match_the_host_calls(which):
    hp = capi.HostProblem.read(common.golden_file("small"))
    opt = capi.default_options(verbosity_level=0)
    a = capi.Solver(hp, opt)
    b = capi.Solver(_device_problem(hp, _orders(hp.num_obs)[3]), opt)
    if which == capi.STATE_JOINT:
        a.to_homogeneous()
        b.to_homogeneous()
    P0, X0 = a.get_state(which)
    rng = np.random.default_rng(3)
    P1 = P0 + 1e-3 * rng.standard_normal(P0.shape)
    X1 = X0 + 1e-3 * rng.standard_normal(X0.shape)
    # set: the perturbed state is produced on the current stream behind a long kernel, no synchronise
    Pd, Xd = torch.from_numpy(P1).cuda(), torch.from_numpy(X1).cuda()
    torch.cuda._sleep(200_000_000)
    Pt, Xt = Pd * 1.0, Xd * 1.0
    b.set_state_device(which, Pt, Xt)
    a.set_state(which, P1, X1)
    ra = a.compute_error_homogeneous() if which == capi.STATE_JOINT else a.compute_error_pOSE(0.1)
    rb = b.compute_error_homogeneous() if which == capi.STATE_JOINT else b.compute_error_pOSE(0.1)
    for f, _ in capi.ResidualInfo._fields_:
        assert getattr(ra, f) == getattr(rb, f), f
    # get: consumed on the current stream without a synchronise
    torch.cuda._sleep(200_000_000)
    P, X = b.get_state_device(which)
    Pc, Xc = (P * 1.0).cpu().numpy(), (X * 1.0).cpu().numpy()
    Ph, Xh = a.get_state(which)
    assert np.array_equal(Pc, Ph) and np.array_equal(Xc, Xh)
    assert np.array_equal(b.get_state(capi.STATE_JOINT)[1], a.get_state(capi.STATE_JOINT)[1])   # w written on set
    a.close()
    b.close()
