"""povar_bundle_adjust_async on the B200: the solve as one graph launch on the caller's stream gives the host driver's
run -- log, summary and final state bit for bit wherever every trust-region radius agrees (the device's cube of the
lambda update is correctly rounded, the host's comes from libm), the same decisions otherwise -- its terminations
and failures, stream order, graph reuse and rebuild, sharded runs, and bad output pointers."""
import ctypes
import os

import numpy as np
import pytest
import torch

import povar_testlib as common
from povar_b200 import capi

pytestmark = pytest.mark.gpu

TIME_COLUMNS = {"iteration_time", "cumulative_time", "residual_evaluation_time", "jacobian_evaluation_time",
                "prepare_time", "solve_reduced_system_time", "back_substitution_time"}
COLUMNS = [f for f, _ in capi.Iteration._fields_ if f not in TIME_COLUMNS]
SUMMARY = ("num_iterations", "termination_type_step_1", "termination_type_step_2", "num_successful_steps",
           "num_unsuccessful_steps", "initial_cost", "final_cost", "power_terms")
DECISIONS = ("step", "iteration", "step_is_valid", "step_is_successful", "linear_solver_iterations")

SOLVERS = {"povar": [], "poba": ["--solver-type-step-1", "POWER_SCHUR_COMPLEMENT"],
           "pcg_ripcg": ["--solver-type-step-1", "PCG", "--solver-type-step-2", "RIPCG"],
           "cholesky": ["--solver-type-step-1", "CHOLESKY"],
           "huber": ["--residual-robust-norm", "HUBER", "--residual-huber-parameter", "30"],
           "error_valid": ["--optimized-cost", "ERROR_VALID"],
           "error_valid_avg": ["--optimized-cost", "ERROR_VALID_AVG"]}
CASES = ([(shape, name) for shape in ("tiny", "small") for name in SOLVERS if name != "error_valid_avg"]
         + [("small", "error_valid_avg"), ("small", "cholesky_tiles"), ("ladybug49", "povar")])


def _options(shape, name, **over):
    meta = common.traces()["traces"].get(f"{shape}_{name}")
    flags = meta["flags"] if meta else SOLVERS["cholesky" if name == "cholesky_tiles" else name]
    return meta, capi.default_options(verbosity_level=0, **{**common.flags_to_options(flags), **over})


def _run(s, opt, route):
    if route == "host":
        its, summary = s.bundle_adjust(opt)
    else:
        its, summary = s.bundle_adjust_async(opt).result()
    P, X = s.get_state(capi.STATE_JOINT)
    return its, summary, P, X


def _val(e, f):
    v = getattr(e, f)
    return v.decode() if isinstance(v, bytes) else v


def _same_bits(a, b):
    return np.array_equal(np.asarray(a, dtype=np.float64).view(np.int64), np.asarray(b, dtype=np.float64).view(np.int64))


def assert_same_run(got, ref, label, meta=None):
    """bitwise where every radius agrees; the same decisions and close costs where the cube differs"""
    (gi, gs, gP, gX), (ri, rs, rP, rX) = got, ref
    assert len(gi) == len(ri), f"{label}: {len(gi)} entries, host {len(ri)}"
    for f in DECISIONS:
        assert [_val(e, f) for e in gi] == [_val(e, f) for e in ri], f"{label}: {f} differs"
    for f in ("termination_type_step_1", "termination_type_step_2", "num_iterations", "num_successful_steps",
              "num_unsuccessful_steps", "power_terms"):
        assert getattr(gs, f) == getattr(rs, f), f"{label}: summary.{f}"
    radius_g = [e.trust_region_radius for e in gi]
    radius_r = [e.trust_region_radius for e in ri]
    if _same_bits(radius_g, radius_r):
        for f in COLUMNS:
            a, b = [_val(e, f) for e in gi], [_val(e, f) for e in ri]
            if a and isinstance(a[0], float):
                assert _same_bits(a, b), f"{label}: column {f} differs"
            else:
                assert a == b, f"{label}: column {f} differs"
        for f in SUMMARY:
            assert getattr(gs, f) == getattr(rs, f), f"{label}: summary.{f}"
        assert _same_bits(gP, rP) and _same_bits(gX, rX), f"{label}: final state differs"
    else:
        k = next(i for i, (a, b) in enumerate(zip(radius_g, radius_r)) if a != b)
        print(f"{label}: first radius difference at entry {k}: {radius_g[k]!r} vs {radius_r[k]!r}")
        if meta:
            common.assert_trace_close(meta, [e.cost for e in ri], [e.step_is_successful for e in ri],
                                      [e.linear_solver_iterations for e in ri], label=f"{label} (host)")
        else:
            for a, b in zip(gi, ri):
                assert common.rel(a.cost, b.cost) <= 1e-6, f"{label}: cost {a.cost} vs {b.cost}"
    if meta:
        common.assert_trace_close(meta, [e.cost for e in gi], [e.step_is_successful for e in gi],
                                  [e.linear_solver_iterations for e in gi], label=f"{label} (async)")


def _pair(shape, opt, tiles=False):
    hp = capi.HostProblem.read(common.golden_file(shape))
    out = []
    for _ in range(2):
        s = capi.Solver(hp, opt)
        if tiles:
            s.debug_set_cholesky_storage(1)
        out.append(s)
    return hp, out


@pytest.mark.parametrize("shape,name", CASES)
def test_async_solve_runs_the_host_driver(shape, name):
    meta, opt = _options(shape, name)
    _, (a, b) = _pair(shape, opt, tiles=name == "cholesky_tiles")
    ref = _run(a, opt, "host")
    got = _run(b, opt, "async")
    assert_same_run(got, ref, f"{shape}_{name}", meta)
    a.close()
    b.close()


@pytest.mark.parametrize("over", [dict(max_num_iterations_step_1=3, max_num_iterations_step_2=2),
                                  dict(function_tolerance=1e-2)])
def test_terminations_match(over):
    _, opt = _options("small", "povar", **over)
    _, (a, b) = _pair("small", opt)
    ref = _run(a, opt, "host")
    got = _run(b, opt, "async")
    assert_same_run(got, ref, f"terminations {over}")
    ms, mg = ref[1].message.decode(), got[1].message.decode()
    if ms.startswith("Function tolerance reached."):
        assert mg == "Function tolerance reached."
    else:
        assert mg == ms
    a.close()
    b.close()


def test_numerical_failure_gives_the_host_status():
    hp = capi.HostProblem.read(common.golden_file("small"))
    hp.obs_uv = hp.obs_uv.copy()
    hp.obs_uv.reshape(-1)[5] = np.nan
    opt = capi.default_options(verbosity_level=0)
    a, b = capi.Solver(hp, opt), capi.Solver(hp, opt)
    with pytest.raises(capi.PovarError) as host:
        a.bundle_adjust(opt)
    with pytest.raises(capi.PovarError) as dev:
        b.bundle_adjust_async(opt).result()
    assert f"povar error {capi.NUM_LINEARIZATION}" in str(host.value)
    assert f"povar error {capi.NUM_LINEARIZATION}" in str(dev.value)
    assert "did not expect numerical failure during linearization" in str(dev.value)
    a.close()
    b.close()


def test_stream_order_reuse_and_rebuild():
    _, opt = _options("small", "povar")
    hp, (a, b) = _pair("small", opt)
    P0, X0 = b.get_state(capi.STATE_POSE)
    ref = _run(a, opt, "host")
    first = _run(b, opt, "async")   # builds the graph
    assert_same_run(first, ref, "first")
    # stream order: the state is set behind a long kernel on the current stream, the solve is enqueued behind it
    Pd, Xd = torch.from_numpy(P0).cuda(), torch.from_numpy(X0).cuda()
    torch.cuda._sleep(200_000_000)
    b.set_state_device(capi.STATE_POSE, Pd * 1.0, Xd * 1.0)
    job = b.bundle_adjust_async(opt)
    assert not torch.cuda.current_stream().query()
    P, X = b.get_state_device(capi.STATE_JOINT)
    Pc, Xc = P.cpu().numpy(), X.cpu().numpy()
    second = job.result()
    assert _same_bits(Pc, first[2]) and _same_bits(Xc, first[3])
    assert len(second[0]) == len(first[0])
    for f in COLUMNS:
        now, then = [_val(e, f) for e in second[0]], [_val(e, f) for e in first[0]]
        assert (_same_bits(now, then) if isinstance(now[0], float) else now == then), f"reuse: column {f} differs"
    # rebuild: other options give the host route's result for them
    _, opt2 = _options("small", "povar", max_num_iterations_step_2=3)
    for s in (a, b):
        s.set_state(capi.STATE_POSE, P0, X0)
    assert_same_run(_run(b, opt2, "async"), _run(a, opt2, "host"), "rebuilt")
    a.close()
    b.close()


def test_host_route_follows_a_changed_alpha():
    """a handle's cached power-series graph is captured with the model parameters: a later solve with another alpha
    gives what a fresh handle gives, on both routes"""
    _, opt = _options("small", "povar")
    _, opt2 = _options("small", "povar", alpha=0.01)
    hp = capi.HostProblem.read(common.golden_file("small"))
    for route in ("host", "async"):
        used, fresh = capi.Solver(hp, opt), capi.Solver(hp, opt)
        P0, X0 = used.get_state(capi.STATE_POSE)
        _run(used, opt, route)
        used.set_state(capi.STATE_POSE, P0, X0)
        assert_same_run(_run(used, opt2, route), _run(fresh, opt2, route), f"{route}: alpha changed")
        used.close()
        fresh.close()


def _worker_shards(rank, world, hid, path, kw, out_dir):
    import torch as _torch  # noqa: F401  (initialises CUDA in the spawned process)
    hp = capi.HostProblem.read(path).shard(rank, world)
    runs = {}
    for route in ("host", "async"):
        s = capi.Solver(hp, capi.default_options(verbosity_level=0, **kw), capi.make_comm(rank, world, 0, hid))
        its, summary, P, X = _run(s, s.options, route)
        runs[route] = dict(cost=[e.cost for e in its], succ=[e.step_is_successful for e in its],
                           lin=[e.linear_solver_iterations for e in its],
                           radius=[e.trust_region_radius for e in its], P=P, X=X, final=summary.final_cost)
        s.close()
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"),
             **{f"{r}_{k}": np.asarray(v) for r, d in runs.items() for k, v in d.items()})
    capi.load().povar_comm_finalize()


@pytest.mark.parametrize("name,world", [("small_povar", 2), ("small_poba", 3)])
def test_sharded_async_runs_the_host_sharded_trace(name, world, tmp_path):
    import torch.multiprocessing as mp
    meta = common.traces()["traces"][name]
    kw = common.flags_to_options(meta["flags"])
    mp.spawn(_worker_shards, args=(world, capi.host_id(), common.golden_file(meta["shape"]), kw, str(tmp_path)),
             nprocs=world, join=True)
    for r in range(world):
        z = np.load(tmp_path / f"rank{r}.npz")
        for k in ("succ", "lin"):
            assert np.array_equal(z[f"host_{k}"], z[f"async_{k}"]), f"{name} x{world} rank {r}: {k} differs"
        if _same_bits(z["host_radius"], z["async_radius"]):
            for k in ("cost", "P", "X", "final"):
                assert _same_bits(z[f"host_{k}"], z[f"async_{k}"]), f"{name} x{world} rank {r}: {k} differs"


def _worker_nccl(rank, world, nid, path, out_dir):
    os.environ["POVAR_PEER_EXCHANGE"] = "0"
    hp = capi.HostProblem.read(path).shard(rank, world)
    torch.cuda.set_device(rank)
    s = capi.Solver(hp, capi.default_options(verbosity_level=0), capi.make_comm(rank, world, rank, nid))
    with torch.cuda.device(rank):
        buf = torch.empty(4096, dtype=torch.uint8, device=f"cuda:{rank}")
        rc = s.lib.povar_bundle_adjust_async(s.h, ctypes.byref(s.options), buf.data_ptr(), 1, buf.data_ptr(),
                                             buf.data_ptr(), None)
    np.save(os.path.join(out_dir, f"rc{rank}.npy"), np.array([rc, int(s.peer_exchange_active())]))
    s.close()
    capi.load().povar_comm_finalize()


def test_nccl_reductions_are_unsupported(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_worker_nccl, args=(2, capi.unique_id(), common.golden_file("small"), str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        rc, active = np.load(tmp_path / f"rc{r}.npy")
        assert active == 0 and rc == capi.ERR_UNSUPPORTED


def test_host_output_pointers_are_invalid_and_the_next_call_works():
    _, opt = _options("tiny", "povar")
    hp = capi.HostProblem.read(common.golden_file("tiny"))
    s = capi.Solver(hp, opt)
    lib = s.lib
    cap = opt.max_num_iterations_step_1 + opt.max_num_iterations_step_2 + 2
    log = torch.empty(cap * ctypes.sizeof(capi.Iteration), dtype=torch.uint8, device="cuda")
    summ = torch.empty(ctypes.sizeof(capi.SolveSummary), dtype=torch.uint8, device="cuda")
    st = torch.empty(1, dtype=torch.int32, device="cuda")
    host = np.zeros(1 << 16, dtype=np.uint8)
    stream = torch.cuda.current_stream().cuda_stream
    good = [log.data_ptr(), summ.data_ptr(), st.data_ptr()]
    for i in range(3):
        args = list(good)
        args[i] = host.ctypes.data
        rc = lib.povar_bundle_adjust_async(s.h, ctypes.byref(opt), args[0], cap, args[1], args[2], stream)
        assert rc == capi.ERR_INVALID, i
        assert lib.povar_last_error(s.h)
    assert lib.povar_bundle_adjust_async(s.h, ctypes.byref(opt), good[0], cap, good[1], good[2], stream) == capi.OK
    torch.cuda.synchronize()
    assert int(st.cpu()[0]) == capi.OK
    s.close()
