"""The tile-sparse CHOLESKY (kernels_chol.cu with the SparseTiles / TiledS policies, host/chol_symbolic.cpp): the
direct solver on caller-supplied matrices, parity of the forced tile-sparse path with the reference's golden traces
and with the dense path, and the scene the dense path refuses (10,000 cameras: 115 GB dense).  `pytest -m gpu`."""
import subprocess

import numpy as np
import pytest

import povar_testlib as common
import test_gpu_parity as parity
import test_gpu_parity_large as parity_large
from povar_b200 import build, capi, synthetic

pytestmark = pytest.mark.gpu

TILE = 64


def _block_banded(nb, block, n, width, closure, seed):
    """SPD matrix of order n with the block pattern of a band of `width` blocks (+ the block (nb-1, 0)), and the
    camera problem of the same graph (cholesky_symbolic gives the order the solver uses when block = 12)"""
    rng = np.random.default_rng(seed)
    pairs = [(a, b) for a in range(nb) for b in range(max(0, a - width), a)]
    if closure:
        pairs.append((nb - 1, 0))
    A = np.zeros((nb * block, nb * block))
    for a, b in pairs:
        blk = rng.normal(size=(block, block))
        A[a * block:(a + 1) * block, b * block:(b + 1) * block] = blk
        A[b * block:(b + 1) * block, a * block:(a + 1) * block] = blk.T
    for c in range(nb):
        blk = rng.normal(size=(block, block))
        A[c * block:(c + 1) * block, c * block:(c + 1) * block] = blk @ blk.T
    A = A[:n, :n]
    A += np.diag(np.abs(A).sum(axis=1) * 0.5 + 1.0)
    lms = [[b, a] for a, b in pairs] + [[c] for c in range(nb)]
    lm_ptr = np.concatenate([[0], np.cumsum([len(l) for l in lms])])
    obs_cam = np.concatenate([np.asarray(sorted(l), np.int32) for l in lms])
    hp = capi.HostProblem(nb, len(lms), lm_ptr, obs_cam, np.zeros((obs_cam.size, 2)), np.zeros((nb, 15)))
    return A, hp


@pytest.mark.parametrize("nb,n,closure", [(16, 192, False), (37, 444, False), (37, 444, True), (64, 768, True),
                                          (84, 1000, False), (120, 1440, True)])
def test_sparse_cholesky_solves_like_numpy(nb, n, closure):
    A, _ = _block_banded(nb, 12, n, 3, closure, seed=n + closure)
    b = np.random.default_rng(n).normal(size=n)
    x, info, tiles = capi.sparse_cholesky_solve(A, b)
    assert info == 0
    ref = np.linalg.solve(A, b)
    assert common.rel(x, ref) < 1e-9 * max(1.0, np.linalg.cond(A) / 1e6)
    assert np.linalg.norm(A @ x - b) <= 1e-10 * np.linalg.norm(b) * np.sqrt(n)
    T = -(-n // TILE)
    if T > 4:
        assert 0 < tiles < T * (T + 1) // 2
    # only the lower triangle is read
    U = A.copy()
    U[np.triu_indices(n, 1)] = 123.0
    assert np.array_equal(x, capi.sparse_cholesky_solve(U, b)[0])
    # twice the same bits
    assert np.array_equal(x, capi.sparse_cholesky_solve(A, b)[0])


def test_sparse_cholesky_reports_the_first_bad_tile_in_factor_order():
    nb = 40
    A, hp = _block_banded(nb, 12, 12 * nb, 3, True, seed=3)
    perm, _ = capi.cholesky_symbolic(hp)

    def tile_of(i):
        return (12 * int(perm[i // 12]) + i % 12) // TILE

    B = A.copy()
    B[250, 250] = -1.0
    assert capi.sparse_cholesky_solve(B, np.ones(12 * nb))[1] == tile_of(250) + 1
    B = A.copy()
    B[3, 3] = np.nan
    assert capi.sparse_cholesky_solve(B, np.ones(12 * nb))[1] == tile_of(3) + 1


def _forced_trace(name, **override):
    meta = common.traces()["traces"][name]
    kw = common.flags_to_options(meta["flags"])
    kw.update(override)
    hp = capi.HostProblem.read(common.golden_file(meta["shape"]))
    s = capi.Solver(hp, capi.default_options(verbosity_level=0, **kw))
    s.debug_set_cholesky_storage(1)
    its, summary = s.bundle_adjust()
    assert s.debug_read("chol_tiles")[0] > 0
    s.close()
    return meta, its, summary


def test_small_cholesky_on_tiles_matches_reference_golden(monkeypatch):
    """the bars of test_two_step_trace_matches_reference_golden, with the tile-sparse path forced"""
    monkeypatch.setattr(parity, "_gpu_trace", _forced_trace)
    parity.test_two_step_trace_matches_reference_golden("small_cholesky")


def test_trafalgar257_cholesky_on_tiles_matches_reference_golden():
    name = "trafalgar257_cholesky"
    meta = common.traces_large()["traces"][name]
    hp = capi.HostProblem.read(common.golden_file(meta["shape"]))
    s = capi.Solver(hp, capi.default_options(verbosity_level=0, **common.flags_to_options(meta["flags"])))
    s.debug_set_cholesky_storage(1)
    its, summary = s.bundle_adjust()
    assert s.debug_read("chol_tiles")[0] > 0
    s.close()
    print(parity_large.check_against_reference(name, meta, its, summary))


def _one_solve(hp, storage, lam=1e-2):
    s = capi.Solver(hp, capi.default_options(alpha=0.1, solver_type_step_1=capi.CHOLESKY, verbosity_level=0))
    if storage is not None:
        s.debug_set_cholesky_storage(storage)
    s.initialize_varproj_lm_pOSE(0.1)
    assert s.linearize_pOSE(0.1) == capi.OK
    inc, its, rc = s.solve(lam)
    assert rc == capi.OK and its == 0
    inc2, _, _ = s.solve(lam)
    assert np.array_equal(inc, inc2)
    C = hp.num_cams
    b = s.debug_read("b").reshape(C, 12)
    Bm = s.debug_read("b_mat").reshape(C, 12, 12)
    res = np.einsum("cij,cj->ci", Bm, inc) - s.right_mul_e0(capi.STATE_POSE, inc) + b
    tiles = s.debug_read("chol_tiles")
    perm = s.debug_read("chol_perm")
    s.close()
    return inc, np.linalg.norm(res) / np.linalg.norm(b), tiles, perm


@pytest.mark.parametrize("shape", ["small", "ladybug49"])
def test_sparse_and_dense_solves_agree(shape):
    hp = capi.HostProblem.read(common.golden_file(shape))
    dense, res_d, tiles_d, perm_d = _one_solve(hp, 0)
    sparse, res_s, tiles_s, perm_s = _one_solve(hp, 1)
    assert tiles_d.size == 0 and perm_d.size == 0           # automatic: dense at this size
    assert tiles_s.size == 1 and tiles_s[0] > 0
    assert np.array_equal(np.sort(perm_s), np.arange(hp.num_cams))
    assert res_d <= 1e-8 and res_s <= 1e-8, (res_d, res_s)
    assert common.rel(sparse, dense) <= 1e-9


def test_one_handle_switched_between_the_storages():
    """povar_debug_set_cholesky_storage on a live handle: each solve uses the storage asked for, "chol_tiles" /
    "chol_perm" follow it, and the dense solve after a tile-sparse one gives the bits of a fresh dense handle."""
    hp = capi.HostProblem.read(common.golden_file("ladybug49"))
    fresh = _one_solve(hp, 0)[0]
    s = capi.Solver(hp, capi.default_options(alpha=0.1, solver_type_step_1=capi.CHOLESKY, verbosity_level=0))
    s.initialize_varproj_lm_pOSE(0.1)
    assert s.linearize_pOSE(0.1) == capi.OK
    s.debug_set_cholesky_storage(1)
    tiled = s.solve(1e-2)[0]
    assert s.debug_count("chol_tiles") == 1 and s.debug_count("chol_perm") == hp.num_cams
    s.debug_set_cholesky_storage(0)
    dense = s.solve(1e-2)[0]
    assert s.debug_count("chol_tiles") == 0 and s.debug_count("chol_perm") == 0
    s.debug_set_cholesky_storage(1)
    assert np.array_equal(s.solve(1e-2)[0], tiled)
    s.close()
    assert np.array_equal(dense, fresh)
    assert common.rel(tiled, dense) <= 1e-9


@pytest.fixture(scope="module")
def scene10k():
    sp = synthetic.generate(10000, 200000, 1_000_000, seed=77, window_frac=0.005)
    return sp, capi.HostProblem.from_unordered(sp.num_cams, sp.num_lms, sp.obs_cam, sp.obs_lm, sp.obs_xy,
                                               sp.cam_params)


def test_ten_thousand_cameras_solve_on_tiles(scene10k):
    """12 x 10,000 rows: the dense reduced system would take 115 GB and is refused; automatic mode takes the tiles."""
    _, hp = scene10k
    inc, res, tiles, perm = _one_solve(hp, None)
    T = 12 * 10000 // TILE
    assert tiles.size == 1 and 0 < tiles[0] <= 0.03 * T * (T + 1) // 2
    assert np.array_equal(np.sort(perm), np.arange(hp.num_cams))
    assert np.all(np.isfinite(inc)) and res <= 1e-8, res


def test_ten_thousand_cameras_bundle_adjust(scene10k):
    _, hp = scene10k
    opt = capi.default_options(alpha=0.1, solver_type_step_1=capi.CHOLESKY, verbosity_level=0,
                               max_num_iterations_step_1=5, max_num_iterations_step_2=2)
    s = capi.Solver(hp, opt)
    its, summary = s.bundle_adjust()
    s.close()
    step1 = [e for e in its if e.step == 1]
    step2 = [e for e in its if e.step == 2]
    assert step2 and max(e.iteration for e in step1) <= 5 and max(e.iteration for e in step2) <= 2
    assert summary.num_successful_steps > 0
    accepted = [e.cost for e in step1 if e.step_is_successful]
    assert len(accepted) >= 2
    assert all(b <= a for a, b in zip(accepted, accepted[1:])), accepted


def test_bal_cholesky_runs_on_ten_thousand_cameras(scene10k, tmp_path):
    sp, _ = scene10k
    path = tmp_path / "scene10k.txt"
    synthetic.write_bal(sp, str(path))
    res = subprocess.run([build.BAL, "--input", str(path), "--solver-type-step-1", "CHOLESKY", "--alpha", "0.1",
                          "--max-num-iterations-step-1", "2", "--max-num-iterations-step-2", "1",
                          "--verbosity-level", "0", "--log-log-path", str(tmp_path / "log.json")],
                         capture_output=True, text=True, cwd=tmp_path)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "96 GB" not in res.stdout + res.stderr
