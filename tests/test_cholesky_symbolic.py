"""The host side of the tile-sparse CHOLESKY (host/chol_symbolic.cpp): reverse Cuthill-McKee camera order and the
symbolic factorisation on 64x64 tiles, through povar_debug_cholesky_symbolic.  CPU only.

The fill check factorises, in numpy, random SPD matrices with exactly a scene's 12x12 block pattern in the
library's camera order and asserts that every non-zero of L lies in a tile of the symbolic pattern; the pattern is
recomputed here from the order (tile pattern of S, then right-looking elimination on tiles) and the library must
store exactly as many tiles."""
import numpy as np
import pytest

from povar_b200 import capi, synthetic

TILE = 64


def _problem(num_cams, cams_of_landmark):
    lists = [sorted(set(c)) for c in cams_of_landmark]
    lm_ptr = np.concatenate([[0], np.cumsum([len(c) for c in lists])])
    obs_cam = np.concatenate([np.asarray(c, np.int32) for c in lists])
    n = obs_cam.shape[0]
    return capi.HostProblem(num_cams, len(lists), lm_ptr, obs_cam, np.zeros((n, 2)), np.zeros((num_cams, 15)))


def _named(shape):
    sp = synthetic.generate_named(shape)
    return capi.HostProblem.from_unordered(sp.num_cams, sp.num_lms, sp.obs_cam, sp.obs_lm, sp.obs_xy, sp.cam_params)


def _banded(num_cams, width, closure=False, shuffle=None):
    lms = [list(range(i, i + width + 1)) for i in range(num_cams - width)]
    if closure:
        lms.append([0, num_cams - 1])
    if shuffle is not None:
        sigma = np.random.default_rng(shuffle).permutation(num_cams)
        lms = [[int(sigma[c]) for c in l] for l in lms]
    return _problem(num_cams, lms)


def _pairs(hp):
    """co-observing camera pairs (a, b), a > b"""
    out = set()
    for l in range(hp.num_lms):
        cams = hp.obs_cam[hp.lm_ptr[l]:hp.lm_ptr[l + 1]]
        for i, a in enumerate(cams):
            for b in cams[:i]:
                out.add((max(int(a), int(b)), min(int(a), int(b))))
    return sorted(out)


def _tiles_of(pos):
    return range(12 * pos // TILE, (12 * pos + 11) // TILE + 1)


def _reference_pattern(hp, perm):
    T = -(-12 * hp.num_cams // TILE)
    P = np.eye(T, dtype=bool)
    for c in range(hp.num_cams):
        for I in _tiles_of(perm[c]):
            for J in _tiles_of(perm[c]):
                P[max(I, J), min(I, J)] = True
    for a, b in _pairs(hp):
        for I in _tiles_of(perm[a]):
            for J in _tiles_of(perm[b]):
                P[max(I, J), min(I, J)] = True
    for k in range(T):
        rows = np.nonzero(P[k + 1:, k])[0] + k + 1
        P[np.ix_(rows, rows)] |= np.tril(np.ones((rows.size, rows.size), dtype=bool))
    return P


def _random_spd(hp, rng):
    C = hp.num_cams
    A = np.zeros((12 * C, 12 * C))
    for a, b in _pairs(hp):
        blk = rng.normal(size=(12, 12))
        A[12 * a:12 * a + 12, 12 * b:12 * b + 12] = blk
        A[12 * b:12 * b + 12, 12 * a:12 * a + 12] = blk.T
    for c in range(C):
        blk = rng.normal(size=(12, 12))
        A[12 * c:12 * c + 12, 12 * c:12 * c + 12] = blk + blk.T
    A += np.diag(np.abs(A).sum(axis=1) + 1.0)    # diagonally dominant: SPD
    return A


@pytest.mark.parametrize("case", ["small", "ladybug49", "trafalgar257", "banded_closure"])
def test_symbolic_pattern_covers_the_fill_of_the_factor(case):
    hp = _banded(60, 3, closure=True) if case == "banded_closure" else _named(case)
    perm, tiles = capi.cholesky_symbolic(hp)
    C = hp.num_cams
    assert np.array_equal(np.sort(perm), np.arange(C))
    P = _reference_pattern(hp, perm)
    assert tiles == int(P.sum())
    T = P.shape[0]
    # the matrix in the factor order: row 12 c + k of camera c goes to 12 perm[c] + k, identity on the padding
    q = (12 * perm[:, None] + np.arange(12)[None]).reshape(-1)
    A = np.eye(T * TILE)
    A[np.ix_(q, q)] = _random_spd(hp, np.random.default_rng(C))
    L = np.linalg.cholesky(A)
    nz = (np.abs(L) > 0).reshape(T, TILE, T, TILE).any(axis=(1, 3))
    assert not np.any(nz & ~P), np.argwhere(nz & ~P)[:5]


def test_loop_closure_costs_tiles_not_correctness():
    open_band = capi.cholesky_symbolic(_banded(60, 3))[1]
    closed = capi.cholesky_symbolic(_banded(60, 3, closure=True))[1]
    assert closed > open_band


@pytest.mark.parametrize("case", ["ladybug49", "trafalgar257", "banded_shuffled"])
def test_order_does_not_depend_on_the_host_threads(case):
    hp = _banded(300, 4, shuffle=5) if case == "banded_shuffled" else _named(case)
    runs = [capi.cholesky_symbolic(hp, threads=t) for t in (1, 2, 8)]
    for perm, tiles in runs[1:]:
        assert np.array_equal(perm, runs[0][0]) and tiles == runs[0][1]


def test_reverse_cuthill_mckee_recovers_a_narrow_band():
    width = 3
    hp = _banded(400, width, shuffle=7)
    pairs = np.array(_pairs(hp))
    assert np.max(np.abs(pairs[:, 0] - pairs[:, 1])) > 100        # the shuffled labels have no band
    perm, _ = capi.cholesky_symbolic(hp)
    assert np.max(np.abs(perm[pairs[:, 0]] - perm[pairs[:, 1]])) <= width


def test_every_component_is_ordered_isolated_cameras_included():
    # cameras 0..9 a chain, 10..14 a second chain, 15..19 see no landmark shared with another camera
    lms = [[i, i + 1] for i in range(9)] + [[i, i + 1] for i in range(10, 14)] + [[c] for c in range(15, 20)]
    perm, tiles = capi.cholesky_symbolic(_problem(20, lms))
    assert np.array_equal(np.sort(perm), np.arange(20))
    assert tiles >= -(-12 * 20 // TILE)


def test_malformed_index_is_rejected():
    hp = _banded(20, 2)
    bad = capi.HostProblem(hp.num_cams, hp.num_lms, hp.lm_ptr - 1, hp.obs_cam, hp.obs_uv, hp.cam_params)
    with pytest.raises(capi.PovarError):
        capi.cholesky_symbolic(bad)                  # lm_ptr[0] != 0
    cams = hp.obs_cam.copy()
    cams[3] = hp.num_cams
    with pytest.raises(capi.PovarError):
        capi.cholesky_symbolic(capi.HostProblem(hp.num_cams, hp.num_lms, hp.lm_ptr, cams, hp.obs_uv, hp.cam_params))


def test_ten_thousand_camera_scene_keeps_a_few_percent_of_the_tiles():
    """The 10,000-camera sequence whose dense reduced system (115 GB) exceeds the dense path's 96 GB."""
    sp = synthetic.generate(10000, 200000, 1_000_000, seed=77, window_frac=0.005)
    hp = capi.HostProblem.from_unordered(sp.num_cams, sp.num_lms, sp.obs_cam, sp.obs_lm, sp.obs_xy, sp.cam_params)
    perm, tiles = capi.cholesky_symbolic(hp)
    T = 12 * 10000 // TILE
    assert np.array_equal(np.sort(perm), np.arange(10000))
    assert tiles <= 0.03 * T * (T + 1) // 2, tiles
