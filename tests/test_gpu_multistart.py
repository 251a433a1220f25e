"""Multi-start alignment (icpb_run_multistart_host / icp_multistart): every pair aligned from K start
transforms, the best start kept.

* Every problem gives the bits icp_batch gives on the expanded list -- pair p repeated K times with the
  guesses compose_starts(init, starts) -- and the winner is np.argmin over the errors.
* Against the C oracle and the reference's golden outputs with the tolerances of test_gpu_parity.py.
* Ties go to the lowest start index; slices of 2^22 problems; the argument contract; the loop-closure
  callers with a heading sweep.
"""
import ctypes
import functools

import numpy as np
import pytest

from conftest import load_golden, pose_diff

pytestmark = pytest.mark.gpu

EINVAL = 10001


@pytest.fixture(scope="module")
def gicp():
    from icp_slam_b200 import icp as m
    return m


@pytest.fixture(scope="module")
def synth():
    from icp_slam_b200 import synth as m
    return m


@pytest.fixture(scope="module")
def eng(gicp):
    e = gicp.IcpEngine()
    yield e
    e.close()


@functools.lru_cache(maxsize=None)
def _chain(n_scans, n_beams):
    from icp_slam_b200 import synth
    scans, pairs, init, _, _ = synth.make_chain_workload(n_scans, n_beams, seed=8100 + n_beams)
    return scans, pairs, init


CHAIN_SCANS = {360: 10, 1024: 6, 4096: 3}


def _expanded(gicp, init, S, B):
    G = gicp.compose_starts(init, S)
    return np.ascontiguousarray(np.broadcast_to(G, (B,) + G.shape[1:])).reshape(-1, 3, 3)


def _check_expansion(eng, gicp, pairs, init, S, exhaustive=False, **kw):
    """return_all of the multi-start run against the resident-table run of the expanded list."""
    B, K = len(pairs), len(S)
    ms = eng.run_multistart(pairs, S, init, return_all=True, exhaustive=exhaustive, **kw)
    ref = eng.run(np.repeat(pairs, K, axis=0), _expanded(gicp, init, S, B), exhaustive=exhaustive, **kw)
    assert ms.error_all.shape == (B, K) and ms.iters_all.shape == (B, K) and ms.start.dtype == np.int32
    np.testing.assert_array_equal(ms.error_all.reshape(-1), ref.error)
    np.testing.assert_array_equal(ms.iters_all.reshape(-1), ref.iters)
    np.testing.assert_array_equal(ms.start, np.argmin(ref.error.reshape(B, K), axis=1))
    w = np.arange(B) * K + ms.start
    np.testing.assert_array_equal(ms.T, ref.T[w])
    np.testing.assert_array_equal(ms.error, ref.error[w])
    np.testing.assert_array_equal(ms.iters, ref.iters[w])
    return ms


# ------------------------------------------------------------------ bit identity with the expansion
@pytest.mark.parametrize("beams", [360, 1024, 4096])
@pytest.mark.parametrize("K", [1, 2, 7, 32])
@pytest.mark.parametrize("guess", ["odometry", "identity"])
def test_chain_equals_expanded_batch(eng, gicp, beams, K, guess):
    scans, pairs, init = _chain(CHAIN_SCANS[beams], beams)
    eng.set_scans(scans)
    _check_expansion(eng, gicp, pairs, init if guess == "odometry" else None, gicp.heading_starts(K), epsilon=0.05)


def test_proximity_pairs_equal_expanded_batch(eng, gicp, synth):
    rng = np.random.default_rng(8201)
    poses = synth.loop_trajectory(400, step=0.2)
    scans = synth.scans_from_poses(poses, 360, rng, drop_frac=0.03)
    pairs = synth.proximity_pairs(poses, max_pairs=60, seed=8201)
    assert len(pairs) == 60
    eng.set_scans(scans)
    _check_expansion(eng, gicp, pairs, None, gicp.heading_starts(8), epsilon=0.05)


@pytest.mark.parametrize("case", ["rotation_only", "exhaustive", "large", "cluster"])
def test_variants_equal_expanded_batch(eng, gicp, case):
    scans, pairs, init = _chain(CHAIN_SCANS[1024], 1024)
    eng.set_scans(scans)
    S = gicp.heading_starts(7)
    if case == "rotation_only":
        _check_expansion(eng, gicp, pairs, init, S, epsilon=0.05, rotation_only=True)
    elif case == "exhaustive":
        _check_expansion(eng, gicp, pairs, init, S, epsilon=0.05, exhaustive=True)
    elif case == "large":
        eng.set_tuning("large", 1)
        try:
            _check_expansion(eng, gicp, pairs, init, S, epsilon=0.05)
        finally:
            eng.set_tuning("large", -1)
    else:
        # 2 pairs x 7 starts of 1,024 points: few enough problems that each gets a thread-block cluster
        _check_expansion(eng, gicp, pairs[:2], init[:2], S, epsilon=0.05)


def _submap(synth, seed, n_beams=1024, k=16):
    """A 1,024-beam source scan and the k scans before it merged into the frame of the first of them."""
    rng = np.random.default_rng(seed)
    poses = synth.loop_trajectory(k + 1, step=0.04)
    scans = synth.scans_from_poses(poses, n_beams, rng)
    M0inv = np.linalg.inv(synth.pose_to_mat(poses[0]))
    parts = []
    for i in range(k):
        A = M0inv @ synth.pose_to_mat(poses[i])
        parts.append(scans[i] @ A[:2, :2].T + A[:2, 2])
    init = M0inv @ synth.pose_to_mat(poses[k])
    return scans[k], np.ascontiguousarray(np.concatenate(parts)), init


def test_split_table_equals_expanded_batch(eng, gicp, synth):
    """A table holding a 16,384-point submap: every slice is split by scan length, two launches."""
    scans, pairs, init = _chain(CHAIN_SCANS[1024], 1024)
    src, sub, isub = _submap(synth, seed=8301)
    n = len(scans)
    table = list(scans) + [src, sub]
    all_pairs = np.concatenate([pairs, [[n, n + 1], [n + 1, 0]]]).astype(np.int32)
    all_init = np.concatenate([init, [isub, np.eye(3)]])
    eng.set_scans(table)
    S = gicp.heading_starts(7)
    n0 = eng.launch_count
    eng.run_multistart(all_pairs, S, all_init, epsilon=0.05)
    assert eng.launch_count - n0 == 2
    _check_expansion(eng, gicp, all_pairs, all_init, S, epsilon=0.05)


def test_one_identity_start_equals_batch(eng, gicp):
    scans, pairs, init = _chain(CHAIN_SCANS[360], 360)
    eng.set_scans(scans)
    for guess in (init, None):
        ms = eng.run_multistart(pairs, np.eye(3)[None], guess, epsilon=0.05)
        ref = eng.run(pairs, guess, epsilon=0.05)
        np.testing.assert_array_equal(ms.T, ref.T)
        np.testing.assert_array_equal(ms.error, ref.error)
        np.testing.assert_array_equal(ms.iters, ref.iters)
        assert not ms.start.any()


# ------------------------------------------------------------------ oracle and goldens
def test_heading_sweep_matches_oracle(gicp):
    from oracle import c_oracle
    c_oracle.build()
    scans, pairs, _ = _chain(7, 360)
    S = gicp.heading_starts(8)
    ms = gicp.icp_multistart(scans, pairs, S, epsilon=0.05, return_all=True)
    xy, off = c_oracle.pack(scans)
    T, err, passes = c_oracle.icp_batch(xy, off, np.repeat(pairs, 8, axis=0), _expanded(gicp, None, S, 6),
                                        epsilon=0.05)
    np.testing.assert_array_equal(ms.iters_all.reshape(-1), passes)
    np.testing.assert_allclose(ms.error_all.reshape(-1), err, rtol=1e-9, atol=1e-20)
    # The winner is np.argmin over the library's own errors.  Starts that converge to the same minimum
    # have errors equal to ~1e-12 relative, whose last bits the oracle's scalar sums round differently,
    # so the oracle's argmin may name another of them: compare the winner's run with the oracle's run of
    # the same start, and check that it is the oracle's minimum up to that rounding.
    np.testing.assert_array_equal(ms.start, np.argmin(ms.error_all, axis=1))
    w = np.arange(6) * 8 + ms.start
    assert np.abs(ms.T - T[w]).max() < 1e-9
    np.testing.assert_allclose(err[w], err.reshape(6, 8).min(axis=1), rtol=1e-9, atol=1e-20)


def test_golden_L_identity_start_meets_its_golden(gicp, synth):
    case = [c for c in load_golden() if c.name == "L_defaults"][0]
    S = np.stack([np.eye(3), synth.pose_to_mat((0.0, 0.0, np.pi))])
    ms = gicp.icp_multistart([case.src, case.dst], [[0, 1]], S, return_all=True, **case.kwargs)
    assert ms.iters_all[0, 0] == len(case.transforms) - 1
    np.testing.assert_allclose(ms.error_all[0, 0], case.error, rtol=1e-9, atol=1e-20)
    assert ms.start[0] == 0
    np.testing.assert_allclose(ms.T[0], case.transforms[-1], rtol=0, atol=1e-9)


# ------------------------------------------------------------------ ties
def test_ties_go_to_the_lowest_start(eng, gicp, synth):
    scans, pairs, init = _chain(CHAIN_SCANS[360], 360)
    eng.set_scans(scans)
    R = [synth.pose_to_mat((0.0, 0.0, t)) for t in (np.pi / 2, np.pi, -np.pi / 2)]
    S = np.stack([R[0], np.eye(3), R[1], np.eye(3), R[2]])        # the identity at k = 1 and k = 3
    ms = _check_expansion(eng, gicp, pairs, None, S, epsilon=0.05)
    np.testing.assert_array_equal(ms.error_all[:, 1], ms.error_all[:, 3])
    assert (ms.start == 1).any() and not (ms.start == 3).any()
    same = np.tile(synth.pose_to_mat((0.0, 0.0, 0.3)), (6, 1, 1))  # all K identical
    ms = _check_expansion(eng, gicp, pairs, init, same, epsilon=0.05)
    assert not ms.start.any()


# ------------------------------------------------------------------ slices
def test_slices_at_the_real_boundary(eng, gicp):
    """K = 1 and 2^22 + 1 pairs: two slices, one launch each; the results are icp_batch's."""
    scans, pairs, _ = _chain(CHAIN_SCANS[360], 360)
    eng.set_scans(scans)
    B = (1 << 22) + 1
    big = np.ascontiguousarray(np.resize(pairs, (B, 2)))
    eng.run(pairs[:1], None, epsilon=0.05)                       # the table's staging images exist
    n0 = eng.launch_count
    ms = eng.run_multistart(big, np.eye(3)[None], None, epsilon=0.05)
    assert eng.launch_count - n0 == 2
    ref = eng.run(big, None, epsilon=0.05)
    np.testing.assert_array_equal(ms.T, ref.T)
    np.testing.assert_array_equal(ms.error, ref.error)
    np.testing.assert_array_equal(ms.iters, ref.iters)
    assert not ms.start.any()


def test_launches_per_slice(eng, gicp):
    scans, pairs, init = _chain(CHAIN_SCANS[360], 360)
    eng.set_scans(scans)                                          # a new table: no staging images yet
    S = gicp.heading_starts(4)
    n0 = eng.launch_count
    eng.run_multistart(pairs, S, init, epsilon=0.05)
    assert eng.launch_count - n0 == 2                             # the prep launch, then the slice
    n0 = eng.launch_count
    eng.run_multistart(pairs, S, init, epsilon=0.05)
    assert eng.launch_count - n0 == 1


# ------------------------------------------------------------------ contract
def _raw(eng, gicp, pairs, S6, K, init6=None, null_starts=False, **params):
    """icpb_run_multistart_host through ctypes: the status it returns."""
    from icp_slam_b200 import _lib
    p = _lib.default_params()
    p.epsilon = 0.05
    for k, v in params.items():
        setattr(p, k, v)
    pairs = np.ascontiguousarray(pairs, dtype=np.int32)
    B = len(pairs)
    K_out = max(int(K), 1) if int(K) <= 64 else 1
    T, err = np.empty((B, 6)), np.empty(B)
    passes, start = np.empty(B, dtype=np.int32), np.empty(B, dtype=np.int32)
    ptr = gicp._ptr
    return eng._L.icpb_run_multistart_host(eng._h, ptr(pairs), ptr(init6), B, None if null_starts else ptr(S6),
                                           int(K), ctypes.byref(p), ptr(T), ptr(err), ptr(passes), ptr(start),
                                           ptr(np.empty((B, K_out))), ptr(np.empty((B, K_out), dtype=np.int32)))


def test_contract_rejections(eng, gicp, synth):
    scans, pairs, init = _chain(CHAIN_SCANS[360], 360)
    eng.set_scans(scans)
    S = gicp.heading_starts(4)
    before = eng.run_multistart(pairs, S, init, epsilon=0.05, return_all=True)
    S6 = np.ascontiguousarray(S[:, :2].reshape(-1, 6))
    init6 = np.ascontiguousarray(init[:, :2].reshape(-1, 6))
    n_scans = len(scans)
    # init linear part [[1e3, 1e3], [0, 1]] and S = R(pi/4) are each within the bounds; G00 ~ 1414 is not
    wide = np.tile(np.array([[1e3, 1e3, 0.0], [0.0, 1.0, 0.0], [0.0, 0.0, 1.0]]), (len(pairs), 1, 1))
    R45 = synth.pose_to_mat((0.0, 0.0, np.pi / 4))[None]
    nan_init = init6.copy()
    nan_init[2, 4] = np.nan
    far = init6.copy()
    far[0, 2] = 2e12
    bad = {
        "K = 0": dict(S6=S6, K=0),
        "K > 2^22": dict(S6=S6, K=(1 << 22) + 1),
        "null starts": dict(S6=S6, K=4, null_starts=True),
        "pair out of range": dict(pairs=np.r_[pairs, [[0, n_scans]]], S6=S6, K=4),
        "negative pair": dict(pairs=np.r_[pairs, [[-1, 0]]], S6=S6, K=4),
        "hist_cap": dict(S6=S6, K=4, hist_cap=3),
        "corr_stride": dict(S6=S6, K=4, corr_stride=400),
        "pair_mode": dict(S6=S6, K=4, pair_mode=1),
        "composed linear part": dict(S6=np.ascontiguousarray(R45[:, :2].reshape(-1, 6)), K=1,
                                     init6=np.ascontiguousarray(wide[:, :2].reshape(-1, 6))),
        "non-finite guess": dict(S6=S6, K=4, init6=nan_init),
        "composed shift": dict(S6=S6, K=4, init6=far),
    }
    for name, kw in bad.items():
        n0 = eng.launch_count
        kw.setdefault("pairs", pairs)
        assert _raw(eng, gicp, **kw) == EINVAL, name
        assert eng.launch_count == n0, name
    # the same through Python: ValueError, nothing launched
    n0 = eng.launch_count
    for args in [(pairs, S[:0], init), (pairs, S, np.r_[init[:1], init]), (pairs, S[:, :2], init),
                 (np.r_[pairs, [[0, n_scans]]], S, None), (pairs, R45, wide)]:
        with pytest.raises(ValueError):
            eng.run_multistart(*args, epsilon=0.05)
    S_bottom = S.copy()
    S_bottom[1, 2, 0] = 0.5
    S_nan = S.copy()
    S_nan[2, 0, 2] = np.inf
    for starts in (S_bottom, S_nan):
        with pytest.raises(ValueError):
            eng.run_multistart(pairs, starts, init, epsilon=0.05)
    with pytest.raises(ValueError):
        gicp.icp_multistart(gicp.ScanTable(scans), pairs, R45, wide, epsilon=0.05)
    assert eng.launch_count == n0
    # the table still works, with the same results
    after = eng.run_multistart(pairs, S, init, epsilon=0.05, return_all=True)
    for f in ("T", "error", "iters", "start", "error_all", "iters_all"):
        np.testing.assert_array_equal(getattr(after, f), getattr(before, f))


# ------------------------------------------------------------------ callers
def test_proximity_loop_closures_with_starts_equal_host_replay(gicp, synth):
    from icp_slam_b200 import callers
    rng = np.random.default_rng(8401)
    poses = synth.loop_trajectory(500, step=0.2)
    scans = synth.scans_from_poses(poses, 360, rng, drop_frac=0.03)
    S = gicp.heading_starts(8)
    got, res = callers.proximity_loop_closures(poses, scans, starts=S)
    cand = callers.proximity_candidates(poses)
    pairs = np.stack((cand[:, 1], cand[:, 0]), axis=1).astype(np.int32)
    ref = gicp.icp_batch(scans, np.repeat(pairs, 8, axis=0), _expanded(gicp, None, S, len(pairs)),
                         epsilon=0.05, max_iters=100)
    err = ref.error.reshape(-1, 8)
    w = np.arange(len(pairs)) * 8 + np.argmin(err, axis=1)
    used, want = set(), []
    for (i, j), e, T in zip(cand, ref.error[w], ref.T[w]):
        i, j = int(i), int(j)
        if i in used or j in used or not e < 110:
            continue
        want.append((i, j, T))
        used.update((i, j))
    assert len(want) > 0 and len(got) == len(want)
    for (i, j, T), (i2, j2, T2) in zip(got, want):
        assert (i, j) == (i2, j2)
        np.testing.assert_array_equal(T, T2)
    assert np.all(res.error < 110) and len(res.start) == len(res.error)


def test_heading_sweep_accepts_a_flipped_revisit(gicp, synth):
    """Scans taken from nearly the same place facing opposite ways: from the identity ICP settles in a
    wrong minimum far above the threshold; the 8-heading sweep finds the true relative pose."""
    base = synth.loop_trajectory(200, step=0.2)
    scans, truth = [], []
    for i, dxy, dth in [(30, (0.1, -0.05), np.pi - 0.05), (90, (0.05, 0.1), np.pi + 0.1),
                        (140, (-0.1, 0.05), -np.pi + 0.2)]:
        rng = np.random.default_rng(1000 + i)
        pa = base[i]
        pb = pa + np.array([dxy[0], dxy[1], dth])
        scans += [synth.scans_from_poses(pa[None], 360, rng, drop_frac=0.02)[0],
                  synth.scans_from_poses(pb[None], 360, rng, drop_frac=0.02)[0]]
        truth.append(np.linalg.inv(synth.pose_to_mat(pa)) @ synth.pose_to_mat(pb))
    from icp_slam_b200 import callers
    matches = [(1, 0), (3, 2), (5, 4)]                            # source b onto target a
    plain, _ = callers.image_match_loop_closures(matches, scans)
    assert plain == []
    swept, res = callers.image_match_loop_closures(matches, scans, starts=gicp.heading_starts(8))
    assert [(i, j) for i, j, _ in swept] == matches
    for (_, _, T), Tt in zip(swept, truth):
        dt, dth = pose_diff(T, Tt)
        assert dt < 0.05 and dth < 0.01
    assert np.all(res.error < 30)
