"""Scans whose layout does not fit one CTA's shared memory run on the large-scan variant of the
alignment kernel (per-CTA device scratch instead of shared memory).

* On sizes both variants run, the variant forced through the "large" tuning key gives the bits of
  the default kernel: transforms, errors, pass counts, histories and correspondences.
* Above the shared-memory limit the results match the C oracle with the tolerances of
  test_gpu_parity.py: equal pass counts and correspondences, every transform of the history within
  1e-9, errors within 1e-9 relative.
* In a table that holds one long scan, the short pairs give the bits they give on the table without it.
"""
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL = 1e-9


@pytest.fixture(scope="module")
def gicp():
    from icp_slam_b200 import icp as m
    return m


@pytest.fixture(scope="module")
def synth():
    from icp_slam_b200 import synth as m
    return m


@pytest.fixture(scope="module")
def c_oracle():
    from oracle import c_oracle as m
    m.build()
    return m


@pytest.fixture(scope="module")
def eng(gicp):
    e = gicp.IcpEngine()
    yield e
    e.close()


def _chain(synth, n_scans, n_beams, seed):
    scans, pairs, init, poses, _ = synth.make_chain_workload(n_scans, n_beams, seed=seed)
    return scans, pairs, init, poses


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
    target = np.ascontiguousarray(np.concatenate(parts))
    init = np.linalg.inv(synth.pose_to_mat(poses[0])) @ synth.pose_to_mat(poses[k])
    return scans[k], target, init


def _run_both(e, pairs, init, **kw):
    e.set_tuning("large", -1)
    a = e.run(pairs, init, return_history=True, return_correspondences=True, **kw)
    e.set_tuning("large", 1)
    try:
        b = e.run(pairs, init, return_history=True, return_correspondences=True, **kw)
    finally:
        e.set_tuning("large", -1)
    return a, b


def _assert_same(a, b):
    np.testing.assert_array_equal(a.iters, b.iters)
    np.testing.assert_array_equal(a.T, b.T)
    np.testing.assert_array_equal(a.error, b.error)
    np.testing.assert_array_equal(a.history, b.history)
    np.testing.assert_array_equal(a.correspondences, b.correspondences)


# ------------------------------------------------------------------ forced "large" = default, bit for bit
KW_CASES = {
    "default": dict(epsilon=0.05),
    "rotation_only": dict(epsilon=0.05, rotation_only=True),
    "stop_epsilon": dict(epsilon=1e9),
    "stop_max_iters": dict(epsilon=0.0, stopping_thresh=0.0, max_iters=2),
    "stop_thresh": dict(epsilon=0.0, stopping_thresh=1e-3),
    "exhaustive": dict(epsilon=0.05, exhaustive=True),
}


@pytest.mark.parametrize("beams,n_scans", [(360, 24), (1024, 16), (4096, 5)])
@pytest.mark.parametrize("kw", list(KW_CASES), ids=list(KW_CASES))
@pytest.mark.parametrize("guess", ["odometry", "identity"])
def test_forced_large_equals_default(eng, synth, beams, n_scans, kw, guess):
    scans, pairs, init, _ = _chain(synth, n_scans, beams, seed=beams + 7)
    eng.set_scans(scans)
    a, b = _run_both(eng, pairs, init if guess == "odometry" else None, **KW_CASES[kw])
    _assert_same(a, b)


def test_forced_large_ragged_sizes(eng, synth):
    """Scans of 1, 63, 64 and 65 points (partial tiles, partial chunks, a one-point cloud) in every role."""
    rng = np.random.default_rng(11)
    base = synth.scans_from_poses(synth.loop_trajectory(6, step=0.04), 1024, rng)
    lens = [1, 63, 64, 65, 200, 1000]
    scans = [np.ascontiguousarray(s[rng.permutation(len(s))[:m]]) for s, m in zip(base, lens)]
    pairs = np.array([(i, j) for i in range(6) for j in range(6) if i != j], dtype=np.int32)
    eng.set_scans(scans)
    smem = eng.kernel_info()["smem_bytes"]
    eng.set_tuning("large", 1)
    try:
        assert eng.kernel_info()["smem_bytes"] < smem          # the key selects the scratch-backed variant
    finally:
        eng.set_tuning("large", -1)
    for kw in ("default", "exhaustive", "rotation_only"):
        a, b = _run_both(eng, pairs, None, **KW_CASES[kw])
        _assert_same(a, b)


@pytest.mark.parametrize("cluster", [1, 2, 4, 8])
def test_forced_large_cluster_sizes(eng, synth, cluster):
    """One 4,096-beam pair in clusters of 1..8 CTAs: the large variant reads the partial sums of the
    other CTAs from their scratch and must give the bits of the shared-memory kernel."""
    scans, pairs, init, _ = _chain(synth, 3, 4096, seed=41)
    eng.set_scans(scans)
    eng.set_tuning("cluster", 0)
    ref = eng.run(pairs[:1], init[:1], epsilon=0.05, return_history=True, return_correspondences=True)
    eng.set_tuning("cluster", cluster)
    try:
        a, b = _run_both(eng, pairs[:1], init[:1], epsilon=0.05)
    finally:
        eng.set_tuning("cluster", -1)
    _assert_same(ref, a)
    _assert_same(ref, b)


# ------------------------------------------------------------------ above the limit, against the C oracle
def _oracle(c_oracle, jobs):
    """jobs: [(src, dst, init 3x3 or None, kwargs)] -> [(T, err, passes, corr, history)] in parallel."""
    def one(j):
        src, dst, init, kw = j
        return c_oracle.icp_pair(src, dst, init, want_history=True, **kw)
    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), c_oracle.max_threads()))) as ex:
        return list(ex.map(one, jobs))


def _assert_oracle(res, b, ref, n_src):
    T, err, passes, corr, hist = ref
    assert res.iters[b] == passes
    np.testing.assert_array_equal(res.correspondences[b, :n_src], corr)
    assert np.abs(res.history[b, :passes] - hist).max() <= TOL
    assert np.abs(res.T[b] - T).max() <= TOL
    assert abs(res.error[b] - err) <= TOL * max(abs(err), 1e-300)


@pytest.fixture(scope="module")
def long_case(synth):
    """Scans above the shared-memory limit, and pairs across them: 16,384- and 20,000-beam chains, a
    long source onto a short target and the reverse, and a 1,024-beam source onto a 16-scan submap."""
    s16, p16, i16, _ = _chain(synth, 3, 16384, seed=161)
    s20, p20, i20, _ = _chain(synth, 3, 20000, seed=201)
    short = _chain(synth, 2, 1024, seed=202)[0][0]
    src, sub, isub = _submap(synth, seed=203)
    scans = s16 + s20 + [short, src, sub]
    pairs = np.concatenate([p16, p20 + 3, [[3, 6], [6, 4], [7, 8]]]).astype(np.int32)
    init = np.concatenate([i16, i20, [np.eye(3), np.eye(3), isub]])
    return scans, pairs, init


@pytest.fixture(scope="module")
def long_oracle(c_oracle, long_case):
    scans, pairs, init = long_case
    return _oracle(c_oracle, [(scans[s], scans[d], init[b], dict(epsilon=0.05)) for b, (s, d) in enumerate(pairs)])


def test_long_scans_match_oracle(eng, long_case, long_oracle):
    scans, pairs, init = long_case
    eng.set_scans(scans)
    res = eng.run(pairs, init, epsilon=0.05, return_history=True, return_correspondences=True)
    for b, (s, _) in enumerate(pairs):
        _assert_oracle(res, b, long_oracle[b], len(scans[s]))


def test_long_scans_exhaustive_and_clusters_same_bits(eng, long_case):
    scans, pairs, init = long_case
    eng.set_scans(scans)
    ref = eng.run(pairs[:1], init[:1], epsilon=0.05, return_history=True, return_correspondences=True)
    got = [eng.run(pairs[:1], init[:1], epsilon=0.05, return_history=True, return_correspondences=True,
                   exhaustive=True)]
    try:
        for cl in (0, 2, 4, 8):
            eng.set_tuning("cluster", cl)
            got.append(eng.run(pairs[:1], init[:1], epsilon=0.05, return_history=True, return_correspondences=True))
    finally:
        eng.set_tuning("cluster", -1)
    for g in got:
        _assert_same(ref, g)


def test_drop_ins_on_long_pair(gicp, long_case, long_oracle, c_oracle):
    scans, pairs, init = long_case
    s, d = pairs[2]                                           # 20,000 onto 20,000 points
    hom = lambda a: np.c_[a, np.ones(len(a))]
    tfs, err = gicp.icp(hom(scans[s]), hom(scans[d]), init[2].copy(), epsilon=0.05)
    T, e_ref, passes, _, hist = long_oracle[2]
    assert len(tfs) == passes + 1
    assert np.abs(np.array(tfs[1:]) - hist).max() <= TOL
    assert abs(err - e_ref) <= TOL * abs(e_ref)
    T1, corr, e1 = gicp.icp_iteration(hom(scans[s]), hom(scans[d]), init[2].copy())
    T1r, e1r, _, corr_r = c_oracle.icp_pair(scans[s], scans[d], init[2], epsilon=np.inf)
    np.testing.assert_array_equal(corr, corr_r)
    assert np.abs(T1 - T1r).max() <= TOL
    assert abs(e1 - e1r) <= TOL * abs(e1r)


# ------------------------------------------------------------------ a table with one long scan
@pytest.fixture(scope="module")
def mixed_case(synth):
    scans, pairs, init, _ = _chain(synth, 301, 1024, seed=303)
    long_scan = _chain(synth, 2, 20000, seed=304)[0][0]
    n = len(scans)
    mixed = scans + [long_scan]
    lp = np.array([[n, 0], [1, n]], dtype=np.int32)
    all_pairs = np.concatenate([pairs[:150], lp, pairs[150:]]).astype(np.int32)
    all_init = np.concatenate([init[:150], np.repeat(np.eye(3)[None], 2, axis=0), init[150:]])
    short_rows = np.r_[0:150, 152:len(all_pairs)]
    return scans, mixed, pairs, init, all_pairs, all_init, short_rows


@pytest.fixture(scope="module")
def mixed_ref(eng, mixed_case, c_oracle):
    scans, mixed, pairs, init, all_pairs, all_init, _ = mixed_case
    eng.set_scans(scans)
    short = eng.run(pairs, init, epsilon=0.05)
    longs = _oracle(c_oracle, [(mixed[s], mixed[d], all_init[150 + k], dict(epsilon=0.05))
                               for k, (s, d) in enumerate(all_pairs[150:152])])
    return short, longs


def _check_mixed(res, mixed_ref, short_rows, has_corr=False):
    short, longs = mixed_ref
    np.testing.assert_array_equal(res.T[short_rows], short.T)
    np.testing.assert_array_equal(res.error[short_rows], short.error)
    np.testing.assert_array_equal(res.iters[short_rows], short.iters)
    for k, (T, err, passes, _, _) in enumerate(longs):
        b = 150 + k
        assert res.iters[b] == passes
        assert np.abs(res.T[b] - T).max() <= TOL
        assert abs(res.error[b] - err) <= TOL * abs(err)


def test_mixed_table_list_of_arrays(gicp, mixed_case, mixed_ref):
    _, mixed, _, _, all_pairs, all_init, short_rows = mixed_case
    res = gicp.icp_batch(mixed, all_pairs, all_init, epsilon=0.05)            # streaming upload
    _check_mixed(res, mixed_ref, short_rows)


def test_mixed_table_packed(gicp, eng, mixed_case, mixed_ref):
    _, mixed, _, _, all_pairs, all_init, short_rows = mixed_case
    res = eng.align(gicp.ScanTable(mixed), all_pairs, all_init, epsilon=0.05)
    _check_mixed(res, mixed_ref, short_rows)


def test_mixed_table_resident_host_and_device(eng, mixed_case, mixed_ref):
    import torch
    _, mixed, _, _, all_pairs, all_init, short_rows = mixed_case
    eng.set_scans(mixed)
    _check_mixed(eng.run(all_pairs, all_init, epsilon=0.05), mixed_ref, short_rows)
    dev = torch.device("cuda", eng.device)
    B = len(all_pairs)
    pt = torch.from_numpy(all_pairs).to(dev)
    it = torch.from_numpy(np.ascontiguousarray(all_init[:, :2, :].reshape(B, 6))).to(dev)
    oT = torch.empty((B, 6), dtype=torch.float64, device=dev)
    oe = torch.empty(B, dtype=torch.float64, device=dev)
    op = torch.empty(B, dtype=torch.int32, device=dev)
    eng.run_device(pt, it, oT, oe, op, epsilon=0.05)
    torch.cuda.synchronize()
    from icp_slam_b200.icp import BatchResult
    T33 = np.zeros((B, 3, 3))
    T33[:, :2, :] = oT.cpu().numpy().reshape(B, 2, 3)
    T33[:, 2, 2] = 1.0
    _check_mixed(BatchResult(T33, oe.cpu().numpy(), op.cpu().numpy()), mixed_ref, short_rows)


def test_mixed_table_align_accept(eng, mixed_case):
    """Two launches feed one acceptance count: rows and count equal the host filter of the full results."""
    _, mixed, _, _, all_pairs, all_init, _ = mixed_case
    full = eng.align(mixed, all_pairs, all_init, epsilon=0.05)
    for thresh in (float(np.median(full.error)), float(full.error.max()) * 2):
        rows, acc = eng.align_accept(mixed, all_pairs, thresh, all_init, epsilon=0.05)
        keep = np.nonzero(full.error < thresh)[0]
        np.testing.assert_array_equal(rows, keep)
        np.testing.assert_array_equal(acc.T, full.T[keep])
        np.testing.assert_array_equal(acc.error, full.error[keep])
        np.testing.assert_array_equal(acc.iters, full.iters[keep])


def test_mixed_table_rerun_after_missing_counter(gicp, eng, mixed_case, mixed_ref):
    """The streaming rerun of a split batch: when the arrival counter never moves, the CTAs of both
    launches give up after ~0.5 s and the library reruns both parts on the resident table, with the
    results of a call that did not have to."""
    _, mixed, _, _, all_pairs, all_init, short_rows = mixed_case
    n0 = eng.launch_count
    ref = eng.align(gicp.ScanTable(mixed), all_pairs, all_init, epsilon=0.05)
    assert eng.launch_count - n0 == 2                       # one launch per part
    thresh = float(np.median(ref.error))
    rows_ref, acc_ref = eng.align_accept(mixed, all_pairs, thresh, all_init, epsilon=0.05)
    eng.set_tuning("drop_counter", 1)
    try:
        n0 = eng.launch_count
        got = eng.align(gicp.ScanTable(mixed), all_pairs, all_init, epsilon=0.05)
        assert eng.launch_count - n0 == 4                   # both parts, then both again
        rows, acc = eng.align_accept(mixed, all_pairs, thresh, all_init, epsilon=0.05)
    finally:
        eng.set_tuning("drop_counter", 0)
    _check_mixed(got, mixed_ref, short_rows)
    np.testing.assert_array_equal(got.T, ref.T)
    np.testing.assert_array_equal(got.error, ref.error)
    np.testing.assert_array_equal(got.iters, ref.iters)
    assert 0 < len(rows_ref) < len(all_pairs)
    np.testing.assert_array_equal(rows, rows_ref)
    np.testing.assert_array_equal(acc.T, acc_ref.T)
    np.testing.assert_array_equal(acc.error, acc_ref.error)
    np.testing.assert_array_equal(acc.iters, acc_ref.iters)


@pytest.mark.parametrize("n_peers", [1, 5])
def test_mixed_table_fused_gather(eng, mixed_case, mixed_ref, n_peers):
    import torch
    _, mixed, _, _, all_pairs, all_init, short_rows = mixed_case
    eng.set_scans(mixed)
    ref = eng.run(all_pairs, all_init, epsilon=0.05)
    _check_mixed(ref, mixed_ref, short_rows)
    dev = torch.device("cuda", eng.device)
    B = len(all_pairs)
    bufs = [torch.full((B, 8), -1.0, dtype=torch.float64, device=dev) for _ in range(n_peers)]
    ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=dev)
    pt = torch.from_numpy(all_pairs).to(dev)
    it = torch.from_numpy(np.ascontiguousarray(all_init[:, :2, :].reshape(B, 6))).to(dev)
    oT = torch.empty((B, 6), dtype=torch.float64, device=dev)
    oe = torch.empty(B, dtype=torch.float64, device=dev)
    op = torch.empty(B, dtype=torch.int32, device=dev)
    eng.run_device_gather(pt, it, oT, oe, op, ptrs.data_ptr(), n_peers, 0, epsilon=0.05)
    torch.cuda.synchronize()
    for b in bufs:
        got = b.cpu().numpy()
        np.testing.assert_array_equal(got[:, :6].reshape(B, 2, 3), ref.T[:, :2, :])
        np.testing.assert_array_equal(got[:, 6], ref.error)
        np.testing.assert_array_equal(got[:, 7], ref.iters)


# ------------------------------------------------------------------ one pair of about 100k points
def test_100k_pair(eng, synth):
    from scipy.spatial import cKDTree
    scans, pairs, init, _ = _chain(synth, 2, 100000, seed=1000)
    eng.set_scans(scans)
    kw = dict(epsilon=0.05, return_history=True, return_correspondences=True)
    ref = eng.run(pairs, init, **kw)
    _assert_same(ref, eng.run(pairs, init, exhaustive=True, **kw))
    try:
        eng.set_tuning("cluster", 0)
        _assert_same(ref, eng.run(pairs, init, **kw))
    finally:
        eng.set_tuning("cluster", -1)
    # the last pass's matches: nearest neighbours under the transform that pass started from
    src, dst = scans[pairs[0, 0]], scans[pairs[0, 1]]
    passes = int(ref.iters[0])
    T = ref.history[0, passes - 2] if passes >= 2 else init[0]
    P = (T @ np.c_[src, np.ones(len(src))].T).T[:, :2]
    _, cand = cKDTree(dst).query(P, k=8)
    dx = dst[cand, 0] - P[:, :1]
    dy = dst[cand, 1] - P[:, 1:2]
    d = dx * dx + dy * dy
    dmin = d.min(axis=1, keepdims=True)
    idx = np.where(d == dmin, cand, np.iinfo(np.int64).max).min(axis=1)      # first index among ties
    np.testing.assert_array_equal(ref.correspondences[0, :len(src)], idx)
