"""Submap voxel filter (icpb_set_submaps_voxel / IcpEngine.set_submaps(voxel=)): every submap thinned on the
device to the first merged point of every grid cell.

Engine A sets the base table and builds the filtered submaps on the device; engine B uploads the base plus
``merge_scans(..., voxel=)``'s host-built submaps as one table.  Every comparison is bit for bit:

* the table itself (offsets, the points read back with ``read_scans``, the kept lengths, the same call twice);
* alignments onto the filtered submaps under every variant, run_device, pair_mode 1 and multi-start;
* submaps beyond shared memory before the filter and within it after, and still beyond it after;
* adversarial cells (one crowded cell, many distinct cells, coordinates near ICPB_MAX_COORD, non-rigid members);
* voxel 0 against icpb_set_submaps, a voxel that keeps every point against the unfiltered submaps;
* rejections, read_scans ranges, growth, replacement and the return to the base;
* proximity_loop_closures(submap_window=, submap_voxel=) against a host replay.
"""
import ctypes
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EINVAL, ENOSCANS = 10001, 10003


@pytest.fixture(scope="module")
def gicp():
    from icp_slam_b200 import icp as m
    return m


@pytest.fixture(scope="module")
def engines(gicp):
    a, b = gicp.IcpEngine(), gicp.IcpEngine()
    yield a, b
    a.close()
    b.close()


@functools.lru_cache(maxsize=None)
def _base(n_scans, n_beams, seed):
    from icp_slam_b200 import synth
    scans, _, _, poses, _ = synth.make_chain_workload(n_scans, n_beams, seed=seed)
    return tuple(scans), poses


def _windows(poses, targets, w):
    from icp_slam_b200 import callers
    members = callers.submap_window_members(len(poses), targets, w)
    return members, callers.submap_window_transforms(poses, targets, members)


def _ptr(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


def _raw_args(members, transforms):
    off = np.concatenate(([0], np.cumsum([len(m) for m in members]))).astype(np.int64)
    mem = np.ascontiguousarray(np.concatenate(members).astype(np.int32))
    T6 = np.ascontiguousarray(np.concatenate([np.asarray(t)[:, :2].reshape(-1, 6) for t in transforms]))
    return mem, off, T6


def _raw(e, mem, off, T6, n, voxel, lens=None):
    return e._L.icpb_set_submaps_voxel(e._h, _ptr(mem), _ptr(off), _ptr(T6), n, ctypes.c_double(voxel), _ptr(lens))


def _read(e, first, count, n_pts):
    out = np.empty((n_pts, 2))
    rc = e._L.icpb_read_scans(e._h, first, count, _ptr(out))
    return rc, out


def _check_table(gicp, a, base, ids, host):
    """A's table is the base followed by ``host`` (the host-built submaps), bit for bit."""
    n = len(base)
    assert a._L.icpb_scan_count(a._h) == n + len(host)
    np.testing.assert_array_equal(a.table.lengths, [len(s) for s in base] + [len(s) for s in host])
    for s, want in zip(a.read_scans(ids), host):
        assert s.tobytes() == want.tobytes()
    rc, whole = _read(a, 0, n + len(host), int(a.table.offsets[-1]))
    assert rc == 0 and whole.tobytes() == np.concatenate(list(base) + list(host)).tobytes()


def _setup(gicp, engines, base, members, transforms, voxel):
    """Engine A: base, then filtered submaps on the device.  Engine B: base + merge_scans(voxel=) uploaded."""
    a, b = engines
    a.set_scans(list(base))
    ids = a.set_submaps(members, transforms, voxel=voxel)
    host = gicp.merge_scans(list(base), members, transforms, voxel=voxel)
    b.set_scans(list(base) + host)
    n = len(base)
    np.testing.assert_array_equal(ids, np.arange(n, n + len(members)))
    np.testing.assert_array_equal(a.table.offsets, b.table.offsets)
    _check_table(gicp, a, base, ids, host)
    return ids, host


def _same(x, y):
    np.testing.assert_array_equal(x.T, y.T)
    np.testing.assert_array_equal(x.error, y.error)
    np.testing.assert_array_equal(x.iters, y.iters)
    for f in ("history", "correspondences"):
        u, v = getattr(x, f), getattr(y, f)
        assert (u is None) == (v is None), f
        if u is not None:
            np.testing.assert_array_equal(u, v)


def _both(engines, pairs, init=None, **kw):
    a, b = engines
    ra = a.run(pairs, init, epsilon=0.05, return_history=True, return_correspondences=True, **kw)
    rb = b.run(pairs, init, epsilon=0.05, return_history=True, return_correspondences=True, **kw)
    _same(ra, rb)
    return ra


def _role_pairs(poses, ids, targets):
    """(pairs, guesses): scan -> submap and submap -> scan with the true relative pose, and from the identity."""
    from icp_slam_b200 import callers
    M = callers.poses_to_mats(poses)
    s0, s1 = ids[0], ids[1]
    i0, i1 = targets[0], targets[1]
    rows = [(i0 + 5, s0, i0, i0 + 5), (s1, 2, i1, 2), (s1, s0, i1, i0), (1, s1, None, None)]
    pairs = np.array([r[:2] for r in rows], dtype=np.int32)
    init = np.stack([np.eye(3) if r[2] is None else np.linalg.inv(M[r[2]]) @ M[r[3]] for r in rows])
    init[:, 2] = (0.0, 0.0, 1.0)
    return pairs, init


# ------------------------------------------------------------------ the table itself
@pytest.mark.parametrize("voxel", [0.01, 0.05, 0.2])
def test_table_equals_host_restatement(gicp, engines, voxel):
    base, poses = _base(14, 1024, 9301)
    members, transforms = _windows(poses, [3, 7, 10], 3)
    ids, host = _setup(gicp, engines, base, members, transforms, voxel)
    a, _ = engines
    assert all(len(h) < sum(len(base[s]) for s in m) for h, m in zip(host, members))     # the filter thinned
    # the kept lengths the library returns, and the same call twice: the same table
    mem, off, T6 = _raw_args(members, transforms)
    for _ in range(2):
        lens = np.full(len(members), -1, dtype=np.int64)
        assert _raw(a, mem, off, T6, len(members), voxel, lens) == 0
        np.testing.assert_array_equal(lens, [len(h) for h in host])
        rc, whole = _read(a, 0, len(base) + len(host), int(a.table.offsets[-1]))
        assert rc == 0 and whole.tobytes() == np.concatenate(list(base) + host).tobytes()


# ------------------------------------------------------------------ alignments onto filtered submaps
@pytest.mark.parametrize("variant", ["default", "exhaustive", "rotation_only", "large", "cluster"])
def test_alignments_equal_host_built_table(gicp, engines, variant):
    base, poses = _base(14, 1024, 9302)
    targets = [3, 9]
    members, transforms = _windows(poses, targets, 3)
    ids, _ = _setup(gicp, engines, base, members, transforms, 0.02)
    pairs, init = _role_pairs(poses, ids, targets)
    kw = {"exhaustive": variant == "exhaustive", "rotation_only": variant == "rotation_only"}
    tune = {"large": ("large", 1), "cluster": ("cluster", 2)}.get(variant)
    if tune:
        for e in engines:
            e.set_tuning(*tune)
    try:
        if variant == "cluster":
            pairs, init = pairs[:2], init[:2]
        _both(engines, pairs, init, **kw)
        _both(engines, pairs, None, **kw)
    finally:
        if tune:
            for e in engines:
                e.set_tuning(tune[0], -1)


def test_run_device_pair_mode_one_and_multistart(gicp, engines):
    import torch
    base, poses = _base(10, 1024, 9303)
    targets = [2, 6]
    members, transforms = _windows(poses, targets, 2)
    ids, _ = _setup(gicp, engines, base, members, transforms, 0.03)
    a, b = engines
    n = len(base) + len(ids)
    B = n * (n - 1) // 2
    _same(a.run(None, all_pairs=(0, B, 0, B), epsilon=0.05), b.run(None, all_pairs=(0, B, 0, B), epsilon=0.05))
    pairs, init = _role_pairs(poses, ids, targets)
    dev = torch.device("cuda", a.device)
    out_T = torch.empty((len(pairs), 6), dtype=torch.float64, device=dev)
    out_err = torch.empty(len(pairs), dtype=torch.float64, device=dev)
    out_passes = torch.empty(len(pairs), dtype=torch.int32, device=dev)
    init6 = torch.from_numpy(np.ascontiguousarray(init[:, :2].reshape(-1, 6))).to(dev)
    a.run_device(torch.from_numpy(pairs).to(dev), init6, out_T, out_err, out_passes, epsilon=0.05)
    torch.cuda.synchronize(dev)
    ref = b.run(pairs, init, epsilon=0.05)
    np.testing.assert_array_equal(out_T.cpu().numpy(), ref.T[:, :2].reshape(-1, 6))
    np.testing.assert_array_equal(out_err.cpu().numpy(), ref.error)
    np.testing.assert_array_equal(out_passes.cpu().numpy(), ref.iters)
    S = gicp.heading_starts(4)
    for guess in (init, None):
        x = a.run_multistart(pairs, S, guess, epsilon=0.05, return_all=True)
        y = b.run_multistart(pairs, S, guess, epsilon=0.05, return_all=True)
        for f in ("T", "error", "iters", "start", "error_all", "iters_all"):
            np.testing.assert_array_equal(getattr(x, f), getattr(y, f))


# ------------------------------------------------------------------ sizes around the shared-memory limit
@pytest.mark.parametrize("voxel, fits", [(0.01, True), (1e-6, False)])
def test_sizes_around_the_shared_memory_limit(gicp, engines, voxel, fits):
    base, poses = _base(20, 1024, 9103)
    members, transforms = _windows(poses, [8, 10], 8)                          # 17 x 1,024 beams merged
    a, _ = engines
    a.set_scans(list(base))
    a.set_submaps(members, transforms)
    assert a.table.longest > 16 * 1000                                         # beyond shared memory unfiltered
    ids, host = _setup(gicp, engines, base, members, transforms, voxel)
    assert (a.table.longest < 8000) == fits
    pairs = np.array([(1, ids[0]), (ids[1], 0), (ids[0], ids[1]), (2, 3), (ids[1], ids[1])], dtype=np.int32)
    # fits: the first run builds the table's staging images (a launch of its own), then one launch per batch;
    # beyond: no images, and every batch is split by scan length into two launches
    for want in ((2, 1) if fits else (2, 2)):
        n0 = a.launch_count
        a.run(pairs, epsilon=0.05)
        assert a.launch_count - n0 == want
    _both(engines, pairs)


# ------------------------------------------------------------------ adversarial cells
def _adversarial(case):
    rng = np.random.default_rng(9304)
    I = np.eye(3)
    if case == "crowded":           # thousands of points of one cell, across many warps and several members
        s = [rng.uniform(0.0, 0.5, size=(4096, 2)), rng.uniform(0.0, 0.5, size=(3000, 2)),
             rng.uniform(-5, 5, size=(500, 2))]
        members = [np.array([0, 1, 0, 2]), np.array([1])]
        return s, members, [np.stack([I] * 4), I[None]], 1.0
    if case == "distinct":          # a cell per point, pairs of one cell far apart in merged order
        g = np.stack(np.meshgrid(np.arange(64), np.arange(64)), -1).reshape(-1, 2) * 0.1 + 0.01
        s = [g[rng.permutation(len(g))], g[rng.permutation(len(g))] + 0.03, rng.uniform(0, 6.4, size=(2000, 2))]
        return (s, [np.array([0, 1, 2]), np.array([2, 0]), np.array([0])],             # the last at load 0.5
                [np.stack([I] * 3), np.stack([I] * 2), I[None]], 0.1)
    if case == "near_max_coord":    # cells of 1e-6 at |x| ~ 1e10, where x / voxel rounds to even integers
        k = rng.integers(0, 4000, size=(3000, 2))
        sgn = np.where(rng.random((3000, 2)) < 0.5, -1.0, 1.0)
        s = [sgn * (1e10 - k * 1.9073486328125e-06), sgn[::-1] * (1e10 - k[::-1] * 9.5367431640625e-07)]
        return s, [np.array([0, 1]), np.array([1, 0, 1])], [np.stack([I] * 2), np.stack([I] * 3)], 1e-6
    # non-rigid member transforms: shear and scale within the bounds
    s = [rng.uniform(-10, 10, size=(2000, 2)) for _ in range(4)]
    A = np.array([[1.3, 0.4, 2.0], [-0.2, 0.7, -1.0], [0.0, 0.0, 1.0]])
    B = np.array([[0.5, -0.9, 0.1], [1.1, 0.3, 3.0], [0.0, 0.0, 1.0]])
    return s, [np.array([0, 1, 2, 3]), np.array([3, 3, 1])], [np.stack([A, B, A @ B, I]), np.stack([B, A, I])], 0.05


@pytest.mark.parametrize("case", ["crowded", "distinct", "near_max_coord", "non_rigid"])
def test_adversarial_cells_equal_host_restatement(gicp, engines, case):
    base, members, transforms, voxel = _adversarial(case)
    ids, host = _setup(gicp, engines, base, members, transforms, voxel)
    if case == "crowded":
        assert [len(h) for h in host][1] == 1 and len(host[0]) < 600
    if case == "distinct":
        assert len(host[0]) >= 4096
    a, _ = engines
    mem, off, T6 = _raw_args(members, transforms)
    assert _raw(a, mem, off, T6, len(members), voxel) == 0                      # again: the same table
    _check_table(gicp, a, base, ids, host)
    if case != "near_max_coord":
        _both(engines, np.array([(0, ids[0]), (ids[-1], 1), (ids[0], ids[-1])], dtype=np.int32))


# ------------------------------------------------------------------ equivalences
def test_voxel_zero_is_set_submaps_and_a_tiny_voxel_keeps_everything(gicp, engines):
    base, poses = _base(12, 1024, 9305)
    members, transforms = _windows(poses, [3, 8], 2)
    a, b = engines
    mem, off, T6 = _raw_args(members, transforms)
    b.set_scans(list(base))
    assert b._L.icpb_set_submaps(b._h, _ptr(mem), _ptr(off), _ptr(T6), len(members)) == 0
    merged = [len(m) for m in gicp.merge_scans(list(base), members, transforms)]
    n_all = len(base) + len(members)
    rc, want = _read(b, 0, n_all, int(sum(len(s) for s in base)) + sum(merged))
    assert rc == 0
    a.set_scans(list(base))
    lens = np.zeros(len(members), dtype=np.int64)
    assert _raw(a, mem, off, T6, len(members), 0.0, lens) == 0
    np.testing.assert_array_equal(lens, merged)
    rc, got = _read(a, 0, n_all, len(want))
    assert rc == 0 and got.tobytes() == want.tobytes()
    # a voxel small enough that the host keeps every point gives the unfiltered submaps
    host = gicp.merge_scans(list(base), members, transforms, voxel=1e-6)
    assert [len(h) for h in host] == merged
    a.set_submaps(members, transforms, voxel=1e-6)
    rc, got = _read(a, 0, n_all, len(want))
    assert rc == 0 and got.tobytes() == want.tobytes()


# ------------------------------------------------------------------ rejections, reads, growth
def test_rejections_leave_the_table_and_reads_are_checked(gicp, engines):
    base, poses = _base(12, 1024, 9306)
    a, _ = engines
    members, transforms = _windows(poses, [3, 8], 2)
    a.set_scans(list(base))
    ids = a.set_submaps(members, transforms, voxel=0.05)
    n_all = len(base) + len(ids)
    pairs = np.array([(1, ids[0]), (ids[1], 2), (ids[0], ids[1]), (5, 4)], dtype=np.int32)
    before = a.run(pairs, epsilon=0.05, return_history=True, return_correspondences=True)
    rc, table = _read(a, 0, n_all, int(a.table.offsets[-1]))
    assert rc == 0

    def unchanged(name):
        assert a._L.icpb_scan_count(a._h) == n_all, name
        assert a.table.n_scans == n_all, name
        assert _read(a, 0, n_all, len(table))[1].tobytes() == table.tobytes(), name
        _same(a.run(pairs, epsilon=0.05, return_history=True, return_correspondences=True), before)

    mem, off, T6 = _raw_args(members, transforms)
    for v in (np.nan, np.inf, -np.inf, -0.05, -0.0 - 1e-9, 5e-7, 1e-300):
        n0 = a.launch_count
        assert _raw(a, mem, off, T6, len(members), v) == EINVAL, v
        assert a.launch_count == n0, v
        unchanged(v)
        with pytest.raises(ValueError):
            a.set_submaps(members, transforms, voxel=v)
        unchanged(v)
    # a merged coordinate past ICPB_MAX_COORD, with the filter on
    xmax = float(np.max(base[0][:, 0]))
    past = np.array([[1.0, 0.0, 1e10 - xmax + 1.0], [0.0, 1.0, 0.0], [0.0, 0.0, 1.0]])[None]
    pm, po, pT = _raw_args([np.array([0])], [past])
    assert _raw(a, pm, po, pT, 1, 0.05) == EINVAL
    unchanged("merged coordinate")
    with pytest.raises(ValueError):
        a.set_submaps([np.array([0])], [past], voxel=0.05)
    unchanged("merged coordinate")
    # read_scans ranges
    buf = np.empty((len(table), 2))
    for first, count in ((-1, 1), (0, -1), (n_all, 1), (n_all - 1, 2), (2, n_all)):
        assert a._L.icpb_read_scans(a._h, first, count, _ptr(buf)) == EINVAL, (first, count)
    assert a._L.icpb_read_scans(a._h, 0, 1, None) == EINVAL
    assert a._L.icpb_read_scans(a._h, n_all, 0, _ptr(buf)) == 0
    with pytest.raises(ValueError):
        a.read_scans([n_all])
    fresh = gicp.IcpEngine()
    try:
        assert fresh._L.icpb_read_scans(fresh._h, 0, 1, _ptr(buf)) == ENOSCANS
        assert _raw(fresh, mem, off, T6, len(members), 0.05) == ENOSCANS
    finally:
        fresh.close()


def test_growth_replacement_and_back_to_the_base(gicp, engines):
    base, poses = _base(16, 1024, 9307)
    a, b = engines
    base_pairs = np.array([(i + 1, i) for i in range(len(base) - 1)], dtype=np.int32)
    a.set_scans(list(base))
    before = a.run(base_pairs, epsilon=0.05, return_history=True, return_correspondences=True)
    small = _windows(poses, [4, 9], 0)
    large = _windows(poses, [2, 5, 8, 11, 14], 6)                              # several times the base's points
    for (members, transforms), voxel in ((small, 0.05), (large, None), (large, 0.01), (small, 0.2), (large, 0.01)):
        ids = a.set_submaps(members, transforms, voxel=voxel)
        host = gicp.merge_scans(list(base), members, transforms, voxel=voxel)
        b.set_scans(list(base) + host)
        _check_table(gicp, a, base, ids, host)
        pairs = np.array([(1, ids[0]), (ids[-1], 3), (ids[0], ids[-1])] + [tuple(p) for p in base_pairs[:4]],
                         dtype=np.int32)
        _both(engines, pairs)
    assert a.set_submaps([], [], voxel=0.05).size == 0
    assert a._L.icpb_scan_count(a._h) == len(base) and a.table.n_scans == len(base)
    _same(a.run(base_pairs, epsilon=0.05, return_history=True, return_correspondences=True), before)


# ------------------------------------------------------------------ the proximity caller
@functools.lru_cache(maxsize=None)
def _loop(n_poses, beams, seed):
    from icp_slam_b200 import synth
    rng = np.random.default_rng(seed)
    poses = synth.loop_trajectory(n_poses, step=0.2)
    return poses, synth.scans_from_poses(poses, beams, rng, drop_frac=0.03)


def test_caller_equals_host_replay(gicp):
    from icp_slam_b200 import callers
    poses, scans = _loop(500, 360, 9308)
    w, v = 4, 0.05
    got, res = callers.proximity_loop_closures(poses, scans, submap_window=w, submap_voxel=v)
    assert len(got) > 0
    # the host replay: the filtered submaps built by merge_scans, uploaded with the scans
    cand = callers.proximity_candidates(poses)
    targets, sub = np.unique(cand[:, 0], return_inverse=True)
    members = callers.submap_window_members(len(scans), targets, w)
    host = gicp.merge_scans(list(scans), members, callers.submap_window_transforms(poses, targets, members), voxel=v)
    e = gicp.IcpEngine()
    try:
        e.set_scans(list(scans) + host)
        pairs = np.stack((cand[:, 1], len(scans) + sub), axis=1).astype(np.int32)
        ref = e.run(pairs, epsilon=0.05)
    finally:
        e.close()
    rows = np.nonzero(ref.error < 110)[0]
    np.testing.assert_array_equal(res.error, ref.error[rows])
    np.testing.assert_array_equal(res.iters, ref.iters[rows])
    used, want = set(), []
    for (i, j), T in zip(cand[rows], ref.T[rows]):
        i, j = int(i), int(j)
        if i in used or j in used:
            continue
        want.append((i, j, T))
        used.update((i, j))
    assert len(got) == len(want)
    for (i, j, T), (i2, j2, T2) in zip(got, want):
        assert (i, j) == (i2, j2)
        np.testing.assert_array_equal(T, T2)
    # without submap_voxel: today's constraints
    a, _ = callers.proximity_loop_closures(poses, scans, submap_window=w)
    b, _ = callers.proximity_loop_closures(poses, scans, submap_window=w, submap_voxel=None)
    assert len(a) == len(b) > 0
    for (i, j, T), (i2, j2, T2) in zip(a, b):
        assert (i, j) == (i2, j2)
        np.testing.assert_array_equal(T, T2)
