"""Submaps (icpb_set_submaps / IcpEngine.set_submaps): scans of the resident table merged on the device.

Every check is bit for bit (transforms, errors, passes, history, correspondences): engine A sets the base
table and builds its submaps on the device; engine B uploads the base and ``merge_scans``' host-built
submaps as one table.

* Pair roles (scan -> submap, submap -> scan, submap -> submap, scan -> scan) under the default, exhaustive,
  rotation_only, forced large-scan and cluster variants; pair_mode 1 and run_device on the same table.
* Submaps that fit shared memory and ones that do not, ragged and 1-point members, a repeated member,
  non-rigid member transforms; multi-start on submaps.
* Replacement and growth, going back to the base, a borrowed base, every rejection.
* proximity_loop_closures(submap_window=...).
"""
import ctypes
import functools

import numpy as np
import pytest

from conftest import pose_diff

pytestmark = pytest.mark.gpu

EINVAL, ETOOLONG, ENOSCANS = 10001, 10002, 10003


@pytest.fixture(scope="module")
def gicp():
    from icp_slam_b200 import icp as m
    return m


@pytest.fixture(scope="module")
def synth():
    from icp_slam_b200 import synth as m
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


def _setup(gicp, engines, base, members, transforms):
    """Engine A: base, then submaps on the device.  Engine B: base + merge_scans uploaded.  The submap ids."""
    a, b = engines
    a.set_scans(list(base))
    ids = a.set_submaps(members, transforms)
    b.set_scans(list(base) + gicp.merge_scans(list(base), members, transforms))
    n = len(base)
    np.testing.assert_array_equal(ids, np.arange(n, n + len(members)))
    assert a._L.icpb_scan_count(a._h) == b._L.icpb_scan_count(b._h) == n + len(members)
    np.testing.assert_array_equal(a.table.offsets, b.table.offsets)
    return ids


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


def _role_pairs(poses, n, ids, targets):
    """(pairs, guesses): every role, with the true relative pose as the guess where both ends have one."""
    from icp_slam_b200 import callers
    M = callers.poses_to_mats(poses)
    s0, s1 = ids[0], ids[1]
    i0, i1 = targets[0], targets[1]
    rows = [(i0 + 5, s0, i0, i0 + 5),          # scan -> submap (in target i0's frame)
            (s1, 2, i1, 2),                    # submap -> scan
            (s1, s0, i1, i0),                  # submap -> submap
            (3, 1, 1, 3),                      # scan -> scan
            (1, s1, None, None)]               # scan -> submap from the identity
    pairs = np.array([r[:2] for r in rows], dtype=np.int32)
    init = np.stack([np.eye(3) if r[2] is None else np.linalg.inv(M[r[2]]) @ M[r[3]] for r in rows])
    init[:, 2] = (0.0, 0.0, 1.0)
    return pairs, init


# ------------------------------------------------------------------ pair roles and variants
@pytest.mark.parametrize("variant", ["default", "exhaustive", "rotation_only", "large", "cluster"])
def test_pair_roles_equal_host_built_table(gicp, engines, variant):
    base, poses = _base(14, 1024, 9101)
    targets = [3, 9]
    members, transforms = _windows(poses, targets, 2)
    ids = _setup(gicp, engines, base, members, transforms)
    pairs, init = _role_pairs(poses, len(base), ids, targets)
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


def test_all_pairs_and_run_device_see_the_submaps(gicp, engines):
    import torch
    base, poses = _base(10, 1024, 9102)
    members, transforms = _windows(poses, [2, 6], 1)
    ids = _setup(gicp, engines, base, members, transforms)
    a, b = engines
    n = len(base) + len(ids)
    B = n * (n - 1) // 2
    ra = a.run(None, all_pairs=(0, B, 0, B), epsilon=0.05)
    rb = b.run(None, all_pairs=(0, B, 0, B), epsilon=0.05)
    _same(ra, rb)
    pairs, init = _role_pairs(poses, len(base), ids, [2, 6])
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


# ------------------------------------------------------------------ submap sizes and shapes
@pytest.mark.parametrize("case", ["fits", "split", "ragged", "repeated", "non_rigid"])
def test_submap_shapes_equal_host_built_table(gicp, synth, engines, case):
    base, poses = _base(20, 1024, 9103)
    base = list(base)
    if case == "fits":
        members, transforms = _windows(poses, [4, 12], 2)                     # 4 x 1,024 beams
        members, transforms = [m[:4] for m in members], [t[:4] for t in transforms]
    elif case == "split":
        members, transforms = _windows(poses, [8, 10], 8)                     # 16-17 x 1,024 beams
    elif case == "ragged":
        rng = np.random.default_rng(9104)
        base[5] = base[5][:1]                                                  # 1-point scans
        base[6] = base[6][:3]
        base[7] = base[7][::7]
        base[9] = rng.normal(size=(1, 2))
        members = [np.array([5, 6, 7]), np.array([9]), np.array([7, 5, 8, 9, 6])]
        from icp_slam_b200 import callers
        transforms = callers.submap_window_transforms(poses, [6, 9, 3], members)
    elif case == "repeated":
        members, transforms = _windows(poses, [6], 1)
        members = [np.r_[members[0], members[0][1]], np.array([2, 2])]
        transforms = [np.concatenate([transforms[0], transforms[0][1:2]]), np.stack([np.eye(3), np.eye(3)])]
    else:
        members, transforms = _windows(poses, [5, 14], 2)
        A = np.array([[1.2, 0.3, 5.0], [-0.1, 0.8, -2.0], [0.0, 0.0, 1.0]])  # shear and scale, within bounds
        transforms = [A @ t for t in transforms]
        for t in transforms:
            t[:, 2] = (0.0, 0.0, 1.0)
    ids = _setup(gicp, engines, base, members, transforms)
    a, _ = engines
    if case == "split":
        assert a.table.longest > 16 * 1000                                    # beyond shared memory
    pairs = [(1, ids[0]), (ids[-1], 0), (ids[0], ids[-1]), (2, 3), (ids[-1], ids[-1])]
    if case == "split":
        n0 = a.launch_count
        a.run(pairs, epsilon=0.05)
        assert a.launch_count - n0 == 2                                       # split by scan length
    _both(engines, np.array(pairs, dtype=np.int32))


def test_multistart_on_submaps_equals_host_built_table(gicp, engines):
    base, poses = _base(14, 1024, 9105)
    targets = [3, 9]
    members, transforms = _windows(poses, targets, 3)
    ids = _setup(gicp, engines, base, members, transforms)
    pairs, init = _role_pairs(poses, len(base), ids, targets)
    a, b = engines
    S = gicp.heading_starts(4)
    for guess in (init, None):
        x = a.run_multistart(pairs, S, guess, epsilon=0.05, return_all=True)
        y = b.run_multistart(pairs, S, guess, epsilon=0.05, return_all=True)
        for f in ("T", "error", "iters", "start", "error_all", "iters_all"):
            np.testing.assert_array_equal(getattr(x, f), getattr(y, f))


# ------------------------------------------------------------------ replacement, growth, borrowed base
def test_replacement_growth_and_back_to_the_base(gicp, engines):
    base, poses = _base(16, 1024, 9106)
    a, b = engines
    base_pairs = np.array([(i + 1, i) for i in range(len(base) - 1)], dtype=np.int32)
    a.set_scans(list(base))
    before = a.run(base_pairs, epsilon=0.05, return_history=True, return_correspondences=True)
    small = _windows(poses, [4, 9], 0)
    large = _windows(poses, [2, 5, 8, 11, 14], 6)                              # several times the base's points
    for members, transforms in (small, large, small):
        ids = a.set_submaps(members, transforms)
        b.set_scans(list(base) + gicp.merge_scans(list(base), members, transforms))
        pairs = np.array([(1, ids[0]), (ids[-1], 3), (ids[0], ids[-1])] + [tuple(p) for p in base_pairs[:4]],
                         dtype=np.int32)
        _both(engines, pairs)
    assert a.set_submaps([], []).size == 0
    assert a._L.icpb_scan_count(a._h) == len(base) and a.table.n_scans == len(base)
    _same(a.run(base_pairs, epsilon=0.05, return_history=True, return_correspondences=True), before)
    # a new table drops the submaps
    a.set_submaps(*small)
    a.set_scans(list(base[:5]))
    assert a._L.icpb_scan_count(a._h) == 5


def test_borrowed_base_equals_uploaded_base(gicp, engines):
    import torch
    base, poses = _base(12, 1024, 9107)
    a, b = engines
    t = gicp.ScanTable(list(base))
    dev = torch.device("cuda", a.device)
    xy_t, off_t = torch.from_numpy(t.xy).to(dev), torch.from_numpy(t.offsets).to(dev)
    torch.cuda.synchronize(dev)
    xy0, off0 = xy_t.cpu().numpy().tobytes(), off_t.cpu().numpy().tobytes()
    members, transforms = _windows(poses, [3, 8], 2)
    a.set_scans_device(xy_t, off_t, t)
    ids = a.set_submaps(members, transforms)
    b.set_scans(list(base) + gicp.merge_scans(list(base), members, transforms))
    pairs = np.array([(1, ids[0]), (ids[1], 2), (ids[0], ids[1]), (5, 4)], dtype=np.int32)
    ref = _both(engines, pairs)
    torch.cuda.synchronize(dev)
    assert xy_t.cpu().numpy().tobytes() == xy0 and off_t.cpu().numpy().tobytes() == off0
    # the handle reads its own copy from now on
    xy_t.zero_()
    torch.cuda.synchronize(dev)
    _same(a.run(pairs, epsilon=0.05, return_history=True, return_correspondences=True), ref)
    ids2 = a.set_submaps(members[::-1], transforms[::-1])                    # rebuilt from the copied base
    b.set_scans(list(base) + gicp.merge_scans(list(base), members[::-1], transforms[::-1]))
    _both(engines, np.array([(1, ids2[0]), (ids2[1], 2)], dtype=np.int32))


# ------------------------------------------------------------------ rejections
def _raw(e, members, sub_off, T6, n):
    ptr = lambda a: None if a is None else ctypes.c_void_p(a.ctypes.data)   # noqa: E731
    return e._L.icpb_set_submaps(e._h, ptr(members), ptr(sub_off), ptr(T6), n)


def test_rejections_leave_the_table(gicp, engines):
    base, poses = _base(12, 1024, 9108)
    a, _ = engines
    members, transforms = _windows(poses, [3, 8], 2)
    a.set_scans(list(base))
    ids = a.set_submaps(members, transforms)
    n_base, n_all = len(base), len(base) + len(ids)
    pairs = np.array([(1, ids[0]), (ids[1], 2), (ids[0], ids[1]), (5, 4)], dtype=np.int32)
    before = a.run(pairs, epsilon=0.05, return_history=True, return_correspondences=True)

    def unchanged(name):
        assert a._L.icpb_scan_count(a._h) == n_all, name
        assert a.table.n_scans == n_all, name
        _same(a.run(pairs, epsilon=0.05, return_history=True, return_correspondences=True), before)

    I1 = np.eye(3)[None]
    mem = np.array([0, 1], dtype=np.int32)
    off = np.array([0, 2], dtype=np.int64)
    T6 = np.ascontiguousarray(np.tile([1.0, 0.0, 0.0, 0.0, 1.0, 0.0], (2, 1)))
    # one base point's x, pushed just past ICPB_MAX_COORD by an in-bounds shift of an in-bounds scan
    xmax = float(np.max(base[0][:, 0]))
    assert xmax > 0
    past = np.array([[1.0, 0.0, 1e10 - xmax + 1.0], [0.0, 1.0, 0.0], [0.0, 0.0, 1.0]])[None]
    assert np.abs(gicp.merge_scans(list(base), [np.array([0])], [past])[0]).max() > 1e10
    T_past = np.ascontiguousarray(past[:, :2].reshape(-1, 6))
    wide6, far6, nan6 = T6.copy(), T6.copy(), T6.copy()
    wide6[1, 0] = 1.5e3
    far6[0, 5] = -2e12
    nan6[1, 2] = np.inf
    raw = {
        "null offsets": (mem, None, T6, 1, EINVAL),
        "null members": (None, off, T6, 1, EINVAL),
        "null transforms": (mem, off, None, 1, EINVAL),
        "negative count": (mem, off, T6, -1, EINVAL),
        "offsets not from 0": (mem, np.array([1, 2], dtype=np.int64), T6, 1, EINVAL),
        "empty submap": (mem, np.array([0, 2, 2], dtype=np.int64), T6, 2, EINVAL),
        "member past the base": (np.array([0, n_base], dtype=np.int32), off, T6, 1, EINVAL),
        "member is a submap": (np.array([0, ids[0]], dtype=np.int32), off, T6, 1, EINVAL),
        "negative member": (np.array([-1, 0], dtype=np.int32), off, T6, 1, EINVAL),
        "linear bound": (mem, off, wide6, 1, EINVAL),
        "shift bound": (mem, off, far6, 1, EINVAL),
        "non-finite transform": (mem, off, nan6, 1, EINVAL),
        "merged coordinate past 1e10": (np.array([0], dtype=np.int32), np.array([0, 1], dtype=np.int64), T_past, 1,
                                        EINVAL),
        "beyond the 32-bit layout": (np.zeros(200_000, dtype=np.int32), np.array([0, 200_000], dtype=np.int64),
                                     np.ascontiguousarray(np.tile(T6[:1], (200_000, 1))), 1, ETOOLONG),
    }
    for name, (m, o, t, n, want) in raw.items():
        n0 = a.launch_count
        assert _raw(a, m, o, t, n) == want, name
        assert a.launch_count == n0, name
        unchanged(name)
    # the same through Python: ValueError, the table unchanged
    py = {
        "lists of different lengths": ([np.array([0])], []),
        "member is a submap": ([np.array([0, ids[0]])], [np.stack([np.eye(3)] * 2)]),
        "bottom row": ([np.array([0])], [np.array([[[1.0, 0, 0], [0, 1, 0], [0.5, 0, 1]]])]),
        "non-finite": ([np.array([0])], [np.where(np.eye(3) == 1, np.nan, 0.0)[None]]),
        "merged coordinate past 1e10": ([np.array([0])], [past]),
        "beyond the 32-bit layout": ([np.zeros(200_000, dtype=np.int64)], [np.tile(I1, (200_000, 1, 1))]),
    }
    for name, args in py.items():
        with pytest.raises(ValueError):
            a.set_submaps(*args)
        unchanged(name)
    # no table at all
    fresh = gicp.IcpEngine()
    try:
        assert _raw(fresh, mem, off, T6, 1) == ENOSCANS
        with pytest.raises(ValueError):
            fresh.set_submaps([mem], [np.stack([np.eye(3)] * 2)])
    finally:
        fresh.close()


# ------------------------------------------------------------------ the proximity caller
@functools.lru_cache(maxsize=None)
def _loop(n_poses, beams, seed):
    from icp_slam_b200 import synth
    rng = np.random.default_rng(seed)
    poses = synth.loop_trajectory(n_poses, step=0.2)
    return poses, synth.scans_from_poses(poses, beams, rng, drop_frac=0.03)


def test_window_zero_gives_todays_constraints():
    from icp_slam_b200 import callers
    poses, scans = _loop(500, 360, 9201)
    want, wres = callers.proximity_loop_closures(poses, scans)
    got, gres = callers.proximity_loop_closures(poses, scans, submap_window=0)
    assert len(want) > 0 and len(got) == len(want)
    for (i, j, T), (i2, j2, T2) in zip(got, want):
        assert (i, j) == (i2, j2)
        np.testing.assert_array_equal(T, T2)
    np.testing.assert_array_equal(gres.error, wres.error)
    np.testing.assert_array_equal(gres.iters, wres.iters)


def test_window_four_constraints_meet_the_truth(gicp):
    from icp_slam_b200 import callers, synth
    poses, scans = _loop(500, 360, 9202)
    got, res = callers.proximity_loop_closures(poses, scans, submap_window=4)
    assert len(got) > 0 and np.all(res.error < 110)
    for i, j, T in got:
        dt, dth = pose_diff(T, np.linalg.inv(synth.pose_to_mat(poses[i])) @ synth.pose_to_mat(poses[j]))
        assert dt < 0.05 and dth < 0.01, (i, j, dt, dth)
    # the engine is left with the scan table alone
    e = gicp.engine()
    assert e._L.icpb_scan_count(e._h) == len(scans)
    with pytest.raises(ValueError):
        callers.proximity_loop_closures(poses, scans, submap_window=-1)
