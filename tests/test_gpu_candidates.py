"""Loop-closure candidate kernels (icpb_proximity_closest / icpb_proximity_pairs) under adversarial
inputs, bit-exact against oracle/slam_oracle.py (cdist's rounding, tests/test_slam_oracle.py):
P1 ties, P2 the radius boundary, P3 shapes, P4 the input contract of include/icpb.h
(ICPB_MAX_POSE_COORD, a finite non-decreasing `travelled`, a min_dist_along_path that is not NaN)."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def check(poses, min_dist_along_path=2, max_dist=1):
    from icp_slam_b200 import callers
    from oracle import slam_oracle
    poses = np.asarray(poses, dtype=np.float64)
    cand = callers.proximity_candidates(poses, min_dist_along_path, max_dist)
    np.testing.assert_array_equal(cand, slam_oracle.proximity_candidates_ref(poses, min_dist_along_path, max_dist))
    pairs = callers.proximity_pairs(poses, min_dist_along_path, max_dist)
    np.testing.assert_array_equal(pairs, slam_oracle.proximity_pairs_ref(poses, min_dist_along_path, max_dist))
    return cand, pairs


def with_heading(xy, rng):
    xy = np.asarray(xy, dtype=np.float64)
    return np.c_[xy, rng.uniform(-np.pi, np.pi, len(xy))]


# ---- P1: ties ---------------------------------------------------------------------------------------

def stopping_robot(rng, n=400):
    """Integer steps on a 1/8 m lattice with runs of identical poses (the robot stops): travelled has
    plateaus and distances tie exactly."""
    steps = rng.integers(-1, 2, (n, 2)) / 8.0
    steps[rng.random(n) < 0.35] = 0.0
    steps[100:140] = 0.0
    return np.cumsum(steps, axis=0)


def test_p1_plateaus_and_exact_ties():
    rng = np.random.default_rng(1)
    xy = stopping_robot(rng)
    for mdp, md in ((2, 1), (0.0, 0.5), (0.125, 0.25), (1.0, 0.0), (3.0, 2.0)):
        cand, _ = check(with_heading(xy, rng), mdp, md)
    # the plateau: many poses at one place, argmin must pick the first of them
    assert len(cand) > 20


def test_p1_equal_distances_across_lanes_and_warp_blocks():
    """Pose i at the origin; poses j spread over several 32-wide blocks of j all at distance 5 (3-4-5
    and 5-0 offsets), others farther: the kernel's (distance, index) reduction must return the first."""
    rng = np.random.default_rng(2)
    n = 300
    xy = np.c_[np.arange(n) * 0.0 + 40.0, np.arange(n) * 1.0]           # a far line (distance > 5)
    xy[0] = (0.0, 0.0)
    ring = np.array([(3.0, 4.0), (4.0, 3.0), (5.0, 0.0), (0.0, -5.0), (-3.0, 4.0), (-4.0, -3.0)])
    for k, j in enumerate((37, 70, 71, 101, 133, 250, 251, 299)):
        xy[j] = ring[k % len(ring)]
    poses = with_heading(xy, rng)
    for mdp in (2.0, 100.0):
        check(poses, mdp, 5.0)
    cand, pairs = check(poses, 0.0, 5.0)
    assert tuple(cand[-1]) == (0, 37)                                    # row 0: the first of eight ties
    assert ((pairs[:, 1] == 0).sum()) == 8


# ---- P2: the radius boundary ------------------------------------------------------------------------

def test_p2_pairs_on_one_ulp_either_side_of_the_radius():
    rng = np.random.default_rng(3)
    base = np.c_[np.arange(64) * 100.0, np.zeros(64)]                    # far apart: only the planted pairs
    xy = np.repeat(base, 2, axis=0)
    r = 5.0
    offs = [(3.0, 4.0), (4.0, -3.0), (np.nextafter(r, 0), 0.0), (np.nextafter(r, 10), 0.0), (0.0, r),
            (0.0, np.nextafter(r, 10)), (-3.0, np.nextafter(-4.0, -10)), (np.nextafter(3.0, 0), -4.0)]
    for k in range(64):
        xy[2 * k + 1] += offs[k % len(offs)]
    poses = with_heading(xy, rng)
    for md in (r, np.nextafter(r, 0), np.nextafter(r, 10)):
        cand, pairs = check(poses, 0.0, md)
    _, pairs = check(poses, 0.0, r)
    d = np.sqrt(((xy[pairs[:, 0]] - xy[pairs[:, 1]]) ** 2).sum(1))
    assert (d == r).sum() >= 24 and d.max() == r


def test_p2_pairs_that_hypot_rounds_differently_follow_cdist():
    """Pairs whose np.hypot and sqrt(dx*dx + dy*dy) differ in the last bit, with max_dist on one of the
    two values: the kernel follows cdist's sqrt form.  A pair oracle built on hypot (synth.proximity_pairs)
    disagrees with it here, which is why test_candidate_generation_on_gpu no longer uses one."""
    from icp_slam_b200 import synth
    rng = np.random.default_rng(4)
    xy, s_h = [], []
    while len(s_h) < 48:
        a = np.array([1000.0 * len(s_h), 0.0]) + rng.normal(0, 3, 2)
        b = a + rng.normal(0, 3, 2)
        dx, dy = b - a
        s, h = np.sqrt(dx * dx + dy * dy), np.hypot(dx, dy)
        if s != h:
            xy += [a, b]
            s_h.append((s, h))
    poses = with_heading(np.array(xy), rng)
    differs = 0
    for s, h in s_h[:24]:
        for md in (s, h):
            _, pairs = check(poses, 0.0, md)
            differs += not np.array_equal(synth.proximity_pairs(poses, 0.0, md), pairs)
    assert differs >= 24                      # one of the two radii always splits the two roundings


# ---- P3: shapes -------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 255, 256, 257])
def test_p3_pose_counts_around_the_warp(n):
    rng = np.random.default_rng(n)
    xy = np.cumsum(rng.normal(0, 0.3, (n, 2)), axis=0)
    poses = with_heading(xy, rng)
    for mdp, md in ((2, 1), (0.0, 0.5), (-1.0, 0.3), (np.inf, 1.0), (-np.inf, 0.7), (1.0, 0.0), (1.0, np.inf),
                    (0.0, np.inf), (1e9, 1.0)):
        check(poses, mdp, md)


def test_p3_far_coordinates_and_long_rows():
    """Poses 1e6 m and 1e12 m (ICPB_MAX_POSE_COORD) from the origin, and rows with hundreds of
    matches (more than 32 per row: several ballots per row)."""
    rng = np.random.default_rng(7)
    xy = np.cumsum(rng.normal(0, 0.2, (700, 2)), axis=0)
    for shift in (1e6, -1e6, 1e12 - 400.0, -1e12 + 400.0):
        poses = with_heading(xy + shift, rng)
        check(poses, 2, 1)
        _, pairs = check(poses, 0.5, 50.0)
        assert np.bincount(pairs[:, 1]).max() > 100
    corners = np.array([(1e12, 1e12), (-1e12, -1e12), (1e12, -1e12), (-1e12, 1e12), (0.0, 0.0)])
    check(with_heading(corners, rng), 0.0, np.inf)
    check(with_heading(corners, rng), 0.0, 2e12)


# ---- P4: the contract -------------------------------------------------------------------------------

def c_call(xy, trav, mdp, md):
    """Both entry points directly, with a caller-made `travelled`: (closest status, pairs status)."""
    from icp_slam_b200 import _lib, icp as gicp
    e = gicp.engine()
    xy = np.ascontiguousarray(xy, dtype=np.float64)
    trav = np.ascontiguousarray(trav, dtype=np.float64)
    n = len(xy)
    closest, dist = np.full(n, -7, np.int32), np.empty(n)
    rc1 = _lib.lib().icpb_proximity_closest(e._h, ctypes.c_void_p(xy.ctypes.data), ctypes.c_void_p(trav.ctypes.data),
                                            n, mdp, md, ctypes.c_void_p(closest.ctypes.data),
                                            ctypes.c_void_p(dist.ctypes.data))
    total = ctypes.c_int64(-1)
    rc2 = _lib.lib().icpb_proximity_pairs(e._h, ctypes.c_void_p(xy.ctypes.data), ctypes.c_void_p(trav.ctypes.data),
                                          n, mdp, md, 0, None, ctypes.byref(total))
    return rc1, rc2


def test_p4_bad_inputs_are_rejected():
    from icp_slam_b200 import callers
    rng = np.random.default_rng(9)
    xy = np.cumsum(rng.normal(0, 0.3, (80, 2)), axis=0)
    poses = with_heading(xy, rng)
    # a NaN min_dist_along_path: np.searchsorted puts it past the end (no candidates), a binary search
    # with `<=` at the start (every pose paired with itself); it is rejected
    for f in (callers.proximity_candidates, callers.proximity_pairs):
        try:
            got = f(poses, np.nan, 1.0)
        except ValueError:
            pass
        else:
            pytest.fail(f"{f.__name__} accepted a NaN min_dist_along_path and returned {len(got)} rows "
                        f"(the reference returns none), the first {got[:3].tolist()}")
        for bad in (np.nan, np.inf, -np.inf, 1.001e12):
            for r, c in ((0, 0), (40, 1), (79, 0)):
                p = poses.copy()
                p[r, c] = bad
                with pytest.raises(ValueError):
                    f(p, 2, 1)
    p = poses.copy()
    p[3, :2] = (1e12, -1e12)                                           # on the bound: accepted
    check(p, 2, 1)
    trav = np.concatenate(([0.0], np.cumsum(np.sqrt((np.diff(xy, axis=0) ** 2).sum(1)))))
    assert c_call(xy, trav, 2.0, 1.0) == (0, 0)
    for t in (trav[::-1].copy(), np.where(np.arange(80) == 30, trav[29] - 1e-9, trav),
              np.where(np.arange(80) == 50, np.nan, trav), np.where(np.arange(80) == 79, np.inf, trav)):
        assert c_call(xy, t, 2.0, 1.0) == (10001, 10001)
    assert c_call(xy, trav, np.nan, 1.0) == (10001, 10001)
    # NaN max_dist: no pair passes `<=`, as in the reference
    check(poses, 2, np.nan)
