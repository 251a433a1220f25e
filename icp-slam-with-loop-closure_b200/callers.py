"""Batched forms of the reference's ICP call sites (the rows either side of the hot path).

Each function builds the pair list and initial guesses exactly like the reference caller does,
runs ONE ``icp_batch`` launch instead of the caller's loop / joblib fan-out, and hands back what
the caller's remaining host code consumes.  The pose graph container, the SGD relaxation and the
maps stay the reference's own code (out of scope, SURVEY.md section 2).

* ``odometry_chain``            -- scripts/main.py:239-256 (ICP fan-out + chain composition)
* ``proximity_candidates``      -- src/loop_closure_detection.py:12-25 (candidate generation, GPU)
* ``proximity_pairs``           -- the same rule keeping every pair within the radius (config 3)
* ``proximity_loop_closures``   -- src/loop_closure_detection.py:26-39 (ICP + greedy acceptance)
* ``image_match_loop_closures`` -- src/loop_closure_detection.py:134-159 (ICP over image matches)
* ``rotation_only_headings``    -- src/pose_graph_optimization.py:59-74
"""
from __future__ import annotations

import numpy as np

from . import icp as _icp
from .synth import mat_to_pose, pose_to_mat


def chain_pairs(n_scans: int, stride: int = 1, start: int = 0) -> np.ndarray:
    """(source i, target i - stride) for i = start + stride, start + 2*stride, ...
    (scripts/main.py:241-243; stride-k variant scripts/map_proximity_loop_closure.py:50-56)."""
    idx = np.arange(start + stride, n_scans, stride)
    return np.stack((idx, idx - stride), axis=1).astype(np.int32)


def poses_to_mats(poses) -> np.ndarray:
    """``utils.pose_to_mat`` (src/utils.py:28-33) for an (n, 3) array of poses at once: (n, 3, 3).
    numpy's cos/sin give the same bits on arrays as on scalars, so this equals the reference's
    per-pose calls."""
    poses = np.asarray(poses, dtype=np.float64).reshape(-1, 3)
    c, s = np.cos(poses[:, 2]), np.sin(poses[:, 2])
    out = np.zeros((len(poses), 3, 3))
    out[:, 0, 0] = c; out[:, 0, 1] = -s; out[:, 0, 2] = poses[:, 0]
    out[:, 1, 0] = s; out[:, 1, 1] = c; out[:, 1, 2] = poses[:, 1]
    out[:, 2, 2] = 1.0
    return out


def odometry_chain(lidar_points, odometry, max_iters=100, epsilon=0.05, device=None):
    """ICP-corrected poses of the whole trajectory (scripts/main.py:239-256).

    The initial guess of pair (i, i-1) is ``pose_to_mat(odometry[i] - odometry[i-1])`` -- a raw
    global-frame pose difference used as a local transform, as the reference does (:244).
    Returns (corrected_poses (n, 3), BatchResult)."""
    odometry = np.asarray(odometry, dtype=np.float64)
    n = len(odometry)
    pairs = chain_pairs(n)
    init = poses_to_mats(odometry[1:] - odometry[:-1])
    res = _icp.icp_batch(lidar_points, pairs, init, epsilon=epsilon, max_iters=max_iters, device=device)
    # long chains: the device scan (0.11 ms against 0.24 ms for the C host loop at 4,999 steps, equal to
    # 1e-14; tools/compose_bench.py); short ones: the host loop (0.03 ms against 0.06 ms at 500 steps)
    if len(res.T) >= 2000:
        return compose_chain_gpu(odometry[0], res.T, device), res
    return compose_chain(odometry[0], res.T), res


def odometry_chain_strided(lidar_points, odometry, start, skip, max_iters=100, epsilon=0.05, device=None):
    """The serial stride-k scan matching loop of scripts/map_icp.py:44-86 (same loop in
    scripts/map_proximity_loop_closure.py:50-88) as one batch: for i = start, start + skip, ... scan i
    is aligned onto scan i - skip with the odometry difference as the initial guess, and the result is
    composed onto the LAST pose of the list -- which for the first step is ``odometry[start - 1]``, not
    ``odometry[start - skip]`` (the script seeds the list with the raw odometry of poses 0..start-1).
    Returns (corrected_poses as the script builds them: (start + number of steps, 3), BatchResult)."""
    odometry = np.asarray(odometry, dtype=np.float64)
    if not 0 < skip < start:
        raise ValueError("the reference asserts skip < start (scripts/map_icp.py:45)")
    idx = np.arange(start, len(odometry), skip)
    pairs = np.stack((idx, idx - skip), axis=1).astype(np.int32)
    init = poses_to_mats(odometry[idx] - odometry[idx - skip])
    res = _icp.icp_batch(lidar_points, pairs, init, epsilon=epsilon, max_iters=max_iters, device=device)
    tail = compose_chain(odometry[start - 1], res.T)[1:]
    return np.vstack((odometry[:start], tail)), res


def compose_chain(pose0, transforms) -> np.ndarray:
    """Serial SE(2) prefix product of scripts/main.py:249-256:
    ``pose_i = mat_to_pose(pose_to_mat(pose_{i-1}) @ T_{i-1})``; (n + 1, 3) poses from n transforms.
    Runs in the library's C host loop (the reference's Python loop costs ~100 ms at n = 5,000)."""
    T = np.asarray(transforms, dtype=np.float64)
    T6 = np.ascontiguousarray(T[:, :2, :].reshape(-1, 6))
    p0 = np.ascontiguousarray(pose0, dtype=np.float64)
    out = np.empty((len(T6) + 1, 3))
    _icp._lib.check(_icp._lib.lib().icpb_compose_chain(_icp._ptr(p0), _icp._ptr(T6), len(T6), _icp._ptr(out)),
                    "icpb_compose_chain")
    return out


def compose_chain_gpu(pose0, transforms, device=None) -> np.ndarray:
    """`compose_chain` through the device scan (icpb_compose_chain_gpu): same poses to rounding."""
    T = np.asarray(transforms, dtype=np.float64)
    T6 = np.ascontiguousarray(T[:, :2, :].reshape(-1, 6))
    p0 = np.ascontiguousarray(pose0, dtype=np.float64)
    out = np.empty((len(T6) + 1, 3))
    e = _icp.engine(device)
    _icp._lib.check(e._L.icpb_compose_chain_gpu(e._h, _icp._ptr(p0), _icp._ptr(T6), len(T6), _icp._ptr(out)),
                    "icpb_compose_chain_gpu")
    return out


def _travelled(xy: np.ndarray) -> np.ndarray:
    """The reference's ``dist_traveled`` (src/loop_closure_detection.py:13-14): cumulative sum of the
    consecutive pose distances, first entry 0.  O(S) on the host, in numpy's summation order."""
    step = np.sqrt((xy[1:, 0] - xy[:-1, 0]) ** 2 + (xy[1:, 1] - xy[:-1, 1]) ** 2)
    return np.concatenate(([0.0], np.cumsum(step)))


def proximity_candidates(poses, min_dist_along_path=2, max_dist=1, device=None):
    """At most one candidate per pose i: the Euclidean-closest pose j among those at least
    ``min_dist_along_path`` further along the path, kept if within ``max_dist``
    (src/loop_closure_detection.py:12-25).  The S x S cdist matrix of the reference is never
    built: one warp per pose scans its row on the GPU (icpb_proximity_closest).  Returned in the
    reference's processing order (its ``matches.reverse()``), as an (M, 2) array of (i, j)."""
    import ctypes
    xy = np.ascontiguousarray(np.asarray(poses, dtype=np.float64)[:, :2])
    n = len(xy)
    trav = _travelled(xy)
    closest = np.empty(n, dtype=np.int32)
    dist = np.empty(n)
    e = _icp.engine(device)
    _icp._lib.check(e._L.icpb_proximity_closest(e._h, _icp._ptr(xy), _icp._ptr(trav), n,
                                                ctypes.c_double(min_dist_along_path), ctypes.c_double(max_dist),
                                                _icp._ptr(closest), _icp._ptr(dist)), "icpb_proximity_closest")
    i = np.nonzero(closest >= 0)[0]
    out = np.stack((i, closest[i].astype(np.int64)), axis=1)[::-1]
    return np.ascontiguousarray(out, dtype=np.int64).reshape(-1, 2)


def proximity_pairs(poses, min_dist_along_path=2, max_dist=1, device=None) -> np.ndarray:
    """Every pair within the radius (BASELINE config 3's generalisation of detect_proximity): all
    (i, j) with j at least ``min_dist_along_path`` further along the path than i and within
    ``max_dist``, as (source = j, target = i) int32 rows ordered by i then j."""
    import ctypes
    xy = np.ascontiguousarray(np.asarray(poses, dtype=np.float64)[:, :2])
    n = len(xy)
    trav = _travelled(xy)
    e = _icp.engine(device)
    total = ctypes.c_int64()
    args = (e._h, _icp._ptr(xy), _icp._ptr(trav), n, ctypes.c_double(min_dist_along_path), ctypes.c_double(max_dist))
    _icp._lib.check(e._L.icpb_proximity_pairs(*args, 0, None, ctypes.byref(total)), "icpb_proximity_pairs")
    pairs = np.empty((total.value, 2), dtype=np.int32)
    if total.value:
        _icp._lib.check(e._L.icpb_proximity_pairs(*args, total.value, _icp._ptr(pairs), ctypes.byref(total)),
                        "icpb_proximity_pairs")
    return pairs


def _multistart_accept(lidar_points, pairs, starts, thresh, epsilon, max_iters, device):
    """Every candidate aligned from the identity with every start (so its guesses are the starts
    themselves), the best start kept, and the pairs whose best error is below ``thresh``: (rows,
    MultiStartResult of those rows).  The threshold runs on the host over B results, not B * K."""
    res = _icp.icp_multistart(lidar_points, pairs, starts, None, epsilon=epsilon, max_iters=max_iters, device=device)
    rows = np.nonzero(res.error < thresh)[0]
    return rows, _icp.MultiStartResult(res.T[rows], res.error[rows], res.iters[rows], start=res.start[rows])


def proximity_loop_closures(poses, lidar_points, min_dist_along_path=2, max_dist=1, err_thresh=110,
                            max_iters=100, epsilon=0.05, device=None, starts=None):
    """Loop-closure constraints the reference's ``detect_proximity`` would add, in its order.

    ICP is a pure function of its inputs, so every candidate is aligned in one batch
    (source = scan j, target = scan i, identity initial guess, :31-34) and the reference's greedy
    loop -- skip a candidate if either endpoint was already used by an *accepted* one, accept if
    error < err_thresh -- is replayed on the results (:27-39).  Returns a list of
    (i, j, T 3x3) ready for ``pose_graph.add_constraint(i, j, T)``, and the BatchResult of the candidates
    that passed the threshold.

    ``starts`` ((K, 3, 3), e.g. ``icp.heading_starts(8)``): for revisits whose relative heading is
    unknown, every candidate is aligned from each start with ``icp_multistart`` and its best start is
    the one tested against the threshold; the BatchResult is then a MultiStartResult (``start`` says
    which start won)."""
    cand = proximity_candidates(poses, min_dist_along_path, max_dist, device)
    if len(cand) == 0:
        return [], None
    pairs = np.stack((cand[:, 1], cand[:, 0]), axis=1).astype(np.int32)
    if starts is not None:
        rows, res = _multistart_accept(lidar_points, pairs, starts, err_thresh, epsilon, max_iters, device)
    else:
        # the `error < err_thresh` test runs in the kernel epilogue: only the candidates that pass it come
        # back (a candidate that fails it never marks its endpoints as used, so the greedy loop over the
        # passing ones, in the reference's order, accepts exactly what the reference accepts)
        rows, res = _icp.engine(device).align_accept(lidar_points, pairs, err_thresh, None, epsilon=epsilon,
                                                     max_iters=max_iters)
    used = set()
    out = []
    for (i, j), T in zip(cand[rows], res.T):
        i, j = int(i), int(j)
        if i in used or j in used:
            continue
        out.append((i, j, T))
        used.add(i)
        used.add(j)
    return out, res


def image_match_loop_closures(good_matches, lidar_points, image_rate=1, icp_err_thresh=30, max_iters=100,
                              epsilon=0.05, device=None, starts=None):
    """ICP block of the reference's ``detect_images_direct_similarity``
    (src/loop_closure_detection.py:134-159): for every image match (i, j) align scan
    ``i*image_rate`` (source) onto scan ``j*image_rate`` (target) from the identity -- note the
    argument order is the opposite of ``detect_proximity``'s, a reference quirk kept as is -- and
    keep the pairs with error < icp_err_thresh.  Returns [(i*rate, j*rate, T)] in match order, and
    the BatchResult of the accepted pairs.  The ORB/matcher front end that produces ``good_matches`` is out of scope.
    ``starts``: a multi-start sweep per match, as in ``proximity_loop_closures`` (an image match between
    scans taken facing different directions)."""
    gm = np.asarray(good_matches, dtype=np.int64).reshape(-1, 2)
    if len(gm) == 0:
        return [], None
    pairs = (gm * image_rate).astype(np.int32)               # (source = i*rate, target = j*rate)
    if starts is not None:
        rows, res = _multistart_accept(lidar_points, pairs, starts, icp_err_thresh, epsilon, max_iters, device)
    else:
        rows, res = _icp.engine(device).align_accept(lidar_points, pairs, icp_err_thresh, None, epsilon=epsilon,
                                                     max_iters=max_iters)      # filter on the device
    out = [(int(pairs[r, 0]), int(pairs[r, 1]), T) for r, T in zip(rows, res.T)]
    return out, res


def rotation_only_headings(poses, lidar_points, max_iters=100, epsilon=0.05, device=None):
    """Headings re-accumulated from rotation-only ICP between consecutive scans
    (src/pose_graph_optimization.py:59-74, the ``icp_recompute`` branch).  Returns a copy of
    ``poses`` with column 2 rewritten the way the reference's reverse sweep leaves it."""
    poses = np.array(poses, dtype=np.float64)
    n = len(poses)
    pairs = chain_pairs(n)
    init = poses_to_mats(poses[1:] - poses[:-1])
    res = _icp.icp_batch(lidar_points, pairs, init, epsilon=epsilon, max_iters=max_iters,
                         rotation_only=True, device=device)
    # the reference sweeps from the end (:70-74), so pose i-1 still holds its OLD heading when pose i
    # is rewritten: one vector expression
    poses[1:, 2] = poses[:-1, 2].copy() + np.arctan2(res.T[:, 1, 0], res.T[:, 0, 0])
    return poses, res
