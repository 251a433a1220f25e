"""Drop-in for the reference's ``src/pose_graph_optimization.py``: same function names and
arguments, bodies on the GPU (SURVEY.md section 8f-3 and row a10).

* ``pose_graph_optimization_step_sgd(pose_graph, learning_rate=1, loop_closure_uncertainty=0.1)``
  -- one pass of the modified SGD over the loop-closure edges (reference
  src/pose_graph_optimization.py:7-49), ``pose_graph.poses`` updated in place.  The pose graph is
  used exactly as the reference uses it: ``pose_graph.graph.edges(data="object")`` (iteration
  order matters) and ``pose_graph.poses``; the reference's own ``PoseGraph`` works unchanged.
* ``optimise(pose_graph, n_steps)`` -- the loop of scripts/main.py:325-326 (learning rate
  1/(k+1)) in one call: poses and edges cross PCIe once.
* ``recompute_pose_graph_orientation(...)`` -- :51-74; the ``icp_recompute`` branch is one batched
  rotation-only ICP launch (``callers.rotation_only_headings``) instead of the joblib fan-out.

No CPU fallback: without libicpb.so and a B200 these raise.
"""
from __future__ import annotations

import numpy as np

from . import _lib
from . import icp as _icp


def construct_R(pose_graph, idx):
    """src/pose_graph_optimization.py:76-85."""
    theta = pose_graph.poses[idx][2]
    c, s = np.cos(theta), np.sin(theta)
    return np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]])


def edge_arrays(pose_graph):
    """(a, b) int32 rows and 2x3 transforms of the edges the optimiser acts on, in the graph's
    iteration order.  Odometry edges (|a-b| == 1) are skipped by the reference (:14-16, :28-30) and
    edges with b <= a have empty node ranges (:20, :46), so neither is sent to the device."""
    ab, Ts = [], []
    edges = pose_graph.graph.edges(data="object") if hasattr(pose_graph, "graph") else pose_graph
    for a, b, T in edges:
        a, b = int(a), int(b)
        if b - a <= 1:                                         # |a - b| == 1 or b <= a
            continue
        ab.append((a, b))
        Ts.append(T)
    if not ab:
        return np.zeros((0, 2), dtype=np.int32), np.zeros((0, 6), dtype=np.float64)
    # one conversion and one check for all edges; the per-edge walk below only names the offender
    try:
        tf = np.asarray(Ts, dtype=np.float64)
    except ValueError:
        tf = None
    if tf is None or tf.shape != (len(ab), 3, 3) or not (
            (tf[:, 2, 0] == 0.0) & (tf[:, 2, 1] == 0.0) & (tf[:, 2, 2] == 1.0)).all():
        for (a, b), T in zip(ab, Ts):
            T = np.asarray(T, dtype=np.float64)
            if T.shape != (3, 3):
                raise ValueError(f"edge ({a}, {b}) carries a transform of shape {T.shape}; expected (3, 3)")
            if not (T[2, 0] == 0.0 and T[2, 1] == 0.0 and T[2, 2] == 1.0):
                raise ValueError(f"edge ({a}, {b}): the transform's bottom row is not [0, 0, 1]")
    return np.asarray(ab, dtype=np.int32).reshape(-1, 2), _icp._top_rows(tf)


def sgd_steps(poses, edges_ab, edges_T6, learning_rates, loop_closure_uncertainty=0.1, device=None):
    """len(learning_rates) SGD passes over a fixed edge list; returns the new (n, 3) poses."""
    poses = np.array(poses, dtype=np.float64, order="C")
    if poses.ndim != 2 or poses.shape[1] != 3:
        raise ValueError(f"poses has shape {poses.shape}; expected (n, 3)")
    ab = np.ascontiguousarray(edges_ab, dtype=np.int32).reshape(-1, 2)
    T6 = np.ascontiguousarray(edges_T6, dtype=np.float64).reshape(-1, 6)
    if len(ab) != len(T6):
        raise ValueError("edges and transforms differ in length")
    lrs = np.ascontiguousarray(learning_rates, dtype=np.float64).reshape(-1)
    eng = _icp.engine(device)
    _lib.check(_lib.lib().icpb_pose_graph_sgd(eng._h, _lib.ptr(poses), len(poses),
                                               _lib.ptr(ab) if len(ab) else None,
                                               _lib.ptr(T6) if len(ab) else None, len(ab),
                                               _lib.ptr(lrs) if len(lrs) else None, len(lrs),
                                               float(loop_closure_uncertainty)),
               "icpb_pose_graph_sgd")
    return poses


def pose_graph_optimization_step_sgd(pose_graph, learning_rate=1, loop_closure_uncertainty=0.1, device=None):
    """src/pose_graph_optimization.py:7-49; mutates ``pose_graph.poses`` in place, returns None."""
    ab, T6 = edge_arrays(pose_graph)
    pose_graph.poses[...] = sgd_steps(pose_graph.poses, ab, T6, [float(learning_rate)],
                                      loop_closure_uncertainty, device)


def optimise(pose_graph, n_steps, loop_closure_uncertainty=0.1, device=None):
    """``for k in range(n_steps): step_sgd(pg, learning_rate=1/(k+1))`` (scripts/main.py:325-326)."""
    ab, T6 = edge_arrays(pose_graph)
    lrs = [1.0 / float(k + 1) for k in range(int(n_steps))]
    pose_graph.poses[...] = sgd_steps(pose_graph.poses, ab, T6, lrs, loop_closure_uncertainty, device)


def recompute_pose_graph_orientation(pose_graph, lidar_points, icp_max_iters, icp_epsilon, n_jobs=None,
                                     icp_recompute=False, device=None):
    """src/pose_graph_optimization.py:51-74.  Headings of the interior poses from the path tangent
    (:52-57: each uses positions only, so the loop is one vector expression), then optionally the
    rotation-only ICP re-accumulation (:59-74).  ``n_jobs`` is accepted and ignored."""
    poses = pose_graph.poses
    n = len(poses)
    if n > 2:
        vec = poses[2:, 0:2] - poses[1:-1, 0:2]
        norm = np.sqrt(vec[:, 0] ** 2 + vec[:, 1] ** 2)         # np.linalg.norm of a 2-vector
        ok = norm > 0
        unit = vec[ok] / norm[ok][:, None]
        heading = poses[1:-1, 2].copy()
        heading[ok] = np.arctan2(unit[:, 1], unit[:, 0])
        poses[1:-1, 2] = heading
    if icp_recompute:
        from . import callers
        new, _ = callers.rotation_only_headings(poses, lidar_points, max_iters=icp_max_iters,
                                                epsilon=icp_epsilon, device=device)
        poses[:, 2] = new[:, 2]
