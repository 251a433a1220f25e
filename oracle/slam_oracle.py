"""Restatement of the host-side consumers of the ICP path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Used by tests to carry ICP results through to an optimised trajectory (the 1e-4 m ATE criterion)
without the reference tree, which does not exist on the GPU box.  Pinned against
tests/golden/slam_golden.npz, produced by the unmodified reference pipeline
(tests/golden/make_slam_golden.py).

* loop edges in the order ``nx.DiGraph.edges`` yields them for the reference's PoseGraph
  (src/pose_graph.py:22-40): by source node, then insertion order; |a-b| == 1 edges are skipped
  by the optimiser (src/pose_graph_optimization.py:14-16).
* ``sgd_step`` follows src/pose_graph_optimization.py:7-49 with the per-node inner loops
  (:20-24, :44-48) written as slices / cumulative sums.
"""
from __future__ import annotations

import numpy as np


def _rot3(theta):
    c, s = np.cos(theta), np.sin(theta)
    return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])


def _pose_mat(p):
    c, s = np.cos(p[2]), np.sin(p[2])
    return np.array([[c, -s, p[0]], [s, c, p[1]], [0.0, 0.0, 1.0]])


def graph_order(loops):
    """Stable sort by source node: the order the reference's DiGraph iterates added constraints."""
    return sorted(loops, key=lambda e: e[0])


def sgd_step(poses, loops, learning_rate=1.0, loop_closure_uncertainty=0.1, in_graph_order=False):
    """One pass of the reference's modified SGD over the loop edges; mutates and returns poses.
    `in_graph_order`: `loops` is already in the order the graph iterates its edges (a flipped
    graph, src/pose_graph.py:42-52, does not iterate by ascending source node)."""
    n = len(poses)
    sigma = np.eye(3) * loop_closure_uncertainty
    weight = np.zeros((n, 3))
    gamma = np.full(3, np.inf)
    edges = [e for e in (loops if in_graph_order else graph_order(loops)) if abs(e[0] - e[1]) != 1]
    for a, b, _ in edges:                                        # :13-24
        rot = _rot3(poses[a][2])
        dw = np.diag(np.linalg.inv(rot @ sigma @ rot.T))
        if b > a:
            weight[a + 1:b + 1] += dw
            if gamma @ gamma > dw @ dw:
                gamma = dw
    for a, b, tf in edges:                                       # :27-48
        rot = _rot3(poses[a][2])
        pb = _pose_mat(poses[a]) @ tf
        resid = np.array([pb[0, 2], pb[1, 2], np.arctan2(pb[1, 0], pb[0, 0])]) - poses[b]
        resid[2] = resid[2] % (2 * np.pi)
        d = 2 * np.linalg.inv(rot.T @ sigma @ rot) @ resid.reshape(-1, 1)
        for j in range(3):
            alpha = learning_rate / gamma[j]
            total = np.sum(1 / weight[a + 1:b + 1, j])
            beta = (b - a) * d[j, 0] * alpha
            if abs(beta) > abs(resid[j]):
                beta = resid[j]
            inc = np.zeros(n)
            inc[a + 1:b + 1] = beta / weight[a + 1:b + 1, j] / total
            # the reference accumulates dpose sequentially (0 + x1 + x2 ...): cumsum does the same
            poses[a + 1:, j] = poses[a + 1:, j] + np.cumsum(inc[a + 1:])
    return poses


def optimise(poses, loops, steps):
    """scripts/main.py:325-326: `steps` SGD passes with learning rate 1/(k+1)."""
    poses = np.array(poses, dtype=np.float64)
    for k in range(steps):
        sgd_step(poses, loops, learning_rate=1.0 / (k + 1))
    return poses


def ate(a, b):
    """Absolute trajectory error: RMS of the position differences [m]."""
    d = np.asarray(a)[:, :2] - np.asarray(b)[:, :2]
    return float(np.sqrt(np.mean(np.sum(d * d, axis=1))))


def tangent_headings(poses):
    """src/pose_graph_optimization.py:52-57: heading of the interior poses from the path tangent."""
    poses = np.array(poses, dtype=np.float64)
    for i in range(1, len(poses) - 1):
        v = poses[i + 1][0:2] - poses[i][0:2]
        nv = np.linalg.norm(v)
        if nv > 0:
            v = v / nv
            poses[i][2] = np.arctan2(v[1], v[0])
    return poses


def proximity_candidates_ref(poses, min_dist_along_path=2, max_dist=1):
    """src/loop_closure_detection.py:12-25 restated with numpy rows instead of the cdist matrix;
    returns (i, j) rows in the reference's processing order (after its matches.reverse())."""
    xy = np.asarray(poses, dtype=np.float64)[:, :2]
    n = len(xy)
    step = np.sqrt((xy[1:, 0] - xy[:-1, 0]) ** 2 + (xy[1:, 1] - xy[:-1, 1]) ** 2)
    travelled = np.concatenate(([0.0], np.cumsum(step)))
    out = []
    for i in range(n):
        j0 = int(np.searchsorted(travelled, travelled[i] + min_dist_along_path, side="right"))
        if j0 >= n:
            break
        d = np.sqrt((xy[j0:, 0] - xy[i, 0]) ** 2 + (xy[j0:, 1] - xy[i, 1]) ** 2)
        j = j0 + int(np.argmin(d))
        if d[j - j0] <= max_dist:
            out.append((i, j))
    out.reverse()
    return np.asarray(out, dtype=np.int64).reshape(-1, 2)


def proximity_pairs_ref(poses, min_dist_along_path=2, max_dist=1):
    """Every pair the rows of src/loop_closure_detection.py:12-25 consider, kept if within max_dist:
    (source = j, target = i) int32 rows ordered by i then j, with cdist's rounding
    sqrt((dx*dx) + (dy*dy)) -- np.hypot rounds differently in about one entry in six."""
    xy = np.asarray(poses, dtype=np.float64)[:, :2]
    n = len(xy)
    step = np.sqrt((xy[1:, 0] - xy[:-1, 0]) ** 2 + (xy[1:, 1] - xy[:-1, 1]) ** 2)
    travelled = np.concatenate(([0.0], np.cumsum(step)))
    out = []
    for i in range(n):
        j0 = int(np.searchsorted(travelled, travelled[i] + min_dist_along_path, side="right"))
        if j0 >= n:
            break
        dx, dy = xy[j0:, 0] - xy[i, 0], xy[j0:, 1] - xy[i, 1]
        js = j0 + np.nonzero(np.sqrt(dx * dx + dy * dy) <= max_dist)[0]
        out.append(np.stack((js, np.full_like(js, i)), axis=1))
    return np.concatenate(out).astype(np.int32) if out else np.zeros((0, 2), np.int32)
