"""Host-side rows around the ICP path against the end-to-end golden of the unmodified reference
pipeline (tests/golden/slam_golden.npz).  CPU only: ICP results come from the C oracle here."""
import os

import numpy as np

from conftest import GOLDEN
from oracle import c_oracle, slam_oracle


def load():
    z = np.load(os.path.join(GOLDEN, "slam_golden.npz"))
    off = np.concatenate(([0], np.cumsum(z["scan_lengths"])))
    scans = [z["scan_xy"][off[k]:off[k + 1]] for k in range(len(off) - 1)]
    return z, scans


def test_candidates_and_greedy_replay_match_detect_proximity():
    z, scans = load()
    cand = slam_oracle.proximity_candidates_ref(z["corrected"])
    assert len(cand) > len(z["loop_ij"])
    xy, off = c_oracle.pack(scans)
    pairs = np.stack((cand[:, 1], cand[:, 0]), axis=1).astype(np.int32)
    T, err, passes = c_oracle.icp_batch(xy, off, pairs, None, epsilon=0.05, max_iters=100)
    used, loops = set(), []
    for (i, j), Tk, e in zip(cand, T, err):
        if i in used or j in used or not e < 110:
            continue
        loops.append((int(i), int(j), Tk)); used.update((int(i), int(j)))
    loops = slam_oracle.graph_order(loops)
    assert [(a, b) for a, b, _ in loops] == [tuple(r) for r in z["loop_ij"].tolist()]
    np.testing.assert_allclose(np.stack([t for _, _, t in loops]), z["loop_T"], atol=1e-10)


def test_sgd_restatement_matches_reference():
    z, _ = load()
    loops = [(int(a), int(b), T) for (a, b), T in zip(z["loop_ij"], z["loop_T"])]
    out = slam_oracle.optimise(z["corrected"], loops, 5)
    np.testing.assert_allclose(out, z["optimised"], atol=1e-10)
    assert slam_oracle.ate(out, z["optimised"]) < 1e-10
    assert slam_oracle.ate(z["corrected"], z["optimised"]) > 1e-3      # the optimisation does move poses


def test_chain_composition_matches_reference():
    from icp_slam_b200 import synth
    z, scans = load()
    xy, off = c_oracle.pack(scans)
    n = len(scans)
    idx = np.arange(1, n)
    pairs = np.stack((idx, idx - 1), axis=1).astype(np.int32)
    init = np.stack([synth.pose_to_mat(z["odometry"][i] - z["odometry"][i - 1]) for i in idx])
    T, err, passes = c_oracle.icp_batch(xy, off, pairs, init, epsilon=0.05, max_iters=100)
    np.testing.assert_array_equal(passes, z["chain_passes"])
    np.testing.assert_allclose(T, z["chain_T"], atol=1e-11)
    poses = np.zeros((n, 3)); poses[0] = z["odometry"][0]
    for i in range(1, n):
        poses[i] = synth.mat_to_pose(synth.pose_to_mat(poses[i - 1]) @ T[i - 1])
    np.testing.assert_allclose(poses, z["corrected"], atol=1e-9)


def _detect_proximity_cdist(poses, min_dist_along_path=2, max_dist=1):
    """src/loop_closure_detection.py:12-25 written out with scipy's cdist, as the reference does:
    (candidates in its processing order, every pair within the radius as (j, i) rows)."""
    from scipy.spatial.distance import cdist
    positions = np.asarray(poses, dtype=np.float64)[:, :2]
    steps = np.sqrt((positions[1:, 0] - positions[:-1, 0]) ** 2 + (positions[1:, 1] - positions[:-1, 1]) ** 2)
    dist_traveled = np.concatenate(([0.0], np.cumsum(steps)))
    dists = cdist(positions, positions)
    matches, pairs = [], []
    for i in range(len(positions)):
        start = np.searchsorted(dist_traveled, dist_traveled[i] + min_dist_along_path, side="right")
        if start >= len(positions):
            break
        j = start + np.argmin(dists[i, start:])
        if dists[i, j] <= max_dist:
            matches.append((i, j))
        pairs += [(jj, i) for jj in range(start, len(positions)) if dists[i, jj] <= max_dist]
    matches.reverse()
    return (np.asarray(matches, dtype=np.int64).reshape(-1, 2), np.asarray(pairs, dtype=np.int32).reshape(-1, 2))


def boundary_poses(rng, n=300, scale=3.0):
    """A wandering path that stops (runs of identical poses: travelled has plateaus, distances tie)
    and revisits 3-4-5 offsets of earlier poses, so distances sit exactly on radius 5."""
    p = np.cumsum(rng.normal(0, scale / 10, (n, 2)), axis=0)
    p[40:60] = p[40]
    p[100:104] = p[3] + (3.0, 4.0)
    p[150] = p[3] + (-4.0, 3.0)
    p = np.round(p * 64) / 64                                 # exact binary fractions: exact ties
    return np.c_[p, rng.uniform(-np.pi, np.pi, n)]


def test_proximity_refs_equal_a_literal_cdist_implementation():
    from icp_slam_b200 import synth
    from oracle import slam_oracle
    rng = np.random.default_rng(8)
    cases = [(rng.normal(0, 3, (400, 3)), 2, 1), (boundary_poses(rng), 2, 5.0), (boundary_poses(rng), 0.0, 5.0),
             (boundary_poses(rng), -1.0, 0.0), (boundary_poses(rng), np.inf, 5.0), (boundary_poses(rng), 3, np.inf),
             (synth.loop_trajectory(600, step=0.05), 2, 1), (rng.normal(0, 3, (1, 3)), 0, 1)]
    for poses, mdp, md in cases:
        cand, pairs = _detect_proximity_cdist(poses, mdp, md)
        np.testing.assert_array_equal(slam_oracle.proximity_candidates_ref(poses, mdp, md), cand)
        np.testing.assert_array_equal(slam_oracle.proximity_pairs_ref(poses, mdp, md), pairs)
    # on the boundary family the radius is met exactly, and hypot would round some pairs differently
    poses = boundary_poses(np.random.default_rng(9))
    _, pairs = _detect_proximity_cdist(poses, 2, 5.0)
    d = np.sqrt(((poses[pairs[:, 0], :2] - poses[pairs[:, 1], :2]) ** 2).sum(1))
    assert (d == 5.0).sum() >= 5
