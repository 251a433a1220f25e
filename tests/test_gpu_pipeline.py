"""End to end through the batched call sites (icp_slam_b200.callers) on the GPU, against the golden
of the unmodified reference pipeline: corrected poses, loop closures, and the optimised trajectory
(BASELINE.json: within 1e-4 m ATE)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu


def load():
    z = np.load(os.path.join(GOLDEN, "slam_golden.npz"))
    off = np.concatenate(([0], np.cumsum(z["scan_lengths"])))
    scans = [z["scan_xy"][off[k]:off[k + 1]] for k in range(len(off) - 1)]
    return z, scans


def test_pipeline_matches_reference_golden():
    from icp_slam_b200 import callers
    from oracle import slam_oracle
    z, scans = load()
    # scan matching: scripts/main.py:239-256
    corrected, res = callers.odometry_chain(scans, z["odometry"], max_iters=100, epsilon=0.05)
    np.testing.assert_array_equal(res.iters, z["chain_passes"])
    np.testing.assert_allclose(res.T, z["chain_T"], atol=1e-9)
    np.testing.assert_allclose(corrected, z["corrected"], atol=1e-8)
    # loop closure: src/loop_closure_detection.py:11-39
    loops, _ = callers.proximity_loop_closures(z["corrected"], scans)
    loops = slam_oracle.graph_order(loops)
    assert [(a, b) for a, b, _ in loops] == [tuple(r) for r in z["loop_ij"].tolist()]
    np.testing.assert_allclose(np.stack([t for _, _, t in loops]), z["loop_T"], atol=1e-9)
    # optimisation on the GPU-produced constraints: trajectory within 1e-4 m ATE of the reference's
    opt = slam_oracle.optimise(corrected, loops, 5)
    ate = slam_oracle.ate(opt, z["optimised"])
    assert ate < 1e-4, ate
    assert ate < 1e-7, ate                                  # what the kernel actually achieves
    # rotation-only refinement: src/pose_graph_optimization.py:51-74
    start = slam_oracle.tangent_headings(z["optimised"])
    re, _ = callers.rotation_only_headings(start, scans, max_iters=100, epsilon=0.05)
    np.testing.assert_allclose(re, z["reoriented"], atol=1e-8)


def test_image_match_call_site():
    """src/loop_closure_detection.py:134-159: source = scan i*rate, target = scan j*rate, identity
    initial guess, accepted when error < icp_err_thresh."""
    from icp_slam_b200 import callers
    from oracle import c_oracle
    z, scans = load()
    good = [(3, 1), (10, 12), (20, 49), (7, 7)]
    rate = 3
    out, res = callers.image_match_loop_closures(good, scans, image_rate=rate, icp_err_thresh=30)
    xy, off = c_oracle.pack(scans)
    pairs = np.array([(i * rate, j * rate) for i, j in good], dtype=np.int32)
    T, err, passes = c_oracle.icp_batch(xy, off, pairs, None, epsilon=0.05, max_iters=100)
    ok = err < 30                                            # the filter runs on the device: accepted pairs only
    np.testing.assert_array_equal(res.iters, passes[ok])
    np.testing.assert_allclose(res.T, T[ok], atol=1e-9)
    np.testing.assert_allclose(res.error, err[ok], rtol=1e-9)
    keep = [(int(p[0]), int(p[1])) for p, e in zip(pairs, err) if e < 30]
    assert [(a, b) for a, b, _ in out] == keep and (21, 21) in keep
    # a threshold nothing passes, and one everything passes
    none, r0 = callers.image_match_loop_closures(good, scans, image_rate=rate, icp_err_thresh=0.0)
    assert none == [] and len(r0) == 0
    every, r1 = callers.image_match_loop_closures(good, scans, image_rate=rate, icp_err_thresh=1e300)
    assert len(every) == len(good)
    np.testing.assert_allclose(r1.T, T, atol=1e-9)


def test_candidate_generation_on_gpu():
    """icpb_proximity_closest / icpb_proximity_pairs against the numpy restatement of
    src/loop_closure_detection.py:12-25 and against its every-pair form (slam_oracle.proximity_pairs_ref,
    cdist's rounding), on a 5,000-pose loop."""
    from icp_slam_b200 import callers, synth
    from oracle import slam_oracle
    z, _ = load()
    np.testing.assert_array_equal(callers.proximity_candidates(z["corrected"]),
                                  slam_oracle.proximity_candidates_ref(z["corrected"]))
    poses = synth.loop_trajectory(5000, step=0.04)
    for kw in (dict(), dict(min_dist_along_path=5.0, max_dist=0.4), dict(min_dist_along_path=0.0, max_dist=0.1),
               dict(min_dist_along_path=1e9)):
        np.testing.assert_array_equal(callers.proximity_candidates(poses, **kw),
                                      slam_oracle.proximity_candidates_ref(poses, **kw))
    got = callers.proximity_pairs(poses)
    want = slam_oracle.proximity_pairs_ref(poses)
    np.testing.assert_array_equal(got, want)
    assert len(got) > 100000


def test_detect_proximity_drop_in_adds_the_reference_constraints():
    """icp_slam_b200.loop_closure_detection.detect_proximity(pose_graph, lidar_points): same
    signature and side effect as src/loop_closure_detection.py:11-39."""
    from icp_slam_b200 import loop_closure_detection as lcd
    z, scans = load()

    class Graph:
        def __init__(self, poses):
            self.poses, self.added = poses, []

        def add_constraint(self, i, j, tf):
            self.added.append((i, j, tf))

    pg = Graph(z["corrected"].copy())
    out = lcd.detect_proximity(pg, scans)
    assert out == pg.added and len(pg.added) == len(z["loop_ij"])
    # the reference adds them in its greedy processing order; its graph then iterates by source node
    by_source = sorted(pg.added, key=lambda e: e[0])
    assert [(a, b) for a, b, _ in by_source] == [tuple(r) for r in z["loop_ij"].tolist()]
    np.testing.assert_allclose(np.stack([t for _, _, t in by_source]), z["loop_T"], atol=1e-9)
    np.testing.assert_array_equal(pg.poses, z["corrected"])           # poses untouched


def test_pipeline_tool_runs_end_to_end():
    """tools/slam_pipeline.py (scan matching -> loop closure -> SGD -> orientation -> map) on a
    small synthetic run: every stage executes on the GPU and the optimisation does not make the
    trajectory worse than scan matching alone by more than a few centimetres."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "slam_pipeline.py"), "--scans", "400",
                          "--beams", "360", "--sgd-steps", "5", "--cell", "0.1"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    r = json.loads(out.stdout.strip().splitlines()[-1])
    assert set(r["stage_ms"]) == {"scan_matching", "loop_closure", "optimisation", "orientation", "occupancy_grid"}
    assert r["chain_pairs"] == 399 and r["grid"][0] > 50 and r["grid"][1] > 50
    assert np.isfinite(r["ate_m"]["scan_matching"]) and np.isfinite(r["ate_m"]["optimised"])


def test_reference_fan_out_with_loky_workers(monkeypatch):
    """The reference's own fan-out, unchanged except for the import: joblib/loky worker processes
    unpickle ``icp.icp`` by its qualified name and each creates its CUDA handle on first use
    (scripts/main.py:240-247).  The results equal the one-launch ``icp_batch`` bit for bit."""
    from joblib import Parallel, delayed
    from icp_slam_b200 import icp, synth
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    monkeypatch.setenv("PYTHONPATH", root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    scans, pairs, init, _, _ = synth.make_chain_workload(13, 360, seed=467200)
    out = Parallel(n_jobs=2, backend="loky")(
        delayed(icp.icp)(np.c_[scans[i], np.ones(len(scans[i]))], np.c_[scans[j], np.ones(len(scans[j]))],
                         init_transform=init[k], max_iters=100, epsilon=0.05)
        for k, (i, j) in enumerate(pairs))
    res = icp.icp_batch(scans, pairs, init, max_iters=100, epsilon=0.05)
    assert len(out) == len(pairs)
    for k, (tfs, err) in enumerate(out):
        assert len(tfs) == res.iters[k] + 1
        np.testing.assert_array_equal(tfs[0], init[k])
        np.testing.assert_array_equal(tfs[-1], res.T[k])
        assert err == res.error[k]


def test_strided_scan_matching_loop():
    """callers.odometry_chain_strided = the serial loop of scripts/map_icp.py:44-86, including its
    quirk of composing the first step onto odometry[start - 1]; checked against that loop written
    out with the drop-in icp() and the reference's pose <-> matrix formulas (src/utils.py:28-39)."""
    from icp_slam_b200 import callers, icp, synth
    scans, _, _, _, odo = synth.make_chain_workload(60, 360, seed=467300)
    start, skip = 7, 5

    def pose_to_mat(p):
        c, s = np.cos(p[2]), np.sin(p[2])
        return np.array([[c, -s, p[0]], [s, c, p[1]], [0, 0, 1.0]])

    corrected = [odo[i] for i in range(start)]
    for i in range(start, len(odo), skip):
        est = pose_to_mat(odo[i] - odo[i - skip])
        tfs, _ = icp.icp(np.c_[scans[i], np.ones(len(scans[i]))], np.c_[scans[i - skip], np.ones(len(scans[i - skip]))],
                         init_transform=est, max_iters=100, epsilon=0.05)
        m = pose_to_mat(corrected[-1]) @ tfs[-1]
        corrected.append(np.array([m[0, 2], m[1, 2], np.arctan2(m[1, 0], m[0, 0])]))
    got, res = callers.odometry_chain_strided(scans, odo, start, skip)
    assert got.shape == (len(corrected), 3) and len(res) == len(corrected) - start
    np.testing.assert_allclose(got, np.array(corrected), rtol=0, atol=1e-12)
    with pytest.raises(ValueError):
        callers.odometry_chain_strided(scans, odo, 3, 5)


def test_chain_composition_on_the_device():
    """SURVEY 8f-2: the SE(2) prefix product as a parallel scan on the GPU against the reference's
    step-by-step loop (scripts/main.py:249-256): equal to rounding (1e-9 here; the trajectory contract is
    1e-4 m), for chains shorter and longer than the scan's 512 runs."""
    from icp_slam_b200 import callers, synth
    rng = np.random.default_rng(9)
    for n in (0, 1, 7, 511, 512, 513, 4999, 20000):
        T = np.stack([synth.pose_to_mat(p) for p in rng.normal(0, [0.05, 0.05, 0.02], size=(n, 3))]) if n else np.zeros((0, 3, 3))
        pose0 = np.array([1.5, -2.0, 0.3])
        want = callers.compose_chain(pose0, T)
        got = callers.compose_chain_gpu(pose0, T)
        assert got.shape == (n + 1, 3)
        np.testing.assert_allclose(got[:, :2], want[:, :2], rtol=0, atol=1e-9)
        d = np.abs(got[:, 2] - want[:, 2])
        assert np.all(np.minimum(d, 2 * np.pi - d) < 1e-9)
