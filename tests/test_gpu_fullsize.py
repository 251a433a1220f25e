"""Parity at BASELINE.json's full sizes, through size-independent properties (the oracle takes
~15 ms per 1,024-point pair per core, so it checks a seeded subsample; everything else is checked
on every pair)."""
import numpy as np
import pytest

from conftest import pose_diff

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def chain5000():
    from icp_slam_b200 import synth
    return synth.make_chain_workload(5000, 1024, seed=467002, drop_frac=0.03)


def test_config2_full_chain(chain5000):
    """configs[1]: 5,000-scan odometry chain, 1,024 beams, 4,999 pairs in one launch."""
    from icp_slam_b200 import icp as gicp, synth
    from oracle import c_oracle
    scans, pairs, init, poses, odo = chain5000
    e = gicp.IcpEngine()
    table = e.set_scans(scans)
    a = e.run(pairs, init, epsilon=0.05, max_iters=100)
    # (1) idempotence / determinism: a second launch returns the same bits
    b = e.run(pairs, init, epsilon=0.05, max_iters=100)
    np.testing.assert_array_equal(a.T, b.T)
    np.testing.assert_array_equal(a.error, b.error)
    # (2) the exact pruning changes nothing: exhaustive sweep, bit for bit
    c = e.run(pairs, init, epsilon=0.05, max_iters=100, exhaustive=True)
    np.testing.assert_array_equal(a.T, c.T)
    np.testing.assert_array_equal(a.error, c.error)
    np.testing.assert_array_equal(a.iters, c.iters)
    # (3) the pipelined upload+align entry point agrees
    d = e.align(table, pairs, init, epsilon=0.05, max_iters=100)
    np.testing.assert_array_equal(a.T, d.T)
    # (4) structural invariants of the reference on every pair
    assert a.iters.min() >= 1 and a.iters.max() <= 102
    R = a.T[:, :2, :2]
    np.testing.assert_allclose(R @ np.transpose(R, (0, 2, 1)), np.broadcast_to(np.eye(2), R.shape), atol=1e-12)
    np.testing.assert_allclose(np.linalg.det(R), 1.0, atol=1e-12)
    assert np.all(a.T[:, 2] == [0.0, 0.0, 1.0])
    assert np.isfinite(a.error).all() and (a.error >= 0).all()
    # (5) the oracle on a seeded subsample
    sel = np.sort(np.random.default_rng(1).choice(len(pairs), 96, replace=False))
    xy, off = c_oracle.pack(scans)
    T, err, passes = c_oracle.icp_batch(xy, off, pairs[sel], init[sel], epsilon=0.05, max_iters=100)
    np.testing.assert_array_equal(a.iters[sel], passes)
    dt, dth = pose_diff(a.T[sel], T)
    assert dt < 1e-9 and dth < 1e-9
    np.testing.assert_allclose(a.error[sel], err, rtol=1e-9)
    # (6) sanity: the composed trajectory stays near the ground truth (point-to-point ICP on 5 mm
    #     range noise drifts a few mm per step, in the reference as here)
    est = np.zeros((len(scans), 3))
    for i in range(1, len(scans)):
        est[i] = synth.mat_to_pose(synth.pose_to_mat(est[i - 1]) @ a.T[i - 1])
    c0, s0 = np.cos(-poses[0, 2]), np.sin(-poses[0, 2])
    d0 = poses[:, :2] - poses[0, :2]
    truth = np.stack((c0 * d0[:, 0] - s0 * d0[:, 1], s0 * d0[:, 0] + c0 * d0[:, 1]), axis=1)
    assert np.abs(est[:200, :2] - truth[:200]).max() < 0.5
    e.close()


def test_config4_all_pairs_sharded_decode():
    """configs[3] in miniature: all pairs i<j decoded on the device, two interleaved shards; every
    shard's records land where the explicit pair list puts them."""
    from icp_slam_b200 import icp as gicp, synth, dist as d
    rng = np.random.default_rng(5)
    poses = synth.loop_trajectory(64, step=2.5)
    scans = synth.scans_from_poses(poses, 1024, rng, drop_frac=0.03)
    n = len(scans)
    B = synth.all_pairs_count(n)
    e = gicp.IcpEngine()
    e.set_scans(scans)
    ij = synth.all_pairs_decode(np.arange(B), n)
    ref = e.run(np.stack((ij[:, 1], ij[:, 0]), axis=1).astype(np.int32), None, epsilon=0.05, max_iters=100)
    got = np.empty((B, d.RECORD_WIDTH))
    for rank in range(2):
        shard = d.shard_all_pairs(B, rank, 2, block=128)
        r = e.run(None, None, epsilon=0.05, max_iters=100, all_pairs=shard)
        got[d.shard_indices(B, rank, 2, block=128)] = d.pack_records(r.T, r.error, r.iters)
    T, err, passes = d.unpack_records(got)
    np.testing.assert_array_equal(T, ref.T)
    np.testing.assert_array_equal(err, ref.error)
    np.testing.assert_array_equal(passes, ref.iters)
    assert passes.max() == 102                                   # non-overlapping pairs hit the cap
    e.close()


def test_config5_highres_multistart():
    """configs[4]: 4,096-point scans, K initial headings per pair = K independent icp() calls."""
    from icp_slam_b200 import icp as gicp, synth
    from oracle import c_oracle
    rng = np.random.default_rng(6)
    poses = synth.loop_trajectory(3, step=0.05)
    scans = synth.scans_from_poses(poses, 4096, rng, drop_frac=0.02)
    K = 8
    th = -np.pi + 2 * np.pi * np.arange(K) / K
    pairs = np.array([(1, 0)] * K + [(2, 1)] * K, dtype=np.int32)
    init = np.stack([synth.pose_to_mat((0.0, 0.0, t)) for t in np.tile(th, 2)])
    res = gicp.icp_batch(scans, pairs, init, epsilon=0.05, max_iters=100)
    xy, off = c_oracle.pack(scans)
    T, err, passes = c_oracle.icp_batch(xy, off, pairs, init, epsilon=0.05, max_iters=100)
    np.testing.assert_array_equal(res.iters, passes)
    dt, dth = pose_diff(res.T, T)
    assert dt < 1e-9 and dth < 1e-9
    np.testing.assert_allclose(res.error, err, rtol=1e-9)
    best = int(np.argmin(res.error[:K]))
    assert abs(th[best]) < 1.0                                   # the sweep finds the small-motion basin


def test_bench_dump_outputs_device_arm(tmp_path):
    """`bench.py --dump-outputs DIR` on the device: the last timed step's transforms, errors and pass
    counts for every pair of the seeded chain, as the C oracle computes them."""
    import argparse
    import os
    import subprocess
    import sys
    from oracle import c_oracle
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                          "--scans", "120", "--beams", "360", "--no-cpu", "--no-e2e", "--no-sustained",
                          "--no-exhaustive", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    z = {n: np.load(tmp_path / f"{n}.npy") for n in ("T", "error", "passes", "rows")}
    assert all(a.dtype == np.float64 for a in z.values())
    assert z["T"].shape == (119, 6) and z["rows"].tolist() == list(range(119))
    args = argparse.Namespace(workload="chain", scans=120, beams=360, strong=False, pairs=0)
    scans, pairs, init = bench.workload(args, 0, 1)
    xy, off = c_oracle.pack(scans)
    T, err, passes = c_oracle.icp_batch(xy, off, pairs, init, epsilon=bench.EPS, max_iters=bench.MAX_ITERS)
    np.testing.assert_array_equal(z["passes"], passes)
    dt, dth = pose_diff(c_oracle.to33(z["T"]), T)
    assert dt < 1e-9 and dth < 1e-9
    np.testing.assert_allclose(z["error"], err, rtol=1e-9)


def test_parity_campaign_reduced():
    """tools/parity_campaign.py at 4 % of its size (chains, rotation-only, all pairs, ragged clouds
    incl. tie-laden lattices and far-from-origin coordinates): no pass-count mismatch, no differing
    correspondence vector, |dT| < 1e-9; a disagreeing pair is excused only when the numpy oracle
    proves a single-target pass.  The full run (25,172 pairs) is profiles/r01l_parity_campaign.json."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "parity_campaign.py"), "--scale", "0.04",
                          "--corr-sample", "60"], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, (out.stdout[-3000:], out.stderr[-2000:])
    last = json.loads(out.stdout.strip().splitlines()[-1])
    assert last["all_within_contract"] and last["pairs_total"] > 400
