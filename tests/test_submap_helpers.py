"""Host helpers of the submaps (no GPU needed): ``merge_scans`` evaluates the formula of include/icpb.h bit
for bit, its arguments are checked before anything else, and the proximity caller's submaps have the right
members and transforms at both ends of the trajectory."""
import numpy as np
import pytest


def _scans(rng, lengths):
    return [rng.normal(size=(m, 2)) * 10.0 for m in lengths]


def _affine(rng, k):
    T = rng.normal(size=(k, 3, 3)) * [[1, 1, 100], [1, 1, 100], [0, 0, 0]]
    T[:, 2] = (0.0, 0.0, 1.0)
    return T


def test_merge_scans_is_the_header_formula_bit_for_bit():
    from icp_slam_b200 import icp as gicp
    rng = np.random.default_rng(11)
    scans = _scans(rng, [5, 1, 9, 3])
    members = [np.array([2, 0, 2]), np.array([1]), np.array([3, 1, 0, 2])]
    transforms = [_affine(rng, len(m)) for m in members]
    got = gicp.merge_scans(scans, members, transforms)
    assert len(got) == 3
    for mem, T, sub in zip(members, transforms, got):
        assert sub.dtype == np.float64 and sub.shape == (sum(len(scans[s]) for s in mem), 2)
        want = []
        for s, t in zip(mem, T):
            for x, y in scans[s].tolist():
                # one Python float operation at a time: each product and sum rounded on its own
                want.append([(t[0, 0] * x + t[0, 1] * y) + t[0, 2], (t[1, 0] * x + t[1, 1] * y) + t[1, 2]])
        assert sub.tolist() == want
    # the same from a packed table
    table = gicp.ScanTable(scans)
    for a, b in zip(gicp.merge_scans(table, members, transforms), got):
        np.testing.assert_array_equal(a, b)


def test_merge_scans_identity_reproduces_the_scan():
    from icp_slam_b200 import icp as gicp
    rng = np.random.default_rng(12)
    scans = _scans(rng, [7, 4])
    out = gicp.merge_scans(scans, [np.array([1]), np.array([0, 1])], [np.eye(3)[None], np.stack([np.eye(3)] * 2)])
    np.testing.assert_array_equal(out[0], scans[1])
    np.testing.assert_array_equal(out[1], np.concatenate(scans))


def test_submap_arguments_are_checked():
    from icp_slam_b200 import icp as gicp
    rng = np.random.default_rng(13)
    scans = _scans(rng, [3, 3, 3])
    I1 = np.eye(3)[None]
    shear = I1.copy()
    shear[0, 2, 0] = 0.5
    wide = I1.copy()
    wide[0, 0, 0] = 2e3
    far = I1.copy()
    far[0, 1, 2] = 2e12
    nan = I1.copy()
    nan[0, 0, 1] = np.nan
    bad = {
        "lists of different lengths": ([np.array([0])], []),
        "no member": ([np.array([], dtype=np.int64)], [np.zeros((0, 3, 3))]),
        "2-D members": ([np.array([[0]])], [I1]),
        "float ids": ([np.array([0.0])], [I1]),
        "id past the table": ([np.array([3])], [I1]),
        "negative id": ([np.array([-1])], [I1]),
        "one transform short": ([np.array([0, 1])], [I1]),
        "bottom row": ([np.array([0])], [shear]),
        "linear bound": ([np.array([0])], [wide]),
        "shift bound": ([np.array([0])], [far]),
        "non-finite": ([np.array([0])], [nan]),
    }
    for name, (members, transforms) in bad.items():
        with pytest.raises(ValueError):
            gicp.merge_scans(scans, members, transforms)
            pytest.fail(name)


def test_window_members_at_both_ends():
    from icp_slam_b200 import callers
    n = 20
    got = callers.submap_window_members(n, [0, 2, 10, 18, 19], 3)
    want = [range(0, 4), range(0, 6), range(7, 14), range(15, 20), range(16, 20)]
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g, list(w))
    for g, i in zip(callers.submap_window_members(n, [0, 7, 19], 0), [0, 7, 19]):
        np.testing.assert_array_equal(g, [i])


def test_window_transforms_place_members_in_the_target_frame():
    from icp_slam_b200 import callers, synth
    poses = synth.loop_trajectory(12, step=0.3)
    targets = [0, 5, 11]
    members = callers.submap_window_members(len(poses), targets, 2)
    Ts = callers.submap_window_transforms(poses, targets, members)
    for i, mem, T in zip(targets, members, Ts):
        assert T.shape == (len(mem), 3, 3)
        for s, t in zip(mem, T):
            if s == i:
                np.testing.assert_array_equal(t, np.eye(3))        # exact: the target scan keeps its bits
            else:
                want = np.linalg.inv(synth.pose_to_mat(poses[i])) @ synth.pose_to_mat(poses[s])
                np.testing.assert_allclose(t, want, rtol=0, atol=1e-12)
                assert t[2].tolist() == [0.0, 0.0, 1.0]
                # a point of scan s lands where it is in the world, seen from pose i
                p = np.array([1.5, -0.5, 1.0])
                world = synth.pose_to_mat(poses[s]) @ p
                np.testing.assert_allclose(synth.pose_to_mat(poses[i]) @ (t @ p), world, atol=1e-12)
