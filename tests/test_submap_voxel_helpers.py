"""Host side of the submap voxel filter (no GPU needed): ``merge_scans(..., voxel=)`` keeps the first merged
point of every cell floor(x / voxel), in merged order, per submap; the voxel is checked; the library's new
exports are declared."""
import numpy as np
import pytest


def _id(k=1):
    return np.stack([np.eye(3)] * k)


def test_first_point_of_every_cell_in_merged_order():
    from icp_slam_b200 import icp as gicp
    # cells of v = 1: (0,0) (1,0) (0,0) (2,3) (1,0) (0,0) | second scan: (2,3) (5,5) (1,0)
    a = np.array([[0.5, 0.5], [1.2, 0.1], [0.9, 0.9], [2.5, 3.5], [1.9, 0.8], [0.1, 0.2]])
    b = np.array([[2.1, 3.9], [5.0, 5.0], [1.0, 0.0]])
    out = gicp.merge_scans([a, b], [np.array([0, 1]), np.array([1, 0])], [_id(2), _id(2)], voxel=1.0)
    np.testing.assert_array_equal(out[0], np.array([a[0], a[1], a[3], b[1]]))
    np.testing.assert_array_equal(out[1], np.array([b[0], b[1], b[2], a[0]]))    # cells are per submap


def test_points_on_cell_edges_of_both_signs():
    from icp_slam_b200 import icp as gicp
    v = 0.25
    # x = 0.5 opens cell 2; 0.4999 is cell 1; -0.25 is cell -1 (not 0); -0.0 is cell 0 like +0.0
    p = np.array([[0.5, 0.0], [0.4999, 0.0], [0.75 - 1e-17, 0.0], [-0.25, 0.0], [-0.2500001, 0.0],
                  [-0.0, 0.0], [0.0, -0.0], [0.0, -1e-300], [0.2499999, 0.25]])
    merged = gicp.merge_scans([p], [np.array([0])], [_id()])[0]
    got = gicp.merge_scans([p], [np.array([0])], [_id()], voxel=v)[0]
    # 0.75 - 1e-17 is 0.75 in float64: cell 3; -1e-300 / v floors to cell -1
    cx = np.floor(merged[:, 0] / v).astype(np.int64)
    cy = np.floor(merged[:, 1] / v).astype(np.int64)
    assert cx.tolist() == [2, 1, 3, -1, -2, 0, 0, 0, 0]
    assert cy.tolist() == [0, 0, 0, 0, 0, 0, 0, -1, 1]
    keep = [0, 1, 2, 3, 4, 5, 7, 8]                           # row 6 repeats row 5's cell (0, 0)
    assert got.tobytes() == merged[keep].tobytes()           # kept points keep their bits


def test_a_repeated_member_vanishes():
    from icp_slam_b200 import icp as gicp
    rng = np.random.default_rng(5)
    s = rng.uniform(-20, 20, size=(300, 2))
    T = np.array([[0.8, -0.6, 1.5], [0.6, 0.8, -2.0], [0.0, 0.0, 1.0]])
    once = gicp.merge_scans([s], [np.array([0])], [T[None]], voxel=0.05)[0]
    twice = gicp.merge_scans([s], [np.array([0, 0])], [np.stack([T, T])], voxel=0.05)[0]
    np.testing.assert_array_equal(twice, once)


def test_one_cell_holding_everything_leaves_one_point_per_submap():
    from icp_slam_b200 import icp as gicp
    rng = np.random.default_rng(6)
    scans = [rng.uniform(0.0, 0.99, size=(50, 2)), rng.uniform(0.0, 0.99, size=(20, 2))]
    out = gicp.merge_scans(scans, [np.array([0, 1]), np.array([1]), np.array([1, 0])], [_id(2), _id(1), _id(2)],
                           voxel=1.0)
    for sub, first in zip(out, (scans[0][0], scans[1][0], scans[1][0])):
        np.testing.assert_array_equal(sub, first[None])


def test_no_voxel_is_the_unfiltered_merge():
    from icp_slam_b200 import icp as gicp
    rng = np.random.default_rng(7)
    scans = [rng.normal(size=(40, 2)), rng.normal(size=(9, 2))]
    mem, T = [np.array([0, 1, 0])], [_id(3)]
    ref = gicp.merge_scans(scans, mem, T)
    for v in (None, 0, 0.0):
        np.testing.assert_array_equal(gicp.merge_scans(scans, mem, T, voxel=v)[0], ref[0])


def test_packed_key_and_row_unique_agree():
    """Cells too far apart for one int64 key go through the row-wise unique; both keep the same points."""
    from icp_slam_b200 import icp as gicp
    rng = np.random.default_rng(8)
    near = rng.uniform(-1, 1, size=(500, 2))
    far = np.concatenate([near, [[9e9, -9e9], [-9e9, 9e9], [9e9, -9e9]]])
    for p, v in ((near, 0.1), (far, 1e-6), (far, 0.1)):
        c = np.floor(p / v).astype(np.int64)
        _, first = np.unique(c, axis=0, return_index=True)
        np.testing.assert_array_equal(gicp._first_of_cell(p, v), np.sort(first))


@pytest.mark.parametrize("voxel", [np.nan, np.inf, -np.inf, -0.1, 9.9e-7, 1e-300, "x"])
def test_bad_voxels_are_rejected(voxel):
    from icp_slam_b200 import icp as gicp
    with pytest.raises(ValueError):
        gicp.merge_scans([np.zeros((3, 2))], [np.array([0])], [_id()], voxel=voxel)


def test_smallest_voxel_is_accepted_and_far_points_are_rejected():
    from icp_slam_b200 import icp as gicp
    p = np.array([[1e10, -1e10], [-1e10, 1e10], [1e10, -1e10]])
    got = gicp.merge_scans([p], [np.array([0])], [_id()], voxel=gicp.MIN_VOXEL)[0]
    np.testing.assert_array_equal(got, p[:2])
    shift = np.eye(3)[None].copy()
    shift[0, 0, 2] = 1.0
    with pytest.raises(ValueError):                          # 1e10 + 1 has no cell within the bounds
        gicp.merge_scans([p], [np.array([0])], [shift], voxel=1.0)


def test_new_exports_are_declared():
    import ctypes
    from icp_slam_b200 import _lib
    restype, args = _lib.SIGNATURES["icpb_set_submaps_voxel"]
    assert restype is ctypes.c_int
    assert args == [ctypes.c_void_p] * 4 + [ctypes.c_int64, ctypes.c_double, ctypes.c_void_p]
    restype, args = _lib.SIGNATURES["icpb_read_scans"]
    assert restype is ctypes.c_int
    assert args == [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p]
    assert {"icpb_set_submaps_voxel", "icpb_read_scans"} <= set(_lib.EXPORTS)


def test_caller_rejects_a_voxel_without_a_window():
    from icp_slam_b200 import callers
    with pytest.raises(ValueError):
        callers.proximity_loop_closures(np.zeros((3, 3)), [np.zeros((2, 2))] * 3, submap_voxel=0.05)
