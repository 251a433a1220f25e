"""Host helpers of the multi-start alignment (no GPU needed): ``compose_starts`` evaluates the formula
of include/icpb.h bit for bit, and ``heading_starts`` gives bench.py's highres guesses."""
import argparse
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rigid(rng, n, shift=5.0):
    from icp_slam_b200 import synth
    poses = np.c_[rng.uniform(-shift, shift, size=(n, 2)), rng.uniform(-np.pi, np.pi, size=n)]
    return np.stack([synth.pose_to_mat(p) for p in poses])


def test_compose_starts_is_the_header_formula_bit_for_bit():
    from icp_slam_b200 import icp as gicp
    rng = np.random.default_rng(5)
    init = rng.normal(size=(7, 3, 3)) * [[1, 1, 100], [1, 1, 100], [0, 0, 0]]
    init[:, 2] = (0.0, 0.0, 1.0)
    S = rng.normal(size=(5, 3, 3)) * [[1, 1, 10], [1, 1, 10], [0, 0, 0]]
    S[:, 2] = (0.0, 0.0, 1.0)
    G = gicp.compose_starts(init, S)
    assert G.shape == (7, 5, 3, 3) and G.dtype == np.float64
    for p in range(7):
        I = init[p]
        for k in range(5):
            s = S[k]
            for r in range(2):
                # one Python float operation at a time: each product and sum rounded, left to right
                want = (I[r, 0] * s[0, 0] + I[r, 1] * s[1, 0],
                        I[r, 0] * s[0, 1] + I[r, 1] * s[1, 1],
                        (I[r, 0] * s[0, 2] + I[r, 1] * s[1, 2]) + I[r, 2])
                assert tuple(G[p, k, r].tolist()) == want
            assert G[p, k, 2].tolist() == [0.0, 0.0, 1.0]


def test_compose_starts_is_the_matrix_product():
    from icp_slam_b200 import icp as gicp
    rng = np.random.default_rng(6)
    init, S = _rigid(rng, 50), _rigid(rng, 16, shift=1.0)
    G = gicp.compose_starts(init, S)
    want = init[:, None] @ S[None]
    np.testing.assert_allclose(G, want, rtol=1e-15, atol=1e-15 * np.abs(want).max())
    # no init: the identity guess, so G is the starts themselves
    np.testing.assert_array_equal(gicp.compose_starts(None, S), S[None])


def test_compose_starts_rejects_bad_shapes():
    from icp_slam_b200 import icp as gicp
    with pytest.raises(ValueError):
        gicp.compose_starts(np.eye(3)[None], np.eye(3))
    with pytest.raises(ValueError):
        gicp.compose_starts(np.eye(3), np.eye(3)[None])


def test_heading_starts_are_the_highres_guesses():
    from icp_slam_b200 import icp as gicp
    sys.path.insert(0, ROOT)
    import bench
    args = argparse.Namespace(workload="highres", scans=4, beams=64, strong=False, pairs=0)
    _, pairs, init = bench.workload(args, 0, 1)
    S = gicp.heading_starts(32)
    assert S.shape == (32, 3, 3)
    np.testing.assert_array_equal(init, np.tile(S, (3, 1, 1)))
    np.testing.assert_array_equal(pairs[::32], [(1, 0), (2, 1), (3, 2)])
    th = np.arctan2(S[:, 1, 0], S[:, 0, 0])
    np.testing.assert_allclose(th, -np.pi + 2 * np.pi * np.arange(32) / 32, atol=1e-15)
    with pytest.raises(ValueError):
        gicp.heading_starts(0)
