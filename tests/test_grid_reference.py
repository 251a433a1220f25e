"""The C restatement of the occupancy-grid update (oracle/grid_oracle.c) against goldens of the
unmodified reference (tests/golden/make_grid_golden.py): bit-exact int8 grids, bit-exact global
points and grid origin.  CPU only.  Also pins the per-cell closed form the GPU kernel relies on."""
import os
import warnings

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import c_oracle

CASES = ("default", "big_odds", "min_size")


def load():
    z = np.load(os.path.join(GOLDEN, "grid_golden.npz"))
    off = np.concatenate(([0], np.cumsum(z["scan_lengths"]))).astype(np.int64)
    return z, np.ascontiguousarray(z["scan_xy"]), off


def test_global_points_bit_exact():
    z, xy, off = load()
    np.testing.assert_array_equal(c_oracle.global_points(z["poses"], xy, off), z["global_xy"])


@pytest.mark.parametrize("name", CASES)
def test_produce_matches_reference(name):
    z, xy, off = load()
    cell, min_w, min_h, k_hit, k_miss = z[f"{name}/args"]
    grid, origin = c_oracle.produce_grid(z["poses"], xy, off, cell, min_w, min_h, int(k_hit), int(k_miss))
    np.testing.assert_array_equal(np.array(origin), z[f"{name}/origin"])
    assert grid.shape == z[f"{name}/grid"].shape
    np.testing.assert_array_equal(grid, z[f"{name}/grid"])


def test_update_matches_reference():
    z, xy, off = load()
    grid = z["default/grid"].copy()
    n = len(z["update/poses"])
    c_oracle.update_grid(grid, z["update/poses"], xy[:off[n]], off[:n + 1], 0.1, *z["default/origin"], 4, 2)
    np.testing.assert_array_equal(grid, z["update/grid"])


def test_per_cell_closed_form():
    """What a cell holds after any sequence of hits (H) and misses (M) depends only on its initial
    value, the two counts and the type of the LAST event -- the reference's int8 arithmetic
    (src/produce_occupancy_grid.py:109-112, :128-131) makes a miss on a positive cell -128 and a
    hit on a negative cell 127.  The GPU kernel accumulates exactly these per-cell summaries with
    commutative atomics; here the closed form is checked against a literal replay with numpy int8
    scalars, as the reference evaluates it."""
    def miss(g, k):
        return g - k if -128 - g < -k else np.int8(-128)

    def hit(g, k):
        return g + k if 127 - g > k else np.int8(127)

    def closed(g0, seq, k_hit, k_miss):
        n_h, n_m = seq.count("H"), seq.count("M")
        if not seq:
            return g0
        if seq[-1] == "H":
            return 127 if (n_m > 0 or g0 < 0) else min(g0 + n_h * k_hit, 127)
        return -128 if (n_h > 0 or g0 > 0) else max(g0 - n_m * k_miss, -128)

    rng = np.random.default_rng(3)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")                     # the int8 overflow is the point
        for _ in range(4000):
            k_hit, k_miss = int(rng.choice([1, 2, 3, 5, 40, 127])), int(rng.choice([1, 2, 3, 7, 100, 127]))
            g0 = int(rng.choice([0, 0, -128, 127, -1, 1, rng.integers(-128, 128)]))
            n = int(rng.integers(0, 12))
            seq = list(rng.choice(["H", "M"], n)) if rng.random() > 0.3 else [str(rng.choice(["H", "M"]))] * n
            g = np.int8(g0)
            for t in seq:
                g = hit(g, k_hit) if t == "H" else miss(g, k_miss)
            assert int(g) == closed(g0, seq, k_hit, k_miss), (g0, seq, k_hit, k_miss)


# ---- the exact restatement (oracle/grid_exact.py): Python ints, no int64 to overflow ----------------

@pytest.mark.parametrize("name", CASES)
def test_exact_restatement_matches_reference(name):
    from oracle import grid_exact
    z, xy, off = load()
    cell, min_w, min_h, k_hit, k_miss = z[f"{name}/args"]
    grid, origin = grid_exact.produce_grid(z["poses"], xy, off, cell, min_w, min_h, int(k_hit), int(k_miss))
    np.testing.assert_array_equal(np.array(origin), z[f"{name}/origin"])
    np.testing.assert_array_equal(grid, z[f"{name}/grid"])


def test_exact_restatement_update_matches_reference_and_c_oracle():
    from oracle import grid_exact
    z, xy, off = load()
    n = len(z["update/poses"])
    grid = z["default/grid"].copy()
    grid_exact.update_grid(grid, z["update/poses"], xy[:off[n]], off[:n + 1], 0.1, *z["default/origin"], 4, 2)
    np.testing.assert_array_equal(grid, z["update/grid"])
    # random poses around a small pre-filled grid, beams in and out of it, every odds corner
    rng = np.random.default_rng(11)
    for k_hit, k_miss in ((1, 1), (3, 1), (1, 127), (127, 127)):
        poses = np.c_[rng.uniform(-1, 4, (12, 2)), rng.uniform(-np.pi, np.pi, 12)]
        scans = [rng.uniform(-3, 3, (int(rng.integers(1, 70)), 2)) for _ in range(12)]
        sxy, soff = c_oracle.pack(scans)
        g0 = rng.integers(-128, 128, (23, 31)).astype(np.int8)
        g0.flat[:5] = (-128, -1, 0, 1, 127)
        want, got = g0.copy(), g0.copy()
        c_oracle.update_grid(want, poses, sxy, soff, 0.125, -0.5, -0.25, k_hit, k_miss)
        grid_exact.update_grid(got, poses, sxy, soff, 0.125, -0.5, -0.25, k_hit, k_miss)
        np.testing.assert_array_equal(got, want)
        assert (got != g0).sum() > 50


def test_exact_restatement_raises_where_the_reference_raises():
    from oracle import grid_exact
    with pytest.raises(ValueError):
        grid_exact.cell(float("nan"), 0.0, 0.1)
    with pytest.raises(OverflowError):
        grid_exact.cell(0.0, float("-inf"), 0.1)
    assert grid_exact.cell(-1e-300, 0.0, 0.5) == -1 and grid_exact.cell(0.5, 0.0, 0.25) == 2


def _walk_ends(R):
    """Every walk from (0, 0) to an end offset with |dx|, |dy| <= R, vectorised over the offsets:
    the loop of oracle/grid_oracle.c:43-50 without the grid test.  Returns (x1, y1, x_stop, y_stop,
    largest |2 * error| seen per walk, whether each walk stayed in its end cells' bounding box)."""
    x1, y1 = (a.ravel().astype(np.int64) for a in np.meshgrid(np.arange(-R, R + 1), np.arange(-R, R + 1)))
    dx, dy = np.abs(x1), -np.abs(y1)
    sx, sy = np.where(x1 > 0, 1, -1), np.where(y1 > 0, 1, -1)
    x, y = np.zeros_like(x1), np.zeros_like(y1)
    err = dx + dy
    e2max = np.abs(2 * err)
    boxed = np.ones(len(x1), bool)
    live = np.ones(len(x1), bool)
    while live.any():
        e2 = 2 * err
        e2max = np.where(live, np.maximum(e2max, np.abs(e2)), e2max)
        sx_go = live & (e2 >= dy)
        live &= ~(sx_go & (x == x1))
        sx_go &= live
        err = err + np.where(sx_go, dy, 0)
        x = x + np.where(sx_go, sx, 0)
        sy_go = live & (e2 <= dx)
        live &= ~(sy_go & (y == y1))
        sy_go &= live
        err = err + np.where(sy_go, dx, 0)
        y = y + np.where(sy_go, sy, 0)
        boxed &= (np.minimum(0, x1) <= x) & (x <= np.maximum(0, x1)) & (np.minimum(0, y1) <= y) & (y <= np.maximum(0, y1))
    return x1, y1, x, y, e2max, boxed


def test_bresenham_walk_stops_on_its_end_cell():
    """The hit kernel (csrc/icpb_grid.cuh grid_hits_kernel) never walks: when both end cells are in
    the grid it puts the hit on the end cell.  That is the reference's hit cell only if every walk
    stops on (x1, y1) and never leaves the bounding box of its end cells; and the 64-bit walk is exact
    only if |2 * error| stays within 3 * max(|dx|, |dy|) (include/icpb.h, ICPB_MAX_GRID_CELL).  All
    three are checked here for every end offset with |dx|, |dy| <= 300, against the walk of
    oracle/grid_exact.py on a sample."""
    from oracle import grid_exact
    x1, y1, x, y, e2max, boxed = _walk_ends(300)
    assert len(x1) == 601 * 601
    np.testing.assert_array_equal(x, x1)
    np.testing.assert_array_equal(y, y1)
    assert boxed.all()
    assert (e2max <= 3 * np.maximum(np.abs(x1), np.abs(y1))).all()
    big = 1 << 40
    for k in np.random.default_rng(5).choice(len(x1), 300, replace=False):
        visited, end = grid_exact.walk(big, big, big + int(x1[k]), big + int(y1[k]), 1 << 62, 1 << 62)
        assert end == (big + x1[k], big + y1[k]) and visited[-1] == end
        assert len(visited) == 1 + max(abs(int(x1[k])), abs(int(y1[k])))


def test_int64_walk_needs_the_cell_bound():
    """Beyond ICPB_MAX_GRID_CELL the bound of include/icpb.h is not decoration: with end cells near
    6e18, `2 * error` passes 2^63, and a walk in wrapping int64 visits other cells than the exact
    one from its second step.  (tests/test_gpu_grid_edges.py feeds such a beam to the library, which
    must reject it.)"""
    from oracle import grid_exact

    def wrap(v):
        return (v + (1 << 63)) % (1 << 64) - (1 << 63)

    def walk64(x0, y0, x1, y1, w, h):
        dx, dy = abs(x1 - x0), -abs(y1 - y0)
        sx, sy = (1 if x1 > x0 else -1), (1 if y1 > y0 else -1)
        error, out = wrap(dx + dy), []
        while 0 <= x0 < w and 0 <= y0 < h:
            out.append((x0, y0))
            e2 = wrap(error * 2)
            if e2 >= dy:
                if x0 == x1:
                    break
                error, x0 = wrap(error + dy), x0 + sx
            if e2 <= dx:
                if y0 == y1:
                    break
                error, y0 = wrap(error + dx), y0 + sy
        return out

    x1, y1 = 6 * 10 ** 18, -3 * 10 ** 18 + 40
    exact, _ = grid_exact.walk(32, 40, x1, y1, 64, 64)
    assert walk64(32, 40, x1, y1, 64, 64) != exact
    # inside the bound the two agree
    x1, y1 = 1 << 60, -(1 << 60) // 3
    assert walk64(32, 40, x1, y1, 64, 64) == grid_exact.walk(32, 40, x1, y1, 64, 64)[0]
