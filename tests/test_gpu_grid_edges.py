"""Occupancy grid on the GPU under adversarial inputs: bit-exact against the exact restatement
(oracle/grid_exact.py, Python-int cells and walk) or, for the large deterministic sweeps, the C oracle
(equal to it wherever int64 is exact, tests/test_grid_reference.py).  Every case updates a pre-filled
grid whose values cover the whole int8 range, through produce_occupancy_grid / update_occupancy_grid.

G1 beams long enough to take the 64-bit walk, G2 every direction and length from one pose, G3 the
order of hits and misses on shared cells, G4 points on cell edges, G5 warp, scan and grid shapes,
G6 the input contract of include/icpb.h (ICPB_MAX_GRID_CELL, ICPB_MAX_GRID_CELLS, finiteness)."""
import ctypes
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ODDS = ((1, 1), (3, 1), (1, 127), (127, 127))


def prefilled(rng, h, w):
    g = rng.integers(-128, 128, (h, w)).astype(np.int8)
    g.flat[:min(g.size, 7)] = (-128, -1, 0, 1, 127, -127, 126)[:min(g.size, 7)]
    return g


def pack(scans):
    from oracle import c_oracle
    return c_oracle.pack([np.asarray(s, dtype=np.float64).reshape(-1, 2) for s in scans])


def check_update(poses, scans, grid0, cell, min_x, min_y, odds=(3, 1), ref="exact"):
    """update_occupancy_grid on a copy of grid0 against the reference; returns the grid."""
    from icp_slam_b200 import produce_occupancy_grid as pog
    from oracle import c_oracle, grid_exact
    poses = np.asarray(poses, dtype=np.float64).reshape(-1, 3)
    xy, off = pack(scans)
    want = grid0.copy()
    (grid_exact if ref == "exact" else c_oracle).update_grid(want, poses, xy, off, cell, min_x, min_y, *odds)
    got = grid0.copy()
    out = pog.update_occupancy_grid(got, poses, [xy[off[k]:off[k + 1]] for k in range(len(off) - 1)], cell,
                                    min_x, min_y, kHitOdds=odds[0], kMissOdds=odds[1])
    assert out is got
    np.testing.assert_array_equal(got, want)
    return want


# ---- G1: long beams and the int / 64-bit switch --------------------------------------------------

def test_g1_long_beams_take_the_64_bit_walk():
    """A 64 x 64 grid at 5 cm; scans of three warps each: all short, all 1e8..1e10 m, and mixed, in
    every direction, from poses inside and outside the grid."""
    rng = np.random.default_rng(101)
    cell, min_x, min_y = 0.05, -1.6, -1.45
    poses, scans = [], []
    for s in range(8):
        poses.append((rng.uniform(-1.7, 1.7), rng.uniform(-1.6, 1.8), rng.uniform(-np.pi, np.pi)))
        phi = rng.uniform(-np.pi, np.pi, 96)
        r = np.concatenate((rng.uniform(0.01, 3.0, 32), 10 ** rng.uniform(8, 10, 32),
                            np.where(rng.random(32) < 0.5, rng.uniform(0.01, 3.0, 32), 10 ** rng.uniform(8, 10, 32))))
        pts = np.c_[r * np.cos(phi), r * np.sin(phi)]
        pts[40] = (1e10, -1e10)
        pts[41] = (-1e10, 1e10)
        scans.append(np.clip(pts, -1e10, 1e10))
    for odds in ODDS:
        want = check_update(poses, scans, prefilled(rng, 64, 64), cell, min_x, min_y, odds)
        assert len(np.unique(want)) > 20


def test_g1_beams_on_the_switch():
    """End cells exactly 2^28 - 1 and 2^28 cells from the origin along both axes and both signs
    (0.5 m cells and binary-fraction coordinates: the cells are exact), one warp all below the
    switch, one with a single lane on it."""
    from oracle import grid_exact
    cell, min_x, min_y = 0.5, -16.0, -16.0
    rng = np.random.default_rng(102)
    lim = 1 << 28

    def at(cx):                                    # centre of cell cx along an axis whose origin is -16
        return min_x + (cx + 0.5) * cell

    ends = []
    for c in (lim - 1, lim, -(lim - 1), -lim, lim - 2, lim + 1):
        ends += [(at(c), at(rng.integers(0, 64))), (at(rng.integers(0, 64)), at(c)), (at(c), at(c))]
    ends = np.array(ends)
    for xy in ends:
        assert max(abs(grid_exact.cell(xy[0], min_x, cell)), abs(grid_exact.cell(xy[1], min_y, cell))) in \
            (lim - 1, lim, lim - 2, lim + 1)
    below = np.array([(at(lim - 1), at(5)), (at(5), at(-(lim - 1)))] * 16)
    one_on = below.copy()
    one_on[17] = (at(lim), at(9))
    P = np.array([at(30) - 0.125, at(33) + 0.25])
    scans = [ends - P, below - P, one_on - P]
    for odds in ODDS[:2]:
        check_update([(*P, 0.0)] * 3, scans, prefilled(rng, 64, 64), cell, min_x, min_y, odds)


# ---- G2: direction and length coverage ------------------------------------------------------------

def window_scan(pose_cell, R, cell, min_x, min_y):
    """End points at the centre of every cell of the (2R+1)^2 window around pose_cell, in the frame
    of a pose at heading 0 on that cell's centre (so the local points are exact)."""
    ox, oy = np.meshgrid(np.arange(-R, R + 1), np.arange(-R, R + 1))
    pts = np.c_[ox.ravel(), oy.ravel()].astype(np.float64) * cell
    pose = (min_x + (pose_cell[0] + 0.5) * cell, min_y + (pose_cell[1] + 0.5) * cell, 0.0)
    return pose, pts


@pytest.mark.parametrize("where", ["centre", "corner00", "corner10", "corner01", "corner11", "edge_left",
                                   "edge_right", "edge_bottom", "edge_top", "outside"])
def test_g2_every_end_cell_in_a_window(where):
    """One scan of 40,401 beams, one to every cell of a 201 x 201 window: zero-length beams, axis-
    parallel beams, exact diagonals, every slope; the grid is 150 x 110, so most beams also leave it."""
    h, w, cell, min_x, min_y = 110, 150, 0.25, -20.0, -13.75
    pc = {"centre": (75, 55), "corner00": (0, 0), "corner10": (w - 1, 0), "corner01": (0, h - 1),
          "corner11": (w - 1, h - 1), "edge_left": (0, 40), "edge_right": (w - 1, 70), "edge_bottom": (90, 0),
          "edge_top": (20, h - 1), "outside": (-3, 50)}[where]
    pose, pts = window_scan(pc, 100, cell, min_x, min_y)
    rng = np.random.default_rng(len(where))
    odds = ODDS[len(where) % 4]
    grid0 = prefilled(rng, h, w)
    want = check_update([pose], [pts], grid0, cell, min_x, min_y, odds, ref="exact" if where == "centre" else "c")
    changed = int((want != grid0).sum())
    assert changed == 0 if where == "outside" else changed > 1000


# ---- G3: order semantics --------------------------------------------------------------------------

def star(length_order, cell):
    """Beams in 16 directions at lengths 4, 9, 15, 22 cells: a shorter beam's end lies on (or next
    to) a longer beam's path, so cells are hit and crossed within one scan, in the given order."""
    ang = np.arange(16) * (np.pi / 8)
    return np.concatenate([np.c_[np.cos(ang), np.sin(ang)] * (L * cell) for L in length_order])


@pytest.mark.parametrize("odds", ODDS)
def test_g3_hits_and_misses_on_shared_cells_in_both_orders(odds):
    rng = np.random.default_rng(odds[0] * 1000 + odds[1])
    cell, min_x, min_y = 0.1, -3.0, -3.0
    scans = [star((4, 9, 15, 22), cell), star((22, 15, 9, 4), cell), star((9, 22, 4, 15), cell)]
    poses = [(0.03, 0.02, 0.0), (0.53, -0.4, 0.3), (-0.7, 0.45, -1.2)]
    # the same scans again from the same poses in the opposite scan order
    check_update(poses + poses[::-1], scans + scans[::-1], prefilled(rng, 60, 60), cell, min_x, min_y, odds)
    check_update(poses, scans, np.zeros((60, 60), np.int8), cell, min_x, min_y, odds)


# ---- G4: cell boundaries --------------------------------------------------------------------------

@pytest.mark.parametrize("cell", [0.25, 0.5])
def test_g4_points_on_cell_edges(cell):
    """Poses and points on exact multiples of the cell width (global points on cell edges), headings
    k*pi/2 (cos and sin are not exactly 0 and 1: points land one rounding beside an edge), origins
    given as negative multiples."""
    rng = np.random.default_rng(int(cell * 100))
    min_x, min_y = -12 * cell, -7 * cell
    poses, scans = [], []
    for s in range(12):
        k = int(rng.integers(-4, 5))
        poses.append((rng.integers(-14, 50) * cell, rng.integers(-9, 40) * cell, k * np.pi / 2))
        scans.append(rng.integers(-30, 31, (70, 2)) * cell)
    for odds in ODDS[:2]:
        want = check_update(poses, scans, prefilled(rng, 40, 48), cell, min_x, min_y, odds)
    from oracle import c_oracle
    gxy = c_oracle.global_points(np.array(poses), *pack(scans))
    frac = np.abs(gxy / cell - np.round(gxy / cell))
    assert (frac == 0).sum() > 100 and ((frac > 0) & (frac < 1e-12)).sum() > 100


# ---- G5: warp, scan and grid shapes ---------------------------------------------------------------

def test_g5_scan_lengths_around_the_warp_and_cta():
    rng = np.random.default_rng(51)
    lens = (1, 31, 32, 33, 255, 256, 257, 1000)
    scans = [rng.uniform(-4, 4, (m, 2)) for m in lens]
    poses = np.c_[rng.uniform(-1, 1, (len(lens), 2)), rng.uniform(-np.pi, np.pi, len(lens))]
    for odds in ODDS[1:3]:
        check_update(poses, scans, prefilled(rng, 70, 90), 0.1, -4.5, -3.5, odds)


def diverging_pair(k):
    """Two beams from cell (2, 30): one along the x axis to (70, 30), one to (2 + L, 31) with L chosen
    so that the two walks share exactly their first k cells."""
    from oracle import grid_exact
    a, _ = grid_exact.walk(2, 30, 70, 30, 1 << 30, 1 << 30)
    for L in range(k, 200):
        b, _ = grid_exact.walk(2, 30, 2 + L, 31, 1 << 30, 1 << 30)
        first = next(i for i, (p, q) in enumerate(zip(a, b)) if p != q)
        if first == k:
            return L
    raise AssertionError(k)


def test_g5_lanes_sharing_cells_around_the_aggregation_window():
    """kAggregateSteps = 24 (csrc/icpb_grid.cuh): lanes on the same cell elect one leader for the
    first 24 steps.  32 beams into one far cell share every step; pairs of beams diverge at steps
    23, 24 and 25; every group sits in one warp, in both lane orders."""
    cell, min_x, min_y = 0.1, 0.0, 0.0
    pose = (0.25, 3.05, 0.0)                      # cell (2, 30)
    rng = np.random.default_rng(52)

    def end(cx, cy, jitter):
        return ((cx + 0.5 + jitter[0]) * cell - pose[0], (cy + 0.5 + jitter[1]) * cell - pose[1])

    same = [end(70, 55, rng.uniform(-0.4, 0.4, 2)) for _ in range(32)]
    div = []
    for k in (23, 24, 25):
        L = diverging_pair(k)
        div += [end(70, 30, (0, 0)), end(2 + L, 31, (0, 0))] * 8
    div = np.array(div[:96])
    for odds in ODDS:
        check_update([pose, pose, pose], [same, div, div[::-1]], prefilled(rng, 80, 80), cell, min_x, min_y, odds)


@pytest.mark.parametrize("h,w", [(1, 1), (1, 37), (41, 1)])
def test_g5_degenerate_grids(h, w):
    rng = np.random.default_rng(h * 100 + w)
    cell = 0.2
    poses = np.c_[rng.uniform(-0.2, w * cell + 0.2, 9), rng.uniform(-0.2, h * cell + 0.2, 9),
                  rng.uniform(-np.pi, np.pi, 9)]
    scans = [rng.uniform(-2, 2, (40, 2)) for _ in range(9)]
    scans[0][:8] = 0.0
    for odds in ODDS:
        check_update(poses, scans, prefilled(rng, h, w), cell, 0.0, 0.0, odds)


def test_g5_fewer_poses_than_scans_through_the_c_entry_point():
    from icp_slam_b200 import _lib, icp as gicp
    from oracle import grid_exact
    rng = np.random.default_rng(53)
    scans = [rng.uniform(-3, 3, (int(rng.integers(1, 90)), 2)) for _ in range(10)]
    poses = np.ascontiguousarray(np.c_[rng.uniform(-1, 1, (6, 2)), rng.uniform(-np.pi, np.pi, 6)])
    eng = gicp.engine()
    eng.set_scans(scans)
    xy, off = pack(scans)
    grid = prefilled(rng, 50, 60)
    want = grid.copy()
    grid_exact.update_grid(want, poses, xy[:off[6]], off[:7], 0.1, -3.0, -2.5, 3, 1)
    rc = _lib.lib().icpb_occupancy_grid_update(eng._h, ctypes.c_void_p(poses.ctypes.data), 6,
                                               ctypes.c_void_p(grid.ctypes.data), 50, 60, -3.0, -2.5, 0.1, 3, 1)
    assert rc == 0
    np.testing.assert_array_equal(grid, want)


def test_g5_fortran_order_and_strided_grids_are_updated_in_place():
    from icp_slam_b200 import produce_occupancy_grid as pog
    from oracle import grid_exact
    rng = np.random.default_rng(54)
    scans = [rng.uniform(-3, 3, (120, 2)) for _ in range(5)]
    poses = np.c_[rng.uniform(-1, 1, (5, 2)), rng.uniform(-np.pi, np.pi, 5)]
    xy, off = pack(scans)
    base = prefilled(rng, 45, 70)
    want = base.copy()
    grid_exact.update_grid(want, poses, xy, off, 0.1, -3.5, -2.2, 3, 1)
    f = np.asfortranarray(base)
    assert pog.update_occupancy_grid(f, poses, scans, 0.1, -3.5, -2.2) is f
    np.testing.assert_array_equal(f, want)
    big = prefilled(rng, 90, 140)
    view = big[::2, ::2]
    assert view.shape == base.shape
    view[...] = base
    outside = big.copy()
    assert pog.update_occupancy_grid(view, poses, scans, 0.1, -3.5, -2.2) is view
    np.testing.assert_array_equal(view, want)
    outside[::2, ::2] = want
    np.testing.assert_array_equal(big, outside)               # the cells between the strides are untouched


# ---- G6: the input contract -----------------------------------------------------------------------

def expect_rejected(call, grid, exact=None):
    """The call raises ValueError and leaves the grid as it was.  If it is accepted, say whether the
    result even matches the exact reference (`exact`: the grid the exact restatement gives)."""
    before = grid.copy()
    try:
        call()
    except ValueError:
        np.testing.assert_array_equal(grid, before)
        return
    note = "" if exact is None else f"; the grid differs from the exact reference in {(grid != exact).sum()} cells"
    pytest.fail("accepted an input outside the contract" + note)


def reach_cell_width(pose_xy, min_x, min_y, factor):
    """The cell width at which the host bound of include/icpb.h sits at factor * 2^60."""
    reach = max(abs(pose_xy[0]), abs(pose_xy[1])) + max(abs(min_x), abs(min_y)) + math.sqrt(2) * 1e10
    return reach / (factor * 2.0 ** 60)


def test_g6_just_inside_the_cell_bound_matches_the_exact_walk():
    """Beam ends ~2^60 cells away at the smallest cell width the bound admits."""
    from oracle import grid_exact
    rng = np.random.default_rng(61)
    cell = reach_cell_width((0, 0), 0, 0, 1.0) * (1 + 1e-12)
    min_x = min_y = -32 * cell
    pts = np.array([(1e10, 1e10), (1e10, -1e10), (-1e10, 3e9), (7e9, -1e10), (1e10, 0.0)] + [(0.0, 0.0)] * 3)
    poses = [(0.0, 0.0, np.pi / 4), (0.0, 0.0, 0.3), (-5 * cell, 7 * cell, -2.0)]
    want = check_update(poses, [pts] * 3, prefilled(rng, 64, 64), cell, min_x, min_y, (3, 1))
    assert grid_exact.cell(1e10 * math.sqrt(2), min_y, cell) > 2 ** 59 and (want != 0).sum() > 100


def test_g6_outside_the_cell_bound_is_rejected():
    from icp_slam_b200 import produce_occupancy_grid as pog
    rng = np.random.default_rng(62)
    grid = prefilled(rng, 64, 64)
    scans = [np.array([(1e10, -0.5e10), (1.0, 2.0)])]
    # just outside the host bound
    cell = reach_cell_width((0, 0), 0, 0, 1.0) * (1 - 1e-9)
    expect_rejected(lambda: pog.update_occupancy_grid(grid, [(0.0, 0.0, 0.0)], scans, cell, -32 * cell, -32 * cell),
                    grid)
    # an origin or pose far out makes every cell coordinate large
    expect_rejected(lambda: pog.update_occupancy_grid(grid, [(0.0, 0.0, 0.0)], [np.ones((3, 2))], 1e-6, -1e13, 0.0),
                    grid)
    expect_rejected(lambda: pog.update_occupancy_grid(grid, [(3e13, 0.0, 0.0)], [np.ones((3, 2))], 1e-6, 0.0, 0.0),
                    grid)


def test_g6_beams_that_overflow_an_int64_walk_are_rejected():
    """End cells near (6e18, -3e18): 2 * error passes 2^63 in an int64 walk (test_grid_reference.py),
    which would visit other cells than the reference."""
    from icp_slam_b200 import produce_occupancy_grid as pog
    from oracle import grid_exact
    grid = prefilled(np.random.default_rng(64), 64, 64)
    scans = [np.array([(1e10, -0.5e10), (1.0, 2.0)])]
    cell = 1e10 / 6e18
    min_x, min_y = -32 * cell, -40 * cell
    xy, off = pack(scans)
    exact = grid.copy()
    grid_exact.update_grid(exact, np.zeros((1, 3)), xy, off, cell, min_x, min_y, 3, 1)
    assert grid_exact.cell(1e10, min_x, cell) > 2 ** 62
    expect_rejected(lambda: pog.update_occupancy_grid(grid, [(0.0, 0.0, 0.0)], scans, cell, min_x, min_y),
                    grid, exact)


@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
def test_g6_non_finite_inputs_are_rejected(bad):
    from icp_slam_b200 import _lib, icp as gicp, produce_occupancy_grid as pog
    rng = np.random.default_rng(63)
    scans = [rng.uniform(-2, 2, (50, 2)) for _ in range(3)]
    poses = np.c_[rng.uniform(-1, 1, (3, 2)), rng.uniform(-np.pi, np.pi, 3)]
    grid = prefilled(rng, 40, 40)
    for r, c in ((0, 0), (1, 1), (2, 2)):
        p = poses.copy()
        p[r, c] = bad
        expect_rejected(lambda: pog.update_occupancy_grid(grid, p, scans, 0.1, -2.0, -2.0), grid)
        with pytest.raises(ValueError):
            pog.produce_occupancy_grid(p, scans, 0.1)
    expect_rejected(lambda: pog.update_occupancy_grid(grid, poses, scans, 0.1, bad, -2.0), grid)
    expect_rejected(lambda: pog.update_occupancy_grid(grid, poses, scans, 0.1, -2.0, bad), grid)
    expect_rejected(lambda: pog.update_occupancy_grid(grid, poses, scans, bad, -2.0, -2.0), grid)
    for kw in (dict(min_width=bad), dict(min_height=bad), dict(cell_width=bad)):
        args = dict(cell_width=0.1) | kw
        with pytest.raises(ValueError):
            pog.produce_occupancy_grid(poses, scans, **args)
    # the C entry point says ICPB_EINVAL
    eng = gicp.engine()
    eng.set_scans(scans)
    p = np.ascontiguousarray(poses.copy())
    p[1, 0] = bad
    rc = _lib.lib().icpb_occupancy_grid_update(eng._h, ctypes.c_void_p(p.ctypes.data), 3,
                                               ctypes.c_void_p(grid.ctypes.data), 40, 40, -2.0, -2.0, 0.1, 3, 1)
    assert rc == 10001
    mx, my, hh, ww = ctypes.c_double(), ctypes.c_double(), ctypes.c_int64(), ctypes.c_int64()
    rc = _lib.lib().icpb_occupancy_grid_bounds(eng._h, ctypes.c_void_p(poses.ctypes.data), 3, 0.1, bad, 0.0,
                                               ctypes.byref(mx), ctypes.byref(my), ctypes.byref(hh), ctypes.byref(ww))
    assert rc == 10001


def test_g6_oversized_grids_are_reported_before_allocating():
    """A map whose bounding box needs more than ICPB_MAX_GRID_CELLS cells: produce_occupancy_grid
    raises ValueError from the bounds call (before it would allocate)."""
    from icp_slam_b200 import produce_occupancy_grid as pog
    scans = [np.array([(0.0, 0.0), (1e10, 1e10)])]
    with pytest.raises(ValueError):
        pog.produce_occupancy_grid([(0.0, 0.0, 0.0)], scans, 0.05)
    with pytest.raises(ValueError):
        pog.produce_occupancy_grid([(0.0, 0.0, 0.0)], [np.zeros((1, 2))], 0.05, min_width=1e9, min_height=1e9)
    # the largest map allowed passes the bounds call, one more cell per side does not
    from icp_slam_b200 import _lib, icp as gicp
    eng = gicp.engine()
    eng.set_scans([np.array([(0.0, 0.0), (3.0, 0.4)])])
    pose = np.zeros((1, 3))
    for side, ok in ((32.767, True), (32.769, False)):
        mx, my, hh, ww = ctypes.c_double(), ctypes.c_double(), ctypes.c_int64(), ctypes.c_int64()
        rc = _lib.lib().icpb_occupancy_grid_bounds(eng._h, ctypes.c_void_p(pose.ctypes.data), 1, 1e-3, side, side,
                                                   ctypes.byref(mx), ctypes.byref(my), ctypes.byref(hh),
                                                   ctypes.byref(ww))
        assert (rc == 0) == ok, (side, rc)
        if ok:
            assert 32767 <= hh.value <= 32768 and hh.value * ww.value <= 2 ** 30
