"""Drop-in for the reference's ``src/produce_occupancy_grid.py`` (SURVEY.md section 8f-4): same
function names, arguments and return values, the per-beam Bresenham loops on the GPU.

* ``produce_occupancy_grid(poses, lidar_points, cell_width, min_width=0, min_height=0, kHitOdds=3,
  kMissOdds=1) -> (grid int8 (h, w), (min_x, min_y))``                     (reference :11-58)
* ``update_occupancy_grid(occupancy_grid, poses, lidar_points, cell_width, min_x, min_y, kHitOdds=3,
  kMissOdds=1) -> grid`` (updated in place and returned)                    (reference :60-80)
* ``grid_mle(grid, unknown_empty=True)``                                     (reference :140-149)

The grids are bit-identical to the reference's, including the int8 wrap-around of its saturation
tests (see csrc/icpb_grid.cuh).  File output (``save_grid``, ``save_image``) stays with the
reference.  No CPU fallback: without libicpb.so and a B200 these raise.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _lib
from . import icp as _icp


def _odds(v, name):
    if int(v) != v or not 1 <= int(v) <= 127:
        raise ValueError(f"{name} must be an integer in 1..127 (got {v!r})")
    return int(v)


def _stage(poses, lidar_points, device):
    poses = np.ascontiguousarray(poses, dtype=np.float64)
    if poses.ndim != 2 or poses.shape[1] != 3:
        raise ValueError(f"poses has shape {poses.shape}; expected (n, 3)")
    n_scans = lidar_points.n_scans if isinstance(lidar_points, _icp.ScanTable) else len(lidar_points)
    if n_scans != len(poses):
        raise ValueError(f"{len(poses)} poses for {n_scans} scans")
    eng = _icp.engine(device)
    eng.ensure_scans(lidar_points)
    return eng, poses


def _update(eng, poses, grid, cell_width, min_x, min_y, k_hit, k_miss):
    _lib.check(_lib.lib().icpb_occupancy_grid_update(eng._h, _lib.ptr(poses), len(poses),
                                                     _lib.ptr(grid), grid.shape[0], grid.shape[1],
                                                     float(min_x), float(min_y), float(cell_width),
                                                     k_hit, k_miss),
               "icpb_occupancy_grid_update")


def produce_occupancy_grid(poses, lidar_points, cell_width, min_width=0, min_height=0, kHitOdds=3,
                           kMissOdds=1, device=None):
    k_hit, k_miss = _odds(kHitOdds, "kHitOdds"), _odds(kMissOdds, "kMissOdds")
    eng, poses = _stage(poses, lidar_points, device)
    min_x, min_y = ctypes.c_double(), ctypes.c_double()
    h, w = ctypes.c_int64(), ctypes.c_int64()
    _lib.check(_lib.lib().icpb_occupancy_grid_bounds(eng._h, _lib.ptr(poses), len(poses),
                                                     float(cell_width), float(min_width), float(min_height),
                                                     ctypes.byref(min_x), ctypes.byref(min_y),
                                                     ctypes.byref(h), ctypes.byref(w)),
               "icpb_occupancy_grid_bounds")
    grid = np.zeros((h.value, w.value), dtype=np.int8)
    _update(eng, poses, grid, cell_width, min_x.value, min_y.value, k_hit, k_miss)
    return grid, (min_x.value, min_y.value)


def update_occupancy_grid(occupancy_grid, poses, lidar_points, cell_width, min_x, min_y, kHitOdds=3,
                          kMissOdds=1, device=None):
    k_hit, k_miss = _odds(kHitOdds, "kHitOdds"), _odds(kMissOdds, "kMissOdds")
    if not isinstance(occupancy_grid, np.ndarray) or occupancy_grid.dtype != np.int8 or occupancy_grid.ndim != 2:
        raise ValueError("occupancy_grid must be a 2-D int8 array")
    eng, poses = _stage(poses, lidar_points, device)
    work = np.ascontiguousarray(occupancy_grid)
    _update(eng, poses, work, cell_width, min_x, min_y, k_hit, k_miss)
    if work is not occupancy_grid:
        occupancy_grid[...] = work
    return occupancy_grid


def grid_mle(grid, unknown_empty=True):
    grid = grid.copy()
    grid[grid > 0] = 127
    grid[grid < 0] = -128
    return grid
