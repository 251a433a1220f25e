"""Exact restatement of the reference's occupancy-grid update -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The same loops as oracle/grid_oracle.c (reference src/produce_occupancy_grid.py:54-56, :76-78,
:96-138), but every cell coordinate and every Bresenham quantity is a Python int, so the walk is
exact at any magnitude: there is no int64 to overflow.  Global points come from
c_oracle.global_points, which is bit-exact against the goldens.  Cells are
``math.floor((g - min) / cell)``: the same IEEE double subtraction and division as the reference,
then an exact floor, which raises where the reference's ``int(np.floor(...))`` raises (ValueError on
NaN, OverflowError on inf).  Beams are applied one after another in (scan, beam) order.
"""
from __future__ import annotations

import math

import numpy as np

from . import c_oracle


def cell(pos: float, mn: float, cell_width: float) -> int:
    """global_position_to_grid_cell (:133-138) for one coordinate."""
    return math.floor((float(pos) - float(mn)) / float(cell_width))


def walk(x0: int, y0: int, x1: int, y1: int, w: int, h: int):
    """bresenham_update's loop (:100-124): the cells that get a miss, in order, and the cell the walk
    stops on (where the hit lands if it is inside the grid, :127-131)."""
    dx, dy = abs(x1 - x0), -abs(y1 - y0)
    sx, sy = (1 if x1 > x0 else -1), (1 if y1 > y0 else -1)
    error = dx + dy
    visited = []
    while True:
        if x0 < 0 or x0 >= w or y0 < 0 or y0 >= h:
            break
        visited.append((x0, y0))
        e2 = error * 2
        if e2 >= dy:
            if x0 == x1:
                break
            error += dy
            x0 += sx
        if e2 <= dx:
            if y0 == y1:
                break
            error += dx
            y0 += sy
    return visited, (x0, y0)


def update_grid(grid, poses, xy, offsets, cell_width, min_x, min_y, k_hit=3, k_miss=1):
    """update_occupancy_grid (:60-80) on an int8 (h, w) array, in place (any memory layout)."""
    assert grid.dtype == np.int8 and grid.ndim == 2
    poses = np.ascontiguousarray(poses, dtype=np.float64)
    xy = np.ascontiguousarray(xy, dtype=np.float64)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    gxy = c_oracle.global_points(poses, xy, offsets)
    h, w = grid.shape
    g = grid.astype(np.int64).ravel().tolist()            # row-major copy: cell (x, y) is g[y * w + x]
    for i in range(len(poses)):
        x0, y0 = cell(poses[i, 0], min_x, cell_width), cell(poses[i, 1], min_y, cell_width)
        for k in range(int(offsets[i]), int(offsets[i + 1])):
            x1, y1 = cell(gxy[k, 0], min_x, cell_width), cell(gxy[k, 1], min_y, cell_width)
            visited, (xe, ye) = walk(x0, y0, x1, y1, w, h)
            for x, y in visited:                          # :109-112 in int8: a miss on a positive cell wraps to -128
                v = g[y * w + x]
                g[y * w + x] = v - k_miss if v <= 0 and v - k_miss > -128 else -128
            if 0 <= xe < w and 0 <= ye < h:               # :127-131: a hit on a negative cell wraps to 127
                v = g[ye * w + xe]
                g[ye * w + xe] = v + k_hit if v >= 0 and v + k_hit < 127 else 127
    grid[...] = np.asarray(g, dtype=np.int64).reshape(h, w).astype(np.int8)
    return grid


def produce_grid(poses, xy, offsets, cell_width, min_width=0, min_height=0, k_hit=3, k_miss=1):
    """produce_occupancy_grid (:11-58): returns (grid int8 (h, w), (min_x, min_y))."""
    gxy = c_oracle.global_points(poses, np.ascontiguousarray(xy, dtype=np.float64), offsets)
    min_x, min_y, h, w = c_oracle.grid_bounds(gxy, cell_width, min_width, min_height)
    grid = np.zeros((h, w), dtype=np.int8)
    update_grid(grid, poses, xy, offsets, cell_width, min_x, min_y, k_hit, k_miss)
    return grid, (min_x, min_y)
