"""GridMap -- env.py's occupancy grid as a bit-packed HBM tensor: a one-map mpp_map_batch.

Grid convention (env.py:4-7): 0 free, 1 obstacle, 2 start, 3 target; start/target are the
first row-major cells equal to 2 / 3 (MAACO.py:32-41) and are traversable.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib

FREE_SPACE, OBSTACLE, START_NODE_VAL, TARGET_NODE_VAL = 0, 1, 2, 3


def _current_device():
    import torch
    _lib.require_device()
    return torch.cuda.current_device()


class GridMap:
    """`handle` is the batch of one map every entry point takes; the batch is freed by close() or with the last
    object (GridMap, SearchEngine) holding it."""

    def __init__(self, grid, device=None):
        from .batch import _map_set
        g = np.array(grid, dtype=int)  # same coercion as the reference constructors
        if g.ndim != 2:
            raise ValueError("grid must be 2-D")
        self.grid = g
        self.rows, self.cols = g.shape
        self._maps = _map_set(g[None], _current_device() if device is None else int(device))
        self.handle = self._maps.handle
        self.device = self._maps.device_index
        s, t = int(self._maps.start[0]), int(self._maps.target[0])
        self.start_cell, self.target_cell = s, t
        self.start_node = divmod(s, self.cols) if s >= 0 else None
        self.target_node = divmod(t, self.cols) if t >= 0 else None

    def close(self):
        self.handle = None
        self._maps.close()

    def occ_bits(self):
        """(device pointer, pitch in words) of the padded bit-packed occupancy tensor."""
        pitch = C.c_int()
        p = _lib.lib().mpp_map_batch_occ_bits(self.handle, C.byref(pitch))
        return p, pitch.value


def blocks_map(n, frac=0.20, seed=0, rows=None, cols=None):
    """Synthetic block-obstacle map used by the benchmarks (SURVEY.md 8(d)); S=(0,0), T=(n-1,n-1)."""
    rows = rows or n
    cols = cols or n
    rng = np.random.default_rng(seed)
    g = np.zeros((rows, cols), dtype=np.int64)
    m = max(2, min(rows, cols) // 12)
    filled, size = 0, rows * cols                     # (running count: the same decisions as `while g.mean() < frac`)
    while filled / size < frac:
        h, w = rng.integers(1, m, 2)
        r = rng.integers(0, rows - h)
        c = rng.integers(0, cols - w)
        blk = g[r:r + h, c:c + w]
        filled += blk.size - int(blk.sum())
        blk[...] = 1
    g[:2, :2] = 0
    g[-2:, -2:] = 0
    g[0, 0] = START_NODE_VAL
    g[rows - 1, cols - 1] = TARGET_NODE_VAL
    return g
