"""Bisect helper: waypoint fitness vs the oracle for one (size, N, W, use_order) in a subprocess-friendly form."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np, torch
size, N, W, use_order, pso_frac = int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4]), float(sys.argv[5])
from maaco_path_planing_b200 import GridMap, blocks_map
from maaco_path_planing_b200.engine import SearchEngine, make_policy
import pyoracle as O
grid = blocks_map(size, 0.2, seed=size)
rng = np.random.default_rng(size)
wps = rng.integers(0, size * size, (N, W)).astype(np.int32)
free = np.flatnonzero(grid.ravel() != 1)
k = int(N * pso_frac)
wps[k:] = free[rng.integers(0, len(free), (N - k, W))]
eng = SearchEngine(GridMap(grid))
if not use_order:
    eng._chain_order = lambda mi, w: None
cells, ncell, stats = eng.waypoint_fitness(wps, make_policy(0.3, 0.8, 1.8, 100.0))
torch.cuda.synchronize()
ocells, oncell, ostats, oexp = O.waypoint_fitness(grid, wps, 0.3, 0.8, 1.8, 100.0, threads=0)
ok = np.array_equal(ncell.cpu().numpy(), oncell) and np.array_equal(stats.cpu().numpy(), ostats)
print("RESULT", sys.argv[1:], "ok" if ok else "MISMATCH", eng.expansions()[0], oexp, eng.queue_stats(), "heap_cap", eng.heap_cap)
