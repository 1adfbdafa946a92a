"""A* and Dijkstra over the config-5 maps (blocks_map(256, 0.20, seed=5000 + i), i < --maps) with SearchBatch: one
start -> target query per map, all maps in one launch.  Two workloads: the maps' own corners (S=(0,0), T=(255,255)) and
start / target moved to seeded random free cells of each map.  Prints one JSON line with, per (workload, algorithm):

  device_maps_per_s   grids uploaded before the timed window; SearchBatch.search (device tensors in and out, incl. its
                      host checks) --reps times between CUDA events, ending in a synchronise
  host_maps_per_s     end to end from host grids: SearchBatch(grids).solve(algorithm) -- upload, safety tables, launch,
                      Python result tuples -- host clock, ending in a synchronise
  launch_ms           one mpp_astar_batch_maps launch (with its longest-first argsort), CUDA events over --reps launches
  expansions_per_s    node expansions of one launch / launch_ms
  oracle_maps_per_s   the C oracle (AStarOracle, same queries) over a seeded sample of the maps on every host core
  oracle_match        the sample's paths and g equal the GPU's

plus the card's name and power limit, read in the same run.  The maps' occupancy (~11 MB for 1250 maps) stays in L2
between repetitions; the search records (one 2.7 MB slot per query) do not fit there.

    python tools/search_batch_time.py [--maps 1250] [--reps 5] [--oracle-sample 96]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]

import numpy as np  # noqa: E402
import torch  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=60)
        power = float(r.stdout.strip().splitlines()[0])
    except Exception:
        power = None
    return name, power


def moved(grids, seed):
    rng = np.random.default_rng(seed)
    out = grids.copy()
    for g in out:
        g[g >= 2] = 0
        s, t = rng.choice(np.flatnonzero(g.ravel() == 0), 2, replace=False)
        g.flat[s], g.flat[t] = 2, 3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--maps", type=int, default=1250)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--oracle-sample", type=int, default=96)
    args = ap.parse_args()
    import pyoracle as O
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import SearchBatch, _SEARCH_ALGORITHMS
    if not torch.cuda.is_available():
        raise SystemExit("search_batch_time.py measures the GPU: no CUDA device visible")
    torch.cuda.set_device(0)
    name, power = card()
    M = args.maps
    corners = np.stack([blocks_map(256, 0.20, seed=5000 + i) for i in range(M)])
    workloads = {"corners": corners, "random_endpoints": moved(corners, 5000)}
    threads = os.cpu_count() or 1
    sample = np.sort(np.random.default_rng(1).choice(M, min(M, args.oracle_sample), replace=False))
    SearchBatch(corners[:8]).solve("astar")                                  # module load, first launches
    out = {"what": "A*/Dijkstra start->target per map, config-5 maps (blocks_map 256x256, 20% obstacles)",
           "card": name, "power_limit_w": power, "maps": M, "reps": args.reps, "host_threads": threads, "results": {}}
    ev = lambda: torch.cuda.Event(enable_timing=True)
    for wname, grids in workloads.items():
        flat = grids.reshape(M, -1)
        src_h, dst_h = (flat == 2).argmax(axis=1), (flat == 3).argmax(axis=1)
        for algorithm, (variant, _, _) in _SEARCH_ALGORITHMS.items():
            r = {}
            # ---- end to end from host grids ----
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            sb = SearchBatch(grids)
            res = sb.solve(algorithm)
            torch.cuda.synchronize()
            r["host_maps_per_s"] = M / (time.perf_counter() - t0)
            sb.close()
            # ---- device resident ----
            sb = SearchBatch(grids)
            mi = torch.arange(M, dtype=torch.int32, device="cuda")
            src = torch.as_tensor(src_h.astype(np.int32), device="cuda")
            dst = torch.as_tensor(dst_h.astype(np.int32), device="cuda")
            sb.search(variant, mi, src, dst)                                 # warm: safety tables, scratch
            torch.cuda.synchronize()
            e0, e1 = ev(), ev()
            e0.record()
            for _ in range(args.reps):
                sb.search(variant, mi, src, dst)
            e1.record()
            torch.cuda.synchronize()
            r["device_maps_per_s"] = M * args.reps / (e0.elapsed_time(e1) / 1e3)
            x0 = sb.expansions()
            e0.record()
            for _ in range(args.reps):
                sb._launch(variant, mi, src, dst, None, True, sb.allow_diagonal_moves, sb.restrict_corners, sb.policy)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / args.reps
            r["launch_ms"] = ms
            r["expansions_per_launch"] = (sb.expansions() - x0) // args.reps
            r["expansions_per_s"] = r["expansions_per_launch"] / (ms / 1e3)
            r["paths_found"] = sum(p[6] is not None for p in res)
            sb.close()
            # ---- the C oracle on every host core ----
            orcs = {int(k): O.AStarOracle(grids[k], True, True) for k in sample}
            t0 = time.perf_counter()
            with ThreadPoolExecutor(threads) as pool:
                want = list(pool.map(lambda k: orcs[int(k)].solve(variant, int(src_h[k]), int(dst_h[k])), sample))
            r["oracle_maps_per_s"] = len(sample) / (time.perf_counter() - t0)
            r["oracle_sample"] = len(sample)
            r["oracle_match"] = all([(a, b) for a, b in res[k][0]] == [divmod(int(c), 256) for c in w[0]] and
                                    (res[k][6] is None or res[k][6] == w[1]) for k, w in zip(sample, want))
            out["results"][f"{wname}/{algorithm}"] = r
    print(json.dumps(out))


if __name__ == "__main__":
    main()
