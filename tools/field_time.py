"""Exact Dijkstra distance fields (field.py: mpp_dijkstra_fields + mpp_dijkstra_field_paths) against the one-warp-per-
search Dijkstra they can replace.  Three workloads, each timed with CUDA events (ms per call, averaged over --reps calls
after one warm-up call; every call ends in its host read-back, so the events span the whole call):

  single/<map>     one start -> target query: DijkstraSolver.solve() vs DijkstraSolver.solve_targets([target]) (one
                   field + one path) on image5 (256x256) and on blocks_map 512, 1024, 2048 (20% obstacles, S=(0,0),
                   T=(n-1,n-1)); field_ms = the field launch alone
  targets_512      one start -> 1000 seeded free targets on blocks_map 512: DijkstraSolver.solve_batch (one search per
                   target, one launch) vs solve_targets
  config5          the config-5 maps (blocks_map(256, 0.20, seed=5000 + i), start / target moved to seeded free cells as
                   in search_batch_time.py): SearchBatch.search(2, ...) vs SearchBatch.field_paths (device tensors in
                   and out) and, end to end from host grids with the host clock, solve_search_batch(..., "dijkstra") vs
                   SearchBatch(grids).field_paths + read-back

Each workload also checks that both sides return the same results.  Prints one JSON line with the card's name and power
limit, read in the same run.

    python tools/field_time.py [--reps 5] [--maps 1250]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

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


def timed(fn, reps, warm=True):
    """(ms per call over `reps` calls between CUDA events, last result)."""
    if warm:
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


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
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--maps", type=int, default=1250)
    args = ap.parse_args()
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import SearchBatch, solve_search_batch
    from maaco_path_planing_b200.dijkstra import DijkstraSolver
    if not torch.cuda.is_available():
        raise SystemExit("field_time.py measures the GPU: no CUDA device visible")
    torch.cuda.set_device(0)
    name, power = card()
    out = {"what": "exact Dijkstra distance fields vs one warp per search", "card": name, "power_limit_w": power,
           "reps": args.reps, "results": {}}
    env = np.load(os.path.join(ROOT, "tests", "golden", "env_grids.npz"))
    singles = {"image5": env["image5"].astype(int)}
    singles.update({f"blocks{n}": blocks_map(n, 0.20, seed=3000 + n) for n in (512, 1024, 2048)})
    for mname, grid in singles.items():
        s = DijkstraSolver(grid)
        big = grid.size > 512 * 512
        solve_ms, want = timed(s.solve, 1 if big else args.reps, warm=not big)   # (a lone warp: seconds on the big maps)
        both_ms, got = timed(lambda: s.solve_targets([s.target_node]), args.reps)
        field_ms, _ = timed(lambda: s._field(None), args.reps)
        out["results"][f"single/{mname}"] = dict(
            shape=list(grid.shape), solve_ms=solve_ms, field_and_path_ms=both_ms, field_ms=field_ms,
            speedup=solve_ms / both_ms, path_cells=len(want[0]), match=got[0] == want)
        print(mname, out["results"][f"single/{mname}"], file=sys.stderr, flush=True)
    grid = singles["blocks512"]
    s = DijkstraSolver(grid)
    rng = np.random.default_rng(512)
    free = np.argwhere(grid == 0)
    targets = [tuple(int(x) for x in free[i]) for i in rng.choice(len(free), 1000, replace=False)]
    batch_ms, want = timed(lambda: s.solve_batch([s.start_node] * len(targets), targets), args.reps)
    both_ms, got = timed(lambda: s.solve_targets(targets), args.reps)
    want_g = [w[1] for w in want if len(w[0]) > 1]                          # what solve_targets appends to the curve
    out["results"]["targets_512"] = dict(
        targets=len(targets), solve_batch_ms=batch_ms, solve_targets_ms=both_ms, speedup=batch_ms / both_ms,
        match=all(g[0] == w[0] for g, w in zip(got, want)) and s.convergence_curve[-len(want_g):] == want_g)
    print("targets_512", out["results"]["targets_512"], file=sys.stderr, flush=True)
    M = args.maps
    grids = moved(np.stack([blocks_map(256, 0.20, seed=5000 + i) for i in range(M)]), 5000)
    flat = grids.reshape(M, -1)
    src_h, dst_h = (flat == 2).argmax(axis=1).astype(np.int32), (flat == 3).argmax(axis=1).astype(np.int32)
    sb = SearchBatch(grids)
    mi = torch.arange(M, dtype=torch.int32, device="cuda")
    src, dst = torch.as_tensor(src_h, device="cuda"), torch.as_tensor(dst_h, device="cuda")
    search_ms, want = timed(lambda: [x.cpu() for x in sb.search(2, mi, src, dst)], args.reps)
    both_ms, got = timed(lambda: [x.cpu() for x in sb.field_paths(mi, dst)], args.reps)
    fields_ms, _ = timed(lambda: sb._fields(None), args.reps)
    match = all(torch.equal(a, b) for a, b in zip(got[1:], want[1:])) and all(
        torch.equal(got[0][i, :got[1][i]], want[0][i, :want[1][i]]) for i in range(M))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_want = solve_search_batch(list(grids), "dijkstra", {})
    e2e_search_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    b = SearchBatch(grids)
    e2e_got = [x.cpu() for x in b.field_paths(np.arange(M), dst_h)]
    e2e_field_s = time.perf_counter() - t0
    match = match and all(len(w[1]) == int(e2e_got[1][k]) for k, w in enumerate(e2e_want))
    out["results"]["config5"] = dict(
        maps=M, search_ms=search_ms, field_paths_ms=both_ms, fields_ms=fields_ms, speedup=search_ms / both_ms,
        e2e_solve_search_batch_s=e2e_search_s, e2e_field_paths_s=e2e_field_s, match=bool(match))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
