"""PSO and GA over the config-5 maps (blocks_map(256, 0.20, seed=5000 + i), i < --maps) with PSOBatch / GABatch, all maps
in one wave, config-3 parameters (W = 5, policy main.py:21-24, PSO w/c1/c2 main.py:109-118, GA rates main.py:93-103),
--pop individuals per map and --iters iterations / generations.  Prints one JSON line per planner with:

  solve_ms            PSOBatch(...).solve() / GABatch(...).solve() from host grids, CUDA events ending in a synchronise
  init_ms             the same solve with 0 iterations (upload, initialisation rounds, result tuples)
  ms_per_iteration    (solve_ms - init_ms) / iters: one iteration / generation of every map of the wave
  evals_per_s         fitness evaluations of the whole solve (initialisation attempts included) / solve_ms
  launches_per_iteration  kernel launches of an iteration / generation (population kernels, fitness launches and
                      their growth repeats); the per-map loop makes at least one per map
  loop_s, speedup     the same maps solved by a loop of PSOSolver / GASolver, host clock ending in a synchronise, and
                      loop_s over the batch's solve
  match               every map's result tuple, curve and fitness-evaluation count equal the loop's

plus the card's name and power limit, read in the same run.

    python tools/pop_batch_time.py [--maps 32] [--pop 1024] [--iters 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]

import numpy as np  # noqa: E402
import torch  # noqa: E402

POLICY = dict(turn_penalty_factor=0.3, safety_penalty_factor=0.8, min_safe_distance=1.8,
              diagonal_obstacle_penalty_value=100.0, allow_diagonal_moves=True,
              restrict_diagonal_near_obstacle_policy=True)                  # main.py:21-24


def card():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=60)
        power = float(r.stdout.strip().splitlines()[0])
    except Exception:
        power = None
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--maps", type=int, default=32)
    ap.add_argument("--pop", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=3)
    args = ap.parse_args()
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import GABatch, PSOBatch
    from maaco_path_planing_b200.ga_solver import GASolver
    from maaco_path_planing_b200.pso import PSOSolver
    if not torch.cuda.is_available():
        raise SystemExit("pop_batch_time.py measures the GPU: no CUDA device visible")
    torch.cuda.set_device(0)
    name, power = card()
    M, N, K, W = args.maps, args.pop, args.iters, 5
    grids = np.stack([blocks_map(256, 0.20, seed=5000 + i) for i in range(M)])
    seeds = [7000 + i for i in range(M)]
    planners = {
        "pso": (PSOBatch, PSOSolver, dict(w=0.7, c1=1.5, c2=1.5)),
        "ga": (GABatch, GASolver, dict(mutation_rate=0.1, crossover_rate=0.8, tournament_size=3)),
    }
    ev = lambda: torch.cuda.Event(enable_timing=True)
    for planner, (Batch, Solver, params) in planners.items():
        Batch(grids[:2], 1, 64, W, seeds=seeds[:2], **params, **POLICY).solve()          # module load, first launches
        r = {"what": f"{planner.upper()} over config-5 maps (blocks_map 256x256, 20% obstacles), one wave, W=5",
             "card": name, "power_limit_w": power, "maps": M, "pop": N, "iters": K}
        timings = {}
        for k in (0, K):
            torch.cuda.synchronize()
            e0, e1 = ev(), ev()
            e0.record()
            b = Batch(grids, k, N, W, seeds=seeds, **params, **POLICY)
            res = b.solve()
            e1.record()
            torch.cuda.synchronize()
            timings[k] = (e0.elapsed_time(e1), b.launches, sum(b.fitness_evaluations))
            b.close()
        r["solve_ms"], r["init_ms"] = timings[K][0], timings[0][0]
        r["ms_per_iteration"] = (timings[K][0] - timings[0][0]) / max(1, K)
        r["fitness_evaluations"] = timings[K][2]
        r["evals_per_s"] = timings[K][2] / (timings[K][0] / 1e3)
        r["launches_per_iteration"] = (timings[K][1] - timings[0][1]) / max(1, K)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        solos = []
        for m in range(M):
            s = Solver(grids[m], K, N, W, **params, rng_seed=seeds[m], verbose=False, **POLICY)
            solos.append((s, s.solve()))
        torch.cuda.synchronize()
        r["loop_s"] = time.perf_counter() - t0
        r["speedup"] = r["loop_s"] / (r["solve_ms"] / 1e3)
        b_evals = Batch(grids, K, N, W, seeds=seeds, **params, **POLICY)
        res = b_evals.solve()
        r["match"] = all(res[m][:6] == tuple(w) and res[m][6] == s.convergence_curve and
                         b_evals.fitness_evaluations[m] == s.fitness_evaluations for m, (s, w) in enumerate(solos))
        r["paths_found"] = sum(len(x[0]) > 0 for x in res)
        b_evals.close()
        print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
