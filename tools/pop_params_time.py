"""PSO, GA and MPA parameter sweeps in one launch: PSOBatch / GABatch / MPABatch(map_params=...) against a loop of
1-map waves.

The workload, per planner, is --sets parameter sets (default 64, every set its own seed) on one config-5 map
(blocks_map(256, 0.20, seed=5000)), --pop individuals x --iters iterations (PSO / GA: W = 5 waypoints).  PSO varies
w x c1 x c2 x turn_penalty_factor, GA mutation_rate x crossover_rate x tournament_size x safety_penalty_factor, MPA
FADs_rate x P_const x levy_beta x turn_penalty_factor.  Two ways to run a sweep:

  per_map_wave   one batch of --sets copies of the map with map_params (the per-map kernel instantiations)
  one_map_waves  what a sweep did before per-map parameters: one 1-map batch per parameter set

Each arm is timed with the host clock around the whole sweep (it ends in a device synchronise), --rounds rounds with the
arms alternated; medians and the spread (min..max) are reported as maps/s.

Kernel cost of the per-map instantiations: a --sets-map wave whose maps all carry the default parameters is solved with
map_params=None (the existing kernels) and with map_params=[{}] * sets (the _p kernels); both do the same work.
Reported: CUDA-event time of each solve over its iterations, alternated, --rounds rounds (median), and whether the two
give the same results.

Result check: the per-map wave equals the 1-map waves on every set.  Prints one JSON line per planner with the card's
name and power limit, read in the same run.  Needs a GPU; there is no fallback.

    python tools/pop_params_time.py [--planners pso,ga,mpa] [--sets 64] [--pop 1024] [--iters 2] [--rounds 3]
"""
import argparse
import itertools
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]

import numpy as np  # noqa: E402
import torch  # noqa: E402

POLICY = dict(turn_penalty_factor=0.1, safety_penalty_factor=0.05, min_safe_distance=1.5,
              diagonal_obstacle_penalty_value=1000.0)
BASE = {"pso": dict(w=0.7, c1=1.5, c2=1.5, **POLICY), "ga": dict(mutation_rate=0.1, crossover_rate=0.8, **POLICY),
        "mpa": dict(FADs_rate=0.2, P_const=0.5, levy_beta=1.5, turn_penalty_factor=0.1, safety_penalty_factor=0.05)}
GRIDS = {"pso": (("w", (0.4, 0.6, 0.8, 0.9)), ("c1", (1.0, 1.5, 2.0, 2.5)), ("c2", (1.0, 2.0)),
                 ("turn_penalty_factor", (0.1, 0.5))),
         "ga": (("mutation_rate", (0.05, 0.1, 0.2, 0.3)), ("crossover_rate", (0.6, 0.8, 0.9, 1.0)),
                ("tournament_size", (2, 3)), ("safety_penalty_factor", (0.05, 0.5))),
         "mpa": (("FADs_rate", (0.1, 0.2, 0.3, 0.4)), ("P_const", (0.3, 0.5, 0.7, 0.9)), ("levy_beta", (1.2, 1.5)),
                 ("turn_penalty_factor", (0.1, 0.5)))}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=60)
        power = float(r.stdout.strip().splitlines()[0])
    except Exception:
        power = None
    return name, power


def param_sets(planner, n):
    keys, values = zip(*GRIDS[planner])
    return [dict(zip(keys, v)) for v in itertools.islice(itertools.cycle(itertools.product(*values)), n)]


def make(planner, grids, pop, iters, seeds, params, map_params=None):
    from maaco_path_planing_b200.batch import GABatch, MPABatch, PSOBatch
    if planner == "pso":
        return PSOBatch(grids, iters, pop, 5, seeds=seeds, map_params=map_params, **params)
    if planner == "ga":
        return GABatch(grids, iters, pop, 5, seeds=seeds, map_params=map_params, **params)
    return MPABatch(grids, pop, iters, seeds=seeds, map_params=map_params, **params)


def run_planner(planner, g, args):
    P, N, K = args.sets, args.pop, args.iters
    grids = np.stack([g] * P)
    ps = param_sets(planner, P)
    seeds = list(range(P))
    base = BASE[planner]

    def per_map_wave():
        t0 = time.perf_counter()
        out = make(planner, grids, N, K, seeds, base, ps).solve()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, out

    def one_map_waves():
        t0 = time.perf_counter()
        out = []
        for k in range(P):
            out += make(planner, grids[k:k + 1], N, K, [seeds[k]], {**base, **ps[k]}).solve()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, out

    arms = {"per_map_wave": per_map_wave, "one_map_waves": one_map_waves}
    make(planner, grids, N, K, seeds, base, ps).solve()               # warm-up: both launch shapes
    make(planner, grids[:1], N, K, seeds[:1], base).solve()
    times, results = {k: [] for k in arms}, {}
    order = list(arms)
    for r in range(args.rounds):
        for k in (order if r % 2 == 0 else order[::-1]):
            t, out = arms[k]()
            times[k].append(t)
            results[k] = out
    rate = {k: {"maps_per_s_median": P / statistics.median(v), "maps_per_s_min": P / max(v),
                "maps_per_s_max": P / min(v), "seconds": v} for k, v in times.items()}

    # the kernels: one default-parameter wave through the existing and the per-map instantiations
    ev_ms, same = {"existing": [], "per_map": []}, True
    for r in range(args.rounds):
        got = {}
        for k in (("existing", "per_map") if r % 2 == 0 else ("per_map", "existing")):
            b = make(planner, grids, N, K, seeds, base, [{}] * P if k == "per_map" else None)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            got[k] = b.solve()
            e1.record()
            e1.synchronize()
            ev_ms[k].append(e0.elapsed_time(e1) / max(1, K))
        same &= repr(got["existing"]) == repr(got["per_map"])
    return {
        "sets": P, "population": N, "iterations": K, "rounds": args.rounds,
        "map": "blocks_map(256, 0.20, seed=5000)", "arms": rate,
        "speedup_per_map_wave_vs_one_map_waves": rate["per_map_wave"]["maps_per_s_median"] /
        rate["one_map_waves"]["maps_per_s_median"],
        "default_parameter_wave": {"maps": P, "event_ms_per_iteration_median":
                                   {k: statistics.median(v) for k, v in ev_ms.items()}, "event_ms_per_iteration": ev_ms},
        "results_equal": {"per_map_wave_vs_one_map_waves": results["per_map_wave"] == results["one_map_waves"],
                          "default_wave_existing_vs_per_map": bool(same)},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--planners", default="pso,ga,mpa")
    ap.add_argument("--sets", type=int, default=64)
    ap.add_argument("--pop", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pop_params_time.py measures the GPU: no CUDA device visible")
    torch.cuda.set_device(0)
    from maaco_path_planing_b200 import blocks_map
    name, power = card()
    g = blocks_map(256, 0.20, seed=5000)
    for planner in args.planners.split(","):
        print(json.dumps({"tool": "pop_params_time", "planner": planner, "card": name, "power_limit_w": power,
                          **run_planner(planner, g, args)}), flush=True)


if __name__ == "__main__":
    main()
