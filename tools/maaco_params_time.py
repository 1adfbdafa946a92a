"""MAACO parameter sweeps in one launch: MAACOBatch(map_params=...) against a loop of 1-map waves.

The workload is a grid of --sets colony parameter sets (default 128: rho x q0_initial x beta x alpha, every map its own
seed) on one config-5 map (blocks_map(256, 0.20, seed=5000)), --ants ants x --iters passes.  Two ways to run it:

  per_map_wave   one MAACOBatch of --sets copies of the map with map_params (the per-map kernel instantiations)
  one_map_waves  what a sweep did before per-map parameters: one 1-map MAACOBatch per parameter set, buffers reused

Each arm is timed with the host clock around the whole sweep (it ends in a device synchronise), --rounds rounds with the
arms alternated; medians and the spread (min..max) are reported as maps/s.

Kernel cost of the per-map instantiations: a --sets-map wave whose maps all carry the default parameters runs once with
map_params=None (mpp_maaco_pass, the existing kernels) and once with map_params=[{}] * sets (mpp_maaco_pass_maps); the
two do the same work pass by pass.  Reported: CUDA-event time of every pass of both, alternated, --rounds rounds
(median of the per-round totals), and per-kernel device time of one round of each from torch.profiler (a separate run).

Result check: the per-map wave equals the 1-map waves on every set, equals solo MAACO on a seeded sample of
--check-sample sets, and the default-parameter wave gives the same bytes in both forms.  Prints one JSON line with the
card's name and power limit, read in the same run.  Needs a GPU; there is no fallback.

    python tools/maaco_params_time.py [--sets 128] [--ants 1024] [--iters 10] [--rounds 3]
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

PARAMS = dict(alpha=1.0, beta=7.0, rho=0.1, Q=2.5, a_turn_coef=1.0, wh_max=0.9, wh_min=0.2, k_h_adaptive=0.9,
              q0_initial=0.5, C0_initial_pheromone=0.1)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=60)
        power = float(r.stdout.strip().splitlines()[0])
    except Exception:
        power = None
    return name, power


def param_grid(n):
    """The first n sets of rho x q0_initial x beta x alpha (4 x 4 x 4 x 2 = 128), the other keys at PARAMS."""
    grid = itertools.product((1.0, 2.0), (5.0, 6.0, 7.0, 8.0), (0.3, 0.5, 0.7, 0.9), (0.05, 0.1, 0.2, 0.3))
    return [dict(alpha=a, beta=b, q0_initial=q, rho=r) for a, b, q, r in itertools.islice(itertools.cycle(grid), n)]


def kernel_times(prof):
    """{kernel name: (device ms, launches)} of the MAACO pass kernels in a torch.profiler run."""
    out = {}
    for e in prof.key_averages():
        name = e.key
        if "mpp_maaco_" not in name or "tau0" in name or "e01" in name:
            continue
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        ms, n = out.get(name, (0.0, 0))
        out[name] = (ms + t / 1e3, n + e.count)
    return {k: {"device_ms": v[0], "launches": v[1]} for k, v in sorted(out.items())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sets", type=int, default=128)
    ap.add_argument("--ants", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--check-sample", type=int, default=8)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("maaco_params_time.py measures the GPU: no CUDA device visible")
    torch.cuda.set_device(0)
    from maaco_path_planing_b200 import MAACO, blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    name, power = card()
    P, N, K = args.sets, args.ants, args.iters
    g = blocks_map(256, 0.20, seed=5000)
    grids = np.stack([g] * P)
    ps = param_grid(P)
    seeds = list(range(P))
    prev = {}

    def per_map_wave():
        t0 = time.perf_counter()
        b = MAACOBatch(grids, N, K, seeds=seeds, map_params=ps, reuse=prev.get("wave"), **PARAMS)
        out = b.solve()
        torch.cuda.synchronize()
        prev["wave"] = b
        return time.perf_counter() - t0, out

    def one_map_waves():
        t0 = time.perf_counter()
        out = []
        for k in range(P):
            b = MAACOBatch(grids[k:k + 1], N, K, seeds=[seeds[k]], reuse=prev.get("one"), **{**PARAMS, **ps[k]})
            out += b.solve()
            prev["one"] = b
        torch.cuda.synchronize()
        return time.perf_counter() - t0, out

    arms = {"per_map_wave": per_map_wave, "one_map_waves": one_map_waves}
    per_map_wave()                                                    # warm-up: both launch shapes
    MAACOBatch(grids[:1], N, K, seeds=[0], **PARAMS).solve()
    times = {k: [] for k in arms}
    results = {}
    order = list(arms)
    for r in range(args.rounds):
        for k in (order if r % 2 == 0 else order[::-1]):
            t, out = arms[k]()
            times[k].append(t)
            results[k] = out
    rate = {k: {"maps_per_s_median": P / statistics.median(v), "maps_per_s_min": P / max(v),
                "maps_per_s_max": P / min(v), "seconds": v} for k, v in times.items()}

    # the kernels: the same default-parameter wave through the existing and the per-map instantiations
    def wave(per_map, reuse=None):
        return MAACOBatch(grids, N, K, seeds=seeds, map_params=[{}] * P if per_map else None, reuse=reuse, **PARAMS)

    ev_ms = {"existing": [], "per_map": []}
    bytes_equal = True
    for r in range(args.rounds):
        ab = {"existing": wave(False), "per_map": wave(True)}
        tot = {k: 0.0 for k in ab}
        for it in range(1, K + 1):
            for k in (("existing", "per_map") if (r + it) % 2 == 0 else ("per_map", "existing")):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                ab[k].run_iteration(it)
                e1.record()
                e1.synchronize()
                tot[k] += e0.elapsed_time(e1)
            x, y = ab["existing"], ab["per_map"]
            bytes_equal &= all(a.tobytes() == b.tobytes() for a, b in zip(x.last_results(), y.last_results()))
            bytes_equal &= x.pheromone().tobytes() == y.pheromone().tobytes()
        bytes_equal &= ab["existing"].solve() == ab["per_map"].solve()
        for k in ab:
            ev_ms[k].append(tot[k])
    prof_kernels = {}
    from torch.profiler import ProfilerActivity, profile
    for k, per_map in (("existing", False), ("per_map", True)):
        b = wave(per_map)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for it in range(1, K + 1):
                b.run_iteration(it)
            torch.cuda.synchronize()
        prof_kernels[k] = kernel_times(prof)

    # results
    wave_res, one_res = results["per_map_wave"], results["one_map_waves"]
    one_ok = wave_res == one_res
    check = sorted(np.random.default_rng(8).choice(P, min(args.check_sample, P), replace=False).tolist())
    solo_ok = True
    for i in check:
        m = MAACO(g, N, K, rng_seed=seeds[i], verbose=False, **{**PARAMS, **ps[i]})
        path, length, turns = m.solve_path_planning()
        solo_ok &= wave_res[i] == (path, length, turns, m.convergence_curve_data)
    print(json.dumps({
        "tool": "maaco_params_time", "card": name, "power_limit_w": power,
        "sets": P, "ants": N, "passes": K, "rounds": args.rounds, "map": "blocks_map(256, 0.20, seed=5000)",
        "arms": rate,
        "speedup_per_map_wave_vs_one_map_waves": rate["per_map_wave"]["maps_per_s_median"] /
        rate["one_map_waves"]["maps_per_s_median"],
        "default_parameter_wave": {"maps": P, "pass_event_ms_total_median": {k: statistics.median(v) for k, v in ev_ms.items()},
                                   "pass_event_ms_totals": ev_ms, "profiler_kernels_one_round": prof_kernels},
        "results_equal": {"per_map_wave_vs_one_map_waves": one_ok, "per_map_wave_vs_solo_sample": bool(solo_ok),
                          "solo_sample": check, "default_wave_existing_vs_per_map_bytes": bool(bytes_equal)},
    }))


if __name__ == "__main__":
    main()
