"""MAACO sweeps over maps that have their own start and target: solve_maaco_batch(per_map_endpoints=True) against the
default grouping by (shape, start, target).  Config-5 maps (blocks_map(256, 0.20, seed=5000 + i), i < --maps), 1 024
ants x 10 passes, --wave maps per wave, all from host grids.  Two workloads:

  random_endpoints  start / target moved to seeded random free cells of each map: the per-map sweep over all maps,
                    and the default grouping -- one 1-map wave per map -- over a seeded sample of --grouped-sample maps
                    (labelled as a sample: its maps/s is that sample's)
  corners           the maps' own corners (one shared pair): the default sweep and the per-map sweep over all maps (the
                    per-map sweep then takes the shared table, so this shows what the opt-in costs on today's workload)

Every arm is timed with the host clock around the sweep (it ends in a device synchronise), --rounds rounds with the arms
alternated; medians and the spread (min..max) are reported.  For the per-map sweep on random endpoints it also reports,
per wave: the host table build (host clock around mpp_maaco_e01_host on the worker thread), the GPU time (CUDA events
from the wave's construction to the end of its solve) and the exposed host time between one wave's solve and the next
wave's construction (the wait for the tables plus the sweep's own overhead).  Result check: a seeded sample of
--check-sample maps of the per-map sweep against solo MAACO with the same seeds.  Prints one JSON line with the card's
name and power limit, read in the same run.  Needs a GPU; there is no fallback.

    python tools/maaco_endpoints_time.py [--maps 1250] [--wave 128] [--rounds 3] [--grouped-sample 64]
"""
import argparse
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


def moved(grids, seed):
    rng = np.random.default_rng(seed)
    out = grids.copy()
    for g in out:
        g[g >= 2] = 0
        s, t = rng.choice(np.flatnonzero(g.ravel() == 0), 2, replace=False)
        g.flat[s], g.flat[t] = 2, 3
    return out


class _Probe:
    """Per-wave timings of a per-map sweep: patches batch._e01_host and batch.MAACOBatch while active."""

    def __init__(self, batch):
        self.batch, self.table_s, self.gpu_ms, self.exposed_s = batch, [], [], []
        self._last_end = None

    def __enter__(self):
        b, probe = self.batch, self
        self._orig = (b._e01_host, b.MAACOBatch)
        host = b._e01_host

        def timed_tables(*a, **kw):
            t0 = time.perf_counter()
            out = host(*a, **kw)
            probe.table_s.append(time.perf_counter() - t0)
            return out

        class Timed(b.MAACOBatch):
            def __init__(self, *a, **kw):
                now = time.perf_counter()
                if probe._last_end is not None:
                    probe.exposed_s.append(now - probe._last_end)
                self._ev = torch.cuda.Event(enable_timing=True)
                self._ev.record()
                super().__init__(*a, **kw)

            def solve(self):
                out = super().solve()
                end = torch.cuda.Event(enable_timing=True)
                end.record()
                end.synchronize()
                probe.gpu_ms.append(self._ev.elapsed_time(end))
                probe._last_end = time.perf_counter()
                return out

        b._e01_host, b.MAACOBatch = timed_tables, Timed
        self._last_end = time.perf_counter()                 # the first wave's tables are fully exposed
        return self

    def __exit__(self, *exc):
        self.batch._e01_host, self.batch.MAACOBatch = self._orig


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--maps", type=int, default=1250)
    ap.add_argument("--wave", type=int, default=128)
    ap.add_argument("--ants", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--grouped-sample", type=int, default=64)
    ap.add_argument("--check-sample", type=int, default=8)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("maaco_endpoints_time.py measures the GPU: no CUDA device visible")
    torch.cuda.set_device(0)
    from maaco_path_planing_b200 import MAACO, blocks_map
    from maaco_path_planing_b200 import batch
    from maaco_path_planing_b200.batch import solve_maaco_batch
    name, power = card()
    M, N, K, W = args.maps, args.ants, args.iters, args.wave
    corners = np.stack([blocks_map(256, 0.20, seed=5000 + i) for i in range(M)])
    rand = moved(corners, 5000)
    seeds = list(range(M))
    sample = sorted(np.random.default_rng(64).choice(M, min(args.grouped_sample, M), replace=False).tolist())
    rand_sample = [rand[i] for i in sample]

    def sweep(grids, sd, per_map):
        t0 = time.perf_counter()
        out = solve_maaco_batch(grids, N, K, PARAMS, seeds=sd, wave=W, per_map_endpoints=per_map)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, out

    arms = {
        "random_per_map": lambda: sweep(rand, seeds, True),
        "random_grouped_sample": lambda: sweep(rand_sample, [seeds[i] for i in sample], False),
        "corners_default": lambda: sweep(corners, seeds, False),
        "corners_per_map": lambda: sweep(corners, seeds, True),
    }
    # warm-up: every arm's launch shapes (a full wave, 1-map waves, the table builder) once
    sweep(rand[:W], seeds[:W], True)
    sweep(rand_sample[:2], seeds[:2], False)
    sweep(corners[:W], seeds[:W], False)
    times = {k: [] for k in arms}
    results = {}
    probes = []
    order = list(arms)
    for r in range(args.rounds):
        for k in (order if r % 2 == 0 else order[::-1]):
            if k == "random_per_map":
                with _Probe(batch) as probe:
                    t, out = arms[k]()
                probes.append(probe)
            else:
                t, out = arms[k]()
            times[k].append(t)
            results[k] = out
    n_maps = {"random_per_map": M, "random_grouped_sample": len(sample), "corners_default": M, "corners_per_map": M}
    rate = {k: {"maps_per_s_median": n_maps[k] / statistics.median(v),
                "maps_per_s_min": n_maps[k] / max(v), "maps_per_s_max": n_maps[k] / min(v),
                "seconds": v, "maps": n_maps[k]} for k, v in times.items()}
    rate["random_grouped_sample"]["sample"] = f"{len(sample)} of {M} maps (seeded), one 1-map wave each"
    # results: the per-map sweep == the default grouping on the sample, == solo MAACO on a seeded sample, and the corners
    # sweeps agree with each other
    per_map = {r[0]: r[1:] for r in results["random_per_map"]}
    grouped_ok = all(per_map[i] == r[1:] for i, r in zip(sample, results["random_grouped_sample"]))
    check = sorted(np.random.default_rng(8).choice(M, min(args.check_sample, M), replace=False).tolist())
    solo_ok = True
    for i in check:
        m = MAACO(rand[i], N, K, rng_seed=seeds[i], verbose=False, **PARAMS)
        path, length, turns = m.solve_path_planning()
        solo_ok &= per_map[i] == (path, length, turns, m.convergence_curve_data)
    corners_ok = results["corners_default"] == results["corners_per_map"]
    med = lambda v: statistics.median(v) if v else None
    waves = len(probes[-1].gpu_ms)
    print(json.dumps({
        "tool": "maaco_endpoints_time", "card": name, "power_limit_w": power,
        "maps": M, "ants": N, "passes": K, "wave": W, "rounds": args.rounds, "host_cpus": os.cpu_count(),
        "arms": rate,
        "speedup_random_per_map_vs_grouped": rate["random_per_map"]["maps_per_s_median"] /
        rate["random_grouped_sample"]["maps_per_s_median"],
        "per_wave": {"waves": waves,
                     "host_table_ms_median": 1e3 * med([t for p in probes for t in p.table_s]),
                     "gpu_ms_median": med([t for p in probes for t in p.gpu_ms]),
                     "exposed_host_ms_median": 1e3 * med([t for p in probes for t in p.exposed_s]),
                     "exposed_host_ms_total_per_sweep": [1e3 * sum(p.exposed_s) for p in probes]},
        "results_equal": {"per_map_vs_grouped_sample": grouped_ok, "per_map_vs_solo_sample": bool(solo_ok),
                          "solo_sample": check, "corners_default_vs_per_map": corners_ok},
    }))


if __name__ == "__main__":
    main()
