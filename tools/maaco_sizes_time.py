"""MAACO colony-size / pass-count sweeps in one launch: MAACOBatch(map_sizes=...) against the waves a sweep needed
before per-map sizes.

  (a) --settings (num_ants, num_iterations) pairs (default 64: num_ants in 128..4096 x num_iterations in 5..40, every
      map its own seed) on one config-5 map, blocks_map(256, 0.20, seed=5000):
        sized_wave     one MAACOBatch of 64 copies of the map with map_sizes
        one_map_waves  one 1-map MAACOBatch per setting (a wave had to share its sizes), buffers reused where they fit
  (b) --maps config-5 maps (blocks_map(256, 0.20, seed=5000 + i)) x --grid-settings settings (default 16 x 16):
        sized_wave     one MAACOBatch of all 256 (map, setting) pairs with map_sizes
        setting_waves  one 16-map MAACOBatch per setting: what a sweep ran before per-map sizes

Each arm is timed with the host clock around the whole sweep (it ends in a device synchronise), --rounds rounds with the
arms alternated; medians and the spread (min..max) are reported as maps/s.  Result check: the sized wave's results equal
the other arm's on every map, and solo MAACO's on a seeded sample of (a).  Prints one JSON line with the card's name
and power limit, read in the same run.  Needs a GPU; there is no fallback.

    python tools/maaco_sizes_time.py [--rounds 2] [--check-sample 4]
"""
import argparse
import itertools
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

from maaco_params_time import PARAMS, card  # noqa: E402

ANTS = (128, 256, 512, 768, 1024, 1536, 2048, 4096)
PASSES = (5, 10, 15, 20, 25, 30, 35, 40)
GRID_ANTS = (256, 512, 1024, 2048)
GRID_PASSES = (5, 10, 20, 40)


def timed(arms, rounds):
    """Runs every arm `rounds` times, alternating the order; {arm: seconds per round}, {arm: last results}."""
    times, results = {k: [] for k in arms}, {}
    order = list(arms)
    for r in range(rounds):
        for k in (order if r % 2 == 0 else order[::-1]):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = arms[k]()
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)
            results[k] = out
    return times, results


def rates(times, n_maps):
    return {k: {"maps_per_s_median": n_maps / statistics.median(v), "maps_per_s_min": n_maps / max(v),
                "maps_per_s_max": n_maps / min(v), "seconds": v} for k, v in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--check-sample", type=int, default=4)
    ap.add_argument("--maps", type=int, default=16)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("maaco_sizes_time.py measures the GPU: no CUDA device visible")
    torch.cuda.set_device(0)
    from maaco_path_planing_b200 import MAACO, blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    name, power = card()

    # (a) one map, 64 size settings
    sizes = [{"num_ants": n, "num_iterations": k} for n, k in itertools.product(ANTS, PASSES)]
    P = len(sizes)
    g = blocks_map(256, 0.20, seed=5000)
    grids = np.stack([g] * P)
    seeds = list(range(P))
    prev = {}

    def sized_wave():
        b = MAACOBatch(grids, 1, 1, seeds=seeds, map_sizes=sizes, reuse=prev.get("wave"), **PARAMS)
        prev["wave"] = b
        return b.solve()

    def one_map_waves():
        out = []
        for k, s in enumerate(sizes):
            b = MAACOBatch(grids[k:k + 1], s["num_ants"], s["num_iterations"], seeds=[seeds[k]], reuse=prev.get("one"),
                           **PARAMS)
            out += b.solve()
            prev["one"] = b
        return out

    for f in (sized_wave, one_map_waves):                              # warm-up: every launch shape
        f()
    t_a, r_a = timed({"sized_wave": sized_wave, "one_map_waves": one_map_waves}, args.rounds)
    check = sorted(np.random.default_rng(8).choice(P, min(args.check_sample, P), replace=False).tolist())
    solo_ok = True
    for i in check:
        m = MAACO(g, sizes[i]["num_ants"], sizes[i]["num_iterations"], rng_seed=seeds[i], verbose=False, **PARAMS)
        path, length, turns = m.solve_path_planning()
        solo_ok &= r_a["sized_wave"][i] == (path, length, turns, m.convergence_curve_data)
    prev.clear()

    # (b) 16 maps x 16 size settings
    settings = [{"num_ants": n, "num_iterations": k} for n, k in itertools.product(GRID_ANTS, GRID_PASSES)]
    maps = [blocks_map(256, 0.20, seed=5000 + i) for i in range(args.maps)]
    pairs = [(m, s) for s in range(len(settings)) for m in range(len(maps))]          # grouped by setting
    grid_b = np.stack([maps[m] for m, _ in pairs])
    seeds_b = list(range(len(pairs)))
    sizes_b = [settings[s] for _, s in pairs]

    def sized_wave_b():
        b = MAACOBatch(grid_b, 1, 1, seeds=seeds_b, map_sizes=sizes_b, reuse=prev.get("wave"), **PARAMS)
        prev["wave"] = b
        return b.solve()

    def setting_waves():
        out = []
        for s, st in enumerate(settings):
            lo = s * len(maps)
            b = MAACOBatch(grid_b[lo:lo + len(maps)], st["num_ants"], st["num_iterations"],
                           seeds=seeds_b[lo:lo + len(maps)], reuse=prev.get("set"), **PARAMS)
            out += b.solve()
            prev["set"] = b
        return out

    for f in (sized_wave_b, setting_waves):
        f()
    t_b, r_b = timed({"sized_wave": sized_wave_b, "setting_waves": setting_waves}, args.rounds)
    prev.clear()

    ra, rb = rates(t_a, P), rates(t_b, len(pairs))
    print(json.dumps({
        "tool": "maaco_sizes_time", "card": name, "power_limit_w": power, "rounds": args.rounds,
        "a": {"map": "blocks_map(256, 0.20, seed=5000)", "settings": P, "num_ants": ANTS, "num_iterations": PASSES,
              "arms": ra, "speedup_sized_wave_vs_one_map_waves":
                  ra["sized_wave"]["maps_per_s_median"] / ra["one_map_waves"]["maps_per_s_median"],
              "results_equal": {"sized_wave_vs_one_map_waves": r_a["sized_wave"] == r_a["one_map_waves"],
                                "sized_wave_vs_solo_sample": bool(solo_ok), "solo_sample": check}},
        "b": {"maps": len(maps), "settings": len(settings), "num_ants": GRID_ANTS, "num_iterations": GRID_PASSES,
              "arms": rb, "speedup_sized_wave_vs_setting_waves":
                  rb["sized_wave"]["maps_per_s_median"] / rb["setting_waves"]["maps_per_s_median"],
              "results_equal": {"sized_wave_vs_setting_waves": r_b["sized_wave"] == r_b["setting_waves"]}},
    }))


if __name__ == "__main__":
    main()
