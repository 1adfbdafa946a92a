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
per wave: the GPU time (CUDA events from the wave's construction to the end of its solve) and the host time between one
wave's solve and the next wave's construction.  The device table time of one --wave-map wave (CUDA events around
mpp_maaco_e01_maps alone, --table-reps launches after a warm-up, median) is reported next to the host build of the same
tables (host clock around mpp_maaco_e01_host, default thread count).  Result check: a seeded sample of --check-sample maps
of the per-map sweep against solo MAACO with the same seeds.  Prints one JSON line with the card's name and power limit,
read in the same run.  Needs a GPU; there is no fallback.

--ab TREE compares two builds of the project instead: the random-endpoint per-map sweep from TREE (another checkout
whose library is built, e.g. the parent commit) and from this tree, --rounds rounds alternated, each run a fresh process
(`--gpus G`: G ranks under torchrun, maps sharded over them, time = the slowest rank's).

    python tools/maaco_endpoints_time.py [--maps 1250] [--wave 128] [--rounds 3] [--grouped-sample 64]
    python tools/maaco_endpoints_time.py --ab ../parent --maps 1250 [--gpus 8 --maps 10000]
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
    """Per-wave timings of a per-map sweep: patches batch.MAACOBatch while active."""

    def __init__(self, batch):
        self.batch, self.gpu_ms, self.exposed_s = batch, [], []
        self._last_end = None

    def __enter__(self):
        b, probe = self.batch, self
        self._orig = b.MAACOBatch

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

        b.MAACOBatch = Timed
        return self

    def __exit__(self, *exc):
        self.batch.MAACOBatch = self._orig


def table_times(grids, reps):
    """(device ms, host ms): mpp_maaco_e01_maps on one wave of `grids` (CUDA events, median of `reps` launches after a
    warm-up) and mpp_maaco_e01_host on the same maps (host clock, median of 3)."""
    import ctypes as C
    from maaco_path_planing_b200 import _lib
    from maaco_path_planing_b200.batch import _e01_host, _maaco_params, _map_set
    p = _maaco_params(1, **PARAMS)
    maps = _map_set(grids)
    M, n = len(grids), grids[0].size
    e01 = torch.empty((M, 2 * n), dtype=torch.float64, device="cuda")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    launch = lambda: _lib.check(_lib.lib().mpp_maaco_e01_maps(maps.handle, C.byref(p), _lib.ptr(e01), 2 * n, stream),
                                "mpp_maaco_e01_maps")
    launch()
    dev = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        launch()
        b.record()
        b.synchronize()
        dev.append(a.elapsed_time(b))
    host = []
    out = torch.empty(M * 2 * n, dtype=torch.float64, pin_memory=True)
    for _ in range(3):
        t0 = time.perf_counter()
        _e01_host(*grids[0].shape, maps.start, maps.target, p, out)
        host.append(1e3 * (time.perf_counter() - t0))
    same = out.numpy().tobytes() == e01.cpu().numpy().tobytes()
    maps.close()
    return statistics.median(dev), statistics.median(host), same


def child(tree, maps, ants, iters, wave):
    """One per-map sweep over the random-endpoint maps from the project at `tree`; prints {"seconds", "digest"} (rank 0;
    under torchrun the slowest rank's time)."""
    sys.path.insert(0, os.path.abspath(tree))
    import hashlib
    group = None
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
        dist.init_process_group("nccl")
        group = dist.group.WORLD
    else:
        torch.cuda.set_device(0)
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import shard_maps, solve_maaco_batch
    lo, hi = shard_maps(maps, group)
    grids = [None] * maps
    shard = moved(np.stack([blocks_map(256, 0.20, seed=5000 + i) for i in range(lo, hi)]), 5000 + lo)
    grids[lo:hi] = list(shard)
    for i in range(maps):                                     # other ranks' maps: only their shape is read
        if grids[i] is None:
            grids[i] = shard[0]
    solve_maaco_batch(grids[lo:lo + wave] if group is None else grids, ants, 1, PARAMS, seeds=list(range(maps)),
                      wave=wave, group=group, per_map_endpoints=True)       # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = solve_maaco_batch(grids, ants, iters, PARAMS, seeds=list(range(maps)), wave=wave, group=group,
                            per_map_endpoints=True)
    torch.cuda.synchronize()
    t = torch.tensor([time.perf_counter() - t0], device="cuda")
    digest = hashlib.sha256(repr(out).encode()).hexdigest()
    if group is not None:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        digests = [None] * dist.get_world_size()
        dist.all_gather_object(digests, digest)
        digest = hashlib.sha256("".join(digests).encode()).hexdigest()
        dist.destroy_process_group()
    if int(os.environ.get("RANK", "0")) == 0:
        print(json.dumps({"seconds": float(t.item()), "digest": digest}), flush=True)


def ab(args):
    """Alternate child sweeps of the tree at args.ab ("parent") and this tree ("new")."""
    trees = {"parent": os.path.abspath(args.ab), "new": ROOT}
    me = os.path.abspath(__file__)
    times = {k: [] for k in trees}
    digests = {k: set() for k in trees}
    for r in range(args.rounds):
        for k in (("parent", "new") if r % 2 == 0 else ("new", "parent")):
            cmd = [sys.executable, me]
            if args.gpus > 1:
                cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc_per_node={args.gpus}",
                       me]
            cmd += ["--child", trees[k], "--maps", str(args.maps), "--ants", str(args.ants), "--iters", str(args.iters),
                    "--wave", str(args.wave)]
            res = subprocess.run(cmd, capture_output=True, text=True, cwd=trees[k])
            line = [l for l in res.stdout.splitlines() if l.startswith("{")]
            if res.returncode != 0 or not line:
                raise SystemExit(f"{k} run failed ({res.returncode}):\n{res.stdout[-2000:]}\n{res.stderr[-4000:]}")
            d = json.loads(line[-1])
            times[k].append(d["seconds"])
            digests[k].add(d["digest"])
    name, power = card()
    rate = {k: {"maps_per_s_median": args.maps / statistics.median(v), "maps_per_s_min": args.maps / max(v),
                "maps_per_s_max": args.maps / min(v), "seconds": v} for k, v in times.items()}
    print(json.dumps({"tool": "maaco_endpoints_time", "mode": "ab", "card": name, "power_limit_w": power,
                      "gpus": args.gpus, "maps": args.maps, "ants": args.ants, "passes": args.iters, "wave": args.wave,
                      "rounds": args.rounds, "host_cpus": os.cpu_count(), "arms": rate,
                      "speedup_new_vs_parent": rate["new"]["maps_per_s_median"] / rate["parent"]["maps_per_s_median"],
                      "results_equal": len(digests["parent"] | digests["new"]) == 1}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--maps", type=int, default=1250)
    ap.add_argument("--wave", type=int, default=128)
    ap.add_argument("--ants", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--grouped-sample", type=int, default=64)
    ap.add_argument("--check-sample", type=int, default=8)
    ap.add_argument("--table-reps", type=int, default=20)
    ap.add_argument("--ab", default=None)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--child", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        return child(args.child, args.maps, args.ants, args.iters, args.wave)
    if args.ab:
        return ab(args)
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
    table_dev_ms, table_host_ms, tables_equal = table_times(rand[:W], args.table_reps)
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
        "tables_one_wave": {"maps": min(W, M), "device_ms_median": table_dev_ms, "host_ms_median": table_host_ms,
                            "host_threads": min(16, os.cpu_count() or 1), "device_equals_host": tables_equal},
        "per_wave": {"waves": waves,
                     "gpu_ms_median": med([t for p in probes for t in p.gpu_ms]),
                     "exposed_host_ms_median": 1e3 * med([t for p in probes for t in p.exposed_s]),
                     "exposed_host_ms_total_per_sweep": [1e3 * sum(p.exposed_s) for p in probes]},
        "results_equal": {"per_map_vs_grouped_sample": grouped_ok, "per_map_vs_solo_sample": bool(solo_ok),
                          "solo_sample": check, "corners_default_vs_per_map": corners_ok},
    }))


if __name__ == "__main__":
    main()
