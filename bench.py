#!/usr/bin/env python
"""bench.py -- path evaluations / second of the B200 hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Default workload (N=1): BASELINE config 4 -- MAACO, 4096 ants on a 512x512 synthetic block map
(`blocks(512, 0.20, seed=4000)`), parameters of main.py:34-38.  One *step* = one colony pass
(move ranking + tour construction for every ant + best tracking + pheromone update); one path evaluation = one
`_construct_ant_solution_maaco` call incl. its share of the pheromone update (SURVEY 8(d)).
N>1 (torchrun): one process per GPU, the colony is sharded with 4096 ants per GPU (weak scaling) and exchanges one
buffer of move codes + tau slices per pass; the same run also reports the fixed 4096-ant colony (strong scaling)
and BASELINE config 5 (independent maps sharded over the ranks, no collective) under "extra", and checks that the
sharded colony reproduces a single-GPU replay bit for bit ("parity_check").

`--dump-outputs DIR` writes what the last timed pass handed its caller to DIR/<name>.npy (finite float64: -1 stands for
the length of a failed tour; 64 MiB at most), so that two builds can be compared output for output: the inputs depend
only on the arguments.

`--impl reference` times the UNMODIFIED Python reference (baseline/_ref, copied there by build(); one single-threaded
interpreter per host core) on bounded samples of the same workload, and reports the CPU oracle port
(oracle/mpp_oracle.c, OpenMP over ants, every host thread) beside it (`cpu_baseline.port`); without the reference
tree the port is the arm.  The GPU arm's `cpu_baseline` has the same shape (kind "reference" + `port`).
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MAACO_PARAMS = dict(alpha=1.0, beta=7.0, rho=0.1, Q=2.5, a_turn_coef=1.0, wh_max=0.9, wh_min=0.2,
                    k_h_adaptive=0.9, q0_initial=0.5, C0_initial_pheromone=0.1)   # main.py:34-38
MPA_PARAMS = dict(FADs_rate=0.2, P_const=0.5, levy_beta=2.0, turn_penalty_factor=0.1, safety_penalty_factor=0.8,
                  min_safe_distance=1.8, diagonal_obstacle_penalty=100.0)          # main.py:44-52
BYTES_PER_ANT_STEP = 148          # SURVEY 8(d): 8x8 B tau + 8x8 B E-table + 2x8 B uniforms + 4 B path cell
METRIC = "path evals/sec (MAACO ant tours, MPA/PSO/GA fitness) at 1/2/4/8 B200 vs CPU"
CORES = os.cpu_count() or 1


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for _, r in self.rows]
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arms.  (The only place bench.py touches oracle/: as the thing timed on the host, never on the GPU path.)
# ------------------------------------------------------------------------------------------------
def _oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle as O
    return O


def cpu_maaco(grid, n_ants, seconds_budget, threads, max_passes=4096):
    """The C port of the colony pass (OpenMP over ants; `threads` is passed explicitly: torchrun exports
    OMP_NUM_THREADS=1)."""
    O = _oracle()
    orc = O.MaacoOracle(grid, n_ants, 100, seed=4, threads=threads, max_cells=min(grid.size, 8 * sum(grid.shape)),
                        **MAACO_PARAMS)
    orc.iterate(1)                                    # warm-up pass (page faults, OpenMP pool)
    t0 = time.perf_counter()
    passes, it = 0, 2
    steps0 = orc.total_steps
    while True:
        orc.iterate(it)
        it = it + 1 if it < 100 else 2                # (the schedule of q0 has 100 iterations: stay inside it)
        passes += 1
        dt = time.perf_counter() - t0
        if dt >= seconds_budget or passes >= max_passes:
            break
    return {"evals": passes * n_ants, "seconds": dt, "passes": passes, "ant_steps": orc.total_steps - steps0}


def ref_python(kind, size, map_seed, seconds, procs=None):
    """The UNMODIFIED Python reference (baseline/_ref or /root/reference) timed by oracle/ref_timing.py, one process
    per host core.  Returns None when no reference tree is present."""
    procs = procs or CORES
    have = any(os.path.isfile(os.path.join(d, "MAACO.py")) for d in
               (os.environ.get("MAACO_REF_DIR") or "/nonexistent", "/root/reference", os.path.join(ROOT, "baseline", "_ref")))
    if not have:
        return None
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_timing.py"), kind, str(size), str(map_seed), str(seconds)]
    env = dict(os.environ, OMP_NUM_THREADS="1", OPENBLAS_NUM_THREADS="1", MKL_NUM_THREADS="1")
    t0 = time.perf_counter()
    ps = [subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, env=env) for _ in range(procs)]
    outs = []
    for p in ps:
        o, _ = p.communicate()
        try:
            outs.append(json.loads(o.strip().splitlines()[-1]))
        except (ValueError, IndexError):
            pass
    wall = time.perf_counter() - t0
    if not outs:
        return None
    evals = sum(o["evals"] for o in outs)
    per_core = statistics.median(o["evals"] / o["seconds"] for o in outs)
    return {"value": sum(o["evals"] / o["seconds"] for o in outs), "unit": "path evals/s", "cores": len(outs),
            "one_core_value": per_core, "kind": "reference",
            "sample": f"{evals} evaluations by {len(outs)} concurrent single-threaded processes of the unmodified Python "
                      f"reference, {seconds:.0f} s each ({wall:.0f} s wall incl. interpreter start + table build)"}


def workload_config(args, world, total):
    """The same dict in both arms (the driver compares them); how the GPU arm exchanges is reported under "exchange"."""
    return {"workload": f"MAACO colony pass, {total} ants ({total // world}/GPU) on {args.size}x{args.size} "
                        f"blocks(n,0.20,seed=4000), params main.py:34-38 (BASELINE config 4)",
            "ants_total": total, "grid": [args.size, args.size], "l2": "flushed (256 MiB write) between timed steps",
            "parallelism": f"colony sharded over {world} GPU(s)"}


def exchange_note(world, p2p):
    if world == 1:
        return "none (one GPU)"
    return ("the tour kernel stores every visited-set slab straight into the rank that updates its tile row and the update "
            "kernel its tau slice into every rank (NVLink peer memory, two device-side barriers per pass: no pack / "
            "all-gather / replay)" if p2p else
            "per pass one all-gather of results + move codes and one all-gather of tau slices (NCCL)")


def run_reference(args):
    """`--impl reference`: only rank 0 works; the others exit 0.  Same total ant count as the GPU arm at this N."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from maaco_path_planing_b200.gridmap import blocks_map
    world = max(1, int(os.environ.get("WORLD_SIZE", str(args.gpus))))
    total = args.ants * world
    grid = blocks_map(args.size, 0.20, seed=4000)
    per_step = max(1.0, min(20.0, 60.0 / max(1, args.steps + args.warmup)))
    # The reference is Python: when its tree travelled with the repo (baseline/_ref, copied by build()), the arm times the
    # UNMODIFIED code (one single-threaded interpreter per host core: the reference has no threading of its own); the C
    # port is then reported beside it.  Without the tree the port is all there is.
    port = cpu_maaco(grid, total, min(per_step, 4.0), CORES)
    port_v = port["evals"] / port["seconds"]
    port_d = {"value": port_v, "unit": "path evals/s", "cores": CORES, "kind": "port",
              "sample": f"{port['passes']} colony passes of {total} ants, C port of the reference's colony pass, OpenMP over "
                        f"ants on {CORES} threads, {port['seconds']:.1f} s"}
    rp = ref_python("maaco", args.size, 4000, 1.0)                     # (also the warm-up: page cache, .pyc files)
    if rp:
        for _ in range(max(0, args.warmup - 1)):
            ref_python("maaco", args.size, 4000, 1.0)
        vals, cores, evals = [], rp["cores"], 0
        t0 = time.perf_counter()
        for _ in range(args.steps):
            r = ref_python("maaco", args.size, 4000, per_step)
            if r:
                vals.append(r["value"])
                cores = r["cores"]
                evals += int(r["sample"].split()[0])
        wall = time.perf_counter() - t0
        v = statistics.mean(vals)
        ms_step = 1e3 * wall / max(1, args.steps)
        cb = {"value": v, "unit": "path evals/s", "cores": cores, "kind": "reference",
              "sample": f"{args.steps} samples of {per_step:.1f} s on each of {cores} concurrent single-threaded processes of the "
                        f"unmodified Python reference ({evals} tours by MAACO._construct_ant_solution_maaco + one "
                        f"_update_pheromone_trails_maaco per process, charged per tour; same map and parameters)",
              "port": port_d}
    else:
        for _ in range(args.warmup):
            cpu_maaco(grid, total, 0.0, CORES, max_passes=1)
        tot_e, tot_s = 0, 0.0
        for _ in range(args.steps):
            r = cpu_maaco(grid, total, per_step, CORES)
            tot_e += r["evals"]
            tot_s += r["seconds"]
        v = tot_e / tot_s
        ms_step = 1e3 * tot_s / max(1, args.steps)
        cb = dict(port_d, value=v, sample=f"{tot_e // total} colony passes of {total} ants on blocks({args.size},0.20,4000), C port "
                                          f"of the reference's colony pass, OpenMP over ants on {CORES} threads")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "path evals/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world, total),
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "path evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def time_colony(solver, K, W, flush, sync_all, it0=0):
    """W warm-up passes + K timed passes with per-kernel CUDA events; returns (per-pass event times, first free it)."""
    import torch
    it = it0
    for _ in range(W):
        it += 1
        solver.run_iteration(it)
    solver._settle()
    sync_all()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(K)]
    sync_all()
    for k in range(K):
        flush.fill_(k & 0xff)                                   # evict L2 between timed steps (untimed)
        it += 1
        solver._enqueue_iteration(it, events=ev[k])             # events: start / after tours / before pheromone / end / after ranking
    solver._settle()
    sync_all()
    return ev, it


# --dump-outputs: bytes each array may take (64 MiB in all); a larger one is written as a seeded sample of its rows
DUMP_BUDGETS = {"ant_n_cells": 2 << 20, "ant_length": 2 << 20, "ant_turns": 2 << 20, "ant_tours": 32 << 20,
                "pheromone": 24 << 20, "best": 1 << 10, "best_path": 1 << 20}


def last_pass_outputs(solver):
    """What the last colony pass handed a caller of MAACO.run_iteration: every ant's record and tour (last_tours; a
    tour is -1 past its last cell; with N>1 GPUs the tours of this rank's ants), the pheromone field and the best
    length / turns / cell count / path so far.  A length is -1 where the caller receives inf (no tour reached the
    target), as the turns already are, so that every value written is finite.  Collective when the colony is sharded
    (the best path lives on the rank whose ant found it)."""
    import numpy as np
    nc, ln, tn, cells = solver.last_tours()
    cells[np.arange(cells.shape[1])[None, :] >= nc[:, None]] = -1
    ln[~np.isfinite(ln)] = -1.0
    st = solver._read_state()
    if not np.isfinite(st.best_len):
        st.best_len = -1.0
    n_best = min(st.best_n_cells, solver._best_cells.numel())
    if solver.world > 1 and n_best > 0:
        import torch.distributed as dist
        owner = dist.get_global_rank(solver.group, st.best_ant // solver.n_local)
        dist.broadcast(solver._best_cells, src=owner, group=solver.group)
    return {"ant_n_cells": nc, "ant_length": ln, "ant_turns": tn, "ant_tours": cells,
            "pheromone": solver.pheromone_matrix, "best": [st.best_len, st.best_turns, st.best_n_cells],
            "best_path": solver._best_cells[:n_best].cpu().numpy()}


def save_outputs(out_dir, arrays, budgets):
    """arrays[name] -> out_dir/<name>.npy in float64.  An array above budgets[name] bytes is replaced by the rows (first
    axis) of a fixed, seeded sample that fits, and their indices go to <name>_rows.npy.  Every value must be finite."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        if not np.isfinite(a).all():
            raise ValueError(f"--dump-outputs: {name} has values that are not finite")
        row_bytes = 8 * (a.size // max(1, a.shape[0]))
        if row_bytes * a.shape[0] > budgets[name]:
            k = budgets[name] // (row_bytes + 8)
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], k, replace=False))
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def run_gpu(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from maaco_path_planing_b200 import MAACO, blocks_map

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        group = dist.group.WORLD
    dev = torch.device("cuda", local)
    total_ants = args.ants * world
    grid = blocks_map(args.size, 0.20, seed=4000)
    K, W = args.steps, args.warmup
    n = args.size * args.size
    solver = MAACO(grid, total_ants, K + W + 64, rng_seed=4, device=local, group=group, verbose=False, **MAACO_PARAMS)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier(group=group)
            torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
        return float(t.item())

    it = 0
    for _ in range(W):                                              # warm-up passes (untimed)
        it += 1
        solver.run_iteration(it)
    steps_before = solver.total_steps()
    launches_before = solver.kernel_launches
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    t_wall0 = time.time()
    ev, it = time_colony(solver, K, 0, flush, sync_all, it0=it)
    t_wall1 = time.time()
    step_ms = [e[0].elapsed_time(e[3]) for e in ev]
    tour_ms = [e[4].elapsed_time(e[1]) for e in ev]             # the tour kernel alone
    rank_ms = [e[0].elapsed_time(e[4]) for e in ev]             # the move-ranking kernel before it
    pher_ms = [e[2].elapsed_time(e[3]) for e in ev]             # pheromone update (N>1: + the tau all-gather)
    total_ms = max_over_ranks(sum(step_ms))
    ant_steps_local = solver.total_steps() - steps_before
    launches_timed = solver.kernel_launches - launches_before      # kernels of this library inside the timed region
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    nc_last, _, _ = solver.last_results()
    path_cells = int(nc_last[nc_last > 0].sum())                   # cells that receive a deposit in one pass
    if args.dump_outputs:                                          # before the e2e passes below move the colony on
        outputs = last_pass_outputs(solver)
        if rank == 0:
            save_outputs(args.dump_outputs, outputs, DUMP_BUDGETS)

    # ---- e2e: the colony pass through the host-buffer entry point (MAACO.run_iteration_host -> C ABI
    #      mpp_maaco_pass_host): pinned host pheromone field in; per-ant records, best path, updated field out ----
    e2e = None
    if world == 1:
        tau_host = torch.empty(n, dtype=torch.float64).pin_memory()
        tau_host.copy_(solver._tau[:n].cpu())
        res_host = torch.empty((total_ants, 2), dtype=torch.int64).pin_memory()
        best_host = torch.empty(8192, dtype=torch.int32).pin_memory()
        K2 = max(3, min(K, 10))
        sync_all()
        t0 = time.perf_counter()
        for _ in range(K2):
            it += 1
            solver.run_iteration_host(it, tau_in=tau_host, tau_out=tau_host, result_out=res_host, best_out=best_host)
        e2e_s = time.perf_counter() - t0
        e2e = {"value": total_ants * K2 / e2e_s, "unit": "path evals/s", "h2d_bytes_per_step": n * 8,
               "d2h_bytes_per_step": n * 8 + total_ants * 16 + 8192 * 4 + 40, "steps": K2,
               "note": "MAACO.run_iteration_host -> mpp_maaco_pass_host: host pheromone field in; per-ant results, "
                       "colony state, best path and updated field out, synchronous, every pass"}
    else:
        # a sharded colony keeps tau on the devices (it is exchanged between them every pass); end to end = the
        # device-resident passes + reading every pass's per-ant results back to pinned host memory
        res_host = torch.empty((total_ants, 2), dtype=torch.int64).pin_memory()
        K2 = max(3, min(K, 10))
        sync_all()
        t0 = time.perf_counter()
        for _ in range(K2):
            it += 1
            solver.run_iteration(it)
            res_host.copy_(solver._result, non_blocking=True)
        solver._settle()
        sync_all()
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": total_ants * K2 / e2e_s, "unit": "path evals/s", "h2d_bytes_per_step": 0,
               "d2h_bytes_per_step": total_ants * 16, "steps": K2,
               "note": "sharded colony: tau stays on the devices; every pass's per-ant results are read to pinned host memory"}

    parity = parity_check(args, grid, world, rank, local, group, dev)

    extra = {}
    if world > 1:
        extra["strong_scaling"] = strong_scaling(args, grid, world, rank, local, group, dev, flush, sync_all, max_over_ranks)
    if not args.no_extra:
        extra.update(side_workloads(args, dev, world, rank, group, max_over_ranks, sync_all))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = peaks()
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if world == 1 and args.ants == 4096 and args.size == 512 and os.path.exists(tp):
        traffic = json.load(open(tp)).get("mpp_maaco_tour1_kernel", {}).get("dram_bytes_per_launch")   # committed ncu capture
    value = total_ants * K / (total_ms / 1e3)
    tour_avg_ms = sum(tour_ms) / K
    achieved = BYTES_PER_ANT_STEP * (ant_steps_local / K) / (tour_avg_ms / 1e3) / 1e9
    pher_bytes = 16.0 * n + 12.0 * path_cells + 16.0 * total_ants         # SURVEY 8(d): K3 bytes per pass
    out = {
        "metric": METRIC, "value": value, "unit": "path evals/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world, total_ants),
        "exchange": exchange_note(world, getattr(solver, "_p2p", None) is not None),
        "e2e": e2e,
        "gpu_launches": launches_timed,
        "clocks": clocks,
        "parity_check": parity,
        "roofline": {"bound": "hbm", "kernel": "mpp_maaco_tour1_kernel", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_unit": BYTES_PER_ANT_STEP, "units_per_launch": ant_steps_local / K,
                     "kernel_ms": tour_avg_ms,
                     "rank_kernel_ms": sum(rank_ms) / K,
                     "pheromone_kernel": {"kernel": "mpp_maaco_pheromone_kernel" + ("" if world == 1 else " + tau exchange"),
                                          "ms": sum(pher_ms) / K, "algorithmic_bytes": pher_bytes,
                                          "achieved": pher_bytes / (sum(pher_ms) / K / 1e3) / 1e9, "unit": "GB/s",
                                          "frac": pher_bytes / (sum(pher_ms) / K / 1e3) / 1e9 / peak,
                                          "model": "16*R*C + 12*sum(path cells) + 16*N bytes per pass (SURVEY 8(d) K3)"}},
        "ant_steps_per_s": ant_steps_local * world / (total_ms / 1e3),
    }
    if world == 1 and not args.no_cpu:
        r = cpu_maaco(grid, args.ants, 12.0, CORES)
        port = {"value": r["evals"] / r["seconds"], "unit": "path evals/s", "cores": CORES, "kind": "port",
                "sample": f"{r['passes']} colony passes of {args.ants} ants (same map/params), C port of "
                          f"the reference's colony pass, OpenMP over ants, {r['seconds']:.1f} s",
                "ant_steps_per_s": r["ant_steps"] / r["seconds"]}
        r1 = cpu_maaco(grid, args.ants, 4.0, 1)
        port["one_core_value"] = r1["evals"] / r1["seconds"]
        rp = ref_python("maaco", args.size, 4000, 12.0)
        # the reference itself when its tree is here (kind "reference"), the C port beside it; else the port alone
        out["cpu_baseline"] = dict(rp, port=port) if rp else port
    if extra:
        out["extra"] = extra
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    if isinstance(parity, str) and not parity.startswith("ok"):
        sys.exit(3)


def _digest(solver):
    import torch
    n = solver.rows * solver.cols
    solver._settle()
    h = hashlib.sha256()
    h.update(solver._result.cpu().numpy().tobytes())
    h.update(solver._tau[:n].cpu().numpy().tobytes())
    h.update(solver._state.cpu().numpy().tobytes()[:24])        # best_len, best_turns, best_n_cells, best_iter, best_ant
    return h.digest()


def parity_check(args, grid, world, rank, local, group, dev):
    """2 colony passes of a fresh colony: N=1 -> per-ant records + pheromone field + best state bit-identical to the C
    oracle; N>1 -> every rank's (records, field, state) SHA-256 identical to a single-GPU replay of the SAME colony
    (all N x 4096 ants) on rank 0."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from maaco_path_planing_b200 import MAACO
    total = args.ants * world
    seed = 20262
    try:
        s = MAACO(grid, total, 4, rng_seed=seed, device=local, group=group, verbose=False, **MAACO_PARAMS)
        for it in (1, 2):
            s.run_iteration(it)
        mine = _digest(s)
        if world == 1:
            O = _oracle()
            orc = O.MaacoOracle(grid, total, 4, seed=seed, threads=CORES, max_cells=min(grid.size, 8 * sum(grid.shape)),
                                **MAACO_PARAMS)
            for it in (1, 2):
                _, onc, oln, otn, _ = orc.iterate(it)
            nc, ln, tn = s.last_results()
            ok = (np.array_equal(nc, onc) and np.array_equal(ln, oln) and np.array_equal(tn, otn)
                  and np.array_equal(s.pheromone_matrix.ravel(), orc.tau) and s._read_state().best_len == orc.best_len)
            return "ok (2 passes of a fresh 4096-ant colony: records, pheromone field, best bit-identical to the C oracle)" \
                if ok else "MISMATCH vs the C oracle"
        del s
        torch.cuda.empty_cache()
        digs = torch.zeros((world, 32), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(digs, torch.frombuffer(bytearray(mine), dtype=torch.uint8).to(dev), group=group)
        verdict = torch.zeros(1, dtype=torch.int32, device=dev)
        if rank == 0:
            one = MAACO(grid, total, 4, rng_seed=seed, device=local, verbose=False, **MAACO_PARAMS)
            for it in (1, 2):
                one.run_iteration(it)
            want = torch.frombuffer(bytearray(_digest(one)), dtype=torch.uint8).to(dev)
            verdict[0] = int(bool((digs == want[None, :]).all().item()))
            del one
        dist.broadcast(verdict, src=0, group=group)
        torch.cuda.empty_cache()
        return (f"ok (2 passes: records + pheromone field + best state of all {world} ranks SHA-256-identical to a "
                f"single-GPU replay of the same {total}-ant colony)") if int(verdict.item()) else \
            "MISMATCH: sharded colony differs from the single-GPU replay"
    except Exception as e:                                        # noqa: BLE001 -- the bench line must still be printed
        return f"ERROR: {type(e).__name__}: {e}"


def strong_scaling(args, grid, world, rank, local, group, dev, flush, sync_all, max_over_ranks):
    """BASELINE config 4 as written: the SAME 4096-ant colony sharded over the GPUs (fixed total work)."""
    from maaco_path_planing_b200 import MAACO
    K, W = max(5, min(args.steps, 20)), 3
    s = MAACO(grid, args.ants, K + W + 8, rng_seed=4, device=local, group=group, verbose=False, **MAACO_PARAMS)
    ev, _ = time_colony(s, K, W, flush, sync_all)
    ms = max_over_ranks(sum(e[0].elapsed_time(e[3]) for e in ev)) / K
    tour = sum(e[4].elapsed_time(e[1]) for e in ev) / K
    return {"workload": f"the fixed {args.ants}-ant colony of BASELINE config 4 sharded over {world} GPUs "
                        f"({args.ants // world} ants/GPU)", "value": args.ants / (ms / 1e3), "unit": "path evals/s",
            "ms_per_step": ms, "tour_kernel_ms": tour, "scaling": "strong",
            "note": "a pass lasts as long as its longest tour (a dependent chain), however few ants a GPU holds: "
                    "sharding a 4096-ant colony only adds the exchange"}


def side_workloads(args, dev, world, rank, group, max_over_ranks, sync_all):
    """The other configs of BASELINE.json, each with its own CPU baseline (N=1) -- reported under "extra"; the headline
    stays the MAACO colony.  config 3: PSO/GA A*-connector fitness (512x512, N=4096, W=5, policy main.py:21-24);
    config 2: MPA (100x100, N=1024, 100 iterations, params main.py:44-52); config 5: independent 256x256 maps x 1024
    ants (MAACO), maps sharded over the ranks."""
    import numpy as np
    import torch
    from maaco_path_planing_b200 import GridMap, blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch, shard_maps
    out = {}
    peak, _ = peaks()
    # ---- config 5: waves of independent maps, one launch per colony pass of the whole wave; maps sharded over ranks ----
    n_maps, ants, iters, wave = args.batch_maps * world, 1024, args.batch_iters, args.batch_wave
    lo, hi = shard_maps(n_maps, group)
    all_grids = np.stack([blocks_map(256, 0.20, seed=5000 + i) for i in range(lo, hi)])   # the input data (host, untimed)
    b = MAACOBatch(all_grids[:wave], ants, iters, seeds=list(range(lo, lo + min(wave, hi - lo))), **MAACO_PARAMS)
    b.run_iteration(1)                                                     # warm-up pass (module load, allocations)
    torch.cuda.synchronize()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    dev_ms, solved, steps = 0.0, 0, 0
    for w0 in range(lo, hi, wave):
        idx = list(range(w0, min(hi, w0 + wave)))
        b = MAACOBatch(all_grids[w0 - lo:w0 - lo + len(idx)], ants, iters, seeds=idx, reuse=b, **MAACO_PARAMS)   # H2D + tables
        e0.record()
        res = b.solve()
        e1.record()
        torch.cuda.synchronize()
        dev_ms += e0.elapsed_time(e1)
        solved += sum(1 for r in res if r[0])
        steps += b.total_steps()
        b.close()
    wall = max_over_ranks(time.perf_counter() - t0)
    dev_s = max_over_ranks(dev_ms / 1e3)
    tot = torch.tensor([solved, steps], dtype=torch.int64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(tot, group=group)
    evals = n_maps * ants * iters
    out["batched_maps"] = {
        "workload": f"{n_maps} independent 256x256 blocks maps x {ants} ants x {iters} MAACO iterations "
                    f"({n_maps // world} maps/GPU in waves of {wave}: one launch per colony pass of a wave, grid.y = map; "
                    "BASELINE config 5, MAACO part)",
        "value": evals / dev_s, "unit": "path evals/s", "maps_per_s": n_maps / dev_s, "seconds_device": dev_s,
        "e2e": {"value": evals / wall, "unit": "path evals/s", "maps_per_s": n_maps / wall, "seconds": wall,
                "note": "from host grids: map upload + bit-packing, shared host table build, all passes, result read-back "
                        "and path decoding, per wave"},
        "ant_steps_per_s": int(tot[1]) / dev_s, "solved_maps": int(tot[0]), "scaling": "weak",
        "roofline": {"bound": "hbm", "kernel": "whole pass (rank + tours + best + pheromone)",
                     "achieved": BYTES_PER_ANT_STEP * int(tot[1]) / dev_s / 1e9 / world, "peak": peak, "unit": "GB/s",
                     "frac": BYTES_PER_ANT_STEP * int(tot[1]) / dev_s / 1e9 / world / peak,
                     "algorithmic_bytes_per_unit": BYTES_PER_ANT_STEP}}
    # ---- config 5, MPA part: the same maps, MPA populations of 1024 paths, a bounded number of maps / iterations ----
    from maaco_path_planing_b200.batch import MPABatch
    mw, mit = min(args.mpa_batch_maps, hi - lo), args.mpa_batch_iters
    sync_all()
    t0 = time.perf_counter()
    mb = MPABatch(all_grids[:mw], 1024, mit, seeds=list(range(lo, lo + mw)), **MPA_PARAMS)
    mres = mb.solve()
    torch.cuda.synchronize()
    mwall = max_over_ranks(time.perf_counter() - t0)
    mexp = torch.tensor([mb.expansions], dtype=torch.int64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(mexp, group=group)
    out["batched_maps_mpa"] = {
        "workload": f"{mw * world} independent 256x256 blocks maps x 1024 predators x {mit} MPA iterations ({mw} maps/GPU in one "
                    "wave: one launch per iteration for every map; BASELINE config 5, MPA part; from host grids, incl. "
                    "the initial searches and the result read-back = end to end)",
        "value": mw * world * 1024 * mit / mwall, "unit": "predator-iterations/s", "seconds": mwall,
        "astar_expansions_per_s": int(mexp.item()) / mwall, "solved_maps": sum(1 for r in mres if r[0]), "scaling": "weak"}
    mb.close()
    del mb
    torch.cuda.empty_cache()
    if world > 1 or rank != 0:
        return out
    if not args.no_cpu:
        O = _oracle()
        nmaps_cpu = 32
        t0 = time.perf_counter()
        for i in range(nmaps_cpu):
            orc = O.MaacoOracle(blocks_map(256, 0.20, seed=5000 + i), ants, iters, seed=i, threads=CORES, **MAACO_PARAMS)
            orc.solve()
        dt = time.perf_counter() - t0
        out["batched_maps"]["cpu_baseline"] = {"value": nmaps_cpu * ants * iters / dt, "unit": "path evals/s", "cores": CORES, "kind": "port",
                                               "sample": f"{nmaps_cpu} of the maps one after the other, {iters} iterations x {ants} ants each, "
                                                         f"C port (map + tables + passes, OpenMP over ants), {dt:.1f} s"}
    # ---- config 3: fitness evaluation of a population of random free-cell waypoint chromosomes ----
    from maaco_path_planing_b200.engine import SearchEngine, make_policy
    size, N, Wp = args.fit_size, args.fit_pop, 5
    grid = blocks_map(size, 0.20, seed=3000 + size)
    rng = np.random.default_rng(3)
    free = np.flatnonzero(grid.ravel() != 1)
    eng = SearchEngine(GridMap(grid))
    pol = make_policy(0.3, 0.8, 1.8, 100.0)
    wps_host = [free[rng.integers(0, len(free), (N, Wp))].astype(np.int32) for _ in range(3)]
    wps = [torch.as_tensor(w, device=dev) for w in wps_host]
    eng.waypoint_fitness(wps[0], pol)
    torch.cuda.synchronize()
    eng.counters.zero_()
    ms = []
    for k in range(1, 3):
        e0.record()
        cells, ncell, stats = eng.waypoint_fitness(wps[k], pol)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    exp, rel = eng.expansions()
    t = sum(ms) / 1e3
    ach = (72.0 * exp + 25.0 * rel) / t / 1e9
    # end to end: host waypoints in (pinned), host stats out
    wp_pin = torch.as_tensor(wps_host[0]).pin_memory()
    st_pin = torch.empty((N, 5), dtype=torch.float64).pin_memory()
    t0 = time.perf_counter()
    _, _, st = eng.waypoint_fitness(wp_pin.to(dev, non_blocking=True), pol)
    st_pin.copy_(st, non_blocking=True)
    torch.cuda.synchronize()
    e2e_t = time.perf_counter() - t0
    out["pso_ga_fitness"] = {"workload": f"A*-connector fitness, {N} individuals x {Wp} waypoints on {size}x{size} blocks map "
                             "(BASELINE config 3)", "value": 2 * N / t, "unit": "path evals/s", "ms_per_population": 1e3 * t / 2,
                             "e2e": {"value": N / e2e_t, "unit": "path evals/s", "h2d_bytes_per_step": N * Wp * 4,
                                     "d2h_bytes_per_step": N * 40},
                             "astar_expansions_per_s": exp / t, "expansions_per_eval": exp / (2 * N),
                             "valid_fraction": float((ncell > 0).float().mean()),
                             "roofline": {"bound": "hbm", "kernel": "mpp_waypoint_fitness_kernel", "achieved": ach, "peak": peak,
                                          "unit": "GB/s", "frac": ach / peak,
                                          "algorithmic_bytes_per_unit": "72 B/expansion + 25 B/relaxation"}}
    if not args.no_cpu:
        O = _oracle()
        ns = min(N, 128 * max(CORES, 16))             # a bounded sample: a few seconds on the box's cores
        t0 = time.perf_counter()
        O.waypoint_fitness(grid, wps_host[1][:ns], 0.3, 0.8, 1.8, 100.0, threads=CORES)
        dt = time.perf_counter() - t0
        out["pso_ga_fitness"]["cpu_baseline"] = {"value": ns / dt, "unit": "path evals/s", "cores": CORES, "kind": "port",
                                                 "sample": f"{ns} individuals of the same population, C port (OpenMP over individuals), {dt:.1f} s"}
        rp = ref_python("fitness", size, 3000 + size, 10.0)
        if rp:
            out["pso_ga_fitness"]["cpu_baseline"] = dict(rp, port=out["pso_ga_fitness"]["cpu_baseline"])
    del eng
    # ---- config 2: MPA, 100 iterations ----
    from maaco_path_planing_b200.mpa import MPA
    grid = blocks_map(100, 0.20, seed=2000)
    iters2 = args.mpa_iters
    mpa = MPA(grid, num_predators=1024, num_iterations=iters2, rng_seed=2, verbose=False, **MPA_PARAMS)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    mpa.solve_path_planning()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    out["mpa"] = {"workload": f"MPA 1024 predators x {iters2} iterations on 100x100 blocks map (BASELINE config 2), "
                  "host-side sorts + best cascade included (= end to end: the population lives on the device, every "
                  "iteration's fitness column is read back)", "value": mpa.predator_evaluations / dt,
                  "unit": "predator-iterations/s", "seconds": dt, "best_fitness": mpa.best_fitness_overall}
    if not args.no_cpu:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import py_solvers as PS
        t0 = time.perf_counter()
        it_cpu = 10
        PS.MpaOracle(grid, 256, it_cpu, 0.2, 0.5, 2.0, 0.1, 0.8, 1.8, 100.0, seed=2).solve()
        dtc = time.perf_counter() - t0
        out["mpa"]["cpu_baseline"] = {"value": 256 * it_cpu / dtc, "unit": "predator-iterations/s", "cores": 1, "kind": "port",
                                      "sample": f"256 predators x {it_cpu} iterations, sequential mirror over the C port's searches, {dtc:.1f} s"}
        rp = ref_python("mpa", 100, 2000, 8.0)
        if rp:
            rp["unit"] = "predator-iterations/s"
            out["mpa"]["cpu_baseline"] = dict(rp, port=out["mpa"]["cpu_baseline"])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="maaco", choices=["maaco"])
    ap.add_argument("--ants", type=int, default=4096, help="ants per GPU")
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-extra", action="store_true", help="skip the other configs (fitness, MPA, batched maps)")
    ap.add_argument("--fit-size", type=int, default=512)
    ap.add_argument("--fit-pop", type=int, default=4096)
    ap.add_argument("--mpa-iters", type=int, default=100)
    ap.add_argument("--batch-maps", type=int, default=1250, help="independent maps per GPU (config 5 is 10000 over 8 GPUs = 1250)")
    ap.add_argument("--batch-iters", type=int, default=10)
    ap.add_argument("--batch-wave", type=int, default=128)
    ap.add_argument("--mpa-batch-maps", type=int, default=16, help="maps per GPU in the MPA part of config 5 (bounded sample)")
    ap.add_argument("--mpa-batch-iters", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed pass computed to DIR/<name>.npy (float64, at most 64 MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
