"""Config 5 from device-resident grids: the same maps (blocks_map(256, 0.20, seed=5000 + i), i < --maps) given to the
batched solvers as host int64 grids, as a CUDA int64 tensor and as a CUDA uint8 tensor.  Prints one JSON line with, per
input:

  ingest_ms_per_wave   building one wave's map batch (host: uint8 conversion, upload, bit-packing; device:
                       mpp_map_batch_create_device), host clock between device synchronises, median over the waves
  maaco_maps_per_s     solve_maaco_batch end to end: --ants ants x --passes passes, --wave maps per wave
  astar_maps_per_s     solve_search_batch(..., "astar") end to end, all maps in one SearchBatch

each the median of --reps rounds that alternate the three inputs (every value is listed too), plus whether every result
equals the first host-grid run, and the card's name and power limit, read in the same run.

    python tools/device_grids_time.py [--maps 1250] [--ants 1024] [--passes 10] [--wave 128] [--reps 3]
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

MAACO_PARAMS = dict(alpha=1.0, beta=7.0, rho=0.1, Q=2.5, a_turn_coef=1.0, wh_max=0.9, wh_min=0.2, k_h_adaptive=0.9,
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


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--maps", type=int, default=1250)
    ap.add_argument("--ants", type=int, default=1024)
    ap.add_argument("--passes", type=int, default=10)
    ap.add_argument("--wave", type=int, default=128)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import _map_set, solve_maaco_batch, solve_search_batch
    if not torch.cuda.is_available():
        raise SystemExit("device_grids_time.py measures the GPU: no CUDA device visible")
    torch.cuda.set_device(0)
    name, power = card()
    M, W = args.maps, args.wave
    grids = np.stack([blocks_map(256, 0.20, seed=5000 + i) for i in range(M)])
    inputs = {"host_int64": grids, "cuda_int64": torch.as_tensor(grids, device="cuda")}
    inputs["cuda_uint8"] = inputs["cuda_int64"].to(torch.uint8)
    seeds = list(range(M))
    solve_maaco_batch(grids[:8], 64, 1, MAACO_PARAMS, seeds=seeds[:8])     # module load, first launches
    solve_search_batch(inputs["cuda_uint8"][:8], "astar", {})
    out = {"what": f"config 5 from host and device grids: {M} blocks maps 256x256 (20% obstacles), MAACO {args.ants} ants "
                   f"x {args.passes} passes in waves of {W}, A* start -> target per map",
           "card": name, "power_limit_w": power, "maps": M, "results": {}}
    want = None
    runs = {kind: {"ingest_ms_per_wave": [], "maaco_maps_per_s": [], "astar_maps_per_s": [], "equal_to_host_int64": True}
            for kind in inputs}
    for _ in range(args.reps):
        for kind, g in inputs.items():
            r = runs[kind]
            ingest = []
            for w0 in range(0, M, W):
                m, dt = timed(lambda: _map_set(g[w0:w0 + W]))
                m.close()
                ingest.append(dt)
            r["ingest_ms_per_wave"].append(1e3 * float(np.median(ingest)))
            maaco, dt = timed(lambda: solve_maaco_batch(g, args.ants, args.passes, MAACO_PARAMS, seeds=seeds, wave=W))
            r["maaco_maps_per_s"].append(M / dt)
            astar, dt = timed(lambda: solve_search_batch(g, "astar", {}))
            r["astar_maps_per_s"].append(M / dt)
            if want is None:
                want = (maaco, astar)
            r["equal_to_host_int64"] &= (maaco, astar) == want
            torch.cuda.empty_cache()
    for kind, r in runs.items():
        res = {k: float(np.median(v)) for k, v in r.items() if isinstance(v, list)}
        res["maaco_evals_per_s"] = res["maaco_maps_per_s"] * args.ants * args.passes
        res["equal_to_host_int64"] = r["equal_to_host_int64"]
        res["all"] = {k: [round(x, 2) for x in v] for k, v in r.items() if isinstance(v, list)}
        out["results"][kind] = res
    print(json.dumps(out))


if __name__ == "__main__":
    main()
