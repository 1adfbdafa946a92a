"""torchrun helper: solve_pso_batch / solve_ga_batch with the maps sharded over WORLD_SIZE GPUs must give, for every
rank's maps, exactly what the one-GPU sweep gives."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
POLICY = dict(turn_penalty_factor=0.3, safety_penalty_factor=0.8, min_safe_distance=1.8,
              diagonal_obstacle_penalty_value=100.0)


def main():
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import shard_maps, solve_ga_batch, solve_pso_batch
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    grids = [blocks_map(40 if i % 3 else 48, 0.2, seed=120 + i) for i in range(9)]
    seeds = [500 + i for i in range(9)]
    lo, hi = shard_maps(len(grids), dist.group.WORLD)
    pso = dict(w=0.7, c1=1.5, c2=1.5, **POLICY)
    ga = dict(mutation_rate=0.1, crossover_rate=0.8, **POLICY)
    for sweep, params in ((solve_pso_batch, pso), (solve_ga_batch, ga)):
        got = sweep(grids, 3, 32, 4, params, seeds=seeds, wave=2, group=dist.group.WORLD, device=local)
        want = sweep(grids, 3, 32, 4, params, seeds=seeds, device=local)
        assert [r[0] for r in got] == list(range(lo, hi)), (lo, hi)
        assert got == want[lo:hi], sweep.__name__
    dist.barrier()
    dist.destroy_process_group()
    print("multigpu_pop_batch_check ok")


if __name__ == "__main__":
    main()
