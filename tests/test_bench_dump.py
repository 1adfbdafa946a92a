"""bench.py --dump-outputs: the last timed pass written as float64 .npy files within a byte budget, identical from run
to run and equal to the C oracle's replay of the same passes."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from conftest import ROOT


def test_save_outputs_samples_rows_within_budget(tmp_path):
    big = np.arange(1000 * 30, dtype=np.int32).reshape(1000, 30)
    small = np.array([1.5, 0.0, -1.0])
    bench.save_outputs(str(tmp_path), {"big": big, "small": small}, {"big": 64 << 10, "small": 1 << 10})
    assert np.array_equal(np.load(tmp_path / "small.npy"), small)
    assert not (tmp_path / "small_rows.npy").exists()
    got, rows = np.load(tmp_path / "big.npy"), np.load(tmp_path / "big_rows.npy")
    assert got.dtype == np.float64 and rows.dtype == np.float64
    assert got.nbytes + rows.nbytes <= 64 << 10 and len(rows) == (64 << 10) // (8 * 30 + 8)
    assert np.all(np.diff(rows) > 0) and np.array_equal(got, big[rows.astype(int)])
    again = tmp_path / "again"
    bench.save_outputs(str(again), {"big": big}, {"big": 64 << 10})
    assert np.array_equal(np.load(again / "big_rows.npy"), rows)                 # the sample is fixed
    for bad in (np.inf, -np.inf, np.nan):
        with pytest.raises(ValueError, match="not finite"):
            bench.save_outputs(str(tmp_path / "bad"), {"x": np.array([1.0, bad])}, {"x": 1 << 10})


def test_dump_budgets_fit_64_mib():
    assert sum(bench.DUMP_BUDGETS.values()) + 1024 * len(bench.DUMP_BUDGETS) <= 64 << 20


@pytest.mark.gpu
def test_dump_outputs_repeat_and_match_oracle(tmp_path):
    import pyoracle as O
    from maaco_path_planing_b200 import blocks_map
    size, ants, steps, warmup = 64, 256, 2, 3
    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                              "--warmup", str(warmup), "--size", str(size), "--ants", str(ants), "--no-cpu", "--no-extra",
                              "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["parity_check"].startswith("ok")
        files = sorted(glob.glob(str(d / "*.npy")))
        assert sum(os.path.getsize(f) for f in files) <= 64 << 20
        dumps.append({os.path.basename(f)[:-4]: np.load(f) for f in files})
    assert dumps[0].keys() == dumps[1].keys()
    for name, a in dumps[0].items():
        assert a.dtype == np.float64 and np.isfinite(a).all() and np.array_equal(a, dumps[1][name]), name
    # the same colony (bench: rng_seed=4, num_iterations = steps + warmup + 64) replayed by the oracle; the dump is its
    # last timed pass, where ants whose tour failed (length inf) are written with length -1
    d = dumps[0]
    orc = O.MaacoOracle(blocks_map(size, 0.20, seed=4000), ants, steps + warmup + 64, seed=4, **bench.MAACO_PARAMS)
    for it in range(1, warmup + steps + 1):
        cells, nc, ln, tn, _ = orc.iterate(it)
    failed = ~np.isfinite(ln)
    assert failed.any() and np.array_equal(d["ant_length"], np.where(failed, -1.0, ln))
    assert np.array_equal(d["ant_n_cells"], nc)
    assert np.array_equal(d["ant_turns"], tn)
    assert np.array_equal(d["pheromone"].ravel(), orc.tau)
    assert d["best"][0] == orc.best_len and d["best"][1] == orc.best_turns
    assert np.array_equal(d["best_path"], orc.best_path)
    tours = d["ant_tours"]
    rows = d["ant_tours_rows"].astype(int) if "ant_tours_rows" in d else np.arange(ants)
    for r, a in zip(tours, rows):
        assert np.array_equal(r[:nc[a]], cells[a, :nc[a]]) and np.all(r[nc[a]:] == -1), f"ant {a}"
