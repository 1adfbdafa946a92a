"""The drop-in modules as the reference's caller, main.py, uses them: the names it imports from `env` are there with the
reference's demo maps, and the six solvers imported under the reference's module names, built with main.py's
parameters and seeded only through MPP_RNG_SEED, give the anchors the unmodified reference prints (A*, Dijkstra) and
the oracle's results under the same seed (MAACO, PSO, GA, MPA)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import MAACO_DEFAULT, ROOT, load_golden

SEED = 20261
POLICY = dict(turn_penalty_factor=0.3, safety_penalty_factor=0.8, min_safe_distance=1.8,
              diagonal_obstacle_penalty_value=100.0)                               # main.py:21-24

# runs in its own interpreter: the reference's module names (MAACO, pso, env, ...) must not leak into this process
DRIVER = """
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from env import grid_fig7_layout_data, grid_map_fig13_base_data
from MAACO import MAACO
from MPA import MPA
from astar import AStarSolver
from dijkstra import DijkstraSolver
from ga_solver import GASolver
from pso import PSOSolver
POLICY, MAACO_DEFAULT = %r, %r
g7 = np.array(grid_fig7_layout_data)
g7[0, 0], g7[19, 19] = 2, 3
out = {}
def keep(name, grid, res, curve=None):
    out[name + "_path"] = np.array([r * grid.shape[1] + c for r, c in res[0]], np.int32)
    out[name + "_stats"] = np.array([float(x) for x in res[1:]])
    if curve is not None:
        out[name + "_curve"] = np.array([np.inf if v is None else v for v in curve], float)
for name, g in (("maaco_fig7", g7), ("maaco_fig13", np.array(grid_map_fig13_base_data))):
    s = MAACO(g, 50, 100, **MAACO_DEFAULT)
    keep(name, g, s.solve_path_planning(), s.convergence_curve_data)
keep("astar", g7, AStarSolver(g7, **POLICY).solve())
keep("dijkstra", g7, DijkstraSolver(g7, **POLICY).solve())
s = PSOSolver(g7, 50, 100, 5, 0.7, 1.5, 1.5, **POLICY)
keep("pso", g7, s.solve(), s.convergence_curve)
s = GASolver(g7, 100, 50, 5, 0.1, 0.8, 3, **POLICY)
keep("ga", g7, s.solve(), s.convergence_curve)
s = MPA(g7, 50, 100, FADs_rate=0.2, P_const=0.5, levy_beta=2.0, turn_penalty_factor=0.1, safety_penalty_factor=0.8,
        min_safe_distance=1.8, diagonal_obstacle_penalty=100.0)
keep("mpa", g7, s.solve_path_planning())
np.savez(sys.argv[2], **out)
""" % (POLICY, MAACO_DEFAULT)


def test_dropin_env_exports_the_names_main_imports(tmp_path):
    """main.py:9-17 -- CPU check (no kernels): the six grids are there, as list-of-lists, equal to the reference's."""
    code = ("import sys; sys.path.insert(0, %r); import env; import numpy as np;"
            "from env import (grid_fig7_layout_data, grid_map_fig13_base_data, grid_map_from_image_data,"
            "grid_map_from_image_data2, grid_map_from_image_data3, grid_map_from_image_data5,"
            "START_NODE_VAL, TARGET_NODE_VAL, OBSTACLE, FREE_SPACE);"
            "assert isinstance(grid_fig7_layout_data, list) and isinstance(grid_fig7_layout_data[0][0], int);"
            "np.savez(sys.argv[1], **{k: np.array(getattr(env, k)) for k in env.GRID_NAMES})"
            % os.path.join(ROOT, "maaco_path_planing_b200", "dropin"))
    out = str(tmp_path / "env_names.npz")
    subprocess.check_call([sys.executable, "-c", code, out], cwd=ROOT)
    z = np.load(out)
    want = load_golden("env_grids")
    g7 = z["grid_fig7_layout_data"].copy()
    assert g7.dtype.kind == "i" and g7[0, 0] == 0
    g7[0, 0], g7[19, 19] = 2, 3                                      # main.py:27-32
    assert np.array_equal(g7, want["fig7"])
    for a, b in (("grid_map_fig13_base_data", "fig13"), ("grid_map_from_image_data", "image1"),
                 ("grid_map_from_image_data2", "image2"), ("grid_map_from_image_data3", "image3"),
                 ("grid_map_from_image_data5", "image5")):
        assert np.array_equal(z[a], want[b]), a


@pytest.mark.gpu
def test_dropin_solvers_with_main_parameters_under_seed(tmp_path):
    import pyoracle as O
    import py_solvers as PS
    out = str(tmp_path / "dropin.npz")
    env = dict(os.environ, MPP_RNG_SEED=str(SEED))
    log = subprocess.run([sys.executable, "-c", DRIVER, os.path.join(ROOT, "maaco_path_planing_b200", "dropin"), out],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    assert log.returncode == 0, log.stdout[-2000:] + log.stderr[-4000:]
    r = np.load(out)
    grids = load_golden("env_grids")
    g7 = grids["fig7"].astype(int)
    # ---- deterministic solvers: anchors printed by the unmodified reference on fig7 ----
    assert len(r["astar_path"]) == 28 and list(r["astar_stats"]) == [31.556349186104047, 17, 0.34870130201414323, 0.0,
                                                                     36.93531022771536]
    st = r["dijkstra_stats"]
    assert len(r["dijkstra_path"]) == 28 and st[1] == 12 and st[2] == 0.3274397055203064 and st[4] == 35.41830095052029
    # ---- MAACO on fig7 and fig13, PSO / GA / MPA on fig7: the oracle under the same seed ----
    for name, grid in (("maaco_fig7", g7), ("maaco_fig13", grids["fig13"].astype(int))):
        o = O.MaacoOracle(grid, 50, 100, seed=SEED, **MAACO_DEFAULT)
        opath, olen, oturns = o.solve()
        assert np.array_equal(r[name + "_path"], opath) and list(r[name + "_stats"]) == [olen, oturns], name
        assert np.array_equal(r[name + "_curve"], [np.inf if v is None else v for v in o.curve]), name
    pol = (0.3, 0.8, 1.8, 100.0)
    ps = PS.PsoOracle(g7, 50, 100, 5, 0.7, 1.5, 1.5, *pol, seed=SEED)
    ppath, pfit = ps.solve()
    assert np.array_equal(r["pso_path"], ppath) and r["pso_stats"][4] == pfit
    assert np.array_equal(r["pso_curve"], ps.curve)
    ga = PS.GaOracle(g7, 100, 50, 5, 0.1, 0.8, 3, *pol, seed=SEED)
    gpath, gst = ga.solve()
    assert np.array_equal(r["ga_path"], gpath) and r["ga_stats"][4] == gst[4]
    assert np.array_equal(r["ga_curve"], ga.curve)
    mp = PS.MpaOracle(g7, 50, 100, 0.2, 0.5, 2.0, 0.1, 0.8, 1.8, 100.0, seed=SEED)
    mpath, mst = mp.solve()
    assert np.array_equal(r["mpa_path"], np.array(mpath, np.int32)) and r["mpa_stats"][4] == mst[4]
