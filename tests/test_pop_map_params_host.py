"""map_params of PSOBatch / GABatch / MPABatch and their sweeps without a device: how per-map parameters are resolved
and refused, how the sweeps form waves from them, and the mpp_pop_params layout the kernels read."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT

PSO = dict(w=0.7, c1=1.5, c2=1.5)
GA = dict(mutation_rate=0.1, crossover_rate=0.8)


def test_resolve_defaults_and_overrides():
    from maaco_path_planing_b200.batch import resolve_map_params
    got = resolve_map_params(PSO, [{}, {"w": 0.5, "turn_penalty_factor": 1}], 2, "pso")
    assert got[0] == dict(w=0.7, c1=1.5, c2=1.5, turn_penalty_factor=0.1, safety_penalty_factor=0.05,
                          diagonal_obstacle_penalty_value=1000.0, min_safe_distance=1.5, allow_diagonal_moves=True,
                          restrict_diagonal_near_obstacle_policy=True)
    assert got[1] == {**got[0], "w": 0.5, "turn_penalty_factor": 1.0}
    assert type(got[1]["turn_penalty_factor"]) is float and type(got[0]["allow_diagonal_moves"]) is bool
    got = resolve_map_params(dict(GA, safety_penalty_factor=0.8), [{}, {"tournament_size": 5.0}], 2, "ga",
                             population=40)
    assert got[0]["tournament_size"] == 3 and got[0]["safety_penalty_factor"] == 0.8
    assert got[1]["tournament_size"] == 5 and type(got[1]["tournament_size"]) is int
    got = resolve_map_params({}, [{"levy_beta": 2.0, "diagonal_obstacle_penalty": 5}], 1, "mpa")
    assert got[0] == dict(FADs_rate=0.2, P_const=0.5, levy_beta=2.0, turn_penalty_factor=0.1, safety_penalty_factor=0.05,
                          diagonal_obstacle_penalty=5.0, min_safe_distance=1.5, allow_diagonal_moves=True,
                          restrict_diagonal_near_obstacle=True)


@pytest.mark.parametrize("planner, map_params, match", [
    ("pso", [{}, {}], "2 entries for 3 maps"),
    ("pso", [{}, {"alpha": 1.0}, {}], "unknown parameter 'alpha'"),
    ("pso", [{}, {}, {"num_particles": 5}], r"map_params\[2\]: num_particles is common"),
    ("pso", [{"num_iterations": 5}, {}, {}], "num_iterations is common"),
    ("pso", [{}, {}, {"num_waypoints_per_particle": 2}], "num_waypoints_per_particle is common"),
    ("ga", [{}, {"population_size": 8}, {}], "population_size is common"),
    ("ga", [{}, {"num_generations": 8}, {}], "num_generations is common"),
    ("ga", [{"num_waypoints_per_chromosome": 8}, {}, {}], "num_waypoints_per_chromosome is common"),
    ("ga", [{}, {"w": 0.5}, {}], "unknown parameter 'w'"),
    ("ga", [{}, {}, {"tournament_size": 2.5}], r"map_params\[2\]: tournament_size must be an integer"),
    ("ga", [{}, {"tournament_size": 0}, {}], r"map_params\[1\]: tournament_size 0 unsupported"),
    ("ga", [{}, {"tournament_size": 17}, {}], r"map_params\[1\]: tournament_size 17 unsupported"),
    ("ga", [{"tournament_size": 6}, {}, {}], r"map_params\[0\]: tournament_size 6 unsupported with a population of 40"),
    ("mpa", [{}, {}, {"num_predators": 4}], "num_predators is common"),
    ("mpa", [{}, {"num_iterations": 4}, {}], "num_iterations is common"),
    ("mpa", [{}, {"w": 4}, {}], "unknown parameter 'w'"),
    ("mpa", [{}, {}, {"levy_beta": 2.5}], r"map_params\[2\]: levy_beta gives a complex Levy sigma"),
    ("mpa", [{}, 3, {}], r"map_params\[1\] is not a mapping"),
    ("mpa", "abc", "sequence of one mapping per map"),
])
def test_resolve_refuses(planner, map_params, match):
    from maaco_path_planing_b200.batch import resolve_map_params
    defaults = {"pso": PSO, "ga": GA, "mpa": {}}[planner]
    with pytest.raises(ValueError, match=match):
        resolve_map_params(defaults, map_params, 3, planner, population=40)


def test_tournament_limits_follow_the_selection_kernel():
    """min(tournament_size, population) decides, as in mpp_ga_select_batch: 16 takes any population above 85, a
    tournament larger than a population of 4 is a tournament of 4."""
    from maaco_path_planing_b200.batch import resolve_map_params
    assert resolve_map_params(GA, [{"tournament_size": 16}], 1, "ga", population=86)[0]["tournament_size"] == 16
    assert resolve_map_params(GA, [{"tournament_size": 20}], 1, "ga", population=4)[0]["tournament_size"] == 20
    with pytest.raises(ValueError, match="unsupported"):
        resolve_map_params(GA, [{"tournament_size": 16}], 1, "ga", population=85)


def test_per_wave_keys_must_agree_in_a_batch():
    from maaco_path_planing_b200.batch import _wave_params, resolve_map_params
    ok = resolve_map_params(PSO, [{"min_safe_distance": 2.0}, {"min_safe_distance": 2.0, "w": 0.1}], 2, "pso")
    assert _wave_params("pso", ok)["min_safe_distance"] == 2.0
    for planner, key, val in (("pso", "min_safe_distance", 2.0), ("ga", "allow_diagonal_moves", False),
                              ("ga", "restrict_diagonal_near_obstacle_policy", False),
                              ("mpa", "restrict_diagonal_near_obstacle", False)):
        r = resolve_map_params({"pso": PSO, "ga": GA, "mpa": {}}[planner], [{}, {}, {key: val}], 3, planner,
                               population=40)
        with pytest.raises(ValueError, match=rf"map_params\[2\]: {key}=.* differs from map 0's"):
            _wave_params(planner, r)
    # MPA never reads min_safe_distance: it may differ from map to map
    r = resolve_map_params({}, [{}, {"min_safe_distance": 3.0}], 2, "mpa")
    assert _wave_params("mpa", r) == dict(allow_diagonal_moves=True, restrict_diagonal_near_obstacle=True)


@pytest.mark.parametrize("cls_name", ["PSOBatch", "GABatch", "MPABatch"])
def test_batches_refuse_before_device_work(monkeypatch, cls_name):
    from maaco_path_planing_b200 import batch
    monkeypatch.setattr(batch, "_map_set", lambda *a, **k: (_ for _ in ()).throw(AssertionError("device work")))
    grids = np.zeros((3, 8, 8), np.int64)
    args = {"PSOBatch": (2, 8, 2, 0.7, 1.5, 1.5), "GABatch": (2, 40, 2, 0.1, 0.8), "MPABatch": (8, 2)}[cls_name]
    bad = {"PSOBatch": [{}, {"w": 1.0}, {"min_safe_distance": 3.0}], "GABatch": [{}, {"tournament_size": 9}, {}],
           "MPABatch": [{}, {"levy_beta": 2.5}, {}]}[cls_name]
    with pytest.raises(ValueError, match=r"map_params\[[12]\]"):
        getattr(batch, cls_name)(grids, *args, map_params=bad)
    with pytest.raises(ValueError, match="2 entries for 3 maps"):
        getattr(batch, cls_name)(grids, *args, map_params=[{}, {}])


@pytest.mark.parametrize("planner", ["pso", "ga", "mpa"])
def test_sweeps_refuse_before_any_wave(monkeypatch, planner):
    from maaco_path_planing_b200 import batch

    class Never:
        _planner = planner

        def __init__(self, *a, **kw):
            raise AssertionError("a wave ran before map_params were checked")

    for name in ("PSOBatch", "GABatch", "MPABatch"):
        monkeypatch.setattr(batch, name, Never)
    monkeypatch.setattr(batch, "_sweep_maps", lambda *a: (_ for _ in ()).throw(AssertionError("maps were read")))
    grids = [np.zeros((8, 8), np.int64) for _ in range(4)]
    if planner == "pso":
        sweep = lambda mp: batch.solve_pso_batch(grids, 2, 8, 2, dict(PSO), map_params=mp)
        bad = [{}, {}, {"num_particles": 4}, {}]
    elif planner == "ga":
        sweep = lambda mp: batch.solve_ga_batch(grids, 2, 40, 2, dict(GA), map_params=mp)
        bad = [{}, {}, {"tournament_size": 7}, {}]
    else:
        sweep = lambda mp: batch.solve_mpa_batch(grids, 8, 2, {}, map_params=mp)
        bad = [{}, {}, {"levy_beta": 2.5}, {}]
    with pytest.raises(ValueError, match="3 entries for 4 maps"):
        sweep([{}] * 3)
    with pytest.raises(ValueError, match=r"map_params\[2\]"):
        sweep(bad)


def test_waves_by_shape_and_per_wave_keys():
    from maaco_path_planing_b200.batch import _pop_waves, _shape_waves, _wave_key, resolve_map_params
    grids = [np.zeros((8, 8)) if i % 3 else np.zeros((6, 9)) for i in range(12)]
    mp = resolve_map_params(PSO, [{"min_safe_distance": 2.0} if i % 2 else {"w": 0.1 * i} for i in range(12)], 12,
                            "pso")
    key = _wave_key("pso", mp)
    waves = _pop_waves(grids, 0, 12, 1024, wave=2, key=key)
    assert sorted(i for w in waves for i in w) == list(range(12))
    for w in waves:
        assert w == sorted(w) and len(w) <= 2
        assert len({grids[i].shape for i in w}) == 1 and len({key(i) for i in w}) == 1
    assert waves[0] == [0, 6]                                   # (6, 9), even: index order within a group
    assert _pop_waves(grids, 0, 12, 1024, key=None) == _shape_waves(grids, 0, 12)
    mpa = resolve_map_params({}, [{"allow_diagonal_moves": bool(i < 5), "min_safe_distance": float(i)}
                                  for i in range(12)], 12, "mpa")
    waves = _shape_waves(grids, 3, 12, None, _wave_key("mpa", mpa))
    assert waves == [[3], [4], [5, 7, 8, 10, 11], [6, 9]]
    assert _wave_key("mpa", None) is None


def test_pop_params_layout_matches_the_header():
    """The ctypes mirror of mpp_pop_params has the header's size and field offsets (a C program built against
    include/mpp.h prints them)."""
    from maaco_path_planing_b200 import _lib
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    import tempfile
    fields = [f for f, _ in _lib.PopParams._fields_]
    src = ("#include <stdio.h>\n#include <stddef.h>\n#include \"mpp.h\"\nint main(void) {\n"
           '    printf("%zu\\n", sizeof(mpp_pop_params));\n'
           + "".join(f'    printf("%zu\\n", offsetof(mpp_pop_params, {f}));\n' for f in fields) + "    return 0;\n}\n")
    with tempfile.TemporaryDirectory() as d:
        with open(os.path.join(d, "layout.c"), "w") as f:
            f.write(src)
        exe = os.path.join(d, "layout")
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, os.path.join(d, "layout.c")], check=True)
        got = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [ctypes.sizeof(_lib.PopParams)] + [getattr(_lib.PopParams, f).offset for f in fields]


def test_pop_params_rows_carry_each_planners_fields():
    """The rows the per-map kernels read: MPA's penalty under the header's field name and the Levy sigma of each map's
    levy_beta; GA's integer tournament size."""
    from maaco_path_planing_b200 import _lib
    from maaco_path_planing_b200.batch import _pop_params_host, levy_sigma, resolve_map_params
    mp = resolve_map_params({}, [{"levy_beta": 1.2, "diagonal_obstacle_penalty": 7.0}, {"P_const": 0.25}], 2, "mpa")
    raw = _pop_params_host("mpa", mp)
    n = ctypes.sizeof(_lib.PopParams)
    assert len(raw) == 2 * n
    rows = [_lib.PopParams.from_buffer_copy(raw[k * n:(k + 1) * n]) for k in range(2)]
    assert rows[0].levy_beta == 1.2 and rows[0].levy_sigma == levy_sigma(1.2)
    assert rows[0].diagonal_obstacle_penalty_value == 7.0 and rows[0].P_const == 0.5
    assert rows[1].P_const == 0.25 and rows[1].levy_sigma == levy_sigma(1.5) and rows[1].FADs_rate == 0.2
    ga = resolve_map_params(GA, [{"tournament_size": 4, "mutation_rate": 0.3}], 1, "ga", population=40)
    g = _lib.PopParams.from_buffer_copy(_pop_params_host("ga", ga))
    assert (g.tournament_size, g.mutation_rate, g.crossover_rate, g.turn_penalty_factor) == (4, 0.3, 0.8, 0.1)
    p = _lib.PopParams.from_buffer_copy(_pop_params_host("pso", resolve_map_params(PSO, [{"c2": 2.5}], 1, "pso")))
    assert (p.w, p.c1, p.c2, p.safety_penalty_factor, p.diagonal_obstacle_penalty_value) == (0.7, 1.5, 2.5, 0.05, 1000.0)
