"""map_params of MAACOBatch / solve_maaco_batch without a device: how per-map parameters are resolved and refused, and
the q0 table the per-map pass reads (one row per pass, one column per map) against mpp_maaco_q0."""
import numpy as np
import pytest

from conftest import MAACO_DEFAULT


def test_resolve_overrides_and_defaults():
    from maaco_path_planing_b200.batch import MAP_PARAM_KEYS, resolve_map_params
    got = resolve_map_params(MAACO_DEFAULT, [{}, {"alpha": 2, "rho": 0.25}, {"C0_initial_pheromone": 0.5}], 3)
    assert got[0] == {k: float(MAACO_DEFAULT[k]) for k in MAP_PARAM_KEYS}
    assert got[1] == {**got[0], "alpha": 2.0, "rho": 0.25}
    assert got[2] == {**got[0], "C0_initial_pheromone": 0.5}
    assert all(isinstance(v, float) for p in got for v in p.values())
    no_c0 = {k: v for k, v in MAACO_DEFAULT.items() if k != "C0_initial_pheromone"}
    assert resolve_map_params(no_c0, [{}], 1)[0]["C0_initial_pheromone"] == 0.1      # MAACO's default


@pytest.mark.parametrize("map_params, match", [
    ([{}, {}], "2 entries for 3 maps"),
    ([{}, {}, {}, {}], "4 entries for 3 maps"),
    ([{}, {"gamma": 1.0}, {}], "unknown parameter 'gamma'"),
    ([{}, {}, {"num_iterations": 5}], "num_iterations is common"),
    ([{"num_ants": 64}, {}, {}], "num_ants is common"),
    ([{}, 0.5, {}], r"map_params\[1\] is not a mapping"),
    ("abc", "sequence of one mapping per map"),
])
def test_resolve_refuses(map_params, match):
    from maaco_path_planing_b200.batch import resolve_map_params
    with pytest.raises(ValueError, match=match):
        resolve_map_params(MAACO_DEFAULT, map_params, 3)


def test_sweep_refuses_before_any_wave(monkeypatch):
    from maaco_path_planing_b200 import batch
    from maaco_path_planing_b200.batch import solve_maaco_batch

    class Never(batch.MAACOBatch):
        def __init__(self, *a, **kw):
            raise AssertionError("a wave ran before map_params were checked")

    monkeypatch.setattr(batch, "MAACOBatch", Never)
    monkeypatch.setattr(batch, "_sweep_maps", lambda *a: (_ for _ in ()).throw(AssertionError("maps were read")))
    grids = [np.zeros((8, 8), np.int64) for _ in range(4)]
    for mp, match in (([{}] * 3, "3 entries for 4 maps"), ([{}, {}, {"beta2": 1}, {}], "unknown parameter"),
                      ([{}, {"num_iterations": 2}, {}, {}], "num_iterations")):
        with pytest.raises(ValueError, match=match):
            solve_maaco_batch(grids, 16, 2, MAACO_DEFAULT, map_params=mp)


@pytest.mark.parametrize("K", [0, 1, 2, 7, 10, 100, 333])
def test_q0_table_is_mpp_maaco_q0(K):
    from maaco_path_planing_b200 import _lib
    from maaco_path_planing_b200.batch import q0_table
    L = _lib.lib()
    q0i = [0.5, 0.1, 0.9, 0.5, 0.0, 1.0, 0.33, 0.9]
    t = q0_table(K, q0i)
    assert t.shape == (max(1, K), len(q0i)) and t.dtype == np.float64
    want = np.array([[L.mpp_maaco_q0(K, k, q) for q in q0i] for k in range(1, max(1, K) + 1)])
    assert t.tobytes() == want.tobytes()
