"""map_sizes of MAACOBatch / solve_maaco_batch without a device: how per-map colony sizes and pass counts are resolved
and refused, the per-map q0 table against mpp_maaco_q0, and the sized pass entry point of the C ABI."""
import numpy as np
import pytest

from conftest import MAACO_DEFAULT


def test_resolve_sizes_overrides_and_defaults():
    from maaco_path_planing_b200.batch import resolve_map_sizes
    got = resolve_map_sizes(64, 3, [{}, {"num_ants": 5}, {"num_iterations": 0}, {"num_ants": np.int64(7),
                                                                                 "num_iterations": np.int32(9)}], 4)
    assert got == [{"num_ants": 64, "num_iterations": 3}, {"num_ants": 5, "num_iterations": 3},
                   {"num_ants": 64, "num_iterations": 0}, {"num_ants": 7, "num_iterations": 9}]
    assert all(type(v) is int for s in got for v in s.values())


@pytest.mark.parametrize("map_sizes, match", [
    ([{}, {}], "2 entries for 3 maps"),
    ([{}, {}, {}, {}], "4 entries for 3 maps"),
    ("abc", "sequence of one mapping per map"),
    (5, "sequence of one mapping per map"),
    ([{}, 7, {}], r"map_sizes\[1\] is not a mapping"),
    ([{}, {}, {"alpha": 1.0}], r"map_sizes\[2\]: unknown key 'alpha'"),
    ([{"num_ants": 2.0}, {}, {}], "num_ants must be an integer"),
    ([{}, {"num_iterations": "3"}, {}], "num_iterations must be an integer"),
    ([{}, {"num_ants": True}, {}], "num_ants must be an integer"),
    ([{}, {"num_iterations": np.bool_(False)}, {}], "num_iterations must be an integer"),
    ([{}, {}, {"num_ants": 0}], r"map_sizes\[2\]: num_ants 0 < 1"),
    ([{"num_iterations": -1}, {}, {}], r"map_sizes\[0\]: num_iterations -1 < 0"),
])
def test_resolve_sizes_refuses(map_sizes, match):
    from maaco_path_planing_b200.batch import resolve_map_sizes
    with pytest.raises(ValueError, match=match):
        resolve_map_sizes(64, 3, map_sizes, 3)


def test_map_params_still_refuse_sizes():
    from maaco_path_planing_b200.batch import resolve_map_params
    for k in ("num_ants", "num_iterations"):
        with pytest.raises(ValueError, match=f"{k} is common"):
            resolve_map_params(MAACO_DEFAULT, [{k: 4}], 1)


def test_sweep_refuses_bad_sizes_before_any_wave(monkeypatch):
    from maaco_path_planing_b200 import batch
    from maaco_path_planing_b200.batch import solve_maaco_batch

    class Never(batch.MAACOBatch):
        def __init__(self, *a, **kw):
            raise AssertionError("a wave ran before map_sizes were checked")

    monkeypatch.setattr(batch, "MAACOBatch", Never)
    monkeypatch.setattr(batch, "_sweep_maps", lambda *a: (_ for _ in ()).throw(AssertionError("maps were read")))
    grids = [np.zeros((8, 8), np.int64) for _ in range(4)]
    for ms, match in (([{}] * 3, "3 entries for 4 maps"), ([{}, {}, {"rho": 0.1}, {}], "unknown key"),
                      ([{}, {"num_ants": 0}, {}, {}], "num_ants 0 < 1"), ([{"num_iterations": 1.5}] + [{}] * 3,
                                                                          "must be an integer")):
        for pme in (False, True):
            with pytest.raises(ValueError, match=match):
                solve_maaco_batch(grids, 16, 2, MAACO_DEFAULT, per_map_endpoints=pme, map_sizes=ms)
    with pytest.raises(ValueError, match="num_iterations -2 < 0"):
        solve_maaco_batch(grids, 16, 2, MAACO_DEFAULT, map_params=[{}] * 4, map_sizes=[{"num_iterations": -2}] * 4)


def test_q0_table_per_map_counts_is_mpp_maaco_q0():
    from maaco_path_planing_b200 import _lib
    from maaco_path_planing_b200.batch import q0_table
    L = _lib.lib()
    Ks = [0, 1, 2, 7, 10, 1, 0, 333, 7]
    q0i = [0.5, 0.1, 0.9, 0.5, 0.0, 1.0, 0.33, 0.9, 0.5]
    t = q0_table(Ks, q0i)
    assert t.shape == (333, len(q0i)) and t.dtype == np.float64
    for m, (K, q) in enumerate(zip(Ks, q0i)):
        want = np.array([L.mpp_maaco_q0(K, k, q) for k in range(1, 334)])
        assert t[:, m].tobytes() == want.tobytes(), m
    assert q0_table([0, 0], [0.5, 0.2]).shape == (1, 2)
    assert q0_table([4] * 3, [0.5, 0.2, 0.5]).tobytes() == q0_table(4, [0.5, 0.2, 0.5]).tobytes()
    with pytest.raises(ValueError, match="2 pass counts for 3 maps"):
        q0_table([1, 2], [0.5, 0.5, 0.5])


def test_sized_pass_symbol_and_abi_version():
    import ctypes as C
    from maaco_path_planing_b200 import _lib
    L = _lib.lib()
    assert L.mpp_abi_version() == 3
    assert isinstance(L.mpp_maaco_pass_maps_sized, C._CFuncPtr)
    assert len(L.mpp_maaco_pass_maps_sized.argtypes) == 9
