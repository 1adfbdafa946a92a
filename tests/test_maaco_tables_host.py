"""mpp_maaco_e01_host, the host half of MAACO's per-map tables: every map's eta'**beta table, interleaved by turn flag,
equals byte for byte the C oracle's tables for a map with those endpoints (the oracle is pinned to MAACO.py:197-210).
CPU only: the function touches no device."""
import ctypes as C

import numpy as np
import pytest

from conftest import MAACO_DEFAULT, load_golden

PARAM_SETS = {
    "default": MAACO_DEFAULT,
    "beta2.5": dict(MAACO_DEFAULT, beta=2.5),
    "k_h0": dict(MAACO_DEFAULT, k_h_adaptive=0.0),
    "turn0": dict(MAACO_DEFAULT, a_turn_coef=0.0),
    "wh_flat": dict(MAACO_DEFAULT, wh_max=0.5, wh_min=0.5),
}


def _pairs_37x53():
    """40 (start, target) cells of a 37 x 53 map: one row, one column, adjacent (both ways, diagonal too), corners to
    corners, then seeded random pairs."""
    R, Cc = 37, 53
    cell = lambda r, c: r * Cc + c
    fixed = [(cell(5, 3), cell(5, 49)), (cell(30, 40), cell(30, 2)), (cell(2, 17), cell(33, 17)), (cell(36, 8), cell(0, 8)),
             (cell(10, 10), cell(10, 11)), (cell(10, 11), cell(10, 10)), (cell(10, 10), cell(11, 11)),
             (cell(20, 20), cell(19, 21)), (cell(0, 0), cell(36, 52)), (cell(36, 52), cell(0, 0)),
             (cell(0, 52), cell(36, 0)), (cell(36, 0), cell(0, 52)), (cell(0, 0), cell(0, 52)), (cell(36, 52), cell(36, 0))]
    rng = np.random.default_rng(3753)
    while len(fixed) < 40:
        s, t = rng.choice(R * Cc, 2, replace=False)
        fixed.append((int(s), int(t)))
    return (R, Cc), fixed


def _pairs_256():
    rng = np.random.default_rng(256)
    n = 256 * 256
    return (256, 256), [(0, n - 1)] + [tuple(int(x) for x in rng.choice(n, 2, replace=False)) for _ in range(15)]


def _demo_pairs():
    """The endpoints of every env.py demo map, as (shape, [(start, target)]) per shape."""
    out = {}
    for name, g in sorted(load_golden("env_grids").items()):
        flat = g.ravel()
        out.setdefault(g.shape, []).append((int(np.flatnonzero(flat == 2)[0]), int(np.flatnonzero(flat == 3)[0])))
    return list(out.items())


def oracle_e01(shape, start, target, params):
    """The oracle's E0 / E1 of a shape-`shape` map with these endpoints, interleaved like mpp_maaco_e01_host's."""
    import pyoracle as O
    g = np.zeros(shape, np.int64)
    g.flat[start], g.flat[target] = 2, 3
    orc = O.MaacoOracle(g, 1, 1, **params)
    return np.stack([orc.E0, orc.E1], axis=1).ravel()


def e01_host(shape, pairs, params, threads=0):
    from maaco_path_planing_b200.batch import _e01_host, _maaco_params
    out = np.full(len(pairs) * 2 * shape[0] * shape[1], np.nan)
    s, t = (np.array([p[k] for p in pairs], np.int64) for k in (0, 1))
    return _e01_host(*shape, s, t, _maaco_params(1, **params), out, threads).reshape(len(pairs), -1)


CASES = _demo_pairs() + [_pairs_37x53(), _pairs_256()]


@pytest.mark.parametrize("pset", sorted(PARAM_SETS))
@pytest.mark.parametrize("case", range(len(CASES)), ids=[f"{r}x{c}" for (r, c), _ in CASES])
def test_e01_host_equals_oracle(case, pset):
    shape, pairs = CASES[case]
    if shape == (256, 256) and pset != "default":
        pairs = pairs[:3]                                   # the oracle's tables cost ~10 ms per 256x256 map
    got = e01_host(shape, pairs, PARAM_SETS[pset])
    for k, (s, t) in enumerate(pairs):
        want = oracle_e01(shape, s, t, PARAM_SETS[pset])
        assert got[k].tobytes() == want.tobytes(), (shape, k, s, t)


def test_thread_counts_agree():
    """threads = 1 and threads = 7 give the same bytes, on many maps (split over maps) and one map (split over rows)."""
    shape, pairs = _pairs_37x53()
    one = e01_host(shape, pairs, MAACO_DEFAULT, threads=1)
    assert one.tobytes() == e01_host(shape, pairs, MAACO_DEFAULT, threads=7).tobytes()
    assert one.tobytes() == e01_host(shape, pairs, MAACO_DEFAULT).tobytes()
    big, bp = _pairs_256()
    assert e01_host(big, bp[:1], MAACO_DEFAULT, threads=1).tobytes() == \
        e01_host(big, bp[:1], MAACO_DEFAULT, threads=7).tobytes()


def test_e01_host_is_the_shared_table_builder():
    """mpp_maaco_tables' shared table comes from the same code: a pair repeated in a batch gives equal tables."""
    shape, pairs = _pairs_37x53()
    got = e01_host(shape, [pairs[0]] * 3 + [pairs[1]], MAACO_DEFAULT, threads=2)
    assert got[0].tobytes() == got[1].tobytes() == got[2].tobytes() != got[3].tobytes()


def test_empty_batch_and_bad_cells():
    from maaco_path_planing_b200 import _lib
    from maaco_path_planing_b200.batch import _maaco_params
    L = _lib.lib()
    p = _maaco_params(1, **MAACO_DEFAULT)
    out = np.zeros(2 * 12)
    i32 = lambda v: np.array(v, np.int32)
    call = lambda n, s, t: L.mpp_maaco_e01_host(3, 4, n, i32(s).ctypes.data_as(C.c_void_p),
                                                i32(t).ctypes.data_as(C.c_void_p), C.byref(p),
                                                out.ctypes.data_as(C.c_void_p), 0)
    assert call(0, [], []) == 0
    assert call(1, [0], [11]) == 0 and np.isfinite(out).all()
    for s, t in ((12, 0), (0, 12), (-1, 5), (5, -1)):
        assert call(1, [s], [t]) == -1                                          # MPP_EINVAL
        assert b"outside the 3 x 4 map" in L.mpp_last_error()
    assert call(-1, [], []) == -1 and b"n = -1" in L.mpp_last_error()
    with pytest.raises(_lib.MppError, match="mpp_maaco_e01_host.*outside"):
        e01_host((3, 4), [(0, 12)], MAACO_DEFAULT)
