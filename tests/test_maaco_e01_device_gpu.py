"""MAACO's per-map eta'**beta tables on the device (mpp_maaco_e01_maps): the exp / pow replicas it evaluates give, on
sm_100a, the host libm's bits; its tables equal mpp_maaco_e01_host's byte for byte over shapes, endpoint pairs and
parameter sets, for host-built and device-built batches on a side stream; and a process whose libm probe fails builds
per-map tables on the host with the same results."""
import ctypes as C

import numpy as np
import pytest

from conftest import MAACO_DEFAULT

PARAM_SETS = {
    "default": MAACO_DEFAULT,
    **{f"beta{b}": dict(MAACO_DEFAULT, beta=b) for b in (0.0, 1.0, 2.5, 7.0, 60.0)},
    **{f"k_h{k}": dict(MAACO_DEFAULT, k_h_adaptive=k) for k in (0.0, 0.9, 1e3)},
    "turn_clamp": dict(MAACO_DEFAULT, a_turn_coef=-1e6),                  # d1 = base - 1e6 < 1e-9: the 1e-9 clamp
    "wh_flat": dict(MAACO_DEFAULT, wh_max=0.5, wh_min=0.5),
}


@pytest.mark.gpu
def test_device_replica_equals_host_libm():
    import torch
    import libm_cases as L
    from maaco_path_planing_b200 import _lib
    for e, x, y in (L.directed_args(), L.random_args(2_000_000, 11)):
        want = L.host_libm(e, x, y)
        assert L.mismatches(L.replica(e, x, y), want).size == 0
        args = [torch.from_numpy(a).cuda() for a in (e, x, y)]
        got = torch.empty(2 * e.size, dtype=torch.float64, device="cuda")
        _lib.check(_lib.lib().mpp_libm_exp_pow(e.size, *(_lib.ptr(a) for a in args), _lib.ptr(got),
                                               torch.cuda.current_device(), None), "mpp_libm_exp_pow")
        bad = L.mismatches(got.cpu().numpy(), want)
        assert bad.size == 0, [(i, e[i // 2], x[i // 2], y[i // 2]) for i in bad[:5]]


def _grids(shape, pairs):
    g = np.zeros((len(pairs),) + shape, np.uint8)
    for k, (s, t) in enumerate(pairs):
        g[k].flat[s], g[k].flat[t] = 2, 3
    return g


def _cases():
    from test_maaco_per_map_endpoints_gpu import hard_pairs
    from test_maaco_tables_host import _demo_pairs, _pairs_37x53
    rng = np.random.default_rng(2560)
    cell = lambda C_: (lambda rc: rc[0] * C_ + rc[1])
    out = _demo_pairs()
    shape, pairs = _pairs_37x53()
    out.append((shape, pairs + [(cell(53)(a), cell(53)(b)) for a, b in hard_pairs(37, 53)]))
    out.append(((256, 256), [tuple(int(v) for v in rng.choice(256 * 256, 2, replace=False)) for _ in range(128)]))
    out.append(((100, 150), [(0, 100 * 150 - 1), (149, 99 * 150)] +
                [tuple(int(v) for v in rng.choice(100 * 150, 2, replace=False)) for _ in range(6)]))
    out.append(((1024, 1024), [(5 * 1024 + 7, 1000 * 1024 + 1001)]))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("pset", sorted(PARAM_SETS))
def test_e01_maps_equals_e01_host(pset):
    """Host-built and device-built batches, the kernel on a side stream, against mpp_maaco_e01_host."""
    import torch
    from maaco_path_planing_b200 import _lib
    from maaco_path_planing_b200.batch import _e01_host, _maaco_params, _map_set
    p = _maaco_params(1, **PARAM_SETS[pset])
    side = torch.cuda.Stream()
    for shape, pairs in _cases():
        g = _grids(shape, pairs)
        n = shape[0] * shape[1]
        s, t = (np.array([q[k] for q in pairs], np.int64) for k in (0, 1))
        want = _e01_host(*shape, s, t, p, np.empty(len(pairs) * 2 * n)).reshape(len(pairs), -1)
        for src in (g, torch.from_numpy(g).cuda()):
            maps = _map_set(src)
            assert (maps.start == s).all() and (maps.target == t).all()
            with torch.cuda.stream(side):
                e01 = torch.full((len(pairs), 2 * n), float("nan"), dtype=torch.float64, device="cuda")
                _lib.check(_lib.lib().mpp_maaco_e01_maps(maps.handle, C.byref(p), _lib.ptr(e01), 2 * n,
                                                         C.c_void_p(side.cuda_stream)), "mpp_maaco_e01_maps")
                got = e01.cpu().numpy()
            for k in range(len(pairs)):
                assert got[k].tobytes() == want[k].tobytes(), (shape, k, pairs[k], pset)
            maps.close()


@pytest.mark.gpu
def test_e01_maps_rejects_bad_arguments():
    import torch
    from maaco_path_planing_b200 import _lib
    from maaco_path_planing_b200.batch import _maaco_params, _map_set
    L = _lib.lib()
    p = _maaco_params(1, **MAACO_DEFAULT)
    g = _grids((8, 8), [(0, 63), (9, 20)])
    e01 = torch.empty(2 * 2 * 64 + 2, dtype=torch.float64, device="cuda")
    maps = _map_set(g)
    assert L.mpp_maaco_e01_maps(maps.handle, C.byref(p), _lib.ptr(e01), 2 * 64 - 2, None) == -1
    assert L.mpp_maaco_e01_maps(maps.handle, C.byref(p), _lib.ptr(e01), 2 * 64 + 1, None) == -1
    assert L.mpp_maaco_e01_maps(maps.handle, C.byref(p), C.c_void_p(e01.data_ptr() + 8), 2 * 64, None) == -1
    assert b"aligned" in L.mpp_last_error()
    g[1][g[1] == 3] = 0                                                       # map 1 loses its target
    bad = _map_set(g)
    assert L.mpp_maaco_e01_maps(bad.handle, C.byref(p), _lib.ptr(e01), 2 * 64, None) == -1
    assert b"map 1 has no start/target" in L.mpp_last_error()


@pytest.mark.gpu
def test_failed_probe_builds_tables_on_the_host(monkeypatch):
    from maaco_path_planing_b200 import batch
    from maaco_path_planing_b200.batch import solve_maaco_batch
    from test_maaco_per_map_endpoints_gpu import mixed_maps
    grids = mixed_maps(48, 64, 7, 4864)
    N, K, seeds = 128, 3, list(range(7))
    device = solve_maaco_batch(grids, N, K, MAACO_DEFAULT, seeds=seeds, wave=4, per_map_endpoints=True)
    assert batch._DEVICE_E01 is True
    calls = []
    host = batch._e01_host
    monkeypatch.setattr(batch, "_DEVICE_E01", False)
    monkeypatch.setattr(batch, "_e01_host", lambda *a, **kw: calls.append(len(a[2])) or host(*a, **kw))
    monkeypatch.setattr(batch, "_libm_probe", lambda *a: pytest.fail("the probe runs once per process"))
    assert solve_maaco_batch(grids, N, K, MAACO_DEFAULT, seeds=seeds, wave=4, per_map_endpoints=True) == device
    assert calls == [4, 3]
