"""Map batches built from grids that are already on the GPU (mpp_map_batch_create_device, batch.py's device input).

The ingestion kernel must give the bytes the host path gives -- occupancy words, svalid masks, per-map start / target and
the obstacle count -- for uint8, int32 and int64 cells, whatever values the cells hold.  Every batch class and sweep must
return from a CUDA tensor exactly what it returns from the same grids as NumPy (values and Python types), without the
grids going through the host, in stream order, and a repeated wave must not see later writes to the caller's tensor."""
import ctypes as C
import gc

import numpy as np
import pytest

from conftest import MAACO_DEFAULT
from test_batch_sweeps_gpu import MPA_PARAMS, assert_equals_oracle, serpentine, with_endpoints

INF = float("inf")
SEARCH_POLICY = dict(turn_penalty_factor=0.1, safety_penalty_factor=0.05, min_safe_distance=1.5)
PSO_SIZES, PSO_PARAMS = (2, 32, 2), dict(w=0.7, c1=1.5, c2=1.5)            # iterations, particles, waypoints
GA_SIZES, GA_PARAMS = (2, 32, 2), dict(mutation_rate=0.1, crossover_rate=0.8)


def typed(x):
    """x with the type of every leaf next to its value: == on it compares values and Python types."""
    if isinstance(x, dict):
        return "dict", {k: typed(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return type(x).__name__, [typed(v) for v in x]
    if isinstance(x, np.ndarray):
        return "ndarray", x.dtype.str, x.tolist()
    return type(x).__name__, x


def forbid_host_path(monkeypatch):
    """From here on, grids that went through the host ingestion path raise."""
    from maaco_path_planing_b200 import _lib, batch

    def boom(*a, **k):
        raise AssertionError("device grids went through the host path")
    monkeypatch.setattr(batch, "_grids_u8", boom)
    monkeypatch.setattr(_lib.lib(), "mpp_map_batch_create", boom)


def cuda(grids, dtype=None):
    import torch
    t = torch.as_tensor(np.asarray(grids), device="cuda")
    return t if dtype is None else t.to(dtype)


def maps64(n, seed0, ends=None):
    from maaco_path_planing_b200 import blocks_map
    gs = [blocks_map(64, 0.20, seed=seed0 + i) for i in range(n)]
    return gs if ends is None else [with_endpoints(g, *ends[i % len(ends)]) for i, g in enumerate(gs)]


MIXED_ENDS = [((0, 0), (63, 63)), ((0, 63), (63, 0)), ((10, 50), (40, 5)), ((63, 63), (0, 0))]


# ---- ingestion ---------------------------------------------------------------------------------------------------------

def soup(n_maps, rows, cols, dtype, seed):
    """Random cells: mostly 0 / 1, a few 2 and 3 per map, and values the uint8 path clips (negative, above 255, and for
    int64 ones whose low 32 bits are 1, 2 or 3).  Map 1 has no start and map 2 no target."""
    rng = np.random.default_rng(seed)
    odd = {np.uint8: [255, 254, 4], np.int32: [-1, -254, 256, 257, 258, 259, 2 ** 31 - 1, -2 ** 31, 65538],
           np.int64: [-1, -253, 257, 258, 259, 2 ** 32 + 1, 2 ** 32 + 2, 2 ** 32 + 3, -2 ** 63, 2 ** 63 - 1]}[dtype]
    g = rng.choice(np.array([0, 1], dtype), size=(n_maps, rows, cols), p=[0.7, 0.3])
    n = rows * cols
    for v, p in ((2, 4.0 / n), (3, 4.0 / n)):
        g[rng.random(g.shape) < p] = v
    mask = rng.random(g.shape) < 0.05
    g[mask] = rng.choice(np.array(odd, dtype), size=int(mask.sum()))
    g[0, -1, -2:] = 2, 3                                                    # map 0 has both, whatever was drawn
    if n_maps > 1:
        g[1][g[1] == 2] = 0
    if n_maps > 2:
        g[2][g[2] == 3] = 0
    return g


def batch_bytes(h, n_maps, rows, cols):
    """(occupancy words, svalid bytes, starts, targets, obstacle count) of a map batch, read from the device."""
    import torch
    from maaco_path_planing_b200 import _lib
    L = _lib.lib()
    pitch = C.c_int()
    occ_ptr = L.mpp_map_batch_occ_bits(h, C.byref(pitch))
    occ_words = ((rows + 2) * pitch.value + 3) & ~3

    def read(ptr, n, typestr):
        class View:
            __cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3}
        return torch.as_tensor(View(), device="cuda").cpu().numpy().copy()
    return (read(occ_ptr, n_maps * occ_words, "<u4"), read(L.mpp_map_batch_svalid(h), n_maps * rows * cols, "|u1"),
            [L.mpp_map_batch_start(h, k) for k in range(n_maps)], [L.mpp_map_batch_target(h, k) for k in range(n_maps)],
            L.mpp_map_batch_obstacles(h))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(6, 37, 42), (4, 100, 100), (1, 1000, 1000), (128, 256, 256)])
@pytest.mark.parametrize("dtype", [np.uint8, np.int32, np.int64])
def test_device_ingestion_equals_host_ingestion(shape, dtype):
    """mpp_map_batch_create_device on the raw cells == mpp_map_batch_create on the cells clipped to uint8, byte for
    byte: occupancy (border and tail padding included), svalid, start / target of every map, obstacle count."""
    import torch
    from maaco_path_planing_b200 import _lib
    from maaco_path_planing_b200.batch import _grids_u8
    L = _lib.lib()
    g = soup(*shape, dtype, seed=sum(shape) + np.dtype(dtype).itemsize)
    g8 = _grids_u8(g)
    hh, hd = C.c_void_p(), C.c_void_p()
    _lib.check(L.mpp_map_batch_create(g8.ctypes.data_as(C.c_void_p), *shape, 0, C.byref(hh)), "host")
    t = torch.as_tensor(g, device="cuda")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(L.mpp_map_batch_create_device(t.data_ptr(), t.element_size(), *shape, 0, stream, C.byref(hd)), "device")
    try:
        want, got = batch_bytes(hh, *shape), batch_bytes(hd, *shape)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
        assert got[2:] == want[2:]
        if shape[0] > 2:
            assert got[2][1] == -1 and got[3][2] == -1 and min(got[2][0], got[3][0]) >= 0
    finally:
        L.mpp_map_batch_destroy(hh)
        L.mpp_map_batch_destroy(hd)


@pytest.mark.gpu
def test_device_ingestion_rejects_bad_arguments():
    import torch
    from maaco_path_planing_b200 import _lib
    L = _lib.lib()
    h = C.c_void_p()
    t = torch.zeros((2, 8, 8), dtype=torch.int16, device="cuda")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert L.mpp_map_batch_create_device(t.data_ptr(), 2, 2, 8, 8, 0, stream, C.byref(h)) == -1
    assert b"elem_bytes" in L.mpp_last_error()
    host = np.zeros((2, 8, 8), np.uint8)
    assert L.mpp_map_batch_create_device(host.ctypes.data_as(C.c_void_p), 1, 2, 8, 8, 0, stream, C.byref(h)) == -1
    assert b"not memory of device" in L.mpp_last_error()


# ---- the batch classes -------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_maaco_config5_wave_from_device_grids(monkeypatch):
    """MAACOBatch at the config-5 launch shape (128 256x256 maps, 1024 ants) from an int64 CUDA tensor: per-ant records
    and tau after every pass, and the solution, == the same wave from host grids."""
    import torch
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    M, N, K = 128, 1024, 3
    grids = np.stack([blocks_map(256, 0.20, seed=5000 + i) for i in range(M)])
    seeds = list(range(M))
    dev = cuda(grids)
    host = MAACOBatch(grids, N, K, seeds=seeds, **MAACO_DEFAULT)
    forbid_host_path(monkeypatch)
    b = MAACOBatch(dev, N, K, seeds=seeds, **MAACO_DEFAULT)
    assert b.device == dev.device
    for it in (1, 2):
        host.run_iteration(it)
        b.run_iteration(it)
        for x, y in zip(host.last_results(), b.last_results()):
            assert np.array_equal(x, y), it
        assert np.array_equal(host.pheromone(), b.pheromone()), it
    assert typed(b.solve()) == typed(host.solve())
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_mpa_search_pso_ga_from_device_grids(monkeypatch):
    """MPABatch, SearchBatch (solve astar / dijkstra, search with per-map endpoints), PSOBatch and GABatch on maps with
    their own endpoints: a CUDA tensor of each accepted integer width gives what the NumPy grids give."""
    import torch
    from maaco_path_planing_b200.batch import GABatch, MPABatch, PSOBatch, SearchBatch
    grids = np.stack(maps64(4, 640, MIXED_ENDS))
    seeds = [21, 22, 23, 24]
    rng = np.random.default_rng(7)
    mi = rng.integers(0, 4, 64)
    src, dst = rng.integers(0, 64 * 64, 64), rng.integers(0, 64 * 64, 64)

    def run(g):
        out = {"mpa": MPABatch(g, 128, 4, seeds=seeds, **MPA_PARAMS).solve()}
        sb = SearchBatch(g, **SEARCH_POLICY)
        out["astar"], out["dijkstra"] = sb.solve("astar"), sb.solve("dijkstra")
        out["search"] = [x.cpu().numpy() for x in sb.search(0, mi, src, dst)]
        p = PSOBatch(g, *PSO_SIZES, **PSO_PARAMS, seeds=seeds)
        out["pso"] = p.solve()
        out["pso_state"] = [x.cpu().numpy() for x in (p.pos, p.vel, p.pbest_fit)]
        q = GABatch(g, *GA_SIZES, **GA_PARAMS, seeds=seeds)
        out["ga"] = q.solve()
        out["ga_state"] = [x.cpu().numpy() for x in (q.chrom, q.fitness)]
        return typed(out)

    want = run(grids)
    forbid_host_path(monkeypatch)
    for dtype in (torch.uint8, torch.int16, torch.int32, torch.int64):
        assert run(cuda(grids, dtype)) == want, dtype


@pytest.mark.gpu
def test_sweeps_over_mixed_shape_device_sequences(monkeypatch):
    """Every sweep over a sequence of 2-D CUDA tensors of three shapes == the same sweep over the NumPy maps; for
    solve_maaco_batch the waves and which of them reuse the previous wave's buffers are the same too."""
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200 import batch
    ends = [((0, 0), (47, 47)), ((0, 47), (47, 0))]
    grids = []
    for i in range(9):
        n = (48, 40, 48)[i % 3]
        grids.append(with_endpoints(blocks_map(n, 0.20, seed=900 + i), *ends[(i // 3) % 2]) if n == 48 else
                     blocks_map(n, 0.20, seed=900 + i))
    grids.insert(4, with_endpoints(blocks_map(56, 0.20, seed=956)[:, :44], (0, 0), (55, 43)))
    seeds = [300 + i for i in range(len(grids))]

    def run(gs):
        seen = []

        class Recording(batch.MAACOBatch):
            def __init__(self, grids, *args, reuse=None, **kw):
                super().__init__(grids, *args, reuse=reuse, **kw)
                seen.append((self.n_maps, reuse is not None and self._moves.data_ptr() == reuse._moves.data_ptr()))
        monkeypatch.setattr(batch, "MAACOBatch", Recording)
        out = {"maaco": batch.solve_maaco_batch(gs, 64, 2, MAACO_DEFAULT, seeds=seeds, wave=2)}
        monkeypatch.setattr(batch, "MAACOBatch", Recording.__mro__[1])
        out["waves"] = seen
        out["mpa"] = batch.solve_mpa_batch(gs, 64, 3, MPA_PARAMS, seeds=seeds, wave=2)
        out["astar"] = batch.solve_search_batch(gs, "astar", SEARCH_POLICY, wave=2)
        out["dijkstra"] = batch.solve_search_batch(gs, "dijkstra", SEARCH_POLICY)
        out["pso"] = batch.solve_pso_batch(gs, *PSO_SIZES, PSO_PARAMS, seeds=seeds, wave=3)
        out["ga"] = batch.solve_ga_batch(gs, *GA_SIZES, GA_PARAMS, seeds=seeds)
        return out

    want = run(grids)
    assert any(reused for _, reused in want["waves"])
    forbid_host_path(monkeypatch)
    assert typed(run([cuda(g) for g in grids])) == typed(want)


@pytest.mark.gpu
def test_sweeps_over_a_device_tensor_and_its_shards(monkeypatch):
    """A 3-D CUDA tensor is a sequence of maps too; with group= each rank slices its [lo, hi) maps on the device."""
    import torch
    import torch.distributed as dist
    from maaco_path_planing_b200 import batch
    grids = np.stack(maps64(5, 520, MIXED_ENDS[:2]))
    seeds = [50 + i for i in range(5)]
    want_maaco = batch.solve_maaco_batch(grids, 64, 2, MAACO_DEFAULT, seeds=seeds, wave=2)
    want_astar = batch.solve_search_batch(grids, "astar", SEARCH_POLICY)
    forbid_host_path(monkeypatch)
    dev = cuda(grids, torch.int32)
    assert typed(batch.solve_maaco_batch(dev, 64, 2, MAACO_DEFAULT, seeds=seeds, wave=2)) == typed(want_maaco)
    monkeypatch.setattr(dist, "get_world_size", lambda group: 2)
    shards = []
    for rank in (0, 1):
        monkeypatch.setattr(dist, "get_rank", lambda group, r=rank: r)
        shards += batch.solve_search_batch(dev, "astar", SEARCH_POLICY, group=object())
    assert typed(shards) == typed(want_astar)


# ---- repeats, stream order, devices ------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_repeated_waves_do_not_see_later_writes(monkeypatch):
    """The serpentine's best path outgrows the default path capacity, so MAACOBatch.solve() repeats the wave: with the
    caller's tensor overwritten after construction the repeat still returns the oracle's path.  MPABatch's buffer
    regrowth (forced with a tiny heap and path buffer) likewise returns what the host grids give."""
    import pyoracle as O
    from maaco_path_planing_b200.batch import MAACOBatch, MPABatch, default_max_cells
    g = serpentine()
    N, K, seed = 32, 3, 11
    forbid_host_path(monkeypatch)
    dev = cuda(g[None])
    b = MAACOBatch(dev, N, K, seeds=[seed], **MAACO_DEFAULT)
    assert b.max_cells == default_max_cells(48, 48)
    dev.zero_()
    res = b.solve()
    assert b.max_cells == 48 * 48                                           # the wave was repeated
    assert_equals_oracle(res[0], O.MaacoOracle(g, N, K, seed=seed, threads=0, **MAACO_DEFAULT), 48)
    monkeypatch.undo()
    grids = np.stack(maps64(3, 660, MIXED_ENDS))
    kw = dict(seeds=[1, 2, 3], max_cells=16, heap_cap=64, **MPA_PARAMS)
    want = MPABatch(grids, 64, 3, **kw).solve()
    forbid_host_path(monkeypatch)
    dev = cuda(grids)
    m = MPABatch(dev, 64, 3, **kw)
    dev.fill_(1)
    assert typed(m.solve()) == typed(want)
    assert m.max_cells == 16 and m.heap_cap == 64                          # the repeats ran on their own instances


@pytest.mark.gpu
def test_grids_written_on_a_side_stream():
    """Grids produced by torch kernels on a non-default stream and handed to the batch classes under that stream, with
    no synchronise in between, give what the host grids give: ingestion is ordered on torch's current stream."""
    import torch
    from maaco_path_planing_b200.batch import MAACOBatch, SearchBatch
    grids = np.stack(maps64(4, 700, MIXED_ENDS[:1]))
    want_s = SearchBatch(grids, **SEARCH_POLICY).solve("astar")
    want_m = MAACOBatch(grids, 64, 2, seeds=[1, 2, 3, 4], **MAACO_DEFAULT).solve()
    base = cuda(grids)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for cls, args, want in ((SearchBatch, (), want_s), (MAACOBatch, (64, 2), want_m)):
            if hasattr(torch.cuda, "_sleep"):
                torch.cuda._sleep(20_000_000)                               # the writes land late on s
            g = torch.full_like(base, 1)
            g.copy_(base)                                                   # written on s, read right after
            b = cls(g, *args, **(SEARCH_POLICY if cls is SearchBatch else dict(seeds=[1, 2, 3, 4], **MAACO_DEFAULT)))
            got = b.solve("astar") if cls is SearchBatch else b.solve()
            assert typed(got) == typed(want), cls.__name__
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_tensor_on_another_gpu():
    """device= naming another GPU than the tensor's: the maps are copied there device to device."""
    import torch
    from maaco_path_planing_b200.batch import SearchBatch, solve_search_batch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    grids = np.stack(maps64(3, 740, MIXED_ENDS))
    want = SearchBatch(grids, device=1, **SEARCH_POLICY).solve("astar")
    sb = SearchBatch(cuda(grids), device=1, **SEARCH_POLICY)
    assert sb.device == torch.device("cuda", 1)
    assert typed(sb.solve("astar")) == typed(want)
    assert typed([r[1:] for r in solve_search_batch([cuda(g) for g in grids], "astar", SEARCH_POLICY, device=1)]) == \
        typed([tuple(r) for r in want])


# ---- errors ------------------------------------------------------------------------------------------------------------

def _error(fn):
    with pytest.raises(ValueError) as e:
        fn()
    return str(e.value)


@pytest.mark.gpu
def test_missing_endpoints_raise_the_host_errors(monkeypatch):
    """Maps without a start or a target: every class and sweep raises, from CUDA tensors, the message it raises from
    host grids, and a class frees the map batch it built before raising."""
    import torch
    from maaco_path_planing_b200 import _lib, batch
    ok = maps64(1, 780)[0]
    no_s, no_t = ok.copy(), ok.copy()
    no_s[no_s == 2] = 0
    no_t[no_t == 3] = 0
    cases = [[ok, no_s], [ok, no_t], [no_s * 0], [no_t, no_s], [no_s, no_t]]
    runs = {
        "MAACOBatch": lambda g: batch.MAACOBatch(g, 8, 1, **MAACO_DEFAULT),
        "MPABatch": lambda g: batch.MPABatch(g, 8, 1),
        "SearchBatch.astar": lambda g: batch.SearchBatch(g).solve("astar"),
        "SearchBatch.dijkstra": lambda g: batch.SearchBatch(g).solve("dijkstra"),
        "PSOBatch": lambda g: batch.PSOBatch(g, *PSO_SIZES, **PSO_PARAMS),
        "GABatch": lambda g: batch.GABatch(g, *GA_SIZES, **GA_PARAMS),
    }
    sweeps = {
        "solve_maaco_batch": lambda gs: batch.solve_maaco_batch(gs, 8, 1, MAACO_DEFAULT),
        "solve_mpa_batch": lambda gs: batch.solve_mpa_batch(gs, 8, 1, {}),
        "solve_search_batch": lambda gs: batch.solve_search_batch(gs, "dijkstra", {}),
        "solve_pso_batch": lambda gs: batch.solve_pso_batch(gs, *PSO_SIZES, PSO_PARAMS),
        "solve_ga_batch": lambda gs: batch.solve_ga_batch(gs, *GA_SIZES, GA_PARAMS),
    }
    L = _lib.lib()
    created, destroyed = [], []
    create, destroy = L.mpp_map_batch_create_device, L.mpp_map_batch_destroy

    def create_rec(*a):
        rc = create(*a)
        created.append(a[-1]._obj.value)
        return rc

    def destroy_rec(h):
        destroyed.append(h.value if isinstance(h, C.c_void_p) else h)
        destroy(h)
    for grids in cases:
        for name, fn in runs.items():
            want = _error(lambda: fn(np.stack(grids)))
            monkeypatch.setattr(L, "mpp_map_batch_create_device", create_rec)
            monkeypatch.setattr(L, "mpp_map_batch_destroy", destroy_rec)
            gc.collect()                                                    # batches left over from earlier runs
            created.clear(), destroyed.clear()
            assert _error(lambda: fn(cuda(np.stack(grids)))) == want, (name, len(grids))
            if not name.startswith("SearchBatch"):
                # freed before the error propagated (the garbage collector may free other, unreferenced batches meanwhile)
                assert created and set(created) <= set(destroyed), name
            monkeypatch.undo()
        for name, fn in sweeps.items():
            want = _error(lambda: fn(grids))
            assert _error(lambda: fn([cuda(g) for g in grids])) == want, (name, len(grids))
    # bool grids hold no start: the error of the same bool grids on the host
    flag = torch.zeros((2, 8, 8), dtype=torch.bool, device="cuda")
    assert _error(lambda: runs["MAACOBatch"](flag)) == _error(lambda: runs["MAACOBatch"](flag.cpu().numpy()))


@pytest.mark.gpu
def test_float_and_misshapen_tensors_are_rejected():
    import torch
    from maaco_path_planing_b200 import batch
    g = cuda(np.stack(maps64(2, 800)), torch.float32)
    for fn in (lambda x: batch.MAACOBatch(x, 8, 1, **MAACO_DEFAULT), lambda x: batch.SearchBatch(x),
               lambda x: batch.MPABatch(x, 8, 1), lambda x: batch.PSOBatch(x, *PSO_SIZES, **PSO_PARAMS),
               lambda x: batch.solve_search_batch(x, "astar", {}), lambda x: batch.solve_maaco_batch(list(x), 8, 1,
                                                                                                    MAACO_DEFAULT)):
        with pytest.raises(TypeError, match="bool, uint8, int8, int16, int32 or int64"):
            fn(g)
        with pytest.raises(ValueError, match=r"grids must be \[n_maps, rows, cols\]"):
            fn(g[0].long())
