"""Batched sweeps over independent maps (BASELINE config 5: "10k independent 256x256 maps x population 1024,
MPA+MAACO, maps sharded across 8 B200").  Maps are independent units, so they are sharded over the ranks with no
data-path collective, and on each GPU a WAVE of same-shape maps is one mpp_map_batch: every colony pass of the
whole wave is four kernel launches (ranking, tours, best tracking, pheromone update with grid.y = map), enqueued
without host synchronisation.  Results are identical to solving each map alone with the same seed.

The eta'**beta / dist-to-target tables depend only on (shape, start, target, parameters), so by default a MAACO wave
holds maps of one (start, target) pair and shares ONE table computed on the host with libm (bit-identical to the
reference), and tau0 of each map is that shared table with the map's obstacles masked on the device
(mpp_maaco_tables).  With per_map_endpoints=True a wave may mix endpoints: it then holds one eta'**beta table per map,
built on the device with replicas of the host libm's exp / pow (mpp_maaco_e01_maps, bit for bit mpp_maaco_e01_host's),
and tau0 is computed per map on the device (mpp_maaco_tau0_maps).

Every batch class takes `grids` either on the host ([M, rows, cols] cell codes, anything np.asarray takes) or as an
[M, rows, cols] CUDA tensor of bool, uint8, int8, int16, int32 or int64 cells; every sweep also takes a sequence of 2-D
CUDA tensors.  Device grids are packed on the GPU, on torch's current stream (mpp_map_batch_create_device), and never go
through the host; results are the same as from the same grids on the host."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .gridmap import START_NODE_VAL, TARGET_NODE_VAL

INF = float("inf")


def shard_maps(n_maps, group=None):
    """[lo, hi) of the maps this rank owns."""
    if group is None:
        return 0, n_maps
    import torch.distributed as dist
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    per = (n_maps + world - 1) // world
    return min(n_maps, rank * per), min(n_maps, (rank + 1) * per)


def default_max_cells(rows, cols):
    """Per-ant path capacity of MAACO and MAACOBatch when `max_cells` is not given: tours are a few (rows + cols) cells
    long (MAACO.py:278-302 never backtracks); a best path that does not fit makes the solve repeat with rows * cols."""
    return min(rows * cols, max(1024, 8 * (rows + cols)))


def _grids_u8(grids):
    """[n_maps, rows, cols] cell codes as uint8 (what mpp_map_batch_create takes): values clipped to 0..255 like
    np.clip(int grid), written straight into the byte array (an int64 wave of 128 256x256 maps is 67 MB: the
    intermediate int64 copies cost more host time than the wave's passes cost on the GPU)."""
    g = np.asarray(grids)
    if g.ndim != 3:
        raise ValueError("grids must be [n_maps, rows, cols]")
    if g.dtype == np.uint8:
        return np.ascontiguousarray(g)
    if g.dtype.kind not in "iub":
        g = g.astype(int)                                                     # (the reference indexes int grids)
    g8 = np.empty(g.shape, np.uint8)
    np.clip(g, 0, 255, out=g8, casting="unsafe")
    return g8


_DEVICE_DTYPES = "bool, uint8, int8, int16, int32 or int64"


def _on_device(grids):
    """True for device grids: a CUDA tensor, or a sequence whose first map is one."""
    import torch
    if isinstance(grids, torch.Tensor):
        return grids.is_cuda
    return (not isinstance(grids, np.ndarray) and len(grids) > 0 and isinstance(grids[0], torch.Tensor)
            and grids[0].is_cuda)


def _device_cells(g):
    """g (a CUDA tensor of cell codes) with bool / int8 / int16 widened to a width mpp_map_batch_create_device reads
    (uint8 / int32); floating-point and other dtypes raise TypeError."""
    import torch
    widen = {torch.bool: torch.uint8, torch.int8: torch.int32, torch.int16: torch.int32, torch.uint8: None,
             torch.int32: None, torch.int64: None}
    if g.dtype not in widen:
        raise TypeError(f"device grids must hold {_DEVICE_DTYPES} cell codes, not {g.dtype}")
    return g if widen[g.dtype] is None else g.to(widen[g.dtype])


def _first_cells(flat):
    """First row-major start (2) and target (3) cell of every row of `flat` ([n_maps, rows*cols] cell codes on the host),
    -1 = none: what the reference constructors look for (MAACO.py:32-41, astar.py:17-18, ...)."""
    ends = []
    for v in (START_NODE_VAL, TARGET_NODE_VAL):
        hit = flat == v
        ends.append(np.where(hit.any(axis=1), hit.argmax(axis=1), -1))
    return tuple(ends)


class _MapSet:
    """An mpp_map_batch with what Python reads from it: (n_maps, rows, cols), its device and every map's first
    row-major start and target cell (-1 = none).  A wave repeated with more buffer room shares its MapSet, so the handle
    is freed when the last batch object holding it lets go of it (or by close())."""

    def __init__(self, handle, shape, device_index, start, target):
        self.handle, self.shape, self.device_index = handle, tuple(int(x) for x in shape), int(device_index)
        self.start, self.target = np.asarray(start, np.int64), np.asarray(target, np.int64)

    def close(self):
        h, self.handle = self.handle, None
        if h:
            _lib.lib().mpp_map_batch_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _map_set(grids, device=None, check=None):
    """The _MapSet every batch class solves on (a _MapSet is returned as it is).  Host grids ([n_maps, rows, cols] cell
    codes, anything np.asarray takes) go through _grids_u8 and mpp_map_batch_create; a [n_maps, rows, cols] CUDA tensor
    goes through mpp_map_batch_create_device on torch's current stream and never leaves the GPU -- it runs on its own
    device unless `device` names another, which then receives a copy of just these maps.  check(start, target) raises
    the planner's errors for maps without a start or target: for host grids before any device work, for device grids
    from the endpoints the ingestion read back, after freeing the handle."""
    import torch
    if isinstance(grids, _MapSet):
        return grids
    L = _lib.lib()
    h = C.c_void_p()
    if isinstance(grids, torch.Tensor) and grids.is_cuda:
        if grids.dim() != 3:
            raise ValueError("grids must be [n_maps, rows, cols]")
        g = grids if device is None else grids.to(torch.device("cuda", int(device)))
        g = _device_cells(g).contiguous()
        _lib.require_device()
        M, R, Cc = g.shape
        stream = C.c_void_p(torch.cuda.current_stream(g.device).cuda_stream)
        _lib.check(L.mpp_map_batch_create_device(g.data_ptr(), g.element_size(), M, R, Cc, g.device.index, stream,
                                                 C.byref(h)), "mpp_map_batch_create_device")
        maps = _MapSet(h, g.shape, g.device.index, [L.mpp_map_batch_start(h, k) for k in range(M)],
                       [L.mpp_map_batch_target(h, k) for k in range(M)])
        if check is not None:
            try:
                check(maps.start, maps.target)
            except ValueError:
                maps.close()
                raise
        return maps
    g8 = _grids_u8(grids)
    start, target = _first_cells(g8.reshape(g8.shape[0], -1))
    if check is not None:
        check(start, target)
    _lib.require_device()
    dev = torch.cuda.current_device() if device is None else int(device)
    _lib.check(L.mpp_map_batch_create(g8.ctypes.data_as(C.c_void_p), *g8.shape, dev, C.byref(h)), "mpp_map_batch_create")
    return _MapSet(h, g8.shape, dev, start, target)


def _all_endpoints(no_start, no_target):
    """MAACOBatch's / MPABatch's check: any map without a start raises no_start, else any without a target no_target."""
    def check(start, target):
        if (start < 0).any():
            raise ValueError(no_start)
        if (target < 0).any():
            raise ValueError(no_target)
    return check


def _maaco_params(num_iterations, alpha, beta, rho, Q, a_turn_coef, wh_max, wh_min, k_h_adaptive, q0_initial,
                  C0_initial_pheromone=0.1):
    """mpp_maaco_params of MAACO's parameters (MAACO.py:11-14)."""
    return _lib.MaacoParams(alpha, beta, rho, Q, a_turn_coef, wh_max, wh_min, k_h_adaptive, q0_initial,
                            C0_initial_pheromone, num_iterations)


def _e01_host(rows, cols, start, target, params, out, threads=0):
    """eta'**beta tables of the endpoint pairs (start[k], target[k]) of a rows x cols map into `out` (a contiguous
    float64 host tensor or array of at least len(start) * 2 * rows * cols values): mpp_maaco_e01_host."""
    s, t = np.ascontiguousarray(start, np.int32), np.ascontiguousarray(target, np.int32)
    ptr = out.data_ptr() if hasattr(out, "data_ptr") else out.ctypes.data
    _lib.check(_lib.lib().mpp_maaco_e01_host(rows, cols, len(s), s.ctypes.data_as(C.c_void_p),
                                             t.ctypes.data_as(C.c_void_p), C.byref(params), C.c_void_p(ptr), threads),
               "mpp_maaco_e01_host")
    return out


_DEVICE_E01 = None       # per process: do the device's exp / pow match the host's libm?  None = not probed yet


def _libm_probe(device_index):
    """True when mpp_exp / mpp_pow on the GPU -- what mpp_maaco_e01_maps evaluates -- return the host libm's exp / pow
    bit for bit on a fixed seeded probe of 2**16 arguments of each from the tables' domain (exp on [-800, 0]; pow with
    x in [1e-7, 1e9], y in [0, 64], a quarter of the y whole numbers).  The host values come from the C library's exp /
    pow, the functions mpp_maaco_e01_host calls.  A tripwire, not a proof: it catches a host libm other than the build
    the replicas reproduce (glibc 2.39, x86-64, FMA), it cannot show that every argument agrees."""
    import ctypes.util
    import torch
    libm = C.CDLL(ctypes.util.find_library("m"))
    libm.exp.restype, libm.exp.argtypes = C.c_double, [C.c_double]
    libm.pow.restype, libm.pow.argtypes = C.c_double, [C.c_double, C.c_double]
    rng = np.random.default_rng(0x6C69626D)
    n = 1 << 16
    e = rng.uniform(-800.0, 0.0, n)
    x = np.exp(rng.uniform(np.log(1e-7), np.log(1e9), n))
    y = rng.uniform(0.0, 64.0, n)
    y[: n // 4] = np.floor(y[: n // 4])
    want = np.empty(2 * n)
    want[0::2] = [libm.exp(v) for v in e.tolist()]
    want[1::2] = [libm.pow(a, b) for a, b in zip(x.tolist(), y.tolist())]
    dev = torch.device("cuda", device_index)
    args = [torch.from_numpy(a).to(dev) for a in (e, x, y)]
    got = torch.empty(2 * n, dtype=torch.float64, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(_lib.lib().mpp_libm_exp_pow(n, *(_lib.ptr(a) for a in args), _lib.ptr(got), device_index, stream),
               "mpp_libm_exp_pow")
    return bool((got.cpu().numpy().view(np.uint64) == want.view(np.uint64)).all())


def _device_e01(device_index):
    """Whether this process builds per-map eta'**beta tables on the device (mpp_maaco_e01_maps): _libm_probe, run by the
    first per-map wave.  Where it fails every per-map table of the process is built on the host (mpp_maaco_e01_host),
    so the tables stay bit for bit the reference's."""
    global _DEVICE_E01
    if _DEVICE_E01 is None:
        _DEVICE_E01 = _libm_probe(device_index)
    return _DEVICE_E01


class MAACOBatch:
    """M same-shape maps, one colony of `num_ants` ants per map, solved together.  Same parameters as MAACO
    (MAACO.py:11-14); `seeds` = one Philox seed per map.  `max_cells` works as in MAACO: left at its default, solve()
    repeats the whole wave with rows*cols cells of path capacity when a best path did not fit; given explicitly, such a
    wave raises MppError.

    By default the maps must share start and target: they then share one table built once (mpp_maaco_tables), and
    maps with other endpoints raise MppError.  With per_map_endpoints=True each map may have its own start and target:
    the wave then holds one eta'**beta table per map ([M, 2*rows*cols] doubles, 16 B per cell per map, built on the
    device on the wave's stream by mpp_maaco_e01_maps -- or on the host by mpp_maaco_e01_host where _device_e01 says the
    device's exp / pow do not match the host libm), and tau0 is computed on the device from each map's own endpoints
    (mpp_maaco_tau0_maps).  A wave whose maps all share their endpoints takes the shared table
    either way.  Results are those of solo MAACO with the same seed in both modes."""

    def __init__(self, grids, num_ants, num_iterations, alpha, beta, rho, Q, a_turn_coef, wh_max, wh_min, k_h_adaptive,
                 q0_initial, C0_initial_pheromone=0.1, *, seeds=None, device=None, max_cells=None, ants_per_warp=0,
                 reuse=None, per_map_endpoints=False, _e01=None):
        # _e01 (the max_cells repeat): this wave's per-map tables, already built -- an [M, 2 * rows * cols] CUDA tensor
        # on the wave's device, used as it is
        import torch
        L = _lib.lib()
        self._map_set = _map_set(grids, device, _all_endpoints("MAACO: Start node not found.",        # MAACO.py:35-36
                                                               "MAACO: Target node not found."))      # MAACO.py:37-38
        self._maps = self._map_set.handle
        self.n_maps, self.rows, self.cols = self._map_set.shape
        self.device_index = self._map_set.device_index
        self.device = torch.device("cuda", self.device_index)
        self.num_ants, self.num_iterations = int(num_ants), int(num_iterations)
        self.alpha, self.rho, self.Q = alpha, rho, Q
        self._params = _maaco_params(num_iterations, alpha, beta, rho, Q, a_turn_coef, wh_max, wh_min, k_h_adaptive,
                                     q0_initial, C0_initial_pheromone)
        M, R, Cc, N = self.n_maps, self.rows, self.cols, self.num_ants
        start, target = self._map_set.start, self._map_set.target
        # one table per map only where the endpoints differ: a wave that shares them keeps the shared table
        self.per_map_tables = bool(per_map_endpoints) and M > 0 and not (
            (start == start[0]).all() and (target == target[0]).all())
        n = R * Cc
        TR = (R + 31) // 32
        self._auto_cells = max_cells is None
        if max_cells is None:
            max_cells = default_max_cells(R, Cc)
        self.max_cells = int(max_cells)
        self._apw = int(ants_per_warp)
        if seeds is None:
            seeds = [int.from_bytes(np.random.bytes(8), "little") for _ in range(M)]
        self.seeds = [int(s) & (2 ** 64 - 1) for s in seeds]
        self._ctor = dict(num_ants=num_ants, num_iterations=num_iterations, alpha=alpha, beta=beta, rho=rho, Q=Q,
                          a_turn_coef=a_turn_coef, wh_max=wh_max, wh_min=wh_min, k_h_adaptive=k_h_adaptive,
                          q0_initial=q0_initial, C0_initial_pheromone=C0_initial_pheromone, seeds=self.seeds,
                          ants_per_warp=ants_per_warp, per_map_endpoints=per_map_endpoints)
        dev = self.device
        f64, i32, i64, u8 = torch.float64, torch.int32, torch.int64, torch.uint8
        K = max(1, self.num_iterations)
        key = (M, R, Cc, N, self.max_cells, K, self.device_index, self.per_map_tables)   # (the E01 layout)
        if reuse is not None and getattr(reuse, "_key", None) == key:
            # the previous wave's device buffers (same shapes): nothing to allocate, only `touched` / counters to clear
            for name in ("_tau", "_E01", "_dist_t", "_rank", "_slabs", "_touched", "_moves", "_result", "_deposit", "_okbits",
                         "_best_cells", "_steps", "_log"):
                setattr(self, name, getattr(reuse, name))
            self._touched.zero_()
            self._steps.zero_()
        else:
            self._tau = torch.empty((M, n), dtype=f64, device=dev)
            if self.per_map_tables:
                self._E01 = None if _e01 is not None else torch.empty((M, 2 * n), dtype=f64, device=dev)
                self._dist_t = None                                           # nothing in the batch reads it
            else:
                self._E01 = torch.empty(2 * n, dtype=f64, device=dev)         # shared by the whole wave
                self._dist_t = torch.empty(n, dtype=f64, device=dev)
            self._rank = torch.empty(M * L.mpp_maaco_rank_words(R, Cc), dtype=i32, device=dev)
            self._slabs = torch.empty(M * L.mpp_maaco_slab_words(TR, Cc, N), dtype=i32, device=dev)
            self._touched = torch.zeros(M * L.mpp_maaco_touched_words(TR, Cc, N), dtype=i32, device=dev)
            self._moves = torch.empty(M * N * self.max_cells, dtype=u8, device=dev)
            self._result = torch.zeros((M, N, 2), dtype=i64, device=dev)
            self._deposit = torch.zeros((M, N), dtype=f64, device=dev)
            self._okbits = torch.zeros((M, (N + 31) // 32), dtype=i32, device=dev)
            self._best_cells = torch.zeros((M, self.max_cells + 1), dtype=i32, device=dev)
            self._steps = torch.zeros(1, dtype=i64, device=dev)
            self._log = torch.zeros((M, K, 4), dtype=f64, device=dev)
        self._key = key
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        if self.per_map_tables:
            if _e01 is not None:
                if tuple(_e01.shape) != (M, 2 * n) or _e01.device != dev or _e01.dtype != f64:
                    raise ValueError(f"_e01 must be a float64 [{M}, {2 * n}] tensor on {dev}")
                self._E01 = _e01
            elif _device_e01(self.device_index):
                _lib.check(L.mpp_maaco_e01_maps(self._maps, C.byref(self._params), _lib.ptr(self._E01), 2 * n, stream),
                           "mpp_maaco_e01_maps")
            else:
                host = _e01_host(R, Cc, start, target, self._params, torch.empty(M * 2 * n, dtype=f64, pin_memory=True))
                # (a pinned tensor of torch's host allocator is not reused before this copy has run)
                self._E01.view(-1).copy_(host, non_blocking=True)
            _lib.check(L.mpp_maaco_tau0_maps(self._maps, C.byref(self._params), _lib.ptr(self._tau), n, stream),
                       "mpp_maaco_tau0_maps")
        else:
            _lib.check(L.mpp_maaco_tables(self._maps, C.byref(self._params), _lib.ptr(self._tau), n,
                                          _lib.ptr(self._E01), _lib.ptr(self._dist_t), stream), "mpp_maaco_tables")
        self._seeds = torch.from_numpy(np.array(self.seeds, np.uint64).view(np.int64)).to(dev)
        st = bytes(_lib.MaacoState(INF, -1, 0, 0, -1, INF, -1, -1))
        self._state = torch.frombuffer(bytearray(st * M), dtype=u8).to(dev)
        self._colony = _lib.Colony(
            self._tau.data_ptr(), n, self._E01.data_ptr(), 2 * n if self.per_map_tables else 0, self._rank.data_ptr(),
            self._slabs.data_ptr(),
            self._touched.data_ptr(), self._moves.data_ptr(), self.max_cells, K, self._result.data_ptr(),
            self._deposit.data_ptr(), self._okbits.data_ptr(), self._state.data_ptr(), self._best_cells.data_ptr(),
            self._log.data_ptr(), self._steps.data_ptr(), self._seeds.data_ptr(), None)
        self._iter_done = 0
        self.kernel_launches = 0

    def close(self):
        self._maps = self._map_set = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def run_iteration(self, it):
        """Enqueue one colony pass of every map of the wave (asynchronous)."""
        import torch
        if not 1 <= it <= max(1, self.num_iterations):
            raise ValueError(f"iteration {it} outside 1..{self.num_iterations}")
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        _lib.check(_lib.lib().mpp_maaco_pass(self._maps, C.byref(self._colony), C.byref(self._params), it, self.num_ants,
                                             self._apw, stream), "mpp_maaco_pass")
        self.kernel_launches += 4
        self._iter_done = max(self._iter_done, it)

    def pheromone(self):
        return self._tau.cpu().numpy().reshape(self.n_maps, self.rows, self.cols)

    def last_results(self):
        """(n_cells, length, turns), each [n_maps, num_ants], of the last pass."""
        import torch
        torch.cuda.synchronize(self.device)
        rec = self._result.cpu().numpy().view(np.dtype([("length", "<f8"), ("n_cells", "<i4"), ("turns", "<i4")]))
        rec = rec.reshape(self.n_maps, self.num_ants)
        return rec["n_cells"].copy(), rec["length"].copy(), rec["turns"].copy()

    def total_steps(self):
        return int(self._steps.cpu().item())

    def solve(self):
        """Runs the remaining iterations; returns one (path, length, turns, convergence_curve) per map -- the values
        MAACO.solve_path_planning (MAACO.py:334-371) returns / stores for that map."""
        import torch
        for it in range(self._iter_done + 1, self.num_iterations + 1):
            self.run_iteration(it)
        torch.cuda.synchronize(self.device)
        M, K = self.n_maps, self.num_iterations
        st = np.frombuffer(self._state.cpu().numpy().tobytes(), dtype=np.dtype(
            [("best_len", "<f8"), ("best_turns", "<i4"), ("best_n_cells", "<i4"), ("best_iter", "<i4"), ("best_ant", "<i4"),
             ("iter_best_len", "<f8"), ("iter_best_turns", "<i4"), ("iter_best_ant", "<i4")]))
        if (st["best_n_cells"] - 1 > self.max_cells).any():
            if not self._auto_cells or self.max_cells >= self.rows * self.cols:
                raise _lib.MppError(f"a tour outgrew max_cells={self.max_cells} (best path: "
                                    f"{int(st['best_n_cells'].max())} cells); re-run with a larger max_cells")
            # the solve is a deterministic function of (maps, parameters, seeds): repeat the wave with full path capacity
            # on the same map batch (not on the caller's grids, which may have changed since) and per-map tables
            again = type(self)(self._map_set, max_cells=self.rows * self.cols,
                               _e01=self._E01 if self.per_map_tables else None, **self._ctor)
            again.kernel_launches = self.kernel_launches
            self.__dict__.update(again.__dict__)
            return self.solve()
        best = self._best_cells.cpu().numpy()
        log = self._log.cpu().numpy()[:, :K]
        out = []
        for k in range(M):
            nb = int(st["best_n_cells"][k])
            pr, pc = np.divmod(best[k, :nb], self.cols)
            path = list(zip(pr.tolist(), pc.tolist()))
            turns = int(st["best_turns"][k]) if st["best_turns"][k] >= 0 else INF
            curve = [float(v) if v != INF else None for v in log[k, :, 2]]
            out.append((path, float(st["best_len"][k]), turns, curve))
        return out


class _HostSweep:
    """The maps lo..hi-1 of a sweep over host grids: a wave is stacked on the host and uploaded by its batch."""

    def __init__(self, grids, lo, hi):
        self.grids, self.lo, self.hi = grids, lo, hi

    def wave(self, idx):
        return np.stack([np.asarray(self.grids[i]) for i in idx])

    def first_cells(self):
        """(start, target) of maps lo..hi-1: first row-major cell, -1 = none."""
        ends = [_first_cells(np.asarray(self.grids[i]).reshape(1, -1)) for i in range(self.lo, self.hi)]
        return tuple(np.array([e[k][0] for e in ends], np.int64) for k in (0, 1))


class _DeviceSweep:
    """The maps lo..hi-1 of a sweep over device grids (a [n_maps, rows, cols] CUDA tensor or a sequence of 2-D CUDA
    tensors), grouped by shape and stacked on their device once -- the shard of a 3-D tensor is a slice of it -- so a
    wave is a slice of its group (a gather for MAACO's endpoint groups) and no grid goes through the host."""

    def __init__(self, grids, lo, hi):
        import torch
        if isinstance(grids, torch.Tensor):
            if grids.dim() != 3:
                raise ValueError("grids must be [n_maps, rows, cols]")
            self.groups = [(list(range(lo, hi)), grids[lo:hi])] if hi > lo else []
        else:
            self.groups = [(idx, torch.stack([grids[i] for i in idx])) for idx in _shape_waves(grids, lo, hi)]
        for _, g in self.groups:
            _device_cells(g[:0])                                             # dtype check before any work
        self._at = {i: (g, k) for idx, g in self.groups for k, i in enumerate(idx)}
        self.lo, self.hi = lo, hi

    def wave(self, idx):
        import torch
        g, k0 = self._at[idx[0]]
        pos = [self._at[i][1] for i in idx]
        if pos == list(range(k0, k0 + len(idx))):
            return g[k0:k0 + len(idx)]
        return g[torch.as_tensor(pos, device=g.device)]

    def first_cells(self):
        """(start, target) of maps lo..hi-1: first row-major cell, -1 = none; computed on the device, one read back."""
        import torch
        if not self.groups:
            return np.zeros(0, np.int64), np.zeros(0, np.int64)
        ends = []
        for idx, g in self.groups:
            flat = g.reshape(len(idx), -1)
            for v in (START_NODE_VAL, TARGET_NODE_VAL):
                hit = flat == v
                ends.append(torch.where(hit.any(dim=1), hit.to(torch.uint8).argmax(dim=1), -1).to(self.groups[0][1].device))
        ends = torch.cat(ends).cpu().numpy()
        start, target = np.empty(self.hi - self.lo, np.int64), np.empty(self.hi - self.lo, np.int64)
        o = 0
        for idx, _ in self.groups:
            at = np.asarray(idx) - self.lo
            start[at], target[at] = ends[o:o + len(idx)], ends[o + len(idx):o + 2 * len(idx)]
            o += 2 * len(idx)
        return start, target


def _sweep_maps(grids, lo, hi):
    return (_DeviceSweep if _on_device(grids) else _HostSweep)(grids, lo, hi)


def _waves(keys, wave):
    """Group maps into waves of same shape / start / target (what one mpp_map_batch needs); keys: map index -> key."""
    groups = {}
    for i, key in keys.items():
        groups.setdefault(key, []).append(i)
    for idx in groups.values():
        for w0 in range(0, len(idx), wave):
            yield idx[w0:w0 + wave]


def solve_maaco_batch(grids, num_ants, num_iterations, params, seeds=None, wave=256, group=None, device=None,
                      max_cells=None, per_map_endpoints=False):
    """Run MAACO on every grid of `grids` (this rank's shard when `group` is given), `wave` maps per launch.  `grids`:
    host maps, a [n_maps, rows, cols] CUDA tensor or a sequence of 2-D CUDA tensors (which never leave the GPU).

    By default a wave holds maps of one shape and one (start, target) pair, so a sweep whose maps have their own
    endpoints runs one small wave per pair.  With per_map_endpoints=True waves are formed by shape only, in index order
    (MAACOBatch(per_map_endpoints=True), whose per-map eta'**beta tables are built on the device).  A map without a
    start or target then raises before any wave runs.

    Returns a list of (map_index, path, length, turns, convergence_curve) for the maps of this rank; results
    are identical to solving each map alone (same seeds => same Philox streams)."""
    lo, hi = shard_maps(len(grids), group)
    maps = _sweep_maps(grids, lo, hi)
    start, target = maps.first_cells()
    if per_map_endpoints:
        _all_endpoints("MAACO: Start node not found.", "MAACO: Target node not found.")(start, target)
        waves = _shape_waves(grids, lo, hi, wave)
    else:
        waves = _waves({i: (_map_shape(grids[i]), start[i - lo], target[i - lo]) for i in range(lo, hi)}, wave)
    out = []
    prev = None
    for idx in waves:
        b = MAACOBatch(maps.wave(idx), num_ants, num_iterations,
                       seeds=None if seeds is None else [seeds[i] for i in idx], device=device, max_cells=max_cells,
                       reuse=prev, per_map_endpoints=per_map_endpoints, **params)
        for i, (path, length, turns, curve) in zip(idx, b.solve()):
            out.append((i, path, length, turns, curve))
        b.close()
        prev = b
    out.sort(key=lambda r: r[0])
    return out


class MPABatch:
    """M same-shape maps, one MPA population of `num_predators` paths per map, every iteration of every map in one
    launch (mpp_mpa_iteration_batch); the stable sorts (MPA.py:333,412) are a batched device argsort whose index
    the kernel reads through, and the best-so-far cascade (MPA.py:415-437) is a few vector operations over the maps --
    no host round trip inside the solve.  Same parameters as MPA (MPA.py:10-18); `seeds` = one Philox seed per map."""

    def __init__(self, grids, num_predators, num_iterations, FADs_rate=0.2, P_const=0.5, levy_beta=1.5,
                 turn_penalty_factor=0.1, safety_penalty_factor=0.05, min_safe_distance=1.5, allow_diagonal_moves=True,
                 restrict_diagonal_near_obstacle=True, diagonal_obstacle_penalty=1000.0, *, seeds=None, device=None,
                 max_cells=None, heap_cap=None, warps_per_map=None):
        import math
        import torch
        from .engine import make_policy
        self._map_set = _map_set(grids, device, _all_endpoints("MPA: Start node not found in grid.",      # MPA.py:36-37
                                                               "MPA: Target node not found in grid."))    # MPA.py:38-39
        self._maps = self._map_set.handle
        self.n_maps, self.rows, self.cols = self._map_set.shape
        self.device_index = self._map_set.device_index
        self.device = torch.device("cuda", self.device_index)
        self.num_predators, self.num_iterations = int(num_predators), int(num_iterations)
        self.FADs_rate, self.P_const, self.levy_beta = FADs_rate, P_const, levy_beta
        self.policy = make_policy(turn_penalty_factor, safety_penalty_factor, min_safe_distance, diagonal_obstacle_penalty,
                                  restrict_diagonal_near_obstacle, allow_diagonal_moves, mode=1)
        b = levy_beta                                                         # Levy sigma MPA.py:251-253
        num = math.gamma(1 + b) * math.sin(math.pi * b / 2)
        den = math.gamma((1 + b) / 2) * b * (2 ** ((b - 1) / 2))
        sig = (num / den) ** (1 / b) if den > 1e-9 else 1.0
        if isinstance(sig, complex):
            raise ValueError("levy_beta gives a complex Levy sigma in the reference expression (MPA.py:253)")
        self._levy_sigma = float(sig)
        n = self.rows * self.cols
        self.max_cells = int(max_cells or min(n, max(1024, 4 * (self.rows + self.cols))))
        self.heap_cap = int(heap_cap or min(8 * n, max(4096, n // 4)))
        if seeds is None:
            seeds = [int.from_bytes(np.random.bytes(8), "little") for _ in range(self.n_maps)]
        self.seeds = [int(s) & (2 ** 64 - 1) for s in seeds]
        sm = torch.cuda.get_device_properties(self.device).multi_processor_count
        # search slots (one warp each): three CTAs of 8 warps per SM in total, split evenly over the maps (at least one CTA each)
        self.warps_per_map = int(warps_per_map or max(8, ((sm * 24) // self.n_maps) // 8 * 8))
        self._ctor = dict(num_predators=num_predators, num_iterations=num_iterations, FADs_rate=FADs_rate,
                          P_const=P_const, levy_beta=levy_beta, turn_penalty_factor=turn_penalty_factor,
                          safety_penalty_factor=safety_penalty_factor, min_safe_distance=min_safe_distance,
                          allow_diagonal_moves=allow_diagonal_moves,
                          restrict_diagonal_near_obstacle=restrict_diagonal_near_obstacle,
                          diagonal_obstacle_penalty=diagonal_obstacle_penalty, seeds=self.seeds,
                          warps_per_map=warps_per_map)
        self.predator_evaluations = 0
        self.kernel_launches = 0

    def close(self):
        self._maps = self._map_set = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def solve(self):
        """Returns one (path, length, turns, safety_p, diag_p, fitness, convergence_curve) per map -- what
        MPA.solve_path_planning (MPA.py:320-448) returns / stores for that map."""
        import torch
        t = torch
        L = _lib.lib()
        dev = self.device
        M, N, K, mc = self.n_maps, self.num_predators, self.num_iterations, self.max_cells
        words = (self.rows * self.cols + 31) // 32
        slots = self.warps_per_map * M
        slot_bytes = L.mpp_astar_slot_bytes(self.rows, self.cols, self.heap_cap)
        scratch = t.zeros(256 + max(slots, M) * slot_bytes, dtype=t.uint8, device=dev)
        cells = [t.zeros((M, N, mc), dtype=t.int32, device=dev) for _ in range(2)]
        ncell = [t.zeros((M, N), dtype=t.int32, device=dev) for _ in range(2)]
        stats = [t.zeros((M, N, 5), dtype=t.float64, device=dev) for _ in range(2)]
        tmp = t.empty((slots, mc), dtype=t.int32, device=dev)
        avoid = t.empty((slots, words), dtype=t.int32, device=dev)
        queue = t.zeros(M, dtype=t.int32, device=dev)
        status = t.zeros(1, dtype=t.int32, device=dev)
        counters = t.zeros(4, dtype=t.int64, device=dev)
        seeds = t.from_numpy(np.array(self.seeds, np.uint64).view(np.int64)).to(dev)
        stream = C.c_void_p(t.cuda.current_stream(dev).cuda_stream)
        # ---- initial population: one search per map, replicated (MPA.py:231-245) ----
        _lib.check(L.mpp_mpa_init_batch(self._maps, C.byref(self.policy), N, mc, _lib.ptr(cells[0]), _lib.ptr(ncell[0]),
                                        _lib.ptr(stats[0]), _lib.ptr(scratch), scratch.numel(), self.heap_cap,
                                        _lib.ptr(status), _lib.ptr(counters), stream), "mpp_mpa_init_batch")
        cells[0][:, 1:] = cells[0][:, :1]
        ncell[0][:, 1:] = ncell[0][:, :1]
        stats[0][:, 1:] = stats[0][:, :1]
        self.kernel_launches += 1
        rows = t.arange(M, device=dev)

        def elite(buf):
            order = t.sort(stats[buf][:, :, 4], dim=1, stable=True).indices.to(t.int32).contiguous()   # list.sort is stable
            e = order[:, 0].long()
            return order, stats[buf][rows, e], cells[buf][rows, e], ncell[buf][rows, e]

        order, best_stats, best_cells, best_n = elite(0)                       # MPA.py:322-330
        best_stats, best_cells, best_n = best_stats.clone(), best_cells.clone(), best_n.clone()
        curve = t.empty((K + 1, M), dtype=t.float64, device=dev)
        curve[0] = best_stats[:, 4]
        cur = 0
        for it in range(1, K + 1):
            ratio = it / K
            CF = 0.0 if ratio >= 1.0 else ((1.0 - ratio) ** (2.0 * ratio) if ratio > 0 else 1.0)   # MPA.py:336
            phase = 1 if it <= K / 3 else (2 if it <= 2 * K / 3 else 3)
            nxt = cur ^ 1
            _lib.check(L.mpp_mpa_iteration_batch(
                self._maps, C.byref(self.policy), N, 0, N, it, phase, self.P_const, CF, self.FADs_rate, self._levy_sigma,
                self.levy_beta, _lib.ptr(seeds), _lib.ptr(order), _lib.ptr(cells[cur]), _lib.ptr(ncell[cur]),
                _lib.ptr(stats[cur]), mc, _lib.ptr(cells[nxt]), _lib.ptr(ncell[nxt]), _lib.ptr(stats[nxt]), _lib.ptr(tmp),
                _lib.ptr(avoid), _lib.ptr(scratch), scratch.numel(), self.warps_per_map, self.heap_cap, _lib.ptr(queue),
                _lib.ptr(status), _lib.ptr(counters), stream), "mpp_mpa_iteration_batch")
            self.kernel_launches += 1
            self.predator_evaluations += M * N
            cur = nxt
            order, cs, cc, cn = elite(cur)                                      # sort :412, population[0]
            # best-so-far cascade MPA.py:415-437, for every map at once (columns: length, turns, safety, diag, fitness)
            eq = lambda a, b: (a - b).abs() < 1e-9
            better = cs[:, 4] < best_stats[:, 4]
            tie = eq(cs[:, 4], best_stats[:, 4]) & ~better
            eL, eT, eS = eq(cs[:, 0], best_stats[:, 0]), eq(cs[:, 1], best_stats[:, 1]), eq(cs[:, 2], best_stats[:, 2])
            casc = (cs[:, 0] < best_stats[:, 0]) | (eL & (cs[:, 1] < best_stats[:, 1])) | \
                   (eL & eT & (cs[:, 2] < best_stats[:, 2])) | (eL & eT & eS & (cs[:, 3] < best_stats[:, 3]))
            upd = better | (tie & casc)
            best_stats = t.where(upd[:, None], cs, best_stats)
            best_cells = t.where(upd[:, None], cc, best_cells)
            best_n = t.where(upd, cn, best_n)
            curve[it] = best_stats[:, 4]
        t.cuda.synchronize(dev)
        st = int(status.item())
        if st:                                                                   # a heap or a path buffer overflowed: the solve
            kw = dict(self._ctor)                                                # is deterministic -- repeat it with more room
            if st == 1:
                if self.heap_cap >= 8 * self.rows * self.cols:
                    raise _lib.MppError("A* heap overflow at maximum capacity")
                kw.update(heap_cap=min(8 * self.rows * self.cols, self.heap_cap * 4), max_cells=self.max_cells)
            else:
                if self.max_cells >= 2 * self.rows * self.cols:
                    raise _lib.MppError("path buffer overflow at maximum capacity")
                kw.update(max_cells=min(2 * self.rows * self.cols, 2 * self.max_cells), heap_cap=self.heap_cap)
            again = MPABatch(self._map_set, **kw)                                # the same map batch
            again.predator_evaluations, again.kernel_launches = self.predator_evaluations, self.kernel_launches
            out = again.solve()
            self.predator_evaluations, self.kernel_launches = again.predator_evaluations, again.kernel_launches
            again.close()
            return out
        self.expansions = int(counters[0].item())
        bs, bc, bn, cv = best_stats.cpu().numpy(), best_cells.cpu().numpy(), best_n.cpu().numpy(), curve.cpu().numpy()
        out = []
        for k in range(M):
            n = int(bn[k])
            path = [(int(c) // self.cols, int(c) % self.cols) for c in bc[k, :n]]
            length = float(bs[k, 0]) if n > 1 else 0
            col = [float(v) if v != INF else None for v in cv[:, k]]
            out.append((path, length, int(bs[k, 1]), float(bs[k, 2]), float(bs[k, 3]), float(bs[k, 4]), col))
        return out


def solve_mpa_batch(grids, num_predators, num_iterations, params, seeds=None, wave=32, group=None, device=None):
    """MPA over this rank's shard of the maps (host maps or device grids, as solve_maaco_batch takes), `wave` maps per
    launch (grouped by shape).  Returns (map_index, path, length, turns, safety_p, diag_p, fitness, convergence_curve)
    per map of this rank."""
    lo, hi = shard_maps(len(grids), group)
    maps = _sweep_maps(grids, lo, hi)
    out = []
    for idx in _shape_waves(grids, lo, hi, wave):
        b = MPABatch(maps.wave(idx), num_predators, num_iterations,
                     seeds=None if seeds is None else [seeds[i] for i in idx], device=device, **params)
        for i, r in zip(idx, b.solve()):
            out.append((i,) + tuple(r))
        b.close()
    out.sort(key=lambda r: r[0])
    return out


# ---- A* / Dijkstra over a batch of maps (astar.py, dijkstra.py) ------------------------------------------------------
# algorithm -> (connector variant, the reference's errors for a map without start / target)
_SEARCH_ALGORITHMS = {
    "astar": (0, "AStar: Start node not found in grid.", "AStar: Target node not found in grid."),      # astar.py:19-20
    "dijkstra": (2, "Dijkstra: Start node not found.", "Dijkstra: Target node not found."),           # dijkstra.py:19-20
}


def _search_algorithm(algorithm):
    if algorithm not in _SEARCH_ALGORITHMS:
        raise ValueError(f"algorithm must be 'astar' or 'dijkstra', not {algorithm!r}")
    return _SEARCH_ALGORITHMS[algorithm]


# planner -> the reference constructor's errors for a map without start / target
_ENDPOINT_ERRORS = {name: msgs for name, (_, *msgs) in _SEARCH_ALGORITHMS.items()}
_ENDPOINT_ERRORS.update(pso=("PSO: Start node not found.", "PSO: Target node not found."),              # pso.py:19-20
                        ga=("GA: Start node not found.", "GA: Target node not found."))                 # ga_solver.py:19-20


def _endpoint_check(algorithm):
    """check(start, target) (per-map first start / target cell, -1 = none) raising the reference constructor's
    ValueError for the first map that has no start or no target -- what a loop of AStarSolver / DijkstraSolver /
    PSOSolver / GASolver constructors over the maps would raise."""
    if algorithm not in _ENDPOINT_ERRORS:
        _search_algorithm(algorithm)
    no_start, no_target = _ENDPOINT_ERRORS[algorithm]

    def check(start, target):
        bad = np.flatnonzero((start < 0) | (target < 0))
        if bad.size:
            raise ValueError(no_start if start[bad[0]] < 0 else no_target)
    return check


def _check_endpoints(flat, algorithm):
    """_endpoint_check on host maps, one per row of `flat` (cell codes)."""
    _endpoint_check(algorithm)(*_first_cells(np.asarray(flat)))


def _valid_queries(map_index, src, dst, n_maps, n_cells):
    """Bool tensor: query i names a map of the batch and both its endpoints are cells of that map.  The others get the
    empty result without a search (astar.py:37-39)."""
    if not (map_index.dim() == src.dim() == dst.dim() == 1):
        raise ValueError("map_index, src and dst must be 1-D")
    if not (map_index.numel() == src.numel() == dst.numel()):
        raise ValueError(f"map_index, src and dst differ in length ({map_index.numel()}, {src.numel()}, {dst.numel()})")
    return (map_index >= 0) & (map_index < n_maps) & (src >= 0) & (src < n_cells) & (dst >= 0) & (dst < n_cells)


def _map_shape(g):
    return tuple(g.shape) if hasattr(g, "shape") else np.shape(g)


def _shape_waves(grids, lo, hi, wave=None):
    """Maps lo..hi-1 grouped by shape (one mpp_map_batch each), `wave` maps per group at most (None: all of them)."""
    shapes = {}
    for i in range(lo, hi):
        shapes.setdefault(_map_shape(grids[i]), []).append(i)
    out = []
    for idx in shapes.values():
        step = wave or len(idx)
        out += [idx[w0:w0 + step] for w0 in range(0, len(idx), step)]
    return out


class SearchBatch:
    """M same-shape maps for the deterministic baselines: `search` runs any number of A* / Dijkstra queries, each on
    its own map with its own endpoints and avoid set, in one launch with the statistics of every path fused in
    (mpp_astar_batch_maps); `solve` is AStarSolver(grid).solve() / DijkstraSolver(grid).solve() for every map at once;
    `distance_fields` / `field_paths` give exact Dijkstra fields and the paths read from them (field.py).
    Same parameters and defaults as AStarSolver (astar.py:11-14); start and target may differ from map to map."""

    def __init__(self, grids, turn_penalty_factor=0.1, safety_penalty_factor=0.05, min_safe_distance=1.5,
                 allow_diagonal_moves=True, restrict_diagonal_near_obstacle_policy=True,
                 diagonal_obstacle_penalty_value=1000.0, *, device=None, max_cells=None, heap_cap=None, n_slots=None):
        import torch
        from .engine import make_policy
        L = _lib.lib()
        self._map_set = _map_set(grids, device)
        self._maps = self._map_set.handle
        self.n_maps, self.rows, self.cols = self._map_set.shape
        self.device_index = self._map_set.device_index
        self.device = torch.device("cuda", self.device_index)
        self.allow_diagonal_moves = bool(allow_diagonal_moves)
        self.restrict_corners = bool(restrict_diagonal_near_obstacle_policy)   # astar_strictly_restricts_corners
        self.policy = make_policy(turn_penalty_factor, safety_penalty_factor, min_safe_distance,
                                  diagonal_obstacle_penalty_value, restrict_diagonal_near_obstacle_policy,
                                  allow_diagonal_moves, mode=0)
        self.n = self.rows * self.cols
        self.words = (self.n + 31) // 32
        # a search's open set is a frontier: a few thousand entries on the largest maps; overflow is reported
        # (n_cells = -1) and the search is repeated with a larger heap
        self.heap_cap = int(heap_cap or min(8 * self.n, max(4096, self.n // 4)))
        self.max_cells = int(max_cells or min(self.n, max(4096, 16 * (self.rows + self.cols))))
        self.max_slots = L.mpp_map_batch_max_slots(self._maps)
        self.n_slots = int(n_slots or self.max_slots)
        self.counters = torch.zeros(4, dtype=torch.int64, device=self.device)  # expansions, relaxations, ring / heap pushes
        self.launches = 0
        self._scratch, self._scratch_key, self._visited = None, None, None
        self._start_dev, self._target_dev = (torch.as_tensor(e.astype(np.int32), device=self.device)
                                             for e in (self._map_set.start, self._map_set.target))

    def close(self):
        self._maps = self._map_set = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def expansions(self):
        return int(self.counters[0].item())

    def _i32(self, a):
        import torch
        if isinstance(a, torch.Tensor):
            return a.to(device=self.device, dtype=torch.int32).contiguous()
        return torch.as_tensor(np.ascontiguousarray(a, dtype=np.int32), device=self.device)

    def _stream(self):
        import torch
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _grow_from(self, mn, mx):
        """Heap overflow (mn < 0) or truncated paths (mx > max_cells) -> enlarge; True: the caller repeats."""
        grew = False
        if mn < 0:
            if self.heap_cap >= 8 * self.n:
                raise _lib.MppError("A* heap overflow at maximum capacity")
            self.heap_cap = min(8 * self.n, self.heap_cap * 4)
            grew = True
        if mx > self.max_cells:
            self.max_cells = min(2 * self.n, max(mx, 2 * self.max_cells))
            grew = True
        return grew

    def _scratch_for(self, n):
        """(scratch, search slots) for a launch over n queries / individuals with the current heap_cap."""
        import torch as t
        slots = max(1, min(self.n_slots, n))
        if self._scratch_key != (slots, self.heap_cap):                   # zero-filled once: search stamps live in it
            nbytes = 256 + slots * _lib.lib().mpp_astar_slot_bytes(self.rows, self.cols, self.heap_cap)
            self._scratch = t.zeros(nbytes, dtype=t.uint8, device=self.device)
            self._scratch_key = (slots, self.heap_cap)
        return self._scratch, slots

    def _launch(self, variant, mi, src, dst, avoid, longest_first, allow_diagonal, restrict_corner, policy):
        """One mpp_astar_batch_maps launch over the given (valid) queries with the current sizes; stats is None when
        policy is."""
        import torch as t
        n, mc = mi.numel(), self.max_cells
        _, slots = self._scratch_for(n)
        order = None
        if longest_first and n > slots:
            # a search costs roughly the square of its endpoint distance; the launch ends with its slowest query
            dr = t.div(src, self.cols, rounding_mode="floor") - t.div(dst, self.cols, rounding_mode="floor")
            dc = src % self.cols - dst % self.cols
            order = t.argsort(dr.long() ** 2 + dc.long() ** 2, descending=True).to(t.int32).contiguous()
        cells = t.empty((n, mc), dtype=t.int32, device=self.device)
        ncell = t.empty(n, dtype=t.int32, device=self.device)
        g = t.empty(n, dtype=t.float64, device=self.device)
        stats = None if policy is None else t.empty((n, 5), dtype=t.float64, device=self.device)
        _lib.check(_lib.lib().mpp_astar_batch_maps(
            self._maps, int(variant), _lib.ptr(mi), _lib.ptr(src), _lib.ptr(dst), _lib.ptr(avoid), n,
            int(bool(allow_diagonal)), int(bool(restrict_corner)), None if policy is None else C.byref(policy),
            _lib.ptr(cells), mc, _lib.ptr(ncell), _lib.ptr(g), _lib.ptr(stats), _lib.ptr(self._scratch),
            self._scratch.numel(), slots, self.heap_cap, _lib.ptr(self.counters), _lib.ptr(order), self._stream()),
            "mpp_astar_batch_maps")
        self.launches += 1
        return cells, ncell, g, stats

    def _chain_order(self, mi, wps):
        """Individuals ordered by the Euclidean length of their waypoint chain, longest first (those outside the batch
        last): a chain costs roughly the sum of its squared hop lengths, and the launch ends with its slowest
        individual."""
        import torch as t
        ok = (mi >= 0) & (mi < self.n_maps)
        m = mi.clamp(0, self.n_maps - 1).long()
        chain = t.cat([self._start_dev[m][:, None], wps, self._target_dev[m][:, None]], dim=1).to(t.float64)
        r, c = t.div(chain, self.cols, rounding_mode="floor"), chain % self.cols
        d = ((r[:, 1:] - r[:, :-1]) ** 2 + (c[:, 1:] - c[:, :-1]) ** 2).sqrt().sum(dim=1)
        return t.argsort(t.where(ok, d, -1.0), descending=True).to(t.int32).contiguous()

    def _chain_launch(self, mi, wps, policy):
        """One mpp_waypoint_fitness_maps launch over individuals mi [n] (map index, -1 = not searched), wps [n, W] with the
        current sizes, longest chains first."""
        import torch as t
        n, W = wps.shape
        mc = self.max_cells
        scratch, slots = self._scratch_for(n)
        if self._visited is None or self._visited.shape[0] < slots:
            self._visited = t.empty((slots, self.words), dtype=t.int32, device=self.device)
        order = self._chain_order(mi, wps) if n > slots // 2 else None
        cells = t.empty((n, mc), dtype=t.int32, device=self.device)
        ncell = t.empty(n, dtype=t.int32, device=self.device)
        stats = t.empty((n, 5), dtype=t.float64, device=self.device)
        _lib.check(_lib.lib().mpp_waypoint_fitness_maps(
            self._maps, _lib.ptr(mi), _lib.ptr(wps), n, W, C.byref(policy), _lib.ptr(cells), mc, _lib.ptr(ncell),
            _lib.ptr(stats), _lib.ptr(self._visited), _lib.ptr(scratch), scratch.numel(), slots, self.heap_cap,
            _lib.ptr(self.counters), _lib.ptr(order), self._stream()), "mpp_waypoint_fitness_maps")
        self.launches += 1
        return cells, ncell, stats

    def _chain_repeat(self, mi, wps, cells, ncell, stats):
        """After _grow_from enlarged the buffers: repeats the individuals whose heap overflowed or whose path was truncated
        (the searches are deterministic) until none is; returns the patched (cells, n_cells, stats)."""
        import torch as t
        while True:
            bad = ((ncell < 0) | (ncell > cells.shape[1])).nonzero().squeeze(1)
            c, nc, st = self._chain_launch(mi.index_select(0, bad).contiguous(), wps.index_select(0, bad).contiguous(),
                                           self.policy)
            if c.shape[1] > cells.shape[1]:                                  # max_cells grew: widen the earlier rows
                cells = t.nn.functional.pad(cells, (0, c.shape[1] - cells.shape[1]))
            cells[bad, :c.shape[1]] = c
            ncell[bad], stats[bad] = nc, st
            if not self._grow_from(*t.stack([nc.min(), nc.max()]).tolist()):
                return cells, ncell, stats

    def chains(self, map_index, waypoints):
        """Waypoint-chain fitness (pso.py:56-94 / ga_solver.py:58-93 + helper.py:98-113): individual i runs on map
        map_index[i] from that map's start through the W cells waypoints[i] to its target.  Returns device tensors
        (cells [n, max_cells] int32, n_cells [n] int32, stats [n, 5] float64).  n_cells = 0: an invalid chain, or a map
        index outside the batch (not searched).  A heap overflow or a truncated path grows the buffers and repeats only
        those individuals."""
        import torch as t
        mi, wps = self._i32(map_index), self._i32(waypoints)
        cells, ncell, stats = self._chain_launch(mi, wps, self.policy)
        if self._grow_from(*t.stack([ncell.min(), ncell.max()]).tolist()):
            cells, ncell, stats = self._chain_repeat(mi, wps, cells, ncell, stats)
        return cells, ncell, stats

    def search(self, variant, map_index, src, dst, avoid_bits=None, *, longest_first=True):
        """Query i: connector `variant` (0 = astar.py, 1 = MPA.py's private A*, 2 = dijkstra.py) from cell src[i] to
        cell dst[i] of map map_index[i], avoiding the cells set in avoid_bits[i] (n x ceil(rows*cols/32) bitmap words,
        or None).  Returns device tensors (cells [n, max_cells] int32, n_cells [n] int32, g [n] float64 = g of the
        popped target, stats [n, 5] float64 = (length, turns, safety, diag, fitness) of the path).  n_cells = 0: no
        path, or an endpoint / map index outside the batch (not searched).  A heap overflow or a truncated path grows
        the buffers and repeats only those queries (the searches are deterministic)."""
        import torch as t
        mi, src, dst = self._i32(map_index), self._i32(src), self._i32(dst)
        valid = _valid_queries(mi, src, dst, self.n_maps, self.n)
        n = mi.numel()
        avoid = None
        if avoid_bits is not None:
            if isinstance(avoid_bits, np.ndarray):
                avoid_bits = np.ascontiguousarray(avoid_bits).view(np.int32)
            avoid = t.as_tensor(avoid_bits, device=self.device).contiguous().view(t.int32)   # (uint32 words as int32)
            if avoid.numel() != n * self.words:
                raise ValueError(f"avoid_bits must hold {n} x {self.words} words, not {avoid.numel()}")
            avoid = avoid.reshape(n, self.words).contiguous()
        cells = t.zeros((n, self.max_cells), dtype=t.int32, device=self.device)
        ncell = t.zeros(n, dtype=t.int32, device=self.device)
        g = t.full((n,), INF, dtype=t.float64, device=self.device)
        stats = t.tensor([INF, 0.0, 0.0, 0.0, INF], dtype=t.float64, device=self.device).repeat(n, 1)   # helper.py:104-105
        idx = valid.nonzero().squeeze(1)
        while idx.numel():
            sub = lambda x: None if x is None else x.index_select(0, idx).contiguous()
            c, nc, gg, st = self._launch(variant, sub(mi), sub(src), sub(dst), sub(avoid), longest_first,
                                         self.allow_diagonal_moves, self.restrict_corners, self.policy)
            if c.shape[1] > cells.shape[1]:                                  # max_cells grew: widen the earlier rows
                wide = t.zeros((n, c.shape[1]), dtype=t.int32, device=self.device)
                wide[:, :cells.shape[1]] = cells
                cells = wide
            cells[idx, :c.shape[1]] = c
            ncell[idx], g[idx], stats[idx] = nc, gg, st
            bad = (nc < 0) | (nc > c.shape[1])
            if not self._grow_from(int(nc.min().item()), int(nc.max().item())):
                break
            idx = idx[bad]
        return cells, ncell, g, stats

    def _fields(self, src):
        from .field import dijkstra_fields
        s = self._start_dev if src is None else self._i32(src)
        if s.shape != (self.n_maps,):
            raise ValueError(f"src must hold one cell per map ({self.n_maps}), not shape {tuple(s.shape)}")
        return dijkstra_fields(self, self._maps, (self.n_maps, self.rows, self.cols), s, self.allow_diagonal_moves,
                               self.restrict_corners)

    def distance_fields(self, src=None):
        """[M, rows, cols] float64 CUDA tensor: map k's exact Dijkstra distance field from cell src[k] (None: every map's
        own start) -- at each cell the g that search(2, ...) from src[k] to that cell returns (+inf at obstacles and
        unreachable cells; all +inf when the source is outside the map or an obstacle)."""
        return self._fields(src)[0]

    def field_paths(self, map_index, dst, src=None):
        """What search(2, map_index, src[map_index], dst) returns -- (cells, n_cells, g, stats) device tensors, bit for
        bit -- from one distance field per map (from src[k], None: every map's own start) and one path-reading launch.
        A truncated path grows max_cells and repeats only the truncated queries."""
        from .field import field_paths
        mi, dst = self._i32(map_index), self._i32(dst)
        if not (mi.dim() == dst.dim() == 1) or mi.numel() != dst.numel():
            raise ValueError(f"map_index and dst must be 1-D and of one length, not {tuple(mi.shape)}, {tuple(dst.shape)}")
        g, parent = self._fields(src)
        return field_paths(self, self._maps, g, parent, mi, dst, self.policy)

    def solve(self, algorithm="astar"):
        """One start -> target query per map.  Returns, per map, what AStarSolver(grid, ...).solve() (algorithm
        "astar") or DijkstraSolver(grid, ...).solve() ("dijkstra") returns -- (path, length, turns, safety_p, diag_p,
        fitness) -- followed by the value that solver appends to its convergence_curve (g, or None when the path has
        at most one cell)."""
        variant = _search_algorithm(algorithm)[0]
        src, dst = self._map_set.start, self._map_set.target              # first row-major 2 / 3 (astar.py:17-18)
        _endpoint_check(algorithm)(src, dst)
        cells, ncell, g, stats = self.search(variant, np.arange(self.n_maps), src, dst)
        cells, ncell, g, stats = cells.cpu().numpy(), ncell.cpu().numpy(), g.cpu().numpy(), stats.cpu().numpy()
        out = []
        for k in range(self.n_maps):
            n = int(ncell[k])
            if n == 0:
                out.append(([], INF, 0, 0.0, 0.0, INF, None))               # helper.py:104-105
                continue
            r, c = np.divmod(cells[k, :n], self.cols)
            path = list(zip(r.tolist(), c.tolist()))
            st = stats[k]
            out.append((path, float(st[0]) if n > 1 else 0, int(st[1]), float(st[2]), float(st[3]), float(st[4]),
                        float(g[k]) if n > 1 else None))                      # astar.py:70 (path and len(path) > 1)
        return out


def solve_search_batch(grids, algorithm, params, wave=None, group=None, device=None):
    """A* or Dijkstra (algorithm "astar" / "dijkstra") start -> target on every grid of `grids` (this rank's shard when
    `group` is given), grouped by shape, `wave` maps per launch (None: all of a shape).  `params` = SearchBatch's keyword
    arguments.  Returns (map_index, path, length, turns, safety_p, diag_p, fitness, g) per map of this rank, g being the
    convergence-curve value (None for a path of at most one cell)."""
    _search_algorithm(algorithm)
    lo, hi = shard_maps(len(grids), group)
    maps = _sweep_maps(grids, lo, hi)
    _endpoint_check(algorithm)(*maps.first_cells())                         # before any search
    out = []
    for idx in _shape_waves(grids, lo, hi, wave):
        b = SearchBatch(maps.wave(idx), device=device, **params)
        for i, r in zip(idx, b.solve(algorithm)):
            out.append((i,) + tuple(r))
        b.close()
    out.sort(key=lambda r: r[0])
    return out


# ---- PSO / GA over a batch of maps (pso.py, ga_solver.py) -------------------------------------------------------------
def default_pop_wave(rows, cols, population):
    """Maps per wave of solve_pso_batch / solve_ga_batch: one [maps, population, max_cells] int32 array of paths (the
    population's evaluation; GA keeps a second one, the sorted population) stays near 1 GiB.  At 256x256 max_cells is
    8192 (32 KB per individual): 32 maps of 1024 individuals."""
    n = rows * cols
    max_cells = min(n, max(4096, 16 * (rows + cols)))                      # SearchBatch's default
    return max(1, (1 << 30) // (population * max_cells * 4))


class _WaypointBatch:
    """What PSOBatch and GABatch share: M same-shape maps (start and target may differ from map to map) behind one
    SearchBatch (map batch, policy, buffer sizes and their growth), one Philox seed per map, and the population
    initialisation of pso.py:97-161 / ga_solver.py:95-133 for every map at once."""
    _planner = None        # "pso" / "ga"
    _pad_class = None      # RNG class of the padding draws

    def __init__(self, grids, num_waypoints, policy, seeds, device, max_cells, heap_cap, n_slots):
        import torch
        endpoints = _endpoint_check(self._planner)

        def check(start, target):                                            # (host grids: before any device work)
            endpoints(start, target)
            if seeds is not None and len(seeds) != len(start):
                raise ValueError(f"seeds holds {len(seeds)} values for {len(start)} maps")
        maps = _map_set(grids, device, check)
        self.n_maps, self.rows, self.cols = maps.shape
        if seeds is None:
            seeds = [int.from_bytes(np.random.bytes(8), "little") for _ in range(self.n_maps)]
        self.seeds = [int(s) & (2 ** 64 - 1) for s in seeds]
        self.num_waypoints = int(num_waypoints)
        self._search = SearchBatch(maps, max_cells=max_cells, heap_cap=heap_cap, n_slots=n_slots, **policy)
        self.device = self._search.device
        self._seeds = torch.from_numpy(np.array(self.seeds, np.uint64).view(np.int64)).to(self.device)
        self.fitness_evaluations = [0] * self.n_maps
        self.init_attempts = [0] * self.n_maps
        self.kernel_launches = 0

    def close(self):
        self._search.close()

    @property
    def launches(self):
        """Kernel launches so far: population kernels and fitness / connector searches."""
        return self.kernel_launches + self._search.launches

    def _stream(self):
        import torch
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _solve_direct(self):
        """num_waypoints == 0 (pso.py:165-170, ga_solver.py:163-168): one start -> target connector per map and the
        statistics of its path; the curve holds that fitness."""
        return [r[:6] + ([r[5]],) for r in self._search.solve("astar")]

    def _initialize(self, generate, n):
        """pso.py:97-161 / ga_solver.py:95-133 for every map.  Each round generates one block of attempts for every map
        that still needs individuals -- generate(offsets [M] device int32, B) enqueues attempts [offsets[m],
        offsets[m] + B) of every map with offsets[m] >= 0 and returns (tensors [M, B, ...] an individual keeps,
        waypoint cells [M, B, W]) -- and evaluates them in one launch; each map accepts valid attempts in attempt
        order until it has n or has used 20 n.  A map without any valid chain gets its direct start -> target path
        (pso.py:128-145, ga_solver.py:111-117).  Returns (n_acc [M] before padding, direct [M] bool, kept [M, n, ...]
        tensors, stats [M, n, 5], cells [M, n, mc], n_cells [M, n]) with every map's rows padded to n (pso.py:159-160,
        ga_solver.py:129-130)."""
        import torch as t
        from . import rng
        M, W, dev = self.n_maps, self.num_waypoints, self.device
        max_total = 20 * n
        n_acc, attempts = np.zeros(M, np.int64), np.zeros(M, np.int64)
        kept = stats = cells = ncell = None
        rows = t.arange(M, device=dev)
        while True:
            need = (n_acc < n) & (attempts < max_total)
            if not need.any():
                break
            block = np.where(need, np.minimum(max_total - attempts, np.maximum(32, (1.25 * (n - n_acc)).astype(np.int64) + 8)),
                             0)
            B = int(block.max())
            offs = t.as_tensor(np.where(need, attempts, -1).astype(np.int32), device=dev)
            k_r, wp = generate(offs, B)
            self.kernel_launches += 1
            mi = t.where(t.arange(B, device=dev)[None, :] < t.as_tensor(block, device=dev)[:, None], rows[:, None], -1)
            c_r, nc_r, st_r = self._search.chains(mi.reshape(-1), wp.reshape(M * B, W))
            valid = (nc_r > 0).reshape(M, B).cpu().numpy()
            src, dst = [], []
            for m in np.flatnonzero(need):
                take = np.flatnonzero(valid[m, :block[m]])
                room = n - n_acc[m]
                if take.size >= room:
                    take = take[:room]
                    attempts[m] += int(take[-1]) + 1                         # the loop stops right after the n-th accept
                else:
                    attempts[m] += block[m]
                self.fitness_evaluations[m] += int(block[m])
                src.append(m * B + take)
                dst.append(m * n + n_acc[m] + np.arange(take.size))
                n_acc[m] += take.size
            if kept is None:
                kept = [t.zeros((M * n,) + x.shape[2:], dtype=x.dtype, device=dev) for x in k_r]
                stats = t.zeros((M * n, 5), dtype=t.float64, device=dev)
                cells = t.zeros((M * n, c_r.shape[1]), dtype=t.int32, device=dev)
                ncell = t.zeros(M * n, dtype=t.int32, device=dev)
            if c_r.shape[1] > cells.shape[1]:
                cells = t.nn.functional.pad(cells, (0, c_r.shape[1] - cells.shape[1]))
            si = t.as_tensor(np.concatenate(src), device=dev)
            di = t.as_tensor(np.concatenate(dst), device=dev)
            for buf, x in zip(kept, k_r):
                buf[di] = x.reshape((M * B,) + x.shape[2:])[si]
            stats[di], ncell[di] = st_r[si], nc_r[si]
            cells[di, :c_r.shape[1]] = c_r[si]
        self.init_attempts = attempts.tolist()
        direct = np.zeros(M, bool)
        lost = np.flatnonzero(n_acc == 0)
        if lost.size:                                                        # the direct path as the one individual
            s, g = self._search._start_dev[lost], self._search._target_dev[lost]
            c_d, nc_d, _, st_d = self._search.search(0, lost, s, g)
            found = (nc_d > 0).cpu().numpy()
            if found.any():
                if c_d.shape[1] > cells.shape[1]:
                    cells = t.nn.functional.pad(cells, (0, c_d.shape[1] - cells.shape[1]))
                fi = t.as_tensor(np.flatnonzero(found), device=dev)
                di = t.as_tensor(lost[found] * n, device=dev)
                stats[di], ncell[di] = st_d[fi], nc_d[fi]
                cells[di, :c_d.shape[1]] = c_d[fi, :cells.shape[1]]
                for buf in kept:
                    buf[di] = 0                                              # position = velocity = [[0.0, 0.0]] * W
                direct[lost[found]] = True
        # padding: random.choice(population).copy() with draws from (seed, PAD, 0, len(population))
        have = np.where(direct, 1, n_acc)
        idx = np.tile(np.arange(n), (M, 1))
        for m in np.flatnonzero((have > 0) & (have < n)):
            k0 = int(have[m])
            u = rng.stream_block(self.seeds[m], self._pad_class, 0, np.arange(k0, n), 1)[:, 0]
            for j, k in enumerate(range(k0, n)):
                idx[m, k] = idx[m, min(int(u[j] * k), k - 1)]
        flat = t.as_tensor((idx + np.arange(M)[:, None] * n).reshape(-1), device=dev)
        view = lambda x: x[flat].reshape((M, n) + x.shape[1:])
        return n_acc, direct, [view(b) for b in kept], view(stats), view(cells), view(ncell)

    def _result(self, n, cells, stats, curve):
        """One map's (path, length, turns, safety_p, diag_p, fitness, convergence_curve) from its best individual."""
        r, c = np.divmod(cells[:n], self.cols)
        return (list(zip(r.tolist(), c.tolist())), float(stats[0]), int(stats[1]), float(stats[2]), float(stats[3]),
                float(stats[4]), curve)


_FAILED = ([], INF, 0, 0.0, 0.0, INF, [])                                    # pso.py:147-157 / ga_solver.py:120-126


class PSOBatch(_WaypointBatch):
    """M same-shape maps, one PSO swarm per map, solved together: PSOSolver (pso.py:8-240) for every map with the same
    arguments and defaults, `grids` [M, rows, cols] in place of `grid` and `seeds` = one Philox seed per map (row m
    draws what PSOSolver(grid, ..., rng_seed=seeds[m]) draws).  Start and target may differ from map to map.  An
    iteration is the speculative repair of PSOSolver._iterate for all maps at once: every map's active suffix is
    updated and evaluated in one update launch and one fitness launch (mpp_pso_update_batch, mpp_waypoint_fitness_maps),
    each map's first global-best improver is found on the device, and only the rest of that map's swarm is restored
    and re-run in the next round; one host synchronise per round."""
    _planner = "pso"

    def __init__(self, grids, num_iterations, num_particles, num_waypoints_per_particle, w, c1, c2,
                 turn_penalty_factor=0.1, safety_penalty_factor=0.05, min_safe_distance=1.5, allow_diagonal_moves=True,
                 restrict_diagonal_near_obstacle_policy=True, diagonal_obstacle_penalty_value=1000.0, *, seeds=None,
                 device=None, max_cells=None, heap_cap=None, n_slots=None):
        from . import rng
        self._pad_class = rng.CLS_PSO_PAD
        policy = dict(turn_penalty_factor=turn_penalty_factor, safety_penalty_factor=safety_penalty_factor,
                      min_safe_distance=min_safe_distance, allow_diagonal_moves=allow_diagonal_moves,
                      restrict_diagonal_near_obstacle_policy=restrict_diagonal_near_obstacle_policy,
                      diagonal_obstacle_penalty_value=diagonal_obstacle_penalty_value)
        super().__init__(grids, num_waypoints_per_particle, policy, seeds, device, max_cells, heap_cap, n_slots)
        self.num_iterations, self.num_particles = int(num_iterations), int(num_particles)
        self.w, self.c1, self.c2 = w, c1, c2
        self.max_vel = max(1.0, 0.15 * max(self.rows, self.cols))            # pso.py:34
        self.pos = self.vel = self.pbest_fit = None

    def _generate(self, offs, B):
        import torch as t
        M, W = self.n_maps, self.num_waypoints
        pos = t.empty((M, B, W, 2), dtype=t.float64, device=self.device)
        vel = t.empty((M, B, W, 2), dtype=t.float64, device=self.device)
        wp = t.empty((M, B, W), dtype=t.int32, device=self.device)
        _lib.check(_lib.lib().mpp_pso_init_batch(self._search._maps, B, _lib.ptr(offs), W, self.max_vel, _lib.ptr(self._seeds),
                                                 _lib.ptr(pos), _lib.ptr(vel), _lib.ptr(wp), self._stream()),
                   "mpp_pso_init_batch")
        return (pos, vel), wp

    def solve(self):
        """Returns, per map, what PSOSolver(grid, ..., rng_seed=seeds[m]).solve() returns followed by that solver's
        convergence_curve.  After it, pos / vel / pbest_fit hold every swarm's final state ([M, N, W, 2], [M, N])."""
        import torch as t
        if self.num_waypoints == 0:
            return self._solve_direct()
        M, N, W, K, dev = self.n_maps, self.num_particles, self.num_waypoints, self.num_iterations, self.device
        n_acc, direct, (pos, vel), stats, cells, ncell = self._initialize(self._generate, N)
        live = t.as_tensor((n_acc > 0) | direct, device=dev)
        fit = stats[..., 4]
        rows, ar = t.arange(M, device=dev), t.arange(N, device=dev)
        gi = (fit == fit.min(dim=1, keepdim=True).values).int().argmax(dim=1)   # first strictly-best, pso.py:121
        g_pos, g_stats, g_cells, g_n = pos[rows, gi], stats[rows, gi], cells[rows, gi], ncell[rows, gi]
        pbest_pos, pbest_fit = pos.clone(), fit.clone()
        curve = t.empty((K + 1, M), dtype=t.float64, device=dev)
        curve[0] = g_stats[:, 4]
        L = _lib.lib()
        idle = np.where(live.cpu().numpy(), 0, N)
        for it in range(K):
            pos0, vel0 = pos.clone(), vel.clone()
            start = idle.copy()
            while (start < N).any():
                st_d = t.as_tensor(start.astype(np.int32), device=dev)
                wp = t.empty((M, N, W), dtype=t.int32, device=dev)
                _lib.check(L.mpp_pso_update_batch(self._search._maps, _lib.ptr(pos), _lib.ptr(vel), _lib.ptr(pbest_pos),
                                                  _lib.ptr(g_pos), N, _lib.ptr(st_d), W, self.w, self.c1, self.c2,
                                                  self.max_vel, _lib.ptr(self._seeds), it, _lib.ptr(wp), self._stream()),
                           "mpp_pso_update_batch")
                self.kernel_launches += 1
                act = ar[None, :] >= st_d[:, None]
                mi = t.where(act, rows[:, None], -1).to(t.int32).reshape(-1)
                wp = wp.reshape(M * N, W)
                c_r, nc_r, s_r = self._search._chain_launch(mi, wp, self._search.policy)
                for m in np.flatnonzero(start < N):
                    self.fitness_evaluations[m] += N - int(start[m])
                while True:
                    nc = nc_r.reshape(M, N)
                    f = s_r[:, 4].reshape(M, N)
                    imp_p = act & (nc > 0) & (f < pbest_fit)                  # pso.py:216
                    imp_g = imp_p & (f < g_stats[:, 4:5])                     # pso.py:222
                    hit = imp_g.any(dim=1)
                    q = t.where(hit, imp_g.int().argmax(dim=1), N - 1)       # the last particle final this round
                    nxt = t.where(hit, q + 1, N)
                    # the round's one host synchronise: buffer growth flags and the next round's start of every map
                    flags = t.cat([t.stack([nc_r.min(), nc_r.max()]).to(t.int64), nxt.to(t.int64)]).tolist()
                    if not self._search._grow_from(flags[0], flags[1]):
                        break
                    c_r, nc_r, s_r = self._search._chain_repeat(mi, wp, c_r, nc_r, s_r)
                upd = imp_p & (ar[None, :] <= q[:, None])                     # pso.py:217-220 for the final particles
                pbest_fit = t.where(upd, f, pbest_fit)
                pbest_pos = t.where(upd[..., None, None], pos, pbest_pos)
                if c_r.shape[1] > g_cells.shape[1]:
                    g_cells = t.nn.functional.pad(g_cells, (0, c_r.shape[1] - g_cells.shape[1]))
                fq = rows * N + q                                             # pso.py:223-229
                g_pos = t.where(hit[:, None, None], pos[rows, q], g_pos)
                g_stats = t.where(hit[:, None], s_r[fq], g_stats)
                g_cells[hit, :c_r.shape[1]] = c_r[fq][hit]
                g_n = t.where(hit, nc_r[fq], g_n)
                rest = (ar[None, :] > q[:, None]) & hit[:, None]             # speculated with the old gbest: re-run
                pos = t.where(rest[..., None, None], pos0, pos).contiguous()
                vel = t.where(rest[..., None, None], vel0, vel).contiguous()
                pbest_pos = pbest_pos.contiguous()
                start = np.array(flags[2:], np.int64)
            curve[it + 1] = g_stats[:, 4]
        self.pos, self.vel, self.pbest_fit = pos, vel, pbest_fit
        g_stats, g_cells, g_n, curve = g_stats.cpu().numpy(), g_cells.cpu().numpy(), g_n.cpu().numpy(), curve.cpu().numpy()
        return [self._result(int(g_n[m]), g_cells[m], g_stats[m], [float(v) for v in curve[:, m]]) if idle[m] == 0
                else _FAILED[:6] + ([],) for m in range(M)]


class GABatch(_WaypointBatch):
    """M same-shape maps, one GA population per map, solved together: GASolver (ga_solver.py:8-223) for every map with
    the same arguments and defaults, `grids` [M, rows, cols] in place of `grid` and `seeds` = one Philox seed per map
    (row m draws what GASolver(grid, ..., rng_seed=seeds[m]) draws).  Start and target may differ from map to map.  A
    generation is one selection, one breeding and one fitness launch for every map (mpp_ga_select_batch,
    mpp_ga_breed_batch, mpp_waypoint_fitness_maps); the invalid-child replacement (:204-205), the stable sort
    (:208-209) and the best-so-far update (:211-213) are torch operations over all maps."""
    _planner = "ga"

    def __init__(self, grids, num_generations, population_size, num_waypoints_per_chromosome, mutation_rate,
                 crossover_rate, tournament_size=3, turn_penalty_factor=0.1, safety_penalty_factor=0.05,
                 min_safe_distance=1.5, allow_diagonal_moves=True, restrict_diagonal_near_obstacle_policy=True,
                 diagonal_obstacle_penalty_value=1000.0, *, seeds=None, device=None, max_cells=None, heap_cap=None,
                 n_slots=None):
        from . import rng
        self._pad_class = rng.CLS_GA_PAD
        policy = dict(turn_penalty_factor=turn_penalty_factor, safety_penalty_factor=safety_penalty_factor,
                      min_safe_distance=min_safe_distance, allow_diagonal_moves=allow_diagonal_moves,
                      restrict_diagonal_near_obstacle_policy=restrict_diagonal_near_obstacle_policy,
                      diagonal_obstacle_penalty_value=diagonal_obstacle_penalty_value)
        super().__init__(grids, num_waypoints_per_chromosome, policy, seeds, device, max_cells, heap_cap, n_slots)
        self.num_generations, self.population_size = int(num_generations), int(population_size)
        self.mutation_rate, self.crossover_rate, self.tournament_size = mutation_rate, crossover_rate, tournament_size
        self.chrom = self.fitness = None

    def _generate(self, offs, B):
        import torch as t
        chrom = t.empty((self.n_maps, B, self.num_waypoints), dtype=t.int32, device=self.device)
        _lib.check(_lib.lib().mpp_ga_init_batch(self._search._maps, B, _lib.ptr(offs), self.num_waypoints,
                                                _lib.ptr(self._seeds), _lib.ptr(chrom), self._stream()), "mpp_ga_init_batch")
        return (chrom,), chrom

    def solve(self):
        """Returns, per map, what GASolver(grid, ..., rng_seed=seeds[m]).solve() returns followed by that solver's
        convergence_curve.  After it, chrom / fitness hold every map's final population in sorted order ([M, N, W],
        [M, N]; meaningful for maps whose initialisation found a valid chain)."""
        import torch as t
        if self.num_waypoints == 0:
            return self._solve_direct()
        M, N, W, K, dev = self.n_maps, self.population_size, self.num_waypoints, self.num_generations, self.device
        n_acc, direct, (chrom,), stats, cells, ncell = self._initialize(self._generate, N)
        evolving = n_acc > 0                       # a direct-path population is a fixed point (ga_solver.py:144-160)
        live = t.as_tensor(evolving, device=dev)
        rows = t.arange(M, device=dev)

        def sort(chrom, stats, cells, ncell):                                 # list.sort is stable (:132, :208-209)
            o = t.sort(stats[..., 4], dim=1, stable=True).indices
            return chrom[rows[:, None], o], stats[rows[:, None], o], cells[rows[:, None], o], ncell[rows[:, None], o]

        chrom, stats, cells, ncell = sort(chrom, stats, cells, ncell)
        b_stats, b_cells, b_n = stats[:, 0].clone(), cells[:, 0].clone(), ncell[:, 0].clone()
        curve = t.empty((K + 1, M), dtype=t.float64, device=dev)
        curve[0] = b_stats[:, 4]
        L = _lib.lib()
        mi = t.where(live[:, None], rows[:, None], -1).expand(M, N).to(t.int32).reshape(-1).contiguous()
        for gen in range(K if evolving.any() else 0):
            parents = t.empty((M, N), dtype=t.int32, device=dev)
            fit = stats[..., 4].contiguous()
            _lib.check(L.mpp_ga_select_batch(self._search._maps, _lib.ptr(fit), N, self.tournament_size,
                                             _lib.ptr(self._seeds), gen, _lib.ptr(parents), self._stream()),
                       "mpp_ga_select_batch")
            children = t.empty((M, N, W), dtype=t.int32, device=dev)
            _lib.check(L.mpp_ga_breed_batch(self._search._maps, _lib.ptr(chrom.contiguous()), _lib.ptr(parents), N, W,
                                            self.crossover_rate, self.mutation_rate, _lib.ptr(self._seeds), gen,
                                            _lib.ptr(children), self._stream()), "mpp_ga_breed_batch")
            self.kernel_launches += 2
            c_c, c_n, c_s = self._search.chains(mi, children.reshape(M * N, W))
            for m in np.flatnonzero(evolving):
                self.fitness_evaluations[m] += N
            # an invalid child is replaced by its parent object (:204-205): child slot s of a map has parent parents[s]
            if c_c.shape[1] > cells.shape[2]:
                cells = t.nn.functional.pad(cells, (0, c_c.shape[1] - cells.shape[2]))
                b_cells = t.nn.functional.pad(b_cells, (0, c_c.shape[1] - b_cells.shape[1]))
            pi = (rows[:, None] * N + parents.long()).reshape(-1)
            bad = (c_n <= 0).nonzero().squeeze(1)
            src = pi[bad]
            children = children.reshape(M * N, W)
            children[bad] = chrom.reshape(M * N, W)[src]
            c_s[bad] = stats.reshape(M * N, 5)[src]
            c_c[bad] = cells.reshape(M * N, -1)[src]
            c_n[bad] = ncell.reshape(M * N)[src]
            chrom, stats, cells, ncell = sort(children.reshape(M, N, W), c_s.reshape(M, N, 5), c_c.reshape(M, N, -1),
                                              c_n.reshape(M, N))
            better = live & (stats[:, 0, 4] < b_stats[:, 4])                 # :211-213
            b_stats = t.where(better[:, None], stats[:, 0], b_stats)
            b_cells = t.where(better[:, None], cells[:, 0], b_cells)
            b_n = t.where(better, ncell[:, 0], b_n)
            curve[gen + 1] = b_stats[:, 4]
        self.chrom, self.fitness = chrom, stats[..., 4]
        b_stats, b_cells, b_n = b_stats.cpu().numpy(), b_cells.cpu().numpy(), b_n.cpu().numpy()
        curve = curve.cpu().numpy()
        out = []
        for m in range(M):
            if evolving[m]:
                out.append(self._result(int(b_n[m]), b_cells[m], b_stats[m], [float(v) for v in curve[:, m]]))
            elif direct[m]:                      # every generation reproduces the direct-path individual (:111-117)
                r = self._result(int(b_n[m]), b_cells[m], b_stats[m], None)
                out.append(r[:6] + ([r[5]] * (K + 1),))
            else:
                out.append(_FAILED[:6] + ([],))
        return out


def _pop_waves(grids, lo, hi, population, wave=None):
    """Maps lo..hi-1 grouped by shape, `wave` maps per wave at most (None: default_pop_wave of the shape)."""
    out = []
    for idx in _shape_waves(grids, lo, hi):
        step = wave or default_pop_wave(*_map_shape(grids[idx[0]]), population)
        out += [idx[w0:w0 + step] for w0 in range(0, len(idx), step)]
    return out


def _pop_sweep(cls, grids, sizes, params, seeds, wave, group, device):
    lo, hi = shard_maps(len(grids), group)
    maps = _sweep_maps(grids, lo, hi)
    _endpoint_check(cls._planner)(*maps.first_cells())                      # before any search
    out = []
    for idx in _pop_waves(grids, lo, hi, sizes[1], wave):
        b = cls(maps.wave(idx), *sizes,
                seeds=None if seeds is None else [seeds[i] for i in idx], device=device, **params)
        for i, r in zip(idx, b.solve()):
            out.append((i,) + tuple(r))
        b.close()
    out.sort(key=lambda r: r[0])
    return out


def solve_pso_batch(grids, num_iterations, num_particles, num_waypoints_per_particle, params, seeds=None, wave=None,
                    group=None, device=None):
    """PSO on every grid of `grids` (this rank's shard when `group` is given), grouped by shape, `wave` maps per
    PSOBatch (None: default_pop_wave, about 1 GiB of population paths per wave -- 32 maps of 1024 particles at
    256x256).  `params` = PSOBatch's other arguments (w, c1, c2, the policy, max_cells / heap_cap / n_slots).  Returns
    (map_index, path, length, turns, safety_p, diag_p, fitness, convergence_curve) per map of this rank, sorted by map
    index; identical to PSOSolver(grid, ..., rng_seed=seeds[i]).solve() per map."""
    return _pop_sweep(PSOBatch, grids, (num_iterations, num_particles, num_waypoints_per_particle), params, seeds, wave,
                      group, device)


def solve_ga_batch(grids, num_generations, population_size, num_waypoints_per_chromosome, params, seeds=None, wave=None,
                   group=None, device=None):
    """GA on every grid of `grids` (this rank's shard when `group` is given), like solve_pso_batch.  A wave keeps two
    [maps, population, max_cells] int32 path arrays (the population and its children): about 2 GiB with the default
    wave.  `params` = GABatch's other arguments (mutation_rate, crossover_rate, tournament_size, the policy, ...)."""
    return _pop_sweep(GABatch, grids, (num_generations, population_size, num_waypoints_per_chromosome), params, seeds,
                      wave, group, device)
