"""ctypes front-end to the C oracle (oracle/mpp_oracle.c) -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this module.  The product never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libmpp_oracle.so")
_lib = None


def build(force=False):
    src = os.path.join(_HERE, "mpp_oracle.c")
    if not force and os.path.exists(_SO) and os.path.getmtime(_SO) >= os.path.getmtime(src):
        return _SO
    gcc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    cmd = [gcc, "-O2", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-fvisibility=hidden",
           "-shared", "-o", _SO, src, "-lm"]
    subprocess.check_call(cmd)
    return _SO


class MaacoParams(C.Structure):
    _fields_ = [("rows", C.c_int), ("cols", C.c_int), ("sr", C.c_int), ("sc", C.c_int), ("tr", C.c_int), ("tc", C.c_int),
                ("alpha", C.c_double), ("beta", C.c_double), ("rho", C.c_double), ("Q", C.c_double),
                ("a_turn", C.c_double), ("wh_max", C.c_double), ("wh_min", C.c_double), ("k_h", C.c_double),
                ("q0_initial", C.c_double), ("C0", C.c_double), ("num_iterations", C.c_int)]


class Policy(C.Structure):
    _fields_ = [("tpf", C.c_double), ("spf", C.c_double), ("msd", C.c_double), ("diag_value", C.c_double),
                ("restrict_policy", C.c_int), ("mode", C.c_int)]


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
        _lib.orc_stream_uniform.restype = C.c_double
        _lib.orc_stream_uniform.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
        _lib.orc_maaco_q0.restype = C.c_double
        _lib.orc_maaco_q0.argtypes = [C.c_int, C.c_int, C.c_double]
        _lib.orc_astar_ctx_new.restype = C.c_void_p
        _lib.orc_astar_ctx_new.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
        _lib.orc_astar_ctx_free.argtypes = [C.c_void_p]
        _lib.orc_astar.restype = C.c_int
        _lib.orc_astar.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                   C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.orc_maaco_best_scan.restype = C.c_int
        _lib.orc_ga_select.restype = C.c_int
        _lib.orc_ga_select.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_uint32, C.c_uint32]
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def find_start_target(grid):
    """First row-major cell equal to 2 / 3 (MAACO.py:32-41)."""
    g = np.asarray(grid)
    s = np.argwhere(g == 2)
    t = np.argwhere(g == 3)
    if s.size == 0 or t.size == 0:
        raise ValueError("start/target not found")
    return (int(s[0][0]), int(s[0][1])), (int(t[0][0]), int(t[0][1]))


def philox(ctr, key):
    out = (C.c_uint32 * 4)()
    lib().orc_philox((C.c_uint32 * 4)(*ctr), (C.c_uint32 * 2)(*key), out)
    return tuple(out)


def stream_uniform(seed, cls, it, ind, d):
    return lib().orc_stream_uniform(seed, cls, it, ind, d)


def maaco_params(grid, num_iterations, alpha, beta, rho, Q, a_turn_coef, wh_max, wh_min, k_h_adaptive,
                 q0_initial, C0_initial_pheromone=0.1, **_ignored):
    g = np.asarray(grid)
    (sr, sc), (tr, tc) = find_start_target(g)
    return MaacoParams(g.shape[0], g.shape[1], sr, sc, tr, tc, alpha, beta, rho, Q, a_turn_coef, wh_max, wh_min,
                       k_h_adaptive, q0_initial, C0_initial_pheromone, num_iterations)


class MaacoOracle:
    """Oracle mirror of MAACO.solve_path_planning (MAACO.py:334-371)."""

    def __init__(self, grid, num_ants, num_iterations, seed=0, threads=1, max_cells=None, **params):
        self.grid8 = np.ascontiguousarray(np.asarray(grid), dtype=np.uint8)
        self.R, self.C = self.grid8.shape
        self.N = num_ants
        self.K = num_iterations
        self.seed = seed
        self.threads = threads
        self.p = maaco_params(grid, num_iterations, **params)
        n = self.R * self.C
        self.tau = np.empty(n)
        self.dist_t = np.empty(n)
        self.E0 = np.empty(n)
        self.E1 = np.empty(n)
        lib().orc_maaco_tables(_p(self.grid8), C.byref(self.p), _p(self.tau), _p(self.dist_t), _p(self.E0), _p(self.E1))
        self.max_cells = max_cells or n
        self.words = (n + 31) // 32
        self.best_len = float("inf")
        self.best_turns = -1
        self.best_path = np.zeros(0, np.int32)
        self.curve = []
        self.total_steps = 0

    def q0(self, it):
        return lib().orc_maaco_q0(self.K, it, self.p.q0_initial)

    def tours(self, it, ant0=0, n_ants=None):
        n_ants = n_ants or self.N
        tabu = np.zeros((n_ants, self.words), np.uint32)
        cells = np.zeros((n_ants, self.max_cells), np.int32)
        ncell = np.zeros(n_ants, np.int32)
        length = np.zeros(n_ants)
        turns = np.zeros(n_ants, np.int32)
        steps = C.c_longlong(0)
        lib().orc_maaco_tours(_p(self.grid8), C.byref(self.p), _p(self.tau), _p(self.E0), _p(self.E1),
                              C.c_double(self.q0(it)), C.c_uint64(self.seed), it, ant0, n_ants, _p(tabu),
                              _p(cells), self.max_cells, _p(ncell), _p(length), _p(turns), C.byref(steps),
                              self.threads)
        self.total_steps += steps.value
        return cells, ncell, length, turns, tabu

    def iterate(self, it):
        cells, ncell, length, turns, _ = self.tours(it)
        bl = C.c_double()
        bt = C.c_int()
        bi = lib().orc_maaco_best_scan(_p(length), _p(turns), self.N, C.byref(bl), C.byref(bt))
        # MAACO.py:351-358
        if bl.value < self.best_len:
            self.best_len, self.best_turns = bl.value, bt.value
            self.best_path = cells[bi, :ncell[bi]].copy()
        elif abs(bl.value - self.best_len) < 1e-9 and bt.value < self.best_turns:
            self.best_turns = bt.value
            self.best_path = cells[bi, :ncell[bi]].copy()
        lib().orc_maaco_pheromone(_p(self.grid8), C.byref(self.p), _p(self.tau), _p(cells), self.max_cells, _p(ncell),
                                  _p(length), self.N, C.c_double(self.best_len))
        self.curve.append(self.best_len if np.isfinite(self.best_len) else None)
        return cells, ncell, length, turns, (bi, bl.value, bt.value)

    def solve(self):
        for it in range(1, self.K + 1):
            self.iterate(it)
        return self.best_path, self.best_len, self.best_turns


class AStarOracle:
    def __init__(self, grid, allow_diag=True, restrict_corner=True):
        self.grid8 = np.ascontiguousarray(np.asarray(grid), dtype=np.uint8)
        self.R, self.C = self.grid8.shape
        self.ctx = lib().orc_astar_ctx_new(_p(self.grid8), self.R, self.C, int(allow_diag), int(restrict_corner))
        self.out = np.zeros(self.R * self.C, np.int32)

    def __del__(self):
        ctx, self.ctx = getattr(self, "ctx", None), None
        try:
            if ctx and _lib is not None:
                _lib.orc_astar_ctx_free(ctx)
        except Exception:                             # at interpreter exit the module's globals may be gone already
            pass

    def solve(self, variant, src, dst, avoid_bits=None):
        """Returns (cells int32 array, popped_g, expansions, relaxations)."""
        g = C.c_double()
        e = C.c_longlong()
        r = C.c_longlong()
        n = lib().orc_astar(self.ctx, variant, src, dst, _p(avoid_bits), _p(self.out), self.out.size,
                            C.byref(g), C.byref(e), C.byref(r))
        return self.out[:n].copy(), g.value, e.value, r.value


def cells_to_bits(cells, n_total):
    bits = np.zeros((n_total + 31) // 32, np.uint32)
    for c in cells:
        bits[c >> 5] |= np.uint32(1 << (c & 31))
    return bits


def path_stats(grid, cells, tpf, spf, msd, diag_value, restrict_policy=True, mode=0):
    g8 = np.ascontiguousarray(np.asarray(grid), dtype=np.uint8)
    cells = np.ascontiguousarray(cells, dtype=np.int32)
    out = np.zeros(5)
    pol = Policy(tpf, spf, msd, diag_value, int(restrict_policy), mode)
    lib().orc_path_stats(_p(g8), g8.shape[0], g8.shape[1], _p(cells), len(cells), C.byref(pol), _p(out))
    return out


def waypoint_fitness(grid, wps, tpf, spf, msd, diag_value, allow_diag=True, restrict_policy=True,
                     max_cells=None, threads=1):
    """wps: (N, W) int32 cells. Returns cells, n_cells, stats(N,5), expansions."""
    g8 = np.ascontiguousarray(np.asarray(grid), dtype=np.uint8)
    R, Cc = g8.shape
    (sr, sc), (tr, tc) = find_start_target(grid)
    wps = np.ascontiguousarray(wps, dtype=np.int32)
    N, W = wps.shape
    max_cells = max_cells or R * Cc
    cells = np.zeros((N, max_cells), np.int32)
    ncell = np.zeros(N, np.int32)
    stats = np.zeros((N, 5))
    pol = Policy(tpf, spf, msd, diag_value, int(restrict_policy), 0)
    ex = C.c_longlong()
    lib().orc_waypoint_fitness(_p(g8), R, Cc, int(allow_diag), int(restrict_policy), sr * Cc + sc, tr * Cc + tc,
                               _p(wps), N, W, C.byref(pol), _p(cells), max_cells, _p(ncell), _p(stats),
                               C.byref(ex), threads)
    return cells, ncell, stats, ex.value
