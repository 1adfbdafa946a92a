"""ctypes binding of libmpp_b200.so (the C ABI declared in include/mpp.h).

There is deliberately no fallback: if the shared library is missing or no sm_100
device is visible, every compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libmpp_b200.so")

c_void_p, c_int, c_double, c_u64 = C.c_void_p, C.c_int, C.c_double, C.c_uint64


class MppError(RuntimeError):
    pass


class MaacoParams(C.Structure):
    _fields_ = [("alpha", c_double), ("beta", c_double), ("rho", c_double), ("Q", c_double),
                ("a_turn_coef", c_double), ("wh_max", c_double), ("wh_min", c_double),
                ("k_h_adaptive", c_double), ("q0_initial", c_double), ("C0_initial_pheromone", c_double),
                ("num_iterations", c_int)]


class MaacoState(C.Structure):
    _fields_ = [("best_len", c_double), ("best_turns", C.c_int32), ("best_n_cells", C.c_int32),
                ("best_iter", C.c_int32), ("best_ant", C.c_int32), ("iter_best_len", c_double),
                ("iter_best_turns", C.c_int32), ("iter_best_ant", C.c_int32)]


class Colony(C.Structure):
    """mpp_colony (include/mpp.h): the caller-owned device buffers of a colony / of one colony per map of a batch."""
    _fields_ = [("tau", c_void_p), ("tau_stride", C.c_longlong), ("E01", c_void_p), ("E01_stride", C.c_longlong),
                ("rank", c_void_p), ("slabs", c_void_p), ("touched", c_void_p), ("moves", c_void_p),
                ("max_cells", c_int), ("log_rows", c_int), ("result", c_void_p), ("deposit", c_void_p),
                ("okbits", c_void_p), ("state", c_void_p), ("best_cells", c_void_p), ("log", c_void_p),
                ("steps", c_void_p), ("seeds", c_void_p), ("latch", c_void_p)]


class Policy(C.Structure):
    _fields_ = [("turn_penalty_factor", c_double), ("safety_penalty_factor", c_double),
                ("min_safe_distance", c_double), ("diagonal_obstacle_penalty_value", c_double),
                ("restrict_policy", c_int), ("allow_diagonal", c_int), ("mode", c_int)]


_SIGS = {
    "mpp_abi_version": (c_int, []),
    "mpp_last_error": (C.c_char_p, []),
    "mpp_device_count": (c_int, []),
    "mpp_map_batch_create": (c_int, [c_void_p, c_int, c_int, c_int, c_int, C.POINTER(c_void_p)]),
    "mpp_map_batch_destroy": (None, [c_void_p]),
    "mpp_map_batch_size": (c_int, [c_void_p]),
    "mpp_map_batch_start": (c_int, [c_void_p, c_int]),
    "mpp_map_batch_target": (c_int, [c_void_p, c_int]),
    "mpp_map_batch_create_device": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, C.POINTER(c_void_p)]),
    "mpp_map_batch_occ_bits": (c_void_p, [c_void_p, C.POINTER(c_int)]),
    "mpp_map_batch_svalid": (c_void_p, [c_void_p]),
    "mpp_map_batch_obstacles": (C.c_longlong, [c_void_p]),
    "mpp_maaco_tables": (c_int, [c_void_p, C.POINTER(MaacoParams), c_void_p, C.c_longlong, c_void_p, c_void_p, c_void_p]),
    "mpp_maaco_e01_host": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, C.POINTER(MaacoParams), c_void_p, c_int]),
    "mpp_maaco_tau0_maps": (c_int, [c_void_p, C.POINTER(MaacoParams), c_void_p, C.c_longlong, c_void_p]),
    "mpp_maaco_e01_maps": (c_int, [c_void_p, C.POINTER(MaacoParams), c_void_p, C.c_longlong, c_void_p]),
    "mpp_libm_exp_pow": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "mpp_maaco_q0": (c_double, [c_int, c_int, c_double]),
    "mpp_maaco_rank_words": (C.c_longlong, [c_int, c_int]),
    "mpp_maaco_slab_words": (C.c_longlong, [c_int, c_int, c_int]),
    "mpp_maaco_touched_words": (C.c_longlong, [c_int, c_int, c_int]),
    "mpp_maaco_rank": (c_int, [c_void_p, C.POINTER(Colony), c_double, c_void_p]),
    "mpp_maaco_tours": (c_int, [c_void_p, C.POINTER(Colony), c_int, c_double, c_double, c_int, c_int, c_int, c_int,
                                c_void_p]),
    "mpp_maaco_tours_p2p": (c_int, [c_void_p, C.POINTER(Colony), c_int, c_double, c_double, c_int, c_int, c_int, c_int,
                                    c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "mpp_maaco_best": (c_int, [c_void_p, C.POINTER(Colony), c_int, c_int, c_int, c_double, c_int, c_void_p]),
    "mpp_maaco_pheromone": (c_int, [c_void_p, C.POINTER(Colony), c_void_p, c_void_p, c_int, c_int, c_int, c_double,
                                    c_int, c_int, c_void_p, c_int, c_void_p]),
    "mpp_maaco_pass": (c_int, [c_void_p, C.POINTER(Colony), C.POINTER(MaacoParams), c_int, c_int, c_int, c_void_p]),
    "mpp_maaco_pass_host": (c_int, [c_void_p, C.POINTER(Colony), C.POINTER(MaacoParams), c_int, c_int, c_int, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "mpp_maaco_max_peers": (c_int, []),
    "mpp_maaco_xhdr_bytes": (C.c_longlong, [c_int]),
    "mpp_maaco_xpack": (c_int, [c_void_p, C.POINTER(Colony), c_int, c_int, c_int, c_void_p, c_void_p, C.c_longlong,
                                c_void_p, c_int, c_int, c_void_p]),
    "mpp_maaco_xunpack": (c_int, [c_void_p, C.POINTER(Colony), c_void_p, C.c_longlong, c_int, c_int, c_int, c_void_p,
                                  c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mpp_path_stats": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, C.POINTER(Policy), c_void_p,
                               c_void_p]),
    "mpp_map_batch_safety_table": (c_int, [c_void_p, c_double, c_void_p]),
    "mpp_map_batch_max_slots": (c_int, [c_void_p]),
    "mpp_astar_batch_maps": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                     C.POINTER(Policy), c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                     C.c_size_t, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "mpp_dijkstra_field_scratch_bytes": (C.c_size_t, [c_void_p]),
    "mpp_dijkstra_fields": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, C.c_size_t, c_void_p]),
    "mpp_dijkstra_field_paths": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, C.POINTER(Policy),
                                         c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mpp_astar_slot_bytes": (C.c_size_t, [c_int, c_int, c_int]),
    "mpp_mpa_init_batch": (c_int, [c_void_p, C.POINTER(Policy), c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                   C.c_size_t, c_int, c_void_p, c_void_p, c_void_p]),
    "mpp_mpa_iteration_batch": (c_int, [c_void_p, C.POINTER(Policy), c_int, c_int, c_int, c_int, c_int, c_double, c_double,
                                        c_double, c_double, c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, C.c_size_t, c_int,
                                        c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mpp_waypoint_fitness_maps": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, C.POINTER(Policy), c_void_p, c_int,
                                          c_void_p, c_void_p, c_void_p, c_void_p, C.c_size_t, c_int, c_int, c_void_p,
                                          c_void_p, c_void_p]),
    "mpp_pso_init_batch": (c_int, [c_void_p, c_int, c_void_p, c_int, c_double, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p]),
    "mpp_ga_init_batch": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "mpp_pso_update_batch": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_double,
                                     c_double, c_double, c_double, c_void_p, c_int, c_void_p, c_void_p]),
    "mpp_ga_select_batch": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "mpp_ga_breed_batch": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_double, c_double, c_void_p, c_int,
                                   c_void_p, c_void_p]),
}

_lib = None


def declared_symbols():
    return sorted(_SIGS)


def lib():
    """Load the library (once). Raises MppError when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise MppError(f"{SO_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU/PyTorch fallback)")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in _SIGS.items():
            if not hasattr(L, name):
                continue  # optional symbols are checked by tests/test_abi.py against include/mpp.h
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().mpp_last_error()
        raise MppError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


def ptr(t):
    """Device/host pointer of a torch tensor (or None)."""
    if t is None:
        return None
    return c_void_p(t.data_ptr())


def require_device():
    n = lib().mpp_device_count()
    if n <= 0:
        raise MppError("no sm_100 (B200) device visible; libmpp_b200 has no CPU fallback")
    return n
