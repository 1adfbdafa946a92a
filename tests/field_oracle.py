"""TEST INFRASTRUCTURE: ctypes front-end to dijkstra_field_oracle.c (the C oracle's Dijkstra run over the whole map),
compiled on first use into a temporary directory keyed by the sources' contents."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import pyoracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "dijkstra_field_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha1()
        for f in (_SRC, os.path.join(os.path.dirname(_HERE), "oracle", "mpp_oracle.c")):
            h.update(open(f, "rb").read())
        so = os.path.join(tempfile.gettempdir(), f"libdijkstra_field_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(so):
            gcc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.check_call([gcc, "-O2", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math",
                                   "-fvisibility=hidden", "-shared", "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.orc_astar_ctx_new.restype = C.c_void_p
        L.orc_astar_ctx_new.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_astar_ctx_free.argtypes = [C.c_void_p]
        L.orc_dijkstra_field.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def dijkstra_field(grid, src, allow_diag=True, restrict_corner=True):
    """(g [R, C] float64, parent [R, C] uint8) of the oracle's Dijkstra from cell src over the whole map."""
    g8 = np.ascontiguousarray(np.asarray(grid), dtype=np.uint8)
    R, Cc = g8.shape
    L = lib()
    ctx = L.orc_astar_ctx_new(O._p(g8), R, Cc, int(allow_diag), int(restrict_corner))
    try:
        g = np.empty((R, Cc))
        parent = np.empty((R, Cc), np.uint8)
        L.orc_dijkstra_field(ctx, int(src), O._p(g), O._p(parent))
    finally:
        L.orc_astar_ctx_free(ctx)
    return g, parent


# move order of helper.py:30-36 (the parent codes)
MOVES = [(0, 1), (0, -1), (1, 0), (-1, 0), (1, 1), (1, -1), (-1, 1), (-1, -1)]


def chain(parent, dst):
    """Cells of the parent chain from the source to dst (forward), [] when dst has no chain (parent 0xFF and g inf is
    the caller's test; the source itself gives [src])."""
    R, Cc = parent.shape
    out = [int(dst)]
    t = int(dst)
    while parent.flat[t] != 0xFF:
        dr, dc = MOVES[parent.flat[t]]
        t -= dr * Cc + dc
        out.append(t)
    return out[::-1]
