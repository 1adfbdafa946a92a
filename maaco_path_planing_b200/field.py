"""Exact Dijkstra distance fields (mpp_dijkstra_fields / mpp_dijkstra_field_paths).

One field per map holds, for every cell, the g with which dijkstra.py's search pops it and the move it was reached by
-- bit for bit what DijkstraSolver.solve computes with that cell as its target.  Any number of targets then cost one
path-reading launch instead of one search each.  Used by DijkstraSolver (one map) and SearchBatch (a batch)."""
from __future__ import annotations

import ctypes as C

from . import _lib


def _stream(device):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def dijkstra_fields(owner, batch, shape, src, allow_diagonal, restrict_corner):
    """Fields of every map of the mpp_map_batch `batch` ([n_maps, rows, cols] = shape) from the cells src (int32 CUDA
    tensor [n_maps]; a cell outside the map or an obstacle gives an all-inf field).  Returns (g float64, parent uint8)
    CUDA tensors of that shape on owner.device."""
    import torch as t
    L = _lib.lib()
    g = t.empty(shape, dtype=t.float64, device=owner.device)
    parent = t.empty(shape, dtype=t.uint8, device=owner.device)
    nbytes = L.mpp_dijkstra_field_scratch_bytes(batch)
    scratch = t.empty(nbytes, dtype=t.uint8, device=owner.device)   # (the allocator keeps it for this stream's work)
    _lib.check(L.mpp_dijkstra_fields(batch, _lib.ptr(src), int(bool(allow_diagonal)), int(bool(restrict_corner)),
                                     _lib.ptr(g), _lib.ptr(parent), _lib.ptr(scratch), nbytes, _stream(owner.device)),
               "mpp_dijkstra_fields")
    owner.launches += 1
    return g, parent


def _paths_launch(owner, batch, g, parent, mi, dst, policy):
    import torch as t
    n, mc = mi.numel(), owner.max_cells
    cells = t.empty((n, mc), dtype=t.int32, device=owner.device)
    ncell = t.empty(n, dtype=t.int32, device=owner.device)
    gout = t.empty(n, dtype=t.float64, device=owner.device)
    stats = t.empty((n, 5), dtype=t.float64, device=owner.device)
    _lib.check(_lib.lib().mpp_dijkstra_field_paths(
        batch, _lib.ptr(g), _lib.ptr(parent), _lib.ptr(mi), _lib.ptr(dst), n, C.byref(policy), _lib.ptr(cells), mc,
        _lib.ptr(ncell), _lib.ptr(gout), _lib.ptr(stats), _stream(owner.device)), "mpp_dijkstra_field_paths")
    owner.launches += 1
    return cells, ncell, gout, stats


def field_paths(owner, batch, g, parent, mi, dst, policy):
    """Query i: the path from the source of field mi[i] to cell dst[i] (int32 CUDA tensors [n]), read from the fields
    (g, parent) of dijkstra_fields.  Returns device tensors (cells [n, max_cells] int32, n_cells [n] int32, g [n] float64,
    stats [n, 5] float64) with SearchBatch.search's conventions.  A truncated path grows owner.max_cells and repeats only
    the truncated queries."""
    import torch as t
    n = mi.numel()
    if n == 0:
        return (t.zeros((0, owner.max_cells), dtype=t.int32, device=owner.device),
                t.zeros(0, dtype=t.int32, device=owner.device), t.zeros(0, dtype=t.float64, device=owner.device),
                t.zeros((0, 5), dtype=t.float64, device=owner.device))
    cells, ncell, gout, stats = _paths_launch(owner, batch, g, parent, mi, dst, policy)
    while owner._grow_from(0, int(ncell.max().item())):
        bad = (ncell > cells.shape[1]).nonzero().squeeze(1)
        c, nc, gg, st = _paths_launch(owner, batch, g, parent, mi.index_select(0, bad).contiguous(),
                                      dst.index_select(0, bad).contiguous(), policy)
        cells = t.nn.functional.pad(cells, (0, c.shape[1] - cells.shape[1]))   # max_cells grew: widen every row
        cells[bad] = c
        ncell[bad], gout[bad], stats[bad] = nc, gg, st
    return cells, ncell, gout, stats
