"""An in-process process group for tests: W ranks as W Python threads on one device, run in lockstep.

Every sharded code path of the package -- the MAACO colony's peer-memory and all-gather exchanges, the sharded
PSO / GA / MPA populations -- computes the same thing whether its ranks sit on W GPUs or take turns on one.  A "peer"
pointer to a buffer on the same device is a plain global store and an all-gather is a copy, so one GPU can run all of
them against the single-colony oracle, at any rank count.

A baton lets exactly one rank run at a time: the C library and the device's default stream are never used from two
threads at once.  A rank runs until its next collective, posts its part and hands the baton to rank + 1; the last rank
to arrive completes the collective (on the tensors' device, in stream order) and hands the baton back to rank 0.  The
order of every launch is therefore fixed, and stream order stands in for the barriers between GPUs.  (What serial
emulation cannot see -- the memory ordering of real peer stores, the symmetric-memory barriers, NCCL -- stays with the
torchrun checks tests/multigpu_check.py and tests/multigpu_solvers_check.py.)

    with lockstep_group(monkeypatch, 4) as g:
        results = g.run(lambda rank: MAACO(..., group=g).solve_path_planning())

If a rank raises, the group is aborted: every rank that waits for the baton raises GroupAborted, and run() re-raises
the first error in the calling thread.  Every wait has a timeout.
"""
from __future__ import annotations

import contextlib
import threading
import time

import torch
import torch.distributed as dist

_DONE = "<rank returned>"


class GroupAborted(RuntimeError):
    """Raised in a rank whose group was aborted by an error in another rank."""


class _SymmHandle:
    """What torch.distributed._symmetric_memory.rendezvous returns, as far as the package uses it."""

    def __init__(self, group, ptrs):
        self._group = group
        self.buffer_ptrs = list(ptrs)

    def barrier(self, channel=0, timeout_ms=0):
        self._group._collective(f"symm_barrier:{channel}", None, lambda parts: [None] * len(parts))


class LockstepGroup:
    def __init__(self, world, timeout=300.0):
        if world < 1:
            raise ValueError("world must be >= 1")
        self.world = int(world)
        self.timeout = float(timeout)
        self.log = []                       # names of the completed collectives, in order
        self._cv = threading.Condition()
        self._tls = threading.local()
        self._turn = 0                      # rank holding the baton
        self._posted = [None] * self.world  # (name, part) of every rank in the current round
        self._results = [None] * self.world
        self._error = None                  # first exception raised by a rank

    # ---- the baton -----------------------------------------------------------------------------------------------
    def rank(self):
        r = getattr(self._tls, "rank", None)
        if r is None:
            raise RuntimeError("not called from a rank of the lockstep group")
        return r

    def _wait_turn(self, r):
        """(cv held) until rank r holds the baton."""
        ok = self._cv.wait_for(lambda: self._error is not None or self._turn == r, self.timeout)
        if self._error is not None:
            raise GroupAborted(f"rank {r}: the group was aborted by {type(self._error).__name__}: {self._error}")
        if not ok:
            raise TimeoutError(f"rank {r}: no baton within {self.timeout} s")

    def _collective(self, name, part, complete):
        """Post this rank's `part` of collective `name`; the last rank runs complete([part of every rank]) -> [result of
        every rank].  Returns this rank's result once every rank before it has resumed."""
        r = self.rank()
        with self._cv:
            if self._error is not None:
                raise GroupAborted(f"rank {r}: the group was aborted")
            assert self._turn == r, f"rank {r} runs without the baton (turn {self._turn})"
            self._posted[r] = (name, part)
            if r == self.world - 1:
                names = [p[0] for p in self._posted]
                if any(n != name for n in names):
                    raise RuntimeError(f"the ranks disagree on the collective: {names}")
                parts = [p[1] for p in self._posted]
                self._posted = [None] * self.world
                if name == _DONE:
                    self._turn = -1
                    self._cv.notify_all()
                    return None
                self._results = complete(parts)
                self.log.append(name)
                self._turn = 0
            else:
                self._turn = r + 1
            self._cv.notify_all()
            if name == _DONE:
                return None
            self._wait_turn(r)
            return self._results[r]

    def run(self, fn, *args):
        """fn(rank, *args) on every rank, each in its own thread; returns the W return values in rank order or re-raises
        the first error of any rank."""
        out = [None] * self.world

        def body(r):
            self._tls.rank = r
            try:
                with self._cv:
                    self._wait_turn(r)
                out[r] = fn(r, *args)
                self._collective(_DONE, None, None)
            except BaseException as e:  # noqa: BLE001 -- handed to the calling thread
                with self._cv:
                    if self._error is None:
                        self._error = e
                    self._cv.notify_all()

        threads = [threading.Thread(target=body, args=(r,), name=f"lockstep-rank-{r}", daemon=True)
                   for r in range(self.world)]
        for t in threads:
            t.start()
        deadline = time.monotonic() + self.timeout
        for t in threads:
            t.join(max(0.0, deadline - time.monotonic()))
        if any(t.is_alive() for t in threads):
            with self._cv:
                if self._error is None:
                    self._error = TimeoutError(f"lockstep group of {self.world} ranks still running after {self.timeout} s")
                self._cv.notify_all()
            for t in threads:
                t.join(5.0)
        if self._error is not None:
            raise self._error
        return out

    # ---- torch.distributed ---------------------------------------------------------------------------------------
    def _check_group(self, group):
        if group is not None and group is not self:
            raise ValueError("a collective on a group other than the lockstep group")

    def get_world_size(self, group=None):
        self._check_group(group)
        return self.world

    def get_rank(self, group=None):
        self._check_group(group)
        return self.rank()

    def get_global_rank(self, group, group_rank):
        self._check_group(group)
        return int(group_rank)

    def barrier(self, group=None, async_op=False, device_ids=None):
        self._check_group(group)
        self._collective("barrier", None, lambda parts: [None] * len(parts))

    def all_reduce(self, tensor, op=dist.ReduceOp.SUM, group=None, async_op=False):
        self._check_group(group)
        if op == dist.ReduceOp.MIN:
            red = lambda x: x.amin(0)
        elif op == dist.ReduceOp.MAX:
            red = lambda x: x.amax(0)
        else:
            raise NotImplementedError(f"all_reduce op {op}")

        def complete(parts):
            v = red(torch.stack([t.clone() for t in parts]))
            for t in parts:
                t.copy_(v)
            return [None] * len(parts)
        self._collective(f"all_reduce:{op}", tensor, complete)

    def broadcast(self, tensor, src, group=None, async_op=False):
        self._check_group(group)

        def complete(parts):
            v = parts[src].clone()
            for t in parts:
                t.copy_(v)
            return [None] * len(parts)
        self._collective(f"broadcast:{src}", tensor, complete)

    def all_gather_into_tensor(self, output_tensor, input_tensor, group=None, async_op=False):
        self._check_group(group)
        if not output_tensor.is_contiguous() or output_tensor.numel() != self.world * input_tensor.numel() or \
                output_tensor.dtype != input_tensor.dtype:
            raise ValueError("all_gather_into_tensor: the output must be a contiguous [world * input] of the input's dtype")

        def complete(parts):
            ins = [i.clone().reshape(-1) for _, i in parts]           # inputs may be slices of the outputs (in place)
            for out, _ in parts:
                flat = out.view(-1)
                for r, x in enumerate(ins):
                    flat[r * x.numel():(r + 1) * x.numel()].copy_(x)
            return [None] * len(parts)
        self._collective("all_gather_into_tensor", (output_tensor, input_tensor), complete)

    # ---- torch.distributed._symmetric_memory ---------------------------------------------------------------------
    def symm_empty(self, *size, dtype=None, device=None):
        return torch.empty(*size, dtype=dtype, device=device)

    def rendezvous(self, tensor, group=None):
        self._check_group(group)

        def complete(parts):
            ptrs = [t.data_ptr() for t in parts]
            return [_SymmHandle(self, ptrs) for _ in parts]
        return self._collective("rendezvous", tensor, complete)


_DIST_NAMES = ("get_world_size", "get_rank", "get_global_rank", "barrier", "all_reduce", "broadcast",
               "all_gather_into_tensor")


@contextlib.contextmanager
def lockstep_group(monkeypatch, world, timeout=300.0):
    """A LockstepGroup of `world` ranks whose collectives stand in for torch.distributed's (and for the symmetric-memory
    allocations the sharded colony's peer exchange uses) while the context is open."""
    import torch.distributed._symmetric_memory as symm
    g = LockstepGroup(world, timeout)
    with monkeypatch.context() as mp:
        for name in _DIST_NAMES:
            mp.setattr(dist, name, getattr(g, name))
        mp.setattr(symm, "empty", g.symm_empty)
        mp.setattr(symm, "rendezvous", g.rendezvous)
        yield g
