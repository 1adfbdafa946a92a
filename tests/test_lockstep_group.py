"""CPU checks of the lockstep process group (tests/lockstep_group.py) that the emulated sharded-colony tests run on: its
collectives compute what torch.distributed's do, in a fixed order, and an error in one rank ends the group instead of
hanging it."""
import threading

import pytest
import torch
import torch.distributed as dist

from lockstep_group import GroupAborted, lockstep_group


def test_rank_and_world_size(monkeypatch):
    with lockstep_group(monkeypatch, 3) as g:
        out = g.run(lambda r: (dist.get_rank(g), dist.get_world_size(g), dist.get_global_rank(g, 2)))
    assert out == [(0, 3, 2), (1, 3, 2), (2, 3, 2)]
    assert dist.get_world_size is not g.get_world_size                       # the fakes are gone with the context


def test_gather_in_place(monkeypatch):
    """The input is a slice of the output (what gather_tau and MPA's row blocks do): every rank gets every part."""
    W, n = 4, 5
    with lockstep_group(monkeypatch, W) as g:
        def body(r):
            out = torch.full((W * n,), -1.0, dtype=torch.float64)
            out[r * n:(r + 1) * n] = torch.arange(n, dtype=torch.float64) + 100 * r
            dist.all_gather_into_tensor(out, out[r * n:(r + 1) * n], group=g)
            return out
        outs = g.run(body)
    want = torch.cat([torch.arange(n, dtype=torch.float64) + 100 * r for r in range(W)])
    for o in outs:
        assert torch.equal(o, want)


def test_gather_separate_buffers_and_2d_output(monkeypatch):
    W = 3
    with lockstep_group(monkeypatch, W) as g:
        def body(r):
            inp = torch.tensor([[r, 10 * r]], dtype=torch.int32)
            out = torch.zeros((W, 2), dtype=torch.int32)
            dist.all_gather_into_tensor(out, inp, group=g)
            return out
        outs = g.run(body)
    for o in outs:
        assert o.tolist() == [[0, 0], [1, 10], [2, 20]]


def test_gather_rejects_a_wrong_output_size(monkeypatch):
    with lockstep_group(monkeypatch, 2) as g:
        with pytest.raises(ValueError, match="all_gather_into_tensor"):
            g.run(lambda r: dist.all_gather_into_tensor(torch.zeros(3), torch.zeros(2), group=g))


@pytest.mark.parametrize("op, want", [(dist.ReduceOp.MIN, [-3, 0, 1]), (dist.ReduceOp.MAX, [0, 5, 9])])
def test_all_reduce_min_max(monkeypatch, op, want):
    rows = [[0, 5, 1], [-3, 0, 9], [-1, 2, 4]]
    with lockstep_group(monkeypatch, 3) as g:
        def body(r):
            t = torch.tensor(rows[r], dtype=torch.int64)
            dist.all_reduce(t, op=op, group=g)
            return t.tolist()
        outs = g.run(body)
    assert outs == [want] * 3


def test_all_reduce_refuses_other_ops(monkeypatch):
    with lockstep_group(monkeypatch, 2) as g:
        with pytest.raises(NotImplementedError):
            g.run(lambda r: dist.all_reduce(torch.zeros(1), op=dist.ReduceOp.SUM, group=g))


def test_broadcast_from_a_nonzero_source(monkeypatch):
    with lockstep_group(monkeypatch, 4) as g:
        def body(r):
            t = torch.tensor([r, r * r], dtype=torch.int32)
            dist.broadcast(t, src=dist.get_global_rank(g, 2), group=g)
            return t.tolist()
        outs = g.run(body)
    assert outs == [[2, 4]] * 4


def test_symmetric_memory_handles(monkeypatch):
    import torch.distributed._symmetric_memory as symm
    with lockstep_group(monkeypatch, 3) as g:
        def body(r):
            t = symm.empty(4, dtype=torch.int32, device="cpu")
            h = symm.rendezvous(t, g)
            h.barrier(channel=0)
            return t.data_ptr(), h.buffer_ptrs
        outs = g.run(body)
    ptrs = [p for p, _ in outs]
    assert len(set(ptrs)) == 3 and all(h == ptrs for _, h in outs)


def test_order_is_deterministic(monkeypatch):
    """Between two collectives the ranks run one at a time in rank order, and never two at once."""
    W, rounds = 5, 4
    for _ in range(3):
        trace = []
        busy = threading.Lock()
        with lockstep_group(monkeypatch, W) as g:
            def body(r):
                for k in range(rounds):
                    assert busy.acquire(blocking=False), "two ranks ran at once"
                    trace.append((k, r))
                    busy.release()
                    dist.barrier(group=g)
            g.run(body)
        assert trace == [(k, r) for k in range(rounds) for r in range(W)]
        assert g.log == ["barrier"] * rounds


def test_an_error_in_one_rank_surfaces_without_a_hang(monkeypatch):
    with lockstep_group(monkeypatch, 4, timeout=30) as g:
        def body(r):
            dist.barrier(group=g)
            if r == 2:
                raise KeyError("rank 2 failed")
            dist.barrier(group=g)                                  # the others wait here for rank 2 ...
            dist.barrier(group=g)
        with pytest.raises(KeyError, match="rank 2 failed"):      # ... and the first error is what the caller sees
            g.run(body)


def test_ranks_that_disagree_on_the_collective_fail(monkeypatch):
    with lockstep_group(monkeypatch, 3, timeout=30) as g:
        def body(r):
            if r == 1:
                dist.all_reduce(torch.zeros(1), op=dist.ReduceOp.MAX, group=g)
            else:
                dist.barrier(group=g)
        with pytest.raises(RuntimeError, match="disagree"):
            g.run(body)


def test_a_rank_that_returns_early_fails_the_others(monkeypatch):
    with lockstep_group(monkeypatch, 2, timeout=30) as g:
        def body(r):
            if r == 1:
                dist.barrier(group=g)
        with pytest.raises((RuntimeError, GroupAborted)):
            g.run(body)


def test_a_stuck_rank_times_out(monkeypatch):
    release = threading.Event()
    with lockstep_group(monkeypatch, 2, timeout=1.0) as g:
        def body(r):
            if r == 0:
                release.wait(20)                                   # holds the baton past the group's timeout
            dist.barrier(group=g)
        try:
            with pytest.raises(TimeoutError):
                g.run(body)
        finally:
            release.set()


def test_collectives_outside_a_rank_are_refused(monkeypatch):
    with lockstep_group(monkeypatch, 2) as g:
        with pytest.raises(RuntimeError, match="not called from a rank"):
            dist.get_rank(g)
