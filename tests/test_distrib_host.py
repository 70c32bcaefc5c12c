"""Host-side logic of flashy_b200.distrib on CPU (no GPU): rank helpers, loader sharding, the
count check that must raise on every rank, object broadcast, host barrier -- with W spawned
processes over gloo (bootstrap only) and with virtual ranks (threads).  Mirrors the
reference's tests/test_distrib.py harness; the tensor data path itself needs CUDA and is
covered by the `-m gpu` tests."""
import threading
from collections import defaultdict

import numpy as np
import pytest
import torch

from tests import golden_io as G
from tests.golden import cases
from tests.harness import run_ranks


def _worker(rank, world):
    from flashy_b200 import distrib
    assert distrib.rank() == rank and distrib.world_size() == world
    assert distrib.is_rank_zero() == (rank == 0) and distrib.is_distributed()
    assert [distrib.rank(), distrib.world_size(), int(distrib.is_rank_zero()), int(distrib.is_distributed())] \
        == G.get(world, "rank", rank).tolist()                      # bit-exact vs the reference
    assert distrib.rank_zero_only(lambda: 7)() == (7 if rank == 0 else None)

    # loader shards: bit-exact against the reference's index lists (flashy/distrib.py:227-243)
    data = list(range(cases.LOADER_N))
    for shuffle in (False, True):
        seen = [int(v) for batch in distrib.loader(data, shuffle=shuffle, batch_size=4) for v in batch]
        assert seen == G.get(world, f"loader/shuffle{int(shuffle)}", rank).tolist()

    # tests/test_distrib.py:37-46 -- count mismatch raises on EVERY rank, nobody hangs
    x, y = torch.tensor([1.0]), torch.tensor([0.0])
    for fn in (distrib.broadcast_tensors, distrib.average_tensors):
        try:
            fn([x, y] if rank == world - 1 else [x])
        except RuntimeError as err:
            assert "Mismatch in number of params" in str(err)
        else:
            raise AssertionError("Should have raised")
    # same count, different shapes: also refused (stricter than the reference, never silent)
    try:
        distrib.average_tensors([torch.zeros(3 if rank == 0 else 4)])
    except RuntimeError as err:
        assert "Mismatch" in str(err)
    else:
        raise AssertionError("Should have raised")

    # equal lists of CPU tensors: the check passes, then the data path refuses loudly
    for fn in (distrib.average_tensors, distrib.broadcast_tensors, distrib.all_reduce):
        arg = torch.ones(4) if fn is distrib.all_reduce else [torch.ones(4)]
        with pytest.raises(RuntimeError, match="no gloo/CPU fallback|no CPU fallback"):
            fn(arg)
    # int tensors are skipped before anything else happens (flashy/distrib.py:102)
    distrib.average_tensors([torch.arange(3)])
    distrib.broadcast_tensors([torch.arange(3)])
    distrib.average_tensors([])

    obj = None
    if distrib.rank() == 0:
        obj = defaultdict(int)
        obj["test"] = 42
        obj["youpi"] = 21
    received = distrib.broadcast_object(obj)                       # tests/test_distrib.py:71-79
    assert isinstance(received, defaultdict) and dict(received) == {"test": 42, "youpi": 21}
    assert distrib.broadcast_object(rank * 10, src=world - 1) == (world - 1) * 10
    big = bytes(range(256)) * 5000 if rank == 1 else None          # 1.28 MB: several fabric chunks
    assert distrib.broadcast_object(big, src=1) == bytes(range(256)) * 5000
    assert distrib.broadcast_object(None) is None and distrib.broadcast_object(b"", src=world - 1) == b""
    for _ in range(20):
        distrib.barrier()


@pytest.mark.parametrize("world", (2, 8))
def test_distrib_host_logic_gloo(world):
    run_ranks(world, "tests.test_distrib_host", "_worker", hide_gpus=True)


def test_single_process_is_a_noop():
    """W == 1: nothing moves, nothing is touched (flashy/distrib.py:54-55,100-101,118-119)."""
    from flashy_b200 import distrib
    assert distrib.rank() == 0 and distrib.world_size() == 1 and not distrib.is_distributed()
    metrics = {"loss": 1.5}
    assert distrib.average_metrics(metrics, 3) is metrics
    t = torch.ones(3)
    assert distrib.all_reduce(t) is None and torch.equal(t, torch.ones(3))
    distrib.average_tensors([t]); distrib.broadcast_tensors([t]); distrib.barrier()
    model = torch.nn.Linear(32, 1)                                 # examples/basic: plumbing only
    model(torch.randn(4, 32)).sum().backward()
    g = model.weight.grad.clone()
    distrib.sync_model(model)
    with distrib.eager_sync_model(model):
        pass
    assert torch.equal(model.weight.grad, g)
    assert distrib.wrap(model) is model
    assert distrib.broadcast_object({"a": 1}) == {"a": 1}
    dl = distrib.loader(list(range(10)), batch_size=5)
    assert [b.tolist() for b in dl] == [[0, 1, 2, 3, 4], [5, 6, 7, 8, 9]]
    distrib.init()                                                 # WORLD_SIZE unset -> no-op


def test_virtual_ranks_host_logic():
    """Virtual ranks (threads of one process) see a world of their own; rendezvous works."""
    run_ranks(1, "tests.test_distrib_host", "_virtual_ranks_worker", backend="none", hide_gpus=True)


def _virtual_ranks_worker(proc_rank, proc_world):
    from flashy_b200 import VirtualWorld, distrib
    world = 4
    vw = VirtualWorld(world)
    assert vw.engine.host_only          # this process sees no CUDA device

    def body(rank, w):
        assert (distrib.rank(), distrib.world_size()) == (rank, w) and w == world
        data = list(range(cases.LOADER_N))
        seen = [int(v) for batch in distrib.loader(data, shuffle=False, batch_size=4) for v in batch]
        assert seen == list(range(rank, cases.LOADER_N, world))
        try:
            distrib.average_tensors([torch.ones(1)] * (2 if rank == 1 else 1))
        except RuntimeError as err:
            assert "Mismatch in number of params" in str(err)
        else:
            raise AssertionError("Should have raised")
        assert distrib.broadcast_object({"r": rank}, src=2) == {"r": 2}
        distrib.barrier()
        return distrib.rank_zero_only(lambda: "zero")()

    try:
        assert vw.run(body) == ["zero", None, None, None]
        with pytest.raises(ZeroDivisionError):
            # a failing rank aborts the local rendezvous: the others do not hang
            vw.run(lambda rank, w: 1 / 0 if rank == 2 else distrib.broadcast_object(rank))
    finally:
        vw.close()
    assert distrib.world_size() == 1      # outside the virtual world again


def _abort_worker(rank, world):
    """A rank that fails poisons the communicator: the others error out promptly, nobody hangs."""
    import time
    from flashy_b200 import distrib, context
    from flashy_b200._native import NativeError
    distrib.barrier()                                   # creates the communicator on every rank
    if rank == 1:
        context.current().engine.abort()                # what a failing rank does before it dies
        return
    t0 = time.time()
    try:
        distrib.barrier()
    except NativeError as err:
        assert "aborted" in str(err)
    else:
        raise AssertionError("the barrier should have failed")
    assert time.time() - t0 < 30


def test_abort_wakes_blocked_ranks():
    run_ranks(3, "tests.test_distrib_host", "_abort_worker")
