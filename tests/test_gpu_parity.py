"""Parity of the CUDA path with the oracle, through flashy_b200.distrib -> C ABI -> kernels.

One GPU is enough: the W ranks are virtual ranks of one process (``VirtualWorld``), each on
its own thread calling the unchanged reference-shaped API; their calls leave as single
launches whose CTAs synchronise through the same flag protocol and read each other's arenas
exactly as separate GPUs would (the peer pointers simply resolve to local memory).

Bars (BASELINE.json north_star / BASELINE.md section 5):
  * integers, indices, broadcast: bit-exact;
  * fp32 / fp64 / complex: |out - ref| / (sum_r |x_r| / W) <= 1e-6 against the golden vectors of
    the unmodified reference (gloo), and bit-exact against oracle/numeric.py (same rank-order sum);
  * bf16 / fp16: <= 1 ulp (in practice 0) against ``round(fp32 oracle on the same inputs)``.
"""
import os

import numpy as np
import pytest
import torch

from oracle import numeric
from tests import golden_io as G
from tests.golden import cases

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-6
_worlds = {}


def vworld(world: int):
    from flashy_b200 import VirtualWorld
    if world not in _worlds:
        _worlds[world] = VirtualWorld(world, device=0, arena_mb=160)
    return _worlds[world]


@pytest.fixture(scope="module", autouse=True)
def _cleanup():
    yield
    for vw in _worlds.values():
        vw.close()
    _worlds.clear()


def run(world, fn, *args):
    return vworld(world).run(fn, *args)


# --------------------------------------------------------------------------- reference's own test
def test_reference_test_distrib_on_cuda():
    """/root/reference/tests/test_distrib.py:26-79, same assertions, CUDA tensors, WS = 8."""
    from collections import defaultdict
    from torch import nn
    from flashy_b200 import distrib
    WS = 8

    def worker(rank, world):
        x = torch.tensor([float(rank) + 1], device="cuda")
        distrib.average_tensors([x])
        assert x.item() == sum(range(1, WS + 1)) / WS, x.item()

        x = torch.tensor([float(rank) + 1], device="cuda")
        distrib.broadcast_tensors([x])
        assert x.item() == 1.

        y = torch.tensor([0.], device="cuda")
        try:
            if rank == 5:
                distrib.broadcast_tensors([x, y])
            else:
                distrib.broadcast_tensors([x])
        except RuntimeError:
            pass
        else:
            assert False, "Should have raised"

        mod = nn.Linear(1, 1, bias=False).cuda()
        mod.weight.data.zero_()
        x = torch.ones(1, 1, device="cuda")
        for eager in [False, True]:
            y = mod(x)
            gt = torch.tensor(float(rank), device="cuda").view(-1, 1)
            loss = nn.functional.mse_loss(y, gt)
            if eager:
                with distrib.eager_sync_model(mod):
                    loss.backward()
            else:
                loss.backward()
                distrib.sync_model(mod)
            grad = mod.weight.grad.data.clone()
            mod.weight.grad.data.zero_()
            y = mod(x.expand(WS, 1))
            gt = torch.arange(WS, device="cuda").float().view(-1, 1)
            loss = nn.functional.mse_loss(y, gt)
            loss.backward()
            grad_ref = mod.weight.grad.data
            assert torch.allclose(grad, grad_ref), (eager, grad.item(), grad_ref.item())
            mod.weight.grad.data.zero_()

        obj = None
        if distrib.rank() == 0:
            obj = defaultdict(int)
            obj['test'] = 42
            obj['youpi'] = 21
        received = distrib.broadcast_object(obj)
        assert isinstance(received, defaultdict)
        assert dict(received) == {'test': 42, 'youpi': 21}

    run(WS, worker)


# --------------------------------------------------------------------------- golden vectors
@pytest.mark.parametrize("world", cases.WORLDS)
@pytest.mark.parametrize("name", list(cases.AVG_DTYPES))
def test_average_tensors_golden(world, name):
    from flashy_b200 import distrib
    dtype = cases.AVG_DTYPES[name]
    per_rank = [cases.avg_inputs(r, name) for r in range(world)]
    model = numeric.average_tensors(per_rank)

    def body(rank, w):
        ts = [t.cuda() for t in per_rank[rank]]
        distrib.average_tensors(ts)
        torch.cuda.synchronize()
        return [t.cpu() for t in ts]

    got = run(world, body)
    for r in range(world):
        for i, t in enumerate(got[r]):
            if i == cases.INT_SLOT:
                assert torch.equal(t, per_rank[r][i])                    # skipped, untouched
                continue
            assert torch.equal(t, got[0][i])                             # replicas agree bit for bit
            cols = [per_rank[q][i] for q in range(world)]
            if name in ("fp32", "fp64", "c64"):
                ref = G.golden_tensor(world, f"avg/{name}/out/{i}", dtype)
                assert G.normalised_error(t, ref, cols) <= FP32_TOL      # vs unmodified reference
                assert torch.equal(t, model[r][i])                       # vs rank-order oracle: exact
            elif name == "bf16":
                assert G.ulp_distance_bf16(t, model[r][i]) <= 1
                assert torch.equal(t, model[r][i])
            else:
                assert torch.equal(t, model[r][i])


@pytest.mark.parametrize("world", cases.WORLDS)
def test_broadcast_golden(world):
    from flashy_b200 import distrib
    per_rank = [cases.avg_inputs(r, "fp32") for r in range(world)]
    for src in (0, world - 1):
        def body(rank, w, src=src):
            ts = [t.cuda() for t in per_rank[rank]]
            distrib.broadcast_tensors(ts, src=src)
            torch.cuda.synchronize()
            return [t.cpu() for t in ts]
        got = run(world, body)
        for r in range(world):
            for i, t in enumerate(got[r]):
                assert np.array_equal(G.get(world, f"bcast/src{src}/out/{i}", r), cases.to_np(t)), (src, r, i)


@pytest.mark.parametrize("world", cases.WORLDS)
@pytest.mark.parametrize("variant", ("avg", "bcast", "eager"))
def test_sync_model_golden(world, variant):
    from flashy_b200 import distrib

    def body(rank, w):
        model = cases.make_model().cuda()
        grads, bufs = cases.model_local_state(rank)
        with torch.no_grad():
            for b, v in zip(model.buffers(), bufs):
                b.copy_(v)
        if variant == "eager":
            loss = sum((p * g.cuda()).sum() for p, g in zip(model.parameters(), grads))
            with distrib.eager_sync_model(model):
                loss.backward()
        else:
            for p, g in zip(model.parameters(), grads):
                p.grad = g.cuda()
            distrib.sync_model(model, average_buffers=(variant == "avg"))
        torch.cuda.synchronize()
        return [p.grad.cpu() for p in model.parameters()], [b.cpu() for b in model.buffers()]

    got = run(world, body)
    local = [cases.model_local_state(r) for r in range(world)]
    for r in range(world):
        grads, bufs = got[r]
        for i, g in enumerate(grads):
            ref = G.golden_tensor(world, f"model/{variant}/grad/{i}", torch.float32)
            assert G.normalised_error(g, ref, [local[q][0][i] for q in range(world)]) <= FP32_TOL
            assert torch.equal(g, numeric.average_one([local[q][0][i] for q in range(world)]))
        for i, b in enumerate(bufs):
            ref = cases.from_np(G.get(world, f"model/{variant}/buf/{i}", r), b.dtype)
            if b.dtype == torch.long or variant == "bcast":
                assert torch.equal(b, ref)                               # skipped / bit copy
            else:
                assert G.normalised_error(b, ref, [local[q][1][i] for q in range(world)]) <= FP32_TOL


@pytest.mark.parametrize("world", cases.WORLDS)
def test_metrics_and_allreduce_golden(world):
    from flashy_b200 import distrib

    def body(rank, w):
        metrics, count = cases.metrics_inputs(rank)
        out = distrib.average_metrics(metrics, count)
        f, i = [t.cuda() for t in cases.allreduce_inputs(rank)]
        assert distrib.all_reduce(f) is None
        distrib.all_reduce(i)
        mx = torch.tensor([float(rank), -float(rank)], device="cuda")
        mn = mx.clone()
        distrib.all_reduce(mx, torch.distributed.ReduceOp.MAX)
        distrib.all_reduce(mn, torch.distributed.ReduceOp.MIN)
        torch.cuda.synchronize()
        return out, f.cpu(), i.cpu(), mx.cpu(), mn.cpu()

    got = run(world, body)
    ref_m = G.get(world, "metrics/out")
    cols = [cases.allreduce_inputs(r) for r in range(world)]
    for r in range(world):
        out, f, i, mx, mn = got[r]
        assert list(out.keys()) == list(G.get(world, "metrics/keys"))
        for v, w in zip(out.values(), ref_m):
            assert abs(v - w) <= 1e-6 * max(1.0, abs(w))
        ref = G.golden_tensor(world, "allreduce/out/0", torch.float32)
        assert G.normalised_error(f, ref, [c[0] for c in cols]) <= FP32_TOL * world
        assert torch.equal(f, numeric.all_reduce_sum([c[0] for c in cols]))
        assert np.array_equal(G.get(world, "allreduce/out/1"), i.numpy())           # int64: exact
        assert mx.tolist() == [world - 1.0, 0.0] and mn.tolist() == [0.0, -(world - 1.0)]


# --------------------------------------------------------------------------- full-size buckets
def _resnet18_numels():
    import torchvision
    return [p.numel() for p in torchvision.models.resnet18(num_classes=10).parameters()]


@pytest.mark.parametrize("dtype", (torch.bfloat16, torch.float32))
def test_resnet18_bucket_vs_oracle(dtype):
    """BASELINE configs[1] payload: 62 gradient tensors, 11 181 642 elements, W = 8."""
    from flashy_b200 import distrib
    world = 8
    numels = _resnet18_numels()
    assert len(numels) == 62 and sum(numels) == 11181642
    gens = [torch.Generator().manual_seed(1000 + r) for r in range(world)]
    per_rank = [[(torch.randn(n, generator=gens[r]) * 1e-2).to(dtype) for n in numels] for r in range(world)]
    want = numeric.average_tensors(per_rank)[0]

    def body(rank, w):
        ts = [t.cuda() for t in per_rank[rank]]
        for _ in range(3):                      # repeated calls: alternating staging halves, rolling epochs
            cur = [t.clone() for t in ts]
            distrib.average_tensors(cur)
        torch.cuda.synchronize()
        return [t.cpu() for t in cur]

    got = run(world, body)
    for r in range(world):
        for g, w_ in zip(got[r], want):
            assert torch.equal(g, w_)
    big = [p.info for p in vworld(world).engine.plans.values() if p.info.wire_bytes > (4 << 20)]
    assert big and all(p.algo == 2 for p in big)                # two-shot path was the one exercised


def test_size_independent_properties_at_full_size():
    """Idempotence (the mean of identical replicas is the identity), broadcast-then-average is
    the identity, and scaling by 2^k commutes, on a 64 MiB bucket (cut into several launches).
    The values carry 8 significant bits so that every partial sum k*x (k <= 8) and
    (2^8 - 1)*x is exact in fp32 and the identities hold bit for bit."""
    from flashy_b200 import distrib
    world = 8
    n = 16 * 1024 * 1024 + 3
    g = torch.Generator().manual_seed(7)
    base = torch.randn(n, generator=g).bfloat16().float()

    def body(rank, w):
        x = base.cuda()
        same = x.clone()
        distrib.average_tensors([same])                          # all ranks hold the same values
        assert torch.equal(same, x)
        mine = x * (rank + 1)
        distrib.broadcast_tensors([mine], src=3)
        assert torch.equal(mine, x * 4)
        a = x * float(2 ** rank)
        distrib.average_tensors([a])
        b = x * float(2 ** rank) * 4.0
        distrib.average_tensors([b])
        assert torch.equal(b, a * 4.0)                           # scaling by 2^k commutes exactly
        s = torch.full((n,), float(rank), device="cuda")
        distrib.all_reduce(s)
        assert torch.equal(s, torch.full_like(s, sum(range(w))))
        torch.cuda.synchronize()
        return True

    assert all(run(world, body))


# --------------------------------------------------------------------------- edge cases
@pytest.mark.parametrize("world", (2, 3, 5, 8))
def test_ragged_unaligned_empty_and_odd_worlds(world):
    """Misaligned views, odd lengths, empty tensors, channels_last, world sizes without a
    compile-time specialisation (3, 5).  The lists are small enough for the one-shot kernel, which
    is asserted; the sharded kernels at these layouts and worlds are covered by
    tests/test_gpu_kernel_matrix.py."""
    from flashy_b200 import distrib
    shapes = [(0,), (1,), (3,), (17,), (1023,), (2, 3, 5, 7), (40000,)]

    def make(rank):
        g = torch.Generator().manual_seed(1000 + rank)
        out = []
        for s in shapes:
            n = int(np.prod(s))
            store = torch.randn(n + 3, generator=g)
            out.append(store[1:1 + n].view(*s))               # storage offset 1: not 16-byte aligned
        cl = torch.randn(2, 8, 5, 5, generator=g).contiguous(memory_format=torch.channels_last)
        out.append(cl)
        return out

    per_rank = [make(r) for r in range(world)]
    want = numeric.average_tensors([[t.contiguous() for t in row] for row in per_rank])[0]

    def body(rank, w):
        dev = []
        for t in per_rank[rank]:
            if t.dim() == 4 and t.shape == (2, 8, 5, 5):
                dev.append(t.cuda().contiguous(memory_format=torch.channels_last))
            else:
                store = torch.empty(t.numel() + 3, device="cuda")
                v = store[1:1 + t.numel()].view(t.shape)
                v.copy_(t)
                dev.append(v)
        for dtype in (torch.float32, torch.bfloat16):
            cur = [d.to(dtype) if dtype != torch.float32 else d for d in dev]
            if dtype == torch.bfloat16:                        # rebuild misaligned bf16 views
                cur2 = []
                for d in cur:
                    store = torch.empty(d.numel() + 3, device="cuda", dtype=dtype)
                    v = store[1:1 + d.numel()].view(d.shape)
                    v.copy_(d)
                    cur2.append(v)
                cur = cur2[:-1] + [cur[-1]]
            distrib.average_tensors(cur)
        with pytest.raises(ValueError):
            distrib.average_tensors([torch.ones(4, 4, device="cuda").t()])
        torch.cuda.synchronize()
        return [d.cpu() for d in dev]

    got = run(world, body)
    for r in range(world):
        for g_, w_ in zip(got[r], want):
            assert torch.equal(g_.contiguous(), w_.contiguous())
    numels = tuple(int(np.prod(s)) for s in shapes if np.prod(s)) + (400,)
    plans = [p.info for p in vworld(world).engine.plans.values() if p.key[1] == numels]
    assert len(plans) == 2 and all(info.kernel == 1 for info in plans)        # fp32 and bf16: k_one_shot


def test_mixed_dtypes_and_bucket_splitting(monkeypatch):
    """A list mixing fp32 / bf16 / int64, with a bucket cap small enough to cut single tensors."""
    from flashy_b200 import distrib
    world = 4
    vw = vworld(world)
    old_cap = vw.engine.bucket_cap
    vw.engine.bucket_cap = 1 << 20                                # 1 MiB buckets
    try:
        g = [torch.Generator().manual_seed(50 + r) for r in range(world)]
        per_rank = [[torch.randn(700001, generator=g[r]), torch.arange(4) + r,
                     torch.randn(300, generator=g[r]).bfloat16(), torch.randn(100000, generator=g[r]),
                     torch.randn(1 << 20, generator=g[r]).bfloat16()] for r in range(world)]
        want = numeric.average_tensors(per_rank)

        def body(rank, w):
            ts = [t.cuda() for t in per_rank[rank]]
            distrib.average_tensors(ts)
            big = torch.arange(3 << 20, device="cuda", dtype=torch.int64) * (rank + 1)   # 24 MiB int64
            distrib.all_reduce(big)
            torch.cuda.synchronize()
            assert torch.equal(big, torch.arange(3 << 20, device="cuda", dtype=torch.int64) * sum(range(1, w + 1)))
            return [t.cpu() for t in ts]
        got = run(world, body)
        for r in range(world):
            for a, b in zip(got[r], want[r]):
                assert torch.equal(a, b)
    finally:
        vw.engine.bucket_cap = old_cap


def test_arena_eviction_and_many_plans():
    """More distinct bucket shapes than the arena can hold at once: the plan cache is dropped
    and the arena recycled (with the fencing barrier) without corrupting later results."""
    from flashy_b200 import VirtualWorld, distrib
    world = 4
    vw = VirtualWorld(world, device=0, arena_mb=8)
    try:
        def body(rank, w):
            for step, n in enumerate([200000, 300000, 250000, 400000, 100, 350000, 200000, 450000]):
                x = torch.full((n,), float(rank + step), device="cuda")
                distrib.average_tensors([x])
                expect = sum(r + step for r in range(w)) / w
                assert torch.equal(x, torch.full_like(x, expect)), (step, n)
            torch.cuda.synchronize()
            return True
        assert all(vw.run(body))
    finally:
        vw.close()


def test_wire_bf16_option():
    """Opt-in fp32 -> bf16 wire cast: result == fp32(bf16(sum of bf16-rounded inputs / W))."""
    from flashy_b200 import distrib
    world = 4
    vw = vworld(world)
    vw.engine.wire_bf16 = True
    try:
        g = [torch.Generator().manual_seed(70 + r) for r in range(world)]
        per_rank = [torch.randn(500000, generator=g[r]) * 1e-2 for r in range(world)]
        want = numeric.average_one([t.bfloat16() for t in per_rank]).float()

        def body(rank, w):
            x = per_rank[rank].cuda()
            distrib.average_tensors([x])
            torch.cuda.synchronize()
            return x.cpu()
        for out in run(world, body):
            assert torch.equal(out, want)
    finally:
        vw.engine.wire_bf16 = False


def test_eager_with_unused_parameters_and_two_models():
    """GAN-shaped use (BASELINE configs[3]): two models on one communicator, eager sync of one
    and plain sync of the other in the same step; a parameter that gets no gradient."""
    from torch import nn
    from flashy_b200 import distrib
    world = 4

    def body(rank, w):
        torch.manual_seed(1234)
        gen = nn.Sequential(nn.Linear(16, 32), nn.ReLU(), nn.Linear(32, 16)).cuda()
        adv = nn.Sequential(nn.Linear(16, 64), nn.ReLU(), nn.Linear(64, 1)).cuda()
        unused = nn.Linear(3, 3).cuda()
        distrib.broadcast_model(gen)
        distrib.broadcast_model(adv)
        x = torch.randn(8, 16, generator=torch.Generator().manual_seed(10 + rank)).cuda()
        out = {}
        for step in range(3):
            for p in list(adv.parameters()) + list(gen.parameters()):
                p.grad = None
            with distrib.eager_sync_gradients(list(adv.parameters()) + list(unused.parameters())):
                adv(gen(x).detach()).mean().backward()
            gen(x).pow(2).mean().backward()
            distrib.sync_model(gen)
            out[step] = [p.grad.clone() for p in list(adv.parameters()) + list(gen.parameters())]
        assert all(p.grad is None for p in unused.parameters())
        # local (unsynchronised) gradients for the oracle
        for p in list(adv.parameters()) + list(gen.parameters()):
            p.grad = None
        adv(gen(x).detach()).mean().backward()
        gen(x).pow(2).mean().backward()
        local = [p.grad.clone() for p in list(adv.parameters()) + list(gen.parameters())]
        torch.cuda.synchronize()
        return [t.cpu() for t in out[2]], [t.cpu() for t in local]

    got = run(world, body)
    n = len(got[0][0])
    for i in range(n):
        want = numeric.average_one([got[r][1][i] for r in range(world)])
        for r in range(world):
            assert torch.equal(got[r][0][i], want), i


def test_count_mismatch_raises_on_every_rank_cuda():
    from flashy_b200 import distrib
    world = 8

    def body(rank, w):
        x = torch.ones(5, device="cuda")
        raised = 0
        for fn in (distrib.average_tensors, distrib.broadcast_tensors):
            try:
                fn([x, x.clone()] if rank == 5 else [x])
            except RuntimeError:
                raised += 1
        distrib.average_tensors([x])                # the communicator is still healthy afterwards
        assert torch.equal(x, torch.ones(5, device="cuda"))
        return raised
    assert run(world, body) == [2] * world


@pytest.mark.parametrize("dtype", (torch.bfloat16, torch.float32))
def test_pipelined_kernel_forced_in_loopback(monkeypatch, dtype):
    """The warp-role pipelined kernel k_pipe (default on real multi-GPU buckets) forced on for
    virtual ranks, with small chunks so that every CTA runs several pipeline stages.  The fused
    kernel is switched off: the planner prefers it whenever it is eligible."""
    from flashy_b200 import VirtualWorld, distrib
    import torchvision
    monkeypatch.setenv("FLASHY_B200_FUSE", "0")
    monkeypatch.setenv("FLASHY_B200_PIPE", "2")
    monkeypatch.setenv("FLASHY_B200_CHUNK_BYTES", "2048")
    world = 8
    numels = [p.numel() for p in torchvision.models.resnet18(num_classes=10).parameters()] + [64] * 40
    gens = [torch.Generator().manual_seed(300 + r) for r in range(world)]
    per_rank = [[(torch.randn(n, generator=gens[r]) * 1e-2).to(dtype) for n in numels] for r in range(world)]
    want = numeric.average_tensors(per_rank)[0]
    vw = VirtualWorld(world, device=0, arena_mb=256)
    try:
        def body(rank, w):
            ts = [t.cuda() for t in per_rank[rank]]
            for _ in range(3):
                cur = [t.clone() for t in ts]
                distrib.average_tensors(cur)
            big = torch.full((5 << 20,), float(rank + 1), device="cuda", dtype=dtype)
            distrib.all_reduce(big)
            torch.cuda.synchronize()
            assert torch.equal(big, torch.full_like(big, float(sum(range(1, w + 1)))))
            return [t.cpu() for t in cur]
        got = vw.run(body)
        for r in range(world):
            for g, w_ in zip(got[r], want):
                assert torch.equal(g, w_)
        sharded = [p.info for p in vw.engine.plans.values() if p.info.algo == 2]
        assert sharded and all(info.kernel == 4 and info.chunks > 1 for info in sharded)   # k_pipe<NVLS=false>
    finally:
        vw.close()


def test_cuda_graph_capture_and_replay():
    """A captured all-reduce launch replays correctly: epochs and staging parity live in device
    memory, so every replay is a fresh collective (C ABI driven from one thread, 4 virtual ranks)."""
    from flashy_b200 import _native as N
    from flashy_b200.engine import Engine
    world, n = 4, 300000
    eng = Engine(n_local=world, device=0, arena_mb=64)
    try:
        plan = eng.get_plan("ar", (n, 77), N.FX_F32, N.FX_F32)
        xs = [[torch.zeros(n, device="cuda"), torch.zeros(77, device="cuda")] for _ in range(world)]
        rows = [[t.data_ptr() for t in row] for row in xs]
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            for _ in range(2):                                   # warm the pointer tables
                eng.allreduce(plan, N.FX_AVG, rows, rows, side)
        side.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            eng.allreduce(plan, N.FX_AVG, rows, rows, torch.cuda.current_stream())
        for it in range(5):
            for r, row in enumerate(xs):
                row[0].fill_(float(r + it))
                row[1].fill_(float(2 * r - it))
            torch.cuda.synchronize()
            graph.replay()
            torch.cuda.synchronize()
            for row in xs:
                assert torch.equal(row[0], torch.full_like(row[0], sum(r + it for r in range(world)) / world))
                assert torch.equal(row[1], torch.full_like(row[1], sum(2 * r - it for r in range(world)) / world))
    finally:
        eng.close()
