"""Every all-reduce / broadcast kernel that runs with virtual ranks, driven directly through the C ABI
and compared bit for bit with ``oracle.numeric.reduce_op`` at the layouts where kernels go wrong.

One ``Engine`` per world hosts all W ranks (``n_local = W``), so every call is one cooperative launch
from this thread.  Each case picks its kernel with the ``algo`` argument and the ``FLASHY_B200_*`` knobs
``fx_plan_create`` reads, and asserts the kernel id it reached (``plan.info.kernel``), so a planner
change cannot move a case to another kernel unseen.

Layouts come from the live plan's geometry (grid, shard, slice, chunk):

* ``boundaries``: tensor ends at -1 / 0 / +1 element of 16-byte vector, chunk, slice and shard
  boundaries, with empty and one-element tensors between them;
* ``many_small``: 1100 tensors of 1-40 elements, more than the kernels keep in shared memory
  (FX_SMEM_TENSORS), so the metadata is read from global memory;
* ``flat``: one tensor of 3 MiB plus three elements.

Every tensor is a window at element offset 0, 1 or VEC-1 of a 16-byte aligned region with at least
64 guard bytes on each side, filled with a sentinel pattern; odd calls are out of place (outputs
pre-filled with another sentinel).  Every plan runs four calls with fresh seeded data (the call index
is part of the seed), with another plan launched between the second and the third, so that each of
the plan's two staging halves is reused with different contents after the pad epochs moved on.  Each call checks: bit-exact against ``reduce_op`` (NaN positions by mask), the
float64 error bound of ``sum_error_bound`` (SUM / AVG on floats), all ranks bit-identical, guards and
inputs untouched, and a clean ``engine.poll()``.

NaN is left out of MAX / MIN inputs: ``combine<FX_MAX>`` keeps or drops a NaN depending on its rank
position, and the reduction contract says nothing about NaN for these ops.
"""
import os
import zlib

import numpy as np
import pytest
import torch

from oracle import numeric

pytestmark = pytest.mark.gpu

SUM, AVG, MAX, MIN, PROD = numeric.SUM, numeric.AVG, numeric.MAX, numeric.MIN, numeric.PROD
OP_NAMES = {SUM: "sum", AVG: "avg", MAX: "max", MIN: "min", PROD: "prod"}
WORLDS = (2, 3, 4, 5, 8)
EXTRA_WORLDS = (6, 7, 16)           # no compile-time specialisation; 16 fills both poll half-warps of k_fuse
GUARD = 64
DEV = "cuda"
FLAT_BYTES = 3 << 20
FUSE_SMALL_CHUNK = 1408             # 11 lines: a chunk is one full and one partial 1 KiB reduce unit

# name -> (tensor dtype, fx dtype, fx wire dtype)
F32, BF16, F16, F64, I32, I64, U8 = range(7)
DTYPES = {
    "f32": (torch.float32, F32, F32), "bf16": (torch.bfloat16, BF16, BF16), "f16": (torch.float16, F16, F16),
    "f64": (torch.float64, F64, F64), "i32": (torch.int32, I32, I32), "i64": (torch.int64, I64, I64),
    "f32>bf16": (torch.float32, F32, BF16),
}
ESIZE = {F32: 4, BF16: 2, F16: 2, F64: 8, I32: 4, I64: 8, U8: 1}
WIRE_TORCH = {F32: torch.float32, BF16: torch.bfloat16, F16: torch.float16, F64: torch.float64,
              I32: torch.int32, I64: torch.int64, U8: torch.uint8}
BITS = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}
ALGO_ONE_SHOT, ALGO_TWO_SHOT = 1, 2
K_ONE_SHOT, K_TWO_SHOT, K_PIPE_P2P, K_FUSE_P2P = 1, 2, 4, 6

# (row, dtype name, world, op) of every case that ran; checked against the matrix by the last test
LEDGER = set()


def _ops(name):
    return (SUM, AVG, MAX, MIN, PROD) if DTYPES[name][0].is_floating_point else (SUM, MAX, MIN, PROD)


def _cells(dtypes, worlds, ops=None):
    return [(w, d, op) for w in worlds for d in dtypes for op in (ops or _ops(d))]


ALL_DTYPES = ("f32", "bf16", "f16", "f64", "i32", "i64", "f32>bf16")


# --------------------------------------------------------------------------- engines
_ENGINES = {}


def engine(world):
    from flashy_b200.engine import Engine
    if world not in _ENGINES:
        # a kernel that stops making progress fails its case with FX_ERR_TIMEOUT instead of stalling
        with pytest.MonkeyPatch.context() as mp:
            mp.setenv("FLASHY_B200_DEVICE_TIMEOUT", "30")
            _ENGINES[world] = Engine(n_local=world, device=0, arena_mb=16)
    return _ENGINES[world]


@pytest.fixture(scope="module", autouse=True)
def _engines():
    yield
    for eng in _ENGINES.values():
        eng.close()
    _ENGINES.clear()


def _plan(eng, numels, fx, wire, algo, tag):
    return eng.get_plan("kernel-matrix", tuple(int(n) for n in numels), fx, wire, algo, tag=tag)


def _drop(eng, plan):
    eng.plans.pop(plan.key, None)
    plan.destroy()


def _offsets(plan):
    from flashy_b200 import _native as N
    arr = (N.C.c_int64 * plan.n)()
    N.check(N.lib.fx_plan_offsets(plan.handle, arr))
    return np.array(arr[:], dtype=np.int64)


def _round_up(x, a):
    return (x + a - 1) // a * a


# --------------------------------------------------------------------------- layouts
def _boundaries(info, total, align, sharded, chunked):
    """Bucket positions of each boundary kind, from the live plan's geometry."""
    shard = int(info.shard_elems)
    slice_ = shard // info.grid_x
    shards = info.world if sharded else 1
    kinds = {"vector": [align * k for k in (3, 7, 12)]}
    kinds["slice"] = [s * shard + b * slice_ for s in (0, shards - 1) for b in range(1, min(info.grid_x, 3))]
    if sharded:
        kinds["shard"] = [s * shard for s in range(1, shards)]
    if chunked:
        chunk = int(info.chunk_bytes) // ESIZE[info.wire_dtype]
        kinds["chunk"] = [s * shard + b * slice_ + c * chunk for s in (0, shards - 1) for b in (0, 1) if b < info.grid_x
                          for c in range(1, min(info.chunks, 3))]
    return {k: sorted(t for t in v if 0 < t < total - 4 * align) for k, v in kinds.items()}


def _numels_at(targets, total, align):
    """Tensor sizes whose ends land at target-1 / target / target+1, with empty and one-element
    tensors in between, padded out to exactly `total` bucket elements."""
    numels, cur = [], 0
    for k, t in enumerate(sorted(set(targets))):
        end = t + (-1, 0, 1)[k % 3]
        if end - cur < 1:
            continue
        numels.append(end - cur)
        cur = _round_up(end, align)
        if k % 2 == 0:
            numels += [0, 1]
            cur += align
    if total - cur >= 1:
        numels.append(total - cur)
    return numels


def build_layout(eng, kind, fx, wire, algo, tag, chunked):
    """(plan, numels) of layout `kind`; asserts that the boundary layout really sits on its boundaries."""
    esize, wsize = ESIZE[fx], ESIZE[wire]
    align = 16 // min(esize, wsize)
    if kind == "flat":
        numels = [FLAT_BYTES // esize + 3]
    elif kind == "many_small":
        numels = np.random.default_rng(11).integers(1, 41, 1100).tolist()
    else:
        world = eng.world
        total = _round_up(max(256 << 10, (32 << 10) * world) // wsize, align)
        probe = _plan(eng, (total,), fx, wire, algo, (tag, "probe"))
        info = probe.info
        _drop(eng, probe)
        kinds = _boundaries(info, total, align, algo != ALGO_ONE_SHOT, chunked)
        numels = _numels_at([t for v in kinds.values() for t in v], total, align)
    plan = _plan(eng, numels, fx, wire, algo, (tag, kind))
    if kind == "boundaries":
        info = plan.info
        assert (info.grid_x, info.shard_elems) == (probe.info.grid_x, probe.info.shard_elems)
        ends = _offsets(plan) + np.array(numels)
        live = _boundaries(info, total, align, algo != ALGO_ONE_SHOT, chunked)
        for k, targets in live.items():
            if k == "chunk" and not targets:           # a single chunk per slice (default fused chunk at W = 2)
                continue
            assert targets, (k, "no boundary of this kind inside the bucket")
            near = int(np.abs(ends[:, None] - np.array(targets)[None, :]).min())
            assert near <= align, (k, "no tensor end within one vector of a boundary", near)
    return plan, numels


class Slabs:
    """All tensors of all ranks as windows of one (W, B) byte slab, with guards and a sentinel."""

    def __init__(self, numels, dtype, world, salt):
        esize = torch.empty((), dtype=dtype).element_size()
        vec = 16 // esize
        starts, pos = [], GUARD
        for i, n in enumerate(numels):
            pos = _round_up(pos, 16)
            start = pos + (0, 1, vec - 1)[i % 3] * esize
            starts.append(start)
            pos = start + n * esize + GUARD
        self.B = _round_up(pos, 16)
        self.world, self.dtype, self.esize = world, dtype, esize
        self.starts = np.array(starts, dtype=np.int64)
        numels = np.array(numels, dtype=np.int64)
        self.total = int(numels.sum())
        data_off = np.concatenate([[0], np.cumsum(numels)[:-1]])
        idx = np.arange(self.total) + np.repeat(self.starts // esize - data_off, numels)
        self.idx = torch.from_numpy(idx).to(DEV)
        covered = np.zeros(self.B, dtype=bool)
        covered[(idx[:, None] * esize + np.arange(esize)[None, :]).ravel()] = True
        self.guard = torch.from_numpy(~covered).to(DEV)
        pattern = torch.arange(self.B, device=DEV)[None, :] * 151 + torch.arange(world, device=DEV)[:, None] * 17
        self.sent_in = ((pattern + salt) % 256).to(torch.uint8)
        self.sent_out = ((pattern + salt + 0x40) % 256).to(torch.uint8)
        self.inp = torch.empty(world, self.B, dtype=torch.uint8, device=DEV)
        self.out = torch.empty_like(self.inp)

    def fill(self, data, out_of_place):
        self.inp.copy_(self.sent_in)
        self.inp.view(self.dtype)[:, self.idx] = data
        if out_of_place:
            self.out.copy_(self.sent_out)
        return self.inp, (self.out if out_of_place else self.inp)

    def rows(self, slab):
        base = slab.data_ptr()
        return [(base + r * self.B + self.starts).tolist() for r in range(self.world)]

    def values(self, slab):
        return slab.view(self.dtype)[:, self.idx]


# --------------------------------------------------------------------------- data
def _seed(*parts):
    return zlib.crc32(repr(parts).encode())


def make_data(name, op, world, total, seed):
    """(W, total) inputs of dtype `name` for `op`: magnitude classes, cancellation and special values."""
    dtype = DTYPES[name][0]
    g = torch.Generator(device=DEV).manual_seed(seed)
    if not dtype.is_floating_point:
        if op == PROD:
            return torch.randint(-3, 4, (world, total), generator=g, device=DEV, dtype=dtype)
        x = torch.randint(-(1 << 20), 1 << 20, (world, total), generator=g, device=DEV, dtype=torch.int64)
        if dtype == torch.int64:            # 64-bit magnitudes, alternating signs keep partial sums in range
            sign = 1 - 2 * (torch.arange(world, device=DEV) % 2)
            x = x + sign[:, None] * (1 << 60)
        return x.to(dtype)
    x = torch.randn(world, total, generator=g, device=DEV, dtype=torch.float64)
    third = total // 3
    if op == PROD:
        x = torch.exp2(x.clamp(-3, 3)) * torch.sign(torch.randn(world, total, generator=g, device=DEV, dtype=torch.float64))
    else:
        # per-rank magnitudes 2^+-10 apart: the summation order shows in the result bits
        scale = torch.exp2(10.0 * ((torch.arange(world, device=DEV) % 3) - 1).double())
        x[:, :third] *= scale[:, None]
        # cancellation: the last rank nearly cancels the others
        x[-1, third:2 * third] = -x[:-1, third:2 * third].sum(0) * (1 + 2.0 ** -6)
    wire = WIRE_TORCH[DTYPES[name][2]]
    pos = [(k * 7919 + 13) % total for k in range(8)] if total >= 64 else []
    if pos and op != PROD:
        inf = float("inf")
        if op not in (MAX, MIN):
            x[:, pos[0]] = 1.0
            x[1 % world, pos[0]] = float("nan")
        x[0, pos[1]] = inf
        x[world - 1, pos[2]] = -inf
        x[0, pos[3]], x[world - 1, pos[3]] = inf, -inf          # SUM: NaN
        x[:, pos[4]] = -0.0                                      # SUM: -0.0
        sub = {torch.float16: 2.0 ** -24, torch.bfloat16: 2.0 ** -130}.get(wire, 3 * 2.0 ** -145)
        x[:, pos[5]] = sub * (torch.arange(world, device=DEV) + 1).double()   # subnormals
        if wire == torch.float16:
            x[:, pos[6]] = 6.0e4 + 100.0 * torch.arange(world, device=DEV).double()   # SUM overflows, AVG does not
        if wire in (torch.bfloat16, torch.float16):
            x[:, pos[7]] = 2.0 ** -9 if wire == torch.bfloat16 else 2.0 ** -12    # a quarter ulp of 1.0
            x[0, pos[7]] = 1.0                                   # right only with fp32 accumulation
    return x.to(dtype)


def expected(name, op, data):
    cols = list(data)
    if DTYPES[name][2] != DTYPES[name][1]:
        return numeric.reduce_op_wire_bf16(cols, op)
    return numeric.reduce_op(cols, op)


def check_bound(name, op, data, got):
    """SUM / AVG of floats: inside the float64 error bound of the exact result (finite inputs)."""
    wire = WIRE_TORCH[DTYPES[name][2]]
    cols = [c.to(wire) for c in data]
    ref = numeric.reference64(cols, op)
    bound = numeric.sum_error_bound(cols, op)
    finite = torch.stack([c.isfinite() for c in cols]).all(0)
    over = ref.abs() > torch.finfo(wire).max
    g = got.double()
    assert bool(torch.isinf(g[finite & over]).all()), "a result beyond the dtype's range must be infinite"
    ok = finite & ~over
    err = (g[ok] - ref[ok]).abs()
    bad = err > bound[ok]
    assert not bool(bad.any()), f"outside the float64 bound: err {err[bad][:4].tolist()} bound {bound[ok][bad][:4].tolist()}"


def compare(want, got, numels, what):
    """got (W, total) against want (total,): every rank bit-identical, NaN by mask, the rest by bits."""
    bits = BITS[got.element_size()]
    gb, wb = got.view(bits), want.view(bits)
    assert torch.equal(gb, gb[:1].expand_as(gb)), f"{what}: ranks disagree"
    if got.dtype.is_floating_point:
        wn, gn = want.isnan(), got[0].isnan()
        assert torch.equal(wn, gn), f"{what}: NaN positions differ"
        bad = (gb[0] != wb) & ~wn
    else:
        bad = gb[0] != wb
    if bool(bad.any()):
        where = torch.nonzero(bad).flatten()[:5].cpu().numpy()
        tensor = np.searchsorted(np.cumsum(numels), where, side="right")
        raise AssertionError(f"{what}: {int(bad.sum())} elements differ, first at {where.tolist()} (tensors "
                             f"{tensor.tolist()}): got {got[0][where].tolist()} want {want[where].tolist()}")


# --------------------------------------------------------------------------- one case
def _set_knobs(monkeypatch, knobs):
    for k in ("FUSE", "PIPE", "CHUNK_BYTES", "FUSE_CHUNK", "SLICE_BYTES", "ONE_SHOT_MAX"):
        monkeypatch.delenv(f"FLASHY_B200_{k}", raising=False)
    for k, v in knobs.items():
        monkeypatch.setenv(f"FLASHY_B200_{k}", str(v))


def run_case(monkeypatch, row, world, name, op, algo, knobs, kernel, begin=False,
             layouts=("boundaries", "many_small", "flat"), check_info=None):
    eng = engine(world)
    _set_knobs(monkeypatch, knobs)
    dtype, fx, wire = DTYPES[name]
    tag = (row, tuple(sorted(knobs.items())))
    stream = torch.cuda.current_stream()
    chunked = kernel in (K_PIPE_P2P, K_FUSE_P2P)
    for layout in layouts:
        plan, numels = build_layout(eng, layout, fx, wire, algo, tag, chunked)
        other = _plan(eng, (777, 5), fx, wire, algo, (tag, "other"))
        try:
            reached = plan.info.kernel if (op in (SUM, AVG) or plan.info.algo == ALGO_ONE_SHOT) else K_TWO_SHOT
            assert reached == kernel, (layout, "planner chose kernel", plan.info.kernel)
            if check_info:
                check_info(layout, plan.info)
            slabs = Slabs(numels, dtype, world, salt=_seed(row, name, op) % 256)
            for call in range(4):
                if call == 2:                     # another plan in between: epochs roll, halves are reused
                    o = make_data(name, op, world, 782, _seed("other", call))
                    ob = torch.empty(world, 792, dtype=dtype, device=DEV)
                    ob[:, :777], ob[:, 784:789] = o[:, :777], o[:, 777:]
                    rows = [[ob[r].data_ptr(), ob[r, 784:].data_ptr()] for r in range(world)]
                    if begin:
                        eng.allreduce_begin(other, op, rows, stream)
                        eng.allreduce_finish(other, rows, stream)
                    else:
                        eng.allreduce(other, op, rows, rows, stream)
                data = make_data(name, op, world, slabs.total, _seed(row, name, op, world, layout, call))
                out_of_place = call % 2 == 1
                inp, out = slabs.fill(data, out_of_place)
                before = inp.clone() if out_of_place else None
                if begin:
                    eng.allreduce_begin(plan, op, slabs.rows(inp), stream)
                    eng.allreduce_finish(plan, slabs.rows(out), stream)
                else:
                    eng.allreduce(plan, op, slabs.rows(inp), slabs.rows(out), stream)
                torch.cuda.synchronize()
                eng.poll()
                what = f"{row} {name} W={world} {OP_NAMES[op]} {layout} call {call}"
                got = slabs.values(out)
                want = expected(name, op, data)
                compare(want, got, numels, what)
                if op in (SUM, AVG) and dtype.is_floating_point:
                    check_bound(name, op, data, got[0])
                sent = slabs.sent_out if out_of_place else slabs.sent_in
                assert torch.equal(out[:, slabs.guard], sent[:, slabs.guard]), f"{what}: guard bytes overwritten"
                if out_of_place:
                    assert torch.equal(inp, before), f"{what}: input changed"
        finally:
            _drop(eng, other)
            _drop(eng, plan)
    LEDGER.add((row, name, world, op))


# --------------------------------------------------------------------------- the matrix
ONE_SHOT_CELLS = _cells(ALL_DTYPES, WORLDS)
TWO_SHOT_CELLS = _cells(ALL_DTYPES, WORLDS) + _cells(("f32",), EXTRA_WORLDS, (SUM, AVG))
PIPE_CELLS = _cells(("f32", "bf16", "f16", "f32>bf16"), WORLDS, (SUM, AVG))
FUSE_CELLS = _cells(("f32", "bf16", "f16"), WORLDS, (SUM, AVG)) + _cells(("f32",), EXTRA_WORLDS, (SUM, AVG))
BEGIN_CELLS = [(w, d, op) for w in WORLDS for d in ("f32", "bf16", "f16", "f64", "i64", "f32>bf16")
               for op in ((SUM, AVG) if DTYPES[d][0].is_floating_point else (SUM,))]
MATRIX_ITEMS = (len(ONE_SHOT_CELLS) + len(TWO_SHOT_CELLS) + len(PIPE_CELLS) + len(FUSE_CELLS)
                + 2 * len(BEGIN_CELLS) + len(WORLDS))


@pytest.mark.parametrize("world,name,op", ONE_SHOT_CELLS)
def test_one_shot(monkeypatch, world, name, op):
    run_case(monkeypatch, "one_shot", world, name, op, ALGO_ONE_SHOT, {}, K_ONE_SHOT)


@pytest.mark.parametrize("world,name,op", TWO_SHOT_CELLS)
def test_two_shot(monkeypatch, world, name, op):
    run_case(monkeypatch, "two_shot", world, name, op, ALGO_TWO_SHOT, {"FUSE": 0, "PIPE": 0}, K_TWO_SHOT)


def _three_chunks(layout, info):
    if layout != "many_small":
        assert info.chunks >= 3, info.chunks


@pytest.mark.parametrize("world,name,op", PIPE_CELLS)
def test_pipe(monkeypatch, world, name, op):
    run_case(monkeypatch, "pipe", world, name, op, ALGO_TWO_SHOT, {"FUSE": 0, "PIPE": 2, "CHUNK_BYTES": 2048},
             K_PIPE_P2P, check_info=_three_chunks)


@pytest.mark.parametrize("world,name,op", FUSE_CELLS)
def test_fuse(monkeypatch, world, name, op):
    run_case(monkeypatch, "fuse", world, name, op, ALGO_TWO_SHOT, {"PIPE": 0}, K_FUSE_P2P)

    def partial_units(layout, info):
        if layout != "many_small":
            assert info.chunks >= 3 and info.chunk_bytes % 1024 != 0, (info.chunks, info.chunk_bytes)
    run_case(monkeypatch, "fuse", world, name, op, ALGO_TWO_SHOT, {"PIPE": 0, "FUSE_CHUNK": FUSE_SMALL_CHUNK},
             K_FUSE_P2P, layouts=("boundaries", "flat"), check_info=partial_units)


@pytest.mark.parametrize("pipe", (0, 2))
@pytest.mark.parametrize("world,name,op", BEGIN_CELLS)
def test_begin_unpack(monkeypatch, world, name, op, pipe):
    """fx_allreduce_begin (sharded kernel, result left in the arena) then fx_allreduce_finish (k_unpack)."""
    pipelined = pipe == 2 and DTYPES[name][2] in (F32, BF16, F16)
    kernel = K_PIPE_P2P if pipelined else K_TWO_SHOT
    knobs = {"FUSE": 0, "PIPE": pipe, "CHUNK_BYTES": 2048}
    run_case(monkeypatch, f"begin+{'pipe' if pipelined else 'two_shot'}", world, name, op, ALGO_TWO_SHOT, knobs, kernel,
             begin=True)


@pytest.mark.parametrize("world", WORLDS)
def test_broadcast(monkeypatch, world):
    """k_broadcast: a byte plan; every rank ends with the source's bytes, whatever dtype they hold."""
    eng = engine(world)
    _set_knobs(monkeypatch, {})
    stream = torch.cuda.current_stream()
    for layout in ("boundaries", "many_small", "flat"):
        plan, numels = build_layout(eng, layout, U8, U8, 0, ("broadcast",), False)
        try:
            assert plan.info.algo == ALGO_TWO_SHOT
            slabs = Slabs(numels, torch.uint8, world, salt=world)
            for call, src in enumerate(sorted({0, world // 2, world - 1})):
                g = torch.Generator(device=DEV).manual_seed(_seed("bc", world, layout, call))
                data = torch.randint(0, 256, (world, slabs.total), generator=g, device=DEV, dtype=torch.uint8)
                inp, _ = slabs.fill(data, False)
                eng.broadcast(plan, src, slabs.rows(inp), stream)
                torch.cuda.synchronize()
                eng.poll()
                what = f"broadcast W={world} src={src} {layout}"
                compare(data[src], slabs.values(inp), numels, what)
                assert torch.equal(inp[:, slabs.guard], slabs.sent_in[:, slabs.guard]), f"{what}: guard bytes overwritten"
                LEDGER.add(("broadcast", "u8", world, src))
        finally:
            _drop(eng, plan)


@pytest.mark.parametrize("world", (2, 3))
def test_refused_combinations_launch_nothing(world):
    from flashy_b200 import _native as N
    eng = engine(world)
    stream = torch.cuda.current_stream()
    x = torch.zeros(world, 64, dtype=torch.int64, device=DEV)
    rows = [[x[r].data_ptr()] for r in range(world)]
    cases = [(I32, ALGO_ONE_SHOT, AVG, False), (I64, ALGO_TWO_SHOT, AVG, False), (I64, ALGO_TWO_SHOT, AVG, True),
             (F32, ALGO_ONE_SHOT, SUM, True), (F32, ALGO_TWO_SHOT, 7, False)]
    for fx, algo, op, begin in cases:
        plan = _plan(eng, (64,), fx, fx, algo, ("refused", op, begin))
        try:
            before = eng.native_launches()
            with pytest.raises(N.NativeError):
                if begin:
                    eng.allreduce_begin(plan, op, rows, stream)
                else:
                    eng.allreduce(plan, op, rows, rows, stream)
            assert eng.native_launches() == before
        finally:
            _drop(eng, plan)
    torch.cuda.synchronize()
    eng.poll()


def test_ledger_covers_the_matrix(request):
    """Every cell of the kernel matrix ran; a shrinking parametrisation fails here."""
    matrix = {"test_one_shot", "test_two_shot", "test_pipe", "test_fuse", "test_begin_unpack", "test_broadcast"}
    selected = sum(1 for it in request.session.items if it.module is request.module and it.originalname in matrix)
    if selected < MATRIX_ITEMS:
        pytest.skip(f"only {selected} of the {MATRIX_ITEMS} kernel-matrix cases were selected")
    floats = ("f32", "bf16", "f16", "f64", "f32>bf16")
    every = ("f32", "bf16", "f16", "f64", "i32", "i64", "f32>bf16")
    want = set()
    for w in WORLDS:
        for d in every:
            ops = (SUM, AVG, MAX, MIN, PROD) if d in floats else (SUM, MAX, MIN, PROD)
            want |= {("one_shot", d, w, op) for op in ops} | {("two_shot", d, w, op) for op in ops}
        want |= {("pipe", d, w, op) for d in ("f32", "bf16", "f16", "f32>bf16") for op in (SUM, AVG)}
        want |= {("fuse", d, w, op) for d in ("f32", "bf16", "f16") for op in (SUM, AVG)}
        want |= {("begin+two_shot", d, w, op) for d in floats for op in (SUM, AVG)} | {("begin+two_shot", "i64", w, SUM)}
        want |= {("begin+pipe", d, w, op) for d in ("f32", "bf16", "f16", "f32>bf16") for op in (SUM, AVG)}
        want |= {("broadcast", "u8", w, src) for src in (0, w // 2, w - 1)}
    for w in EXTRA_WORLDS:
        want |= {(row, "f32", w, op) for row in ("fuse", "two_shot") for op in (SUM, AVG)}
    missing, extra = sorted(want - LEDGER), sorted(LEDGER - want)
    print(f"kernel matrix: {len(LEDGER)} cells ran")
    for cell in sorted(LEDGER):
        print("  ", cell)
    assert not missing, f"cells that did not run: {missing}"
    assert not extra, f"cells outside the matrix: {extra}"
