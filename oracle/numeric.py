"""Single-process arithmetic model of the reference's collectives (TEST INFRASTRUCTURE).

Every function takes the inputs of *all* W ranks (index 0 = rank 0) and returns what the
reference leaves in each rank's tensors.  Citations are into /root/reference/.

Arithmetic contract restated from ``flashy/distrib.py``:

* ``average_tensors`` (:96-111): tensors that are neither floating point nor complex are
  skipped (:102); for the others SUM over ranks (:105-108) and afterwards a true division
  by the world size (:111).  Sum first, divide after.
* ``broadcast_tensors`` (:114-127): bit copy of rank ``src``'s float/complex tensors.
* ``average_metrics`` (:50-62): fp32 vector ``[v_1..v_k, 1] * count`` per rank, SUM, then
  ``v_i / last``.
* ``_check_number_of_params`` (:78-89): ``sum(len) != len * W`` on a rank => that rank raises.
* ``loader`` (:227-243): strided ``Subset`` shard for ``shuffle=False``, ``DistributedSampler``
  with its defaults for ``shuffle=True``.

Accumulation precision.  The reference accumulates in whatever ``torch.distributed`` does for
the dtype (gloo: ring in the native dtype; NCCL: tree/ring/NVLS), so the bits of an fp32 sum
depend on the backend.  The parity bar (SURVEY.md 8c, BASELINE.md 5) is therefore defined on
this model: fp32/fp64 summed in rank order in the native dtype; bf16/fp16 summed in fp32 and
rounded once -- ``bf16(fp32 path on the same bf16-valued inputs)``.
"""
from __future__ import annotations

import typing as tp

import torch

_WIDE = {
    torch.float32: torch.float32,
    torch.float64: torch.float64,
    torch.bfloat16: torch.float32,
    torch.float16: torch.float32,
    torch.complex64: torch.complex64,
    torch.complex128: torch.complex128,
}


def is_complex_or_float(t: torch.Tensor) -> bool:
    # flashy/distrib.py:92-93
    return torch.is_floating_point(t) or torch.is_complex(t)


def count_check(lengths: tp.Sequence[int]) -> tp.List[bool]:
    """flashy/distrib.py:78-89 -- per rank: does the rank raise?"""
    world = len(lengths)
    total = sum(int(n) for n in lengths)
    out = []
    for n in lengths:
        if world == 1 or n == 0:        # :81-82
            out.append(False)
        else:
            out.append(total != n * world)   # :86
    return out


def reduce_sum(columns: tp.Sequence[torch.Tensor]) -> torch.Tensor:
    """SUM over ranks of one tensor, rank order, in the wide dtype (not yet rounded)."""
    wide = _WIDE[columns[0].dtype]
    acc = columns[0].detach().to(wide).clone()
    for other in columns[1:]:
        acc += other.detach().to(wide)
    return acc


def average_one(columns: tp.Sequence[torch.Tensor]) -> torch.Tensor:
    """Mean over ranks of one tensor: (sum_r x_r) / W rounded once to the input dtype."""
    world = len(columns)
    acc = reduce_sum(columns)
    acc /= world                         # flashy/distrib.py:111, true division
    return acc.to(columns[0].dtype)


def average_tensors(per_rank: tp.Sequence[tp.Sequence[torch.Tensor]]) -> tp.List[tp.List[torch.Tensor]]:
    """flashy/distrib.py:96-111.  Returns the post-call tensors of every rank."""
    world = len(per_rank)
    if world == 1:                       # :100-101
        return [[t.clone() for t in per_rank[0]]]
    n = len(per_rank[0])
    out: tp.List[tp.List[torch.Tensor]] = [[] for _ in range(world)]
    for i in range(n):
        cols = [per_rank[r][i] for r in range(world)]
        if is_complex_or_float(cols[0]):
            mean = average_one(cols)
            for r in range(world):
                out[r].append(mean.clone())
        else:                            # :102 -- left untouched
            for r in range(world):
                out[r].append(cols[r].clone())
    return out


def all_reduce_sum(columns: tp.Sequence[torch.Tensor]) -> torch.Tensor:
    """flashy/distrib.py:45-47 with the default op (SUM); integer dtypes are exact."""
    if is_complex_or_float(columns[0]):
        return reduce_sum(columns).to(columns[0].dtype)
    acc = columns[0].clone()
    for other in columns[1:]:
        acc += other
    return acc


def broadcast_tensors(per_rank: tp.Sequence[tp.Sequence[torch.Tensor]], src: int = 0):
    """flashy/distrib.py:114-127."""
    world = len(per_rank)
    out = []
    for r in range(world):
        row = []
        for i, t in enumerate(per_rank[r]):
            if world > 1 and is_complex_or_float(t):
                row.append(per_rank[src][i].clone())
            else:
                row.append(t.clone())
        out.append(row)
    return out


def average_metrics(per_rank: tp.Sequence[tp.Dict[str, float]], counts: tp.Sequence[float]):
    """flashy/distrib.py:50-62 -- returns the dict every rank gets back."""
    world = len(per_rank)
    if world == 1:                       # :54-55 -- input returned unchanged
        return dict(per_rank[0])
    keys = list(per_rank[0].keys())
    acc = torch.zeros(len(keys) + 1, dtype=torch.float32)
    for metrics, count in zip(per_rank, counts):
        row = torch.tensor([metrics[k] for k in keys] + [1], dtype=torch.float32)
        row *= count                     # :59
        acc += row                       # :60
    averaged = (acc[:-1] / acc[-1]).tolist()   # :61
    return dict(zip(keys, averaged))


def loader_indices(n: int, rank: int, world: int, shuffle: bool) -> tp.List[int]:
    """Index list rank ``rank`` iterates for a dataset of length ``n`` (flashy/distrib.py:227-243)."""
    if world == 1:
        if shuffle:
            raise ValueError("single-process shuffle order is torch's global RNG; not modelled")
        return list(range(n))
    if not shuffle:
        return list(range(rank, n, world))       # :241
    # DistributedSampler defaults (:236): shuffle=True, seed=0, epoch=0, drop_last=False.
    g = torch.Generator()
    g.manual_seed(0)
    order = torch.randperm(n, generator=g).tolist()
    per = -(-n // world)
    total = per * world
    pad = total - len(order)
    if pad:
        reps = -(-pad // len(order))
        order += (order * reps)[:pad]
    return order[rank:total:world]


# --------------------------------------------------------------------------- kernel reduction contract
# The collective kernels (flashy_b200/csrc) reduce W columns elementwise: accumulate in rank order in
# Acc<T> (fp32 for bf16 / fp16, the dtype itself otherwise), divide once for AVG, round once to the wire
# dtype.  reduce_op restates that arithmetic so that kernel outputs can be compared bit for bit; the
# float64 reference and error bound below check the restatement itself against the exact operation.
SUM, AVG, MAX, MIN, PROD = range(5)          # fx_op values (include/flashy_b200.h)

_ACC = {
    torch.float32: torch.float32, torch.float64: torch.float64,
    torch.bfloat16: torch.float32, torch.float16: torch.float32,
    torch.int32: torch.int32, torch.int64: torch.int64,
}

# unit roundoff u = 2^-p (p = significand bits incl. the implicit one) and the smallest subnormal
UNIT_ROUNDOFF = {torch.float64: 2.0 ** -53, torch.float32: 2.0 ** -24, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
TINY = {torch.float64: 2.0 ** -1074, torch.float32: 2.0 ** -149, torch.bfloat16: 2.0 ** -133, torch.float16: 2.0 ** -24}


def _combine(acc: torch.Tensor, x: torch.Tensor, op: int) -> torch.Tensor:
    # same selection as combine<OP> in fx_device.cuh: ties (+0 / -0) keep the later rank's value
    if op in (SUM, AVG):
        return acc + x
    if op == MAX:
        return torch.where(acc > x, acc, x)
    if op == MIN:
        return torch.where(acc < x, acc, x)
    if op == PROD:
        return acc * x
    raise ValueError(f"unknown op {op}")


def reduce_op(columns: tp.Sequence[torch.Tensor], op: int, acc_dtype: tp.Optional[torch.dtype] = None) -> torch.Tensor:
    """Elementwise reduction of ``columns`` (rank order) as the kernels compute it: accumulate in
    ``Acc<T>`` in rank order, for AVG one true division by W, one rounding to the input dtype.
    ``acc_dtype`` overrides the accumulator (tests use it to model a wrong accumulator width)."""
    dtype = columns[0].dtype
    if op == AVG and not dtype.is_floating_point:
        raise ValueError("AVG is defined for floating-point tensors only")
    acc_t = acc_dtype or _ACC[dtype]
    acc = columns[0].to(acc_t)
    for x in columns[1:]:
        acc = _combine(acc, x.to(acc_t), op)
    if op == AVG:
        # a tensor divisor: torch turns division by a Python scalar into a reciprocal multiply on CUDA
        acc = torch.div(acc, torch.full_like(acc, len(columns)))
    return acc.to(dtype)


def reduce_op_wire_bf16(columns: tp.Sequence[torch.Tensor], op: int) -> torch.Tensor:
    """fp32 tensors sent over a bf16 wire (FLASHY_B200_WIRE=bf16): every input is rounded to bf16,
    reduced as a bf16 bucket (fp32 accumulation, one rounding to bf16) and widened back to fp32."""
    assert columns[0].dtype == torch.float32
    return reduce_op([c.to(torch.bfloat16) for c in columns], op).to(torch.float32)


def reference64(columns: tp.Sequence[torch.Tensor], op: int) -> torch.Tensor:
    """float64 reference of the operation, independent of the kernels' accumulation order and
    width.  SUM / AVG use a compensated (Neumaier) sum, so for inputs of at most 53 significant bits
    the result is the exact sum rounded to float64 up to a few units of 2^-106 relative."""
    xs = [c.to(torch.float64) for c in columns]
    if op in (SUM, AVG):
        s, comp = xs[0].clone(), torch.zeros_like(xs[0])
        for x in xs[1:]:
            t = s + x
            comp += torch.where(s.abs() >= x.abs(), (s - t) + x, (x - t) + s)
            s = t
        s = s + comp
        return s / len(xs) if op == AVG else s
    acc = xs[0]
    for x in xs[1:]:
        acc = torch.maximum(acc, x) if op == MAX else torch.minimum(acc, x) if op == MIN else acc * x
    return acc


def sum_error_bound(columns: tp.Sequence[torch.Tensor], op: int, out_dtype: tp.Optional[torch.dtype] = None,
                    acc_dtype: tp.Optional[torch.dtype] = None) -> torch.Tensor:
    """Largest |out - reference64| a correct SUM / AVG may show, elementwise:

        (W-1) u_acc sum_r |x_r| / d  +  u_acc |ref|  +  u_out |ref|  +  tiny_out  +  u_ref |ref|

    d = W for AVG and 1 for SUM; u is the unit roundoff (2^-24 fp32, 2^-53 fp64, 2^-8 bf16,
    2^-11 fp16) and tiny_out the smallest subnormal of the output dtype.

    Derivation.  Write S = sum_r x_r and s_k for the accumulator after rank k.  Each of the W-1
    additions is one rounding, s_k = (s_{k-1} + x_k)(1 + e_k) with |e_k| <= u_acc, so
    |s_W - S| <= u_acc sum_{k>=2} |s_k| <= (W-1) u_acc sum_r |x_r| to first order (the standard
    recursive-summation bound; every |s_k| is at most sum_r |x_r|).  Division by d is exact
    for d = 1 and one more rounding for AVG: u_acc |S/d|.  Rounding to the output dtype adds
    u_out |S/d|, or at most half a subnormal spacing when the result is below the normal range
    (tiny_out).  Additions of subnormals are exact, so underflow adds nothing before that.
    The float64 reference carries one rounding of its own division (u_ref = 2^-53; its
    compensated sum is exact to second order).  Second-order terms (products of two u) are left
    out: they are below the first-order slack of sum_{k>=2}|s_k| <= (W-1) sum_r |x_r| for every
    input these tests use.  The bound is meaningful for finite results only."""
    dtype = columns[0].dtype
    out_dtype = out_dtype or dtype
    acc_dtype = acc_dtype or _ACC[dtype]
    world = len(columns)
    d = world if op == AVG else 1
    u_acc, u_out = UNIT_ROUNDOFF[acc_dtype], UNIT_ROUNDOFF[out_dtype]
    mag = torch.stack([c.to(torch.float64).abs() for c in columns]).sum(0)
    ref = reference64(columns, op).abs()
    return ((world - 1) * u_acc * mag / d + (u_acc if op == AVG else 0.0) * ref + u_out * ref
            + TINY[out_dtype] + (2.0 ** -53) * ref)
