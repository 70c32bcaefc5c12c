"""Pin the oracle (oracle/numeric.py, oracle/refdistrib.py) to the unmodified reference.

Golden vectors: tests/golden/ref_w{2,4,8}.npz, produced by tests/golden/make_golden.py from
/root/reference/flashy/distrib.py over gloo.  Known answers: reference tests/test_distrib.py:29-46.
"""
import numpy as np
import pytest
import torch

from oracle import numeric
from tests import golden_io as G
from tests.golden import cases
from tests.harness import run_ranks

FP32_TOL = 1e-6      # BASELINE.json north_star: <= 1e-6 rel for fp32 (normalised by summand magnitude)


@pytest.mark.parametrize("world", cases.WORLDS)
def test_known_answers(world):
    cols = [torch.tensor([float(r) + 1]) for r in range(world)]
    mean = numeric.average_one(cols)
    assert mean.item() == sum(range(1, world + 1)) / world          # tests/test_distrib.py:29-31
    assert G.get(world, "known/avg")[0] == mean.item()
    out = numeric.broadcast_tensors([[c] for c in cols])
    assert all(row[0].item() == 1.0 for row in out)                 # tests/test_distrib.py:33-35
    assert G.get(world, "known/bcast")[0] == 1.0


@pytest.mark.parametrize("world", cases.WORLDS)
def test_count_check(world):
    lengths = [1] * world
    lengths[-1] = 2                                                 # tests/test_distrib.py:37-46
    assert all(numeric.count_check(lengths))
    assert not any(numeric.count_check([3] * world))
    for r in range(world):
        assert G.get(world, "mismatch/raised", r)[0] == 1
    assert numeric.count_check([5]) == [False]
    assert numeric.count_check([0] * world) == [False] * world


@pytest.mark.parametrize("world", cases.WORLDS)
@pytest.mark.parametrize("name", list(cases.AVG_DTYPES))
def test_average_tensors_vs_golden(world, name):
    dtype = cases.AVG_DTYPES[name]
    per_rank = [cases.avg_inputs(r, name) for r in range(world)]
    for r in range(world):
        for i, t in enumerate(per_rank[r]):
            G.check_input(world, f"avg/{name}/in/{i}", r, t)
    out = numeric.average_tensors(per_rank)
    for i in range(len(per_rank[0])):
        if i == cases.INT_SLOT:
            for r in range(world):     # int64 tensors are skipped by the reference (distrib.py:102)
                assert np.array_equal(G.get(world, f"avg/{name}/out/{i}", r), cases.to_np(per_rank[r][i]))
                assert torch.equal(out[r][i], per_rank[r][i])
            continue
        ref = G.golden_tensor(world, f"avg/{name}/out/{i}", dtype)
        cols = [per_rank[r][i] for r in range(world)]
        if name in ("fp32", "fp64", "c64"):
            assert G.normalised_error(out[0][i], ref, cols) <= FP32_TOL
        else:
            # gloo accumulates 16-bit floats in the 16-bit type: the reference's own result is
            # several 1e-3 from the exact mean (SURVEY.md 8c).  The model rounds once.
            exact = torch.stack([c.double() for c in cols]).mean(0)
            err_model = (out[0][i].double() - exact).abs().max()
            err_ref = (ref.double() - exact).abs().max()
            assert err_model <= err_ref + 1e-12
            scale = torch.stack([c.double().abs() for c in cols]).mean(0).clamp_min(1e-30)
            assert float(((out[0][i].double() - ref.double()).abs() / scale).max()) < 0.1


@pytest.mark.parametrize("world", cases.WORLDS)
def test_broadcast_vs_golden(world):
    per_rank = [cases.avg_inputs(r, "fp32") for r in range(world)]
    for src in (0, world - 1):
        out = numeric.broadcast_tensors(per_rank, src=src)
        for i in range(len(per_rank[0])):
            for r in (0, world - 1):
                assert np.array_equal(G.get(world, f"bcast/src{src}/out/{i}", r), cases.to_np(out[r][i]))


@pytest.mark.parametrize("world", cases.WORLDS)
def test_metrics_vs_golden(world):
    ins = [cases.metrics_inputs(r) for r in range(world)]
    got = numeric.average_metrics([m for m, _ in ins], [c for _, c in ins])
    assert list(got.keys()) == list(G.get(world, "metrics/keys"))
    ref = G.get(world, "metrics/out")
    for v, w in zip(got.values(), ref):
        assert abs(v - w) <= 1e-6 * max(1.0, abs(w))
    single = {"a": 1.0}
    assert numeric.average_metrics([single], [3.0]) == single


@pytest.mark.parametrize("world", cases.WORLDS)
def test_allreduce_and_loader_vs_golden(world):
    cols = [cases.allreduce_inputs(r) for r in range(world)]
    f = numeric.all_reduce_sum([c[0] for c in cols])
    ref = G.golden_tensor(world, "allreduce/out/0", torch.float32)
    assert G.normalised_error(f, ref, [c[0] for c in cols]) <= FP32_TOL * world
    i = numeric.all_reduce_sum([c[1] for c in cols])
    assert np.array_equal(G.get(world, "allreduce/out/1"), i.numpy())          # integers: exact
    for r in range(world):
        for shuffle in (False, True):
            want = G.get(world, f"loader/shuffle{int(shuffle)}", r).tolist()
            assert numeric.loader_indices(cases.LOADER_N, r, world, shuffle) == want   # bit-exact
        assert G.get(world, "rank", r).tolist() == [r, world, int(r == 0), 1]
        assert G.get(world, "rank_zero_only", r)[0] == (7 if r == 0 else -1)


# ---- oracle/refdistrib.py over gloo against the same golden file --------------------------

def _refdistrib_worker(rank, world):
    from oracle.refdistrib import RefDistrib as R
    for name, dtype in cases.AVG_DTYPES.items():
        ts = cases.avg_inputs(rank, name)
        R.average_tensors(ts)
        for i, t in enumerate(ts):
            assert np.array_equal(G.get(world, f"avg/{name}/out/{i}", rank), cases.to_np(t)), (name, i)
    for src in (0, world - 1):
        ts = cases.avg_inputs(rank, "fp32")
        R.broadcast_tensors(ts, src=src)
        for i, t in enumerate(ts):
            assert np.array_equal(G.get(world, f"bcast/src{src}/out/{i}", rank), cases.to_np(t))
    x = torch.tensor([1.0])
    try:
        R.broadcast_tensors([x, x.clone()] if rank == world - 1 else [x])
    except RuntimeError:
        pass
    else:
        raise AssertionError("count mismatch must raise on every rank")
    for variant in ("avg", "bcast", "eager"):
        model = cases.make_model()
        grads, bufs = cases.model_local_state(rank)
        with torch.no_grad():
            for b, v in zip(model.buffers(), bufs):
                b.copy_(v)
        if variant == "eager":
            loss = sum((p * g).sum() for p, g in zip(model.parameters(), grads))
            with R.eager_sync_model(model):
                loss.backward()
        else:
            for p, g in zip(model.parameters(), grads):
                p.grad = g.clone()
            R.sync_model(model, average_buffers=(variant == "avg"))
        for i, p in enumerate(model.parameters()):
            assert np.array_equal(G.get(world, f"model/{variant}/grad/{i}", rank), cases.to_np(p.grad))
        for i, b in enumerate(model.buffers()):
            assert np.array_equal(G.get(world, f"model/{variant}/buf/{i}", rank), cases.to_np(b))
    metrics, count = cases.metrics_inputs(rank)
    got = R.average_metrics(metrics, count)
    assert [got[k] for k in got] == G.get(world, "metrics/out").tolist()
    for i, t in enumerate(cases.allreduce_inputs(rank)):
        R.all_reduce(t)
        assert np.array_equal(G.get(world, f"allreduce/out/{i}", rank), cases.to_np(t))
    data = list(range(cases.LOADER_N))
    for shuffle in (False, True):
        seen = [int(v) for batch in R.loader(data, shuffle=shuffle, batch_size=4) for v in batch]
        assert seen == G.get(world, f"loader/shuffle{int(shuffle)}", rank).tolist()
    assert R.broadcast_object({"k": 1} if rank == 0 else None) == {"k": 1}
    R.barrier()


@pytest.mark.parametrize("world", (2, 8))
def test_refdistrib_matches_reference_bit_for_bit(world):
    """Same backend (gloo) + same call sequence => the restatement reproduces the golden bits."""
    run_ranks(world, "tests.test_oracle", "_refdistrib_worker")


def test_bench_reference_arm_line():
    """`bench.py --impl reference` (CPU, gloo, oracle/refdistrib.py) prints one well-formed JSON line."""
    import json
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    out = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--world", "2", "--batch", "4"], capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "samples/s" and line["value"] > 0
    assert line["metric"] == "cifar_resnet18_train_samples_per_sec" and line["higher_is_better"] is True
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["cpu_baseline"]["kind"] == "port"
    assert line["cpu_baseline"]["cores"] >= 1 and "gloo" in line["cpu_baseline"]["sample"]


# ---- the kernels' reduction contract (oracle/numeric.py reduce_op) against exact arithmetic ----------
from fractions import Fraction  # noqa: E402

# (significand bits incl. the implicit one, smallest normal exponent, largest exponent)
_FORMATS = {torch.float64: (53, -1022, 1023), torch.float32: (24, -126, 127),
            torch.bfloat16: (8, -126, 127), torch.float16: (11, -14, 15)}
_FLOATS = (torch.float32, torch.float64, torch.bfloat16, torch.float16)


def _round(q, dtype):
    """Exact value q (Fraction, or +-inf) rounded to nearest-even in `dtype`, returned as a Fraction or +-inf."""
    if not isinstance(q, Fraction):
        return q
    if q == 0:
        return Fraction(0)
    p, emin, emax = _FORMATS[dtype]
    a = abs(q)
    e = a.numerator.bit_length() - a.denominator.bit_length()          # 2^e <= a < 2^(e+2)
    if a >= Fraction(2) ** (e + 1):
        e += 1
    elif a < Fraction(2) ** e:
        e -= 1
    quantum = Fraction(2) ** (max(e, emin) - p + 1)
    r = round(a / quantum) * quantum                                      # Fraction.__round__: ties to even
    if r >= Fraction(2) ** (emax + 1):
        return float("inf") if q > 0 else float("-inf")
    return r if q > 0 else -r


def _exact(x: float):
    return Fraction(x) if np.isfinite(x) else x


def _add(a, b):
    if isinstance(a, float) or isinstance(b, float):
        return float(a) + float(b)
    return a + b


def _stepwise(cols, op, acc_dtype, out_dtype):
    """The contract evaluated in exact arithmetic with an explicit rounding after every step."""
    vals = [_exact(float(v)) for v in cols]
    acc = _round(vals[0], acc_dtype)
    for x in vals[1:]:
        if op in (numeric.SUM, numeric.AVG):
            acc = _round(_add(acc, x), acc_dtype)
        elif op == numeric.PROD:
            acc = _round(acc * x, acc_dtype)
        elif op == numeric.MAX:
            acc = acc if acc > x else x
        else:
            acc = acc if acc < x else x
    if op == numeric.AVG:
        acc = _round(acc / len(vals), acc_dtype)
    return _round(acc, out_dtype)


def _columns(dtype, world, n, seed, op):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(world, n, generator=g, dtype=torch.float64)
    x *= 2.0 ** (torch.randint(-12, 13, (world, n), generator=g)).double()   # magnitudes 2^+-12 apart
    if op == numeric.PROD:
        x = 1 + x / (1 + x.abs()) / 4                                        # stay near 1
    x[-1, : n // 4] = -x[:-1, : n // 4].sum(0) * (1 + 2.0 ** -7)             # cancellation columns
    return [c.to(dtype) for c in x]


@pytest.mark.parametrize("world", (2, 3, 5, 8))
@pytest.mark.parametrize("dtype", _FLOATS)
@pytest.mark.parametrize("op", (numeric.SUM, numeric.AVG, numeric.MAX, numeric.MIN, numeric.PROD))
def test_reduce_op_equals_stepwise_exact_rounding(world, dtype, op):
    """reduce_op is the exact result rounded through the kernels' steps; SUM / AVG lie inside the bound."""
    cols = _columns(dtype, world, 64, 1000 * world + op, op)
    got = numeric.reduce_op(cols, op)
    assert got.dtype == dtype
    acc = numeric._ACC[dtype]
    bound = numeric.sum_error_bound(cols, op) if op in (numeric.SUM, numeric.AVG) else None
    ref64 = numeric.reference64(cols, op)
    for j in range(got.numel()):
        want = _stepwise([c[j] for c in cols], op, acc, dtype)
        assert _exact(float(got[j])) == want, (j, float(got[j]), float(want))
        exact_vals = [Fraction(float(c[j])) for c in cols]
        if op in (numeric.SUM, numeric.AVG):
            exact = sum(exact_vals) / (world if op == numeric.AVG else 1)
            assert abs(Fraction(float(got[j])) - exact) <= Fraction(float(bound[j])), j
            assert abs(float(got[j]) - float(ref64[j])) <= float(bound[j]), j
        elif op == numeric.MAX:
            assert float(ref64[j]) == float(max(exact_vals)) == float(got[j])
        elif op == numeric.MIN:
            assert float(ref64[j]) == float(min(exact_vals)) == float(got[j])


@pytest.mark.parametrize("world", (2, 3, 8))
@pytest.mark.parametrize("dtype", (torch.int32, torch.int64))
@pytest.mark.parametrize("op", (numeric.SUM, numeric.MAX, numeric.MIN, numeric.PROD))
def test_reduce_op_integers_exact(world, dtype, op):
    g = torch.Generator().manual_seed(world + 10 * op)
    hi = 4 if op == numeric.PROD else 1 << 20
    cols = [torch.randint(-hi, hi, (50,), generator=g, dtype=dtype) for _ in range(world)]
    if dtype == torch.int64 and op != numeric.PROD:
        cols = [c + (-1) ** r * (1 << 60) for r, c in enumerate(cols)]          # 64-bit magnitudes
    got = numeric.reduce_op(cols, op)
    fold = {numeric.SUM: lambda a, b: a + b, numeric.MAX: max, numeric.MIN: min, numeric.PROD: lambda a, b: a * b}[op]
    for j in range(50):
        want = int(cols[0][j])
        for c in cols[1:]:
            want = fold(want, int(c[j]))
        assert int(got[j]) == want
    with pytest.raises(ValueError):
        numeric.reduce_op(cols, numeric.AVG)


def test_reduce_op_wire_bf16_rounds_inputs_then_reduces_as_bf16():
    g = torch.Generator().manual_seed(3)
    cols = [torch.randn(256, generator=g) for _ in range(5)]
    got = numeric.reduce_op_wire_bf16(cols, numeric.AVG)
    assert got.dtype == torch.float32
    for j in range(256):
        want = _stepwise([c[j].bfloat16() for c in cols], numeric.AVG, torch.float32, torch.bfloat16)
        assert Fraction(float(got[j])) == want
    assert not torch.equal(got, numeric.reduce_op(cols, numeric.AVG))         # the wire rounding is visible


def test_reduce_op_special_values():
    inf, nan = float("inf"), float("nan")
    cols = [torch.tensor([inf, inf, -0.0, nan, 1e-45, 6.0e4]), torch.tensor([1.0, -inf, -0.0, 1.0, 1e-45, 6.0e4])]
    s = numeric.reduce_op(cols, numeric.SUM)
    assert s[0] == inf and torch.isnan(s[1]) and torch.isnan(s[3])
    assert s[2] == 0 and torch.signbit(s[2])                                    # -0 + -0 = -0
    assert s[4] == 2 * cols[0][4] and s[4] < 2.0 ** -126                        # subnormal sum is exact
    half = numeric.reduce_op([c.half() for c in cols], numeric.SUM)
    assert half[5] == inf                                                       # fp16 SUM overflows ...
    assert numeric.reduce_op([c.half() for c in cols], numeric.AVG)[5] == 6.0e4  # ... its mean does not
    m = numeric.reduce_op([torch.tensor([0.0]), torch.tensor([-0.0])], numeric.MAX)
    assert torch.signbit(m[0])                                                  # tie keeps the later rank, as combine<MAX>


@pytest.mark.parametrize("dtype,step", ((torch.bfloat16, 2.0 ** -9), (torch.float16, 2.0 ** -12)))
def test_bound_rejects_16_bit_accumulation(dtype, step):
    """A mean accumulated in the 16-bit type itself falls outside the bound on cancellation and
    small-increment inputs, so the bound tells a wrong accumulator width from a right one."""
    world = 8
    small = [torch.tensor([1.0, 1.0], dtype=dtype)] + [torch.tensor([step, 2 * step], dtype=dtype)] * (world - 2) \
        + [torch.tensor([-1.0, -1.0], dtype=dtype)]
    for op in (numeric.SUM, numeric.AVG):
        ref = numeric.reference64(small, op)
        bound = numeric.sum_error_bound(small, op)
        good = numeric.reduce_op(small, op)
        assert bool(((good.double() - ref).abs() <= bound).all())
        bad = numeric.reduce_op(small, op, acc_dtype=dtype)
        assert bool(((bad.double() - ref).abs() > bound).any()), (op, bad, ref)
