#!/usr/bin/env python
"""Benchmark of the hot path on BASELINE.json's metric: CIFAR ResNet-18 samples/sec with
``distrib.sync_model`` gradient synchronisation (reference: examples/cifar/solver.py:46-53).

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA path)
    python bench.py --impl reference --gpus N --steps K ...  # reference path on the host CPUs
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results as DIR/*.npy

Workload (``config.workload``): the 8-rank data-parallel job of BASELINE configs[1] --
torchvision resnet18(num_classes=10) in bf16, batch 64 per rank, SGD lr 1e-4, synthetic
CIFAR-shaped batches -- run on N GPUs with 8/N ranks per GPU.  On one GPU the 8 ranks are
virtual ranks of one process (one thread + one CUDA stream each); every ``sync_model`` of the
8 ranks is ONE launch of the bucketed all-reduce kernel.  Total work per step is fixed
(global batch 512), so the scaling over N is "strong".  A step per rank is:
    forward, cross_entropy, backward (replayed CUDA graph), flashy_b200.distrib.sync_model(model),
    optim.step()                    [zero_grad: the replayed backward overwrites .grad]
``value`` times K steps with the batch resident in HBM; ``e2e`` times K more steps through the
same public API with the batch copied from pinned host memory and the loss read back each step.

``--overlap`` (one rank per GPU only) captures the step as ONE CUDA graph of forward, backward and
``sync_model`` with backward overlap enabled (``distrib.overlap(model)``: gradient buckets leave on
the communicator's side stream while backward still runs; ``sync_model`` sends the tail bucket and
joins).  It is off by default: on this latency-bound batch-64 step it measured slower than one exposed
``sync_model`` launch (profiles/README.md).  Before anything is timed, at every N, the real 62-tensor bf16 gradient
bucket is averaged once with seeded inputs and compared with ``oracle/numeric.py`` (checker use
only, outside every timed region): the ``parity`` object, and a non-zero exit on mismatch.
``--model resnet50 --image 224 --batch 32`` is BASELINE configs[2].
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

WORLD = 8
BATCH = 64
METRIC = "cifar_resnet18_train_samples_per_sec"
DUMP_ELEMS = 1 << 22          # per dumped array: 16 MB of float32, so that a dump stays below 64 MB


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=("native", "reference"))
    ap.add_argument("--world", type=int, default=WORLD, help="data-parallel ranks of the job")
    ap.add_argument("--batch", type=int, default=BATCH, help="samples per rank per step")
    ap.add_argument("--no-graphs", action="store_true", help="eager forward/backward instead of a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=5)
    ap.add_argument("--kernel-table", default="", help="write a per-kernel device-time table of the timed region (CUPTI) to this file")
    ap.add_argument("--model", default="resnet18", choices=("resnet18", "resnet50"))
    ap.add_argument("--image", type=int, default=32, help="square image size (32: CIFAR, 224: ImageNet-shaped)")
    ap.add_argument("--overlap", action="store_true",
                    help="capture the step with distrib.overlap(model): gradient buckets leave during backward (measured slower "
                         "for this latency-bound step, see profiles/README.md; default: one sync_model launch after backward)")
    ap.add_argument("--no-parity", action="store_true", help="skip the pre-timing parity check against the oracle")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float32): loss (every rank), and "
                         "rank 0's grads (as sync_model averaged them), buffers and params (after optim.step()); "
                         f"arrays above {DUMP_ELEMS} elements are a fixed seeded sample of that many")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs needs --impl native")
    return args


# =========================================================================== reference arm
def reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cpu_train
    res = cpu_train.run(world=args.world, batch=args.batch, steps=max(1, args.steps), warmup=max(0, args.warmup))
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": workload_config(args, args.gpus, cpu=True),
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": res["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


MODELS = {"resnet18": (62, 11181642), "resnet50": (161, 25557032)}


def workload_config(args, n_gpus: int, cpu: bool = False) -> dict:
    """The same object in both arms (the driver compares them)."""
    tensors, elements = MODELS[args.model]
    classes = 10 if args.model == "resnet18" else 1000
    return {
        "workload": (f"examples/cifar-style step, torchvision {args.model} ({classes} classes), distrib.sync_model gradient+buffer "
                     f"all-reduce, {args.world} data-parallel ranks x batch {args.batch}, SGD lr 1e-4"),
        "world": args.world, "global_batch": args.world * args.batch, "image": f"3x{args.image}x{args.image}",
        "grad_tensors": tensors, "grad_elements": elements,
    }


def make_model(args):
    import torchvision
    if args.model == "resnet18":
        return torchvision.models.resnet18(num_classes=10)
    return torchvision.models.resnet50()


# =========================================================================== clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for row in out.strip().splitlines():
            cells = [c.strip() for c in row.split(",")]
            if len(cells) < 7:
                continue
            try:
                sm.append(float(cells[0]))
                mx.append(float(cells[1]))
            except ValueError:
                continue
            for name, cell in zip(names, cells[3:7]):
                if cell.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# =========================================================================== native arm
class Replica:
    """One data-parallel rank: model, optimizer, static batch, captured step.

    ``overlap``: the captured graph holds forward, backward AND ``distrib.sync_model`` with backward
    overlap (gradient buckets launched from post-accumulate hooks on the side stream, joined by
    ``sync_model``).  Otherwise the graph holds forward+backward and ``sync_model`` is an ordinary
    call after the replay.  ``graph_nosync`` (forward+backward only) serves the no-exchange reference
    step of ``aux``."""

    def __init__(self, rank: int, args, device, distrib, overlap: bool):
        import torch
        import torch.nn.functional as F
        self.rank = rank
        self.distrib = distrib
        self.overlap = overlap
        self.stream = torch.cuda.Stream(device=device)
        torch.manual_seed(1234)                                       # same initial weights everywhere
        self.model = make_model(args).to(device=device, dtype=torch.bfloat16)
        self.model = self.model.to(memory_format=torch.channels_last)
        self.optim = torch.optim.SGD(self.model.parameters(), lr=1e-4)
        classes = 10 if args.model == "resnet18" else 1000
        g = torch.Generator().manual_seed(1234 + rank)
        n_host = 4                                                    # rotating pinned batches for the e2e leg
        self.host_img = [torch.randn(args.batch, 3, args.image, args.image, generator=g).to(torch.bfloat16).pin_memory()
                         for _ in range(n_host)]
        self.host_lab = [torch.randint(0, classes, (args.batch,), generator=g).pin_memory() for _ in range(n_host)]
        self.img = self.host_img[0].to(device).contiguous(memory_format=torch.channels_last)
        self.label = self.host_lab[0].to(device)
        self.loss = torch.zeros((), device=device, dtype=torch.bfloat16)
        self.graph = self.graph_nosync = None
        self.launches_per_replay = 0
        self.h2d_bytes = self.host_img[0].numel() * 2 + self.host_lab[0].numel() * 8
        self.d2h_bytes = 2
        self.F = F

    def _fwd_bwd(self):
        loss = self.F.cross_entropy(self.model(self.img), self.label)
        loss.backward()
        return loss

    def capture(self, engine_launches):
        """Collective when ``overlap`` (sync_model runs during warm-up and capture)."""
        import torch
        with torch.cuda.stream(self.stream):
            for _ in range(3):                                        # warm-up on the capture stream
                self.optim.zero_grad(set_to_none=True)
                self._fwd_bwd()
        self.stream.synchronize()
        self.graph_nosync = torch.cuda.CUDAGraph()
        self.optim.zero_grad(set_to_none=True)
        with torch.cuda.graph(self.graph_nosync, stream=self.stream):
            loss = self._fwd_bwd()
            self.loss.copy_(loss.detach())
        self.stream.synchronize()
        if not self.overlap:
            self.graph = self.graph_nosync
            return
        self.distrib.overlap(self.model, True)
        with torch.cuda.stream(self.stream):
            for _ in range(3):        # 1st sync_model installs the hooks; from the 2nd on the buckets leave during backward
                self.optim.zero_grad(set_to_none=True)
                self._fwd_bwd()
                self.distrib.sync_model(self.model)
        self.stream.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        self.optim.zero_grad(set_to_none=True)
        before = engine_launches()
        with torch.cuda.graph(self.graph, stream=self.stream):
            loss = self._fwd_bwd()
            self.distrib.sync_model(self.model)
            self.loss.copy_(loss.detach())
        self.launches_per_replay = engine_launches() - before
        self.stream.synchronize()

    def step(self, e2e: bool, it: int):
        if e2e:
            k = it % len(self.host_img)
            self.img.copy_(self.host_img[k], non_blocking=True)
            self.label.copy_(self.host_lab[k], non_blocking=True)
        if self.graph is not None:
            self.graph.replay()
        else:
            self.optim.zero_grad()                                    # first, so the step's gradients outlive it
            self.loss.copy_(self._fwd_bwd().detach())
        if not (self.overlap and self.graph is not None):
            self.distrib.sync_model(self.model)
        self.optim.step()
        if e2e:
            return self.loss.item()                                   # device -> host read of the step's result
        return None


def bf16_ulp_distance(a, b) -> int:
    """Largest distance, in bf16 units in the last place, between two bf16 tensors."""
    import torch

    def key(t):
        bits = t.contiguous().view(torch.int16).to(torch.int32) & 0xFFFF
        return torch.where(bits >= 0x8000, 0x8000 - bits, bits)
    return int((key(a) - key(b)).abs().max()) if a.numel() else 0


def write_outputs(out_dir: str, snapshot: dict, proc_world: int, proc_rank: int) -> None:
    """``out_dir/<name>.npy`` in float32 for every array of ``snapshot``; ``loss`` gathers every process's
    ranks in rank order.  An array longer than DUMP_ELEMS is cut to the same seeded sample of positions
    on every run, so that two builds can be compared element for element."""
    import numpy as np
    import torch
    import torch.distributed as dist
    arrays = {name: t.float().cpu() for name, t in snapshot.items()}
    if proc_world > 1:
        losses = [None] * proc_world
        dist.all_gather_object(losses, arrays["loss"])
        arrays["loss"] = torch.cat(losses)
    if proc_rank != 0:
        return
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        if t.numel() > DUMP_ELEMS:
            keep = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_ELEMS]
            t = t[keep.sort().values]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.numpy())


def native_arm(args) -> None:
    import torch
    import torch.distributed as dist
    from flashy_b200 import VirtualWorld, distrib
    from flashy_b200 import _native as N
    from flashy_b200 import context as fctx

    n_gpus = args.gpus
    proc_world = int(os.environ.get("WORLD_SIZE", "1"))
    proc_rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert proc_world == n_gpus, f"--gpus {n_gpus} needs {n_gpus} processes (torchrun), got WORLD_SIZE={proc_world}"
    assert args.world % n_gpus == 0
    n_local = args.world // n_gpus
    W = args.world
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if proc_world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("gloo", init_method="env://")        # bootstrap + timing reduction only
    overlap = n_local == 1 and W > 1 and args.overlap and not args.no_graphs

    vw = VirtualWorld(n_local, device=local_rank) if n_local > 1 else None

    def run_ranks(fn):
        if vw is not None:
            return vw.run(fn)
        return [fn(proc_rank, args.world)]

    def engine():
        return vw.engine if vw is not None else fctx.current().engine

    def global_barrier():
        torch.cuda.synchronize()
        if proc_world > 1:
            dist.barrier()

    def reduce_max(x: float) -> float:
        if proc_world > 1:
            t = torch.tensor([x], dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t[0])
        return x

    # ---- parity first: the real gradient bucket, seeded inputs, against the oracle (checker use only)
    numels = [p.numel() for p in make_model(args).parameters()]
    parity = None
    if not args.no_parity and W > 1:
        from oracle import numeric
        gens = [torch.Generator().manual_seed(1000 + r) for r in range(W)]
        per_rank = [[(torch.randn(n, generator=gens[r]) * 1e-2).to(torch.bfloat16) for n in numels] for r in range(W)]
        want = numeric.average_tensors(per_rank)[0]

        def parity_body(rank, world):
            ts = [t.to(device) for t in per_rank[rank]]
            distrib.average_tensors(ts)
            torch.cuda.synchronize()
            return max(bf16_ulp_distance(t.cpu(), w_) for t, w_ in zip(ts, want))
        global_barrier()
        ulp = reduce_max(float(max(run_ranks(parity_body))))
        global_barrier()
        plan = max(engine().plans.values(), key=lambda pl: pl.info.wire_bytes)
        switch_order = plan.info.kernel in (3, 5, 7)                 # NVLS: the switch picks the summation order
        parity = {"checked": True, "kernel": N.KERNEL_NAMES.get(int(plan.info.kernel), "?"),
                  "algo": N.ALGO_NAMES.get(int(plan.info.algo), "?"), "max_ulp": int(ulp),
                  "bar_ulp": 1 if switch_order else 0, "tensors": len(numels), "elements": sum(numels), "dtype": "bf16",
                  "oracle": "oracle/numeric.py: fp32 sum in rank order, /W, rounded once to bf16",
                  "ok": ulp <= (1 if switch_order else 0)}
        del per_rank, want
        if not parity["ok"]:
            if proc_rank == 0:
                print(json.dumps({"metric": METRIC, "parity": parity, "error": "CUDA all-reduce disagrees with the oracle"}), flush=True)
            sys.exit(3)

    replicas = [Replica(proc_rank * n_local + l, args, device, distrib, overlap) for l in range(n_local)]
    if not args.no_graphs:
        if overlap:
            replicas[0].capture(lambda: engine().native_launches())
        else:
            for rep in replicas:
                rep.capture(None)
    torch.cuda.synchronize()

    def timed_region(steps: int, e2e: bool):
        """Every rank runs `steps` steps; returns max-over-ranks device time in ms."""
        def body(rank, world):
            rep = replicas[rank - proc_rank * n_local]
            with torch.cuda.stream(rep.stream):
                distrib.barrier()                                     # all ranks (threads and processes) start together
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(rep.stream)
                for it in range(steps):
                    rep.step(e2e, it)
                e1.record(rep.stream)
                rep.stream.synchronize()
                return e0.elapsed_time(e1)
        global_barrier()
        ms = max(run_ranks(body))
        global_barrier()
        return reduce_max(ms)

    # ---- warm-up (also creates the communicator and the bucket plans)
    timed_region(max(args.warmup, 3), e2e=False)
    timed_region(2, e2e=True)
    eng = engine()

    # ---- timed: K steps, inputs resident
    sampler = ClockSampler(local_rank) if proc_rank == 0 else None
    launches0 = eng.native_launches()
    cuprof = os.environ.get("FX_BENCH_CUPROF") == "1"                 # ncu --profile-from-start off
    if cuprof:
        torch.cuda.profiler.start()
    prof = None
    if args.kernel_table:
        from torch.profiler import profile, ProfilerActivity
        prof = profile(activities=[ProfilerActivity.CUDA])
        prof.__enter__()
    ms_value = timed_region(args.steps, e2e=False)
    if prof is not None:
        torch.cuda.synchronize()
        prof.__exit__(None, None, None)
        if proc_rank == 0:
            events = [e for e in prof.key_averages() if e.device_time_total > 0]
            total = sum(e.device_time_total for e in events)
            with open(args.kernel_table, "w") as fh:
                fh.write(f"# kernels of {args.steps} timed steps (torch.profiler / CUPTI), sorted by device time; total {total:.0f} us\n")
                fh.write("share_pct,device_us,count,name\n")
                for e in sorted(events, key=lambda e: -e.device_time_total):
                    fh.write(f"{100 * e.device_time_total / total:.2f},{e.device_time_total:.1f},{e.count},{e.key[:140]}\n")
    if cuprof:
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    # what the last timed step handed its caller, copied on the device before later steps overwrite it
    snapshot = None
    if args.dump_outputs:
        snapshot = {"loss": torch.stack([rep.loss for rep in replicas])}
        if proc_rank == 0:
            model0 = replicas[0].model
            snapshot["grads"] = torch.cat([p.grad.flatten() for p in model0.parameters()])
            snapshot["buffers"] = torch.cat([b.flatten() for b in model0.buffers() if b.dtype.is_floating_point])
            snapshot["params"] = torch.cat([p.detach().flatten() for p in model0.parameters()])
        torch.cuda.synchronize()
    # kernels of this library inside the timed region: host-side launches plus the ones each graph replay re-issues
    launches = eng.native_launches() - launches0 + args.steps * sum(rep.launches_per_replay for rep in replicas)
    # ---- timed: K steps end to end (H2D batch + D2H loss inside the region)
    ms_e2e = timed_region(args.steps, e2e=True)
    # The timed regions are short (tens of ms at 8 GPUs): keep the same load running until the
    # sampler has had ~0.6 s, so that the median SM clock under load rests on enough samples.
    # Collective: every rank runs the same number of extra (untimed) steps.
    t_load = ms_value + ms_e2e
    extra = 0
    while t_load < 600.0 and extra < 40:
        t_load += timed_region(args.steps, e2e=False)
        extra += 1
    clocks = sampler.stop() if sampler else None
    if clocks is not None:
        clocks["sampled_over_ms"] = t_load
    if snapshot is not None:
        write_outputs(args.dump_outputs, snapshot, proc_world, proc_rank)

    # ---- the dominant kernel of this repo, timed live: the whole gradient+buffer bucket of one sync_model call as
    # ONE launch (backward overlap switched off), CUDA events around every launch on its launch stream
    for rep in replicas:
        distrib.overlap(rep.model, False)

    def kernel_body(rank, world):
        rep = replicas[rank - proc_rank * n_local]
        with torch.cuda.stream(rep.stream):
            if rep.graph_nosync is not None:
                rep.graph_nosync.replay()                             # fresh gradients
            else:
                rep._fwd_bwd()
            for _ in range(3):
                distrib.sync_model(rep.model)
            rep.stream.synchronize()
            distrib.barrier()
            eng.profile, eng.timings = True, []
            for _ in range(args.steps):
                distrib.sync_model(rep.model)
            rep.stream.synchronize()
        return True
    global_barrier()
    run_ranks(kernel_body)
    global_barrier()
    eng.profile = False
    timings = list(eng.timings)

    # ---- auxiliary: one rank alone on this GPU, no sync_model (the W = 1 step of the reference,
    # where the path is a no-op): what the step costs without any gradient exchange
    rep0 = replicas[0]
    torch.cuda.synchronize()
    with torch.cuda.stream(rep0.stream):
        def plain():
            rep0.graph_nosync.replay() if rep0.graph_nosync is not None else rep0._fwd_bwd()
            rep0.optim.step()
            if rep0.graph_nosync is None:
                rep0.optim.zero_grad()
        for _ in range(3):
            plain()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(rep0.stream)
        for _ in range(args.steps):
            plain()
        s1.record(rep0.stream)
        rep0.stream.synchronize()
    single_ms = s0.elapsed_time(s1) / args.steps

    if proc_world > 1:
        t = torch.tensor([launches], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        launches = int(t[0])

    by_plan = {}
    for key, e0, e1 in timings:
        by_plan.setdefault(key, []).append(e0.elapsed_time(e1))
    grad_key = max(by_plan, key=lambda k: sum(k[1])) if by_plan else None
    roofline = None
    allreduce = None
    if grad_key is not None:
        kernel_ms = reduce_max(statistics.mean(by_plan[grad_key]))
        info = eng.plans[grad_key].info
        kernel = N.KERNEL_NAMES.get(int(info.kernel), "?")
        payload = sum(grad_key[1]) * 2                                # bf16 bytes of one rank's bucket (N)
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except OSError:
            pass
        if n_local == W:
            # all ranks on this GPU: every byte moves through HBM.  Per rank: pack 2N, reduce reads N
            # and writes N/W, gather reads N and writes N  ->  (5 + 1/W) N, times the W hosted ranks.
            alg_bytes = W * (5 + 1 / W) * payload
            peak, bound, peak_src = peaks.get("hbm_gbs", 6650.0), "hbm", ("measured" if peaks else "fallback")
        else:
            # NVLink bytes per GPU per direction in the all-reduce bus-bandwidth convention
            # (reduce-scatter + all-gather of the shards held elsewhere): 2 n_local (W - n_local) / W * N
            alg_bytes = 2 * n_local * (W - n_local) / W * payload
            peak, bound, peak_src = 900.0, "nvlink", "nominal NVLink 5 per direction (measured peer copy: 770)"
        achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
        traffic = None
        try:
            traffic = json.loads((ROOT / "profiles" / "traffic.json").read_text()).get(f"{kernel}@n{n_gpus}")
        except (OSError, ValueError):
            pass
        roofline = {"bound": bound, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic,
                    "kernel": f"{kernel} ({N.ALGO_NAMES.get(int(info.algo), '?')}, grid {int(info.grid_x)} x {n_local}, "
                              f"{int(info.chunks)} chunks of {int(info.chunk_bytes)} B per slice): the gradient+buffer bucket of one "
                              f"sync_model call, {len(grad_key[1])} tensors",
                    "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                    "launches_timed": len(by_plan[grad_key]),
                    "how": "CUDA events around each launch on its launch stream, back-to-back sync_model calls after the "
                           "timed steps (overlap off: one launch per call), mean over launches, max over ranks"}
        allreduce = {"payload_bytes_per_rank": payload, "kernel_ms": kernel_ms, "kernel": kernel,
                     "alg_gbs": payload / (kernel_ms * 1e-3) / 1e9,
                     "bus_gbs": 2 * (W - 1) / W * payload / (kernel_ms * 1e-3) / 1e9}

    if proc_rank != 0:
        return
    samples = args.world * args.batch * args.steps
    ms_step = ms_value / args.steps
    line = {
        "metric": METRIC, "value": samples / (ms_value * 1e-3), "unit": "samples/s", "n_gpus": n_gpus,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args, n_gpus),
        "setup": {"ranks_per_gpu": n_local, "cuda_graphs": not args.no_graphs, "backward_overlap": overlap,
                  "step": ("ONE captured graph per step: forward, backward with gradient buckets leaving from "
                           "post-accumulate hooks on the side stream, sync_model (tail bucket + join); then optim.step()"
                           if overlap else
                           "captured graph of forward+backward, then distrib.sync_model(model) (one launch), then optim.step()"),
                  "zero_grad": ("implicit: the captured backward starts from grad=None, so every replay overwrites "
                                ".grad (same state as zero_grad(set_to_none=True) + backward)" if not args.no_graphs
                                else "optim.zero_grad() every step"),
                  "l2": "not flushed: a step touches weights+grads+activations of every hosted replica; the stand-alone "
                        "kernel timing re-reads a bucket that fits the 126 MB L2, as it does right after backward"},
        "e2e": {"value": samples / (ms_e2e * 1e-3), "unit": "samples/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": replicas[0].h2d_bytes * args.world,
                "d2h_bytes_per_step": replicas[0].d2h_bytes * args.world,
                "api": "flashy_b200.distrib.sync_model(model) per rank; pinned-host batch -> device, loss.item()"},
        "gpu_launches": launches,
        "clocks": clocks,
        "parity": parity,
        "roofline": roofline,
        "allreduce": allreduce,
        "aux": {"single_rank_no_sync_ms_per_step": single_ms,
                "single_rank_no_sync_samples_per_s": args.batch / (single_ms * 1e-3),
                "weak_efficiency": (single_ms / ms_step) if n_local == 1 else None,
                "exposed_sync_ms": (ms_step - single_ms) if n_local == 1 else None,
                "note": "one replica alone on one GPU without sync_model (the reference's W=1 step).  With one rank per "
                        "GPU, weak_efficiency = this / ms_per_step is the fraction of ideal linear (per-GPU work fixed) "
                        "scaling the step reaches, and the difference is the exposed gradient-sync cost"},
    }
    if n_gpus == 1 and not args.no_cpu_baseline:
        from oracle import cpu_train
        res = cpu_train.run(world=args.world, batch=args.batch, steps=max(args.cpu_steps, 5), warmup=1)
        line["cpu_baseline"] = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line), flush=True)
    if vw is not None:
        vw.close()


def main():
    args = parse()
    if args.impl == "reference":
        reference_arm(args)
    else:
        native_arm(args)
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:      # noqa: BLE001
        pass


if __name__ == "__main__":
    main()
