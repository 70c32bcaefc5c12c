#!/usr/bin/env python
"""BASELINE configs[3]: the two-optimizer GAN step of ``flashy.adversarial`` on N GPUs.

    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 benchmarks/gan_step.py [--dim 1024 --depth 6]

One step per rank is the loop body of the reference's dummy solver (``tests/dummy/train.py:88-102``)
scaled up: student / teacher / adversary MLPs of ``depth`` x ``dim`` x ``dim`` layers,
    estimate = model(noise); gt = teacher(noise); mse = mse_loss(estimate, gt)
    adv_disc = adv.train_adv(estimate, gt)       # backward inside distrib.eager_sync_model(adversary), adversary optimizer
    adv_gen = adv(estimate); (mse + adv_gen).backward(); distrib.sync_model(model); optim.step()
so two models are synchronised per step over one communicator (eager hooks for the adversary, the bucketed
``sync_model`` for the generator).  ``AdversarialLoss`` is the UNMODIFIED reference class from
``oracle/_ref`` (``flashy/adversarial.py:22-89``) running over ``flashy_b200.distrib``; ``dora`` /
``colorlog`` come from the test-only stand-ins in ``tests/shims``.  Prints one JSON line (rank 0):
samples/s, ms per step (CUDA events, max over ranks), launches of this library per step.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests" / "shims"))
sys.path.append(str(ROOT / "oracle" / "_ref"))

import torch                      # noqa: E402
import torch.distributed as dist  # noqa: E402
from torch import nn              # noqa: E402


def mlp(dim, depth):
    layers = []
    for _ in range(depth):
        layers += [nn.Linear(dim, dim), nn.ReLU()]
    return nn.Sequential(*layers[:-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dim", type=int, default=1024)
    ap.add_argument("--depth", type=int, default=6)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("gloo", init_method="env://")
    import flashy_b200.distrib
    sys.modules["flashy.distrib"] = flashy_b200.distrib          # INTEGRATION.md section 1
    import flashy
    from flashy_b200 import context as fctx
    distrib = flashy.distrib

    torch.manual_seed(1234 + rank)                                # different initial weights: broadcast_model must fix that
    teacher = mlp(args.dim, args.depth).to(dev)
    distrib.broadcast_model(teacher)
    model = mlp(args.dim, args.depth).to(dev)
    distrib.broadcast_model(model)
    optim = torch.optim.Adam(model.parameters())
    adv_model = mlp(args.dim, args.depth).to(dev)
    adv = flashy.adversarial.AdversarialLoss(adv_model, torch.optim.Adam(adv_model.parameters()))
    g = torch.Generator(device=dev).manual_seed(99 + rank)

    def step():
        noise = torch.randn(args.batch, args.dim, device=dev, generator=g)
        estimate = model(noise)
        with torch.no_grad():
            gt = teacher(noise)
        mse = nn.functional.mse_loss(estimate, gt)
        adv_disc = adv.train_adv(estimate, gt)
        adv_gen = adv(estimate)
        loss = mse + adv_gen
        optim.zero_grad()
        loss.backward()
        distrib.sync_model(model)
        optim.step()
        return loss, adv_disc

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    eng = fctx.current().engine
    distrib.barrier()
    launches0 = eng.native_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss, adv_disc = step()
    e1.record()
    torch.cuda.synchronize()
    launches = eng.native_launches() - launches0
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    # replicas must still agree bit for bit
    flat = torch.cat([p.detach().reshape(-1) for m in (model, adv_model) for p in m.parameters()])
    lo, hi = flat.clone(), flat.clone()
    distrib.all_reduce(lo, dist.ReduceOp.MIN)
    distrib.all_reduce(hi, dist.ReduceOp.MAX)
    same = bool(torch.equal(lo, hi))
    params = sum(p.numel() for p in model.parameters())
    if rank == 0:
        ms = float(t[0]) / args.steps
        print(json.dumps({
            "kind": "gan_step", "world": world, "dim": args.dim, "depth": args.depth, "batch_per_rank": args.batch,
            "params_per_model": params, "grad_bytes_per_model": params * 4,
            "ms_per_step": ms, "samples_per_s": world * args.batch / (ms * 1e-3),
            "native_launches_per_step": launches / args.steps,
            "replicas_identical": same, "final_loss": float(loss), "final_adv_disc": float(adv_disc),
            "adversarial_loss_class": flashy.adversarial.AdversarialLoss.__module__ + " @ " + str(Path(flashy.__file__).parent),
        }), flush=True)
    assert same, "replicas diverged"
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
