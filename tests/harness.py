"""Multi-rank harness without a cluster: W spawned processes + gloo on 127.0.0.1.

Same pattern as the reference's tests/test_distrib.py:82-98 (rank 0 runs in the calling
process, ranks 1..W-1 are spawned, every exit code must be 0).
"""
from __future__ import annotations

import importlib
import multiprocessing as mp
import os
import socket
import sys
import traceback
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _entry(rank: int, world: int, port: int, module: str, func: str, args: tuple, backend: str, hide_gpus: bool):
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world),
                      MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    if hide_gpus:
        os.environ["CUDA_VISIBLE_DEVICES"] = ""
    if str(ROOT) not in sys.path:
        sys.path.insert(0, str(ROOT))
    import torch
    import torch.distributed as dist
    torch.set_num_threads(1)
    if backend != "none":
        dist.init_process_group(backend, init_method="env://")
    try:
        getattr(importlib.import_module(module), func)(rank, world, *args)
    except BaseException:
        traceback.print_exc()
        raise
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


def run_ranks(world: int, module: str, func: str, args: tuple = (), backend: str = "gloo", timeout: float = 180.0,
              hide_gpus: bool = False):
    """Run ``module.func(rank, world, *args)`` on ``world`` processes; raise if any fails.
    ``hide_gpus``: the processes see no CUDA device, as on a CPU-only machine, whatever this one has."""
    ctx = mp.get_context("spawn")
    port = free_port()
    procs = [ctx.Process(target=_entry, args=(r, world, port, module, func, args, backend, hide_gpus))
             for r in range(world)]
    for p in procs:
        p.start()
    bad = []
    for r, p in enumerate(procs):
        p.join(timeout)
        if p.is_alive():
            p.kill()
            bad.append((r, "timeout"))
        elif p.exitcode != 0:
            bad.append((r, p.exitcode))
    assert not bad, f"ranks failed: {bad}"
