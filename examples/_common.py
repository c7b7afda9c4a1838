"""Shared helpers of the experiment scripts (one per reference ``main_*.py``).

Every script builds its experiment from the same public API as the reference script of the same
name, runs it on ``GOSSIPY_DEVICE`` (default: ``cuda`` when available) and prints the last evaluation.
There is no network on the target boxes, so the data sets are the shape-compatible synthetic ones
of :mod:`gossipy_b200.data.synthetic` (``load_*`` fall back to them automatically).

Environment: ``GOSSIPY_ROUNDS`` (override the number of rounds), ``GOSSIPY_NODES`` (cap the number
of nodes), ``GOSSIPY_ENGINE=native|python`` (round-loop control plane), ``GOSSIPY_EXECUTOR=native``
(with the native engine: enqueue eligible simulations from the C++ executor), ``GOSSIPY_BATCHED=auto|0|1``
(with the native engine: run bankable set-ups many nodes per launch -- ``auto``: on a GPU or from 512 nodes),
``GOSSIPY_DEVICE``,
``GOSSIPY_COMPAT=1`` (``reference_compat``: reproduce the reference's numbers, Python engine).
Multi-GPU: launch with ``python -m torch.distributed.run --nproc-per-node N examples/<script>.py``.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

import gossipy_b200 as gossipy  # noqa: E402
from gossipy_b200 import GlobalSettings  # noqa: E402


def setup(seed: int):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = os.environ.get("GOSSIPY_DEVICE", "cuda" if torch.cuda.is_available() else "cpu")
    if dev.startswith("cuda"):
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dev = "cuda:%d" % torch.cuda.current_device()
    GlobalSettings().set_device(dev)
    GlobalSettings().reference_compat = os.environ.get("GOSSIPY_COMPAT", "0") == "1"   # the reference's own numbers
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl" if dev.startswith("cuda") else "gloo")
        from gossipy_b200.parallel import runtime as prt
        prt.init(rank, world)
    gossipy.set_seed(seed)
    return rank, world


def rounds(default: int) -> int:
    return int(os.environ.get("GOSSIPY_ROUNDS", default))


def cap_nodes(n: int) -> int:
    return min(n, int(os.environ.get("GOSSIPY_NODES", n)))


def configure(sim):
    sim.engine = os.environ.get("GOSSIPY_ENGINE", "python")
    sim.native_executor = os.environ.get("GOSSIPY_EXECUTOR", "python") == "native"
    sim.progress = os.environ.get("GOSSIPY_PROGRESS", "0") == "1"
    sim.batched = {"auto": "auto", "0": False, "1": True}[os.environ.get("GOSSIPY_BATCHED", "auto")]
    return sim


def finish(report, rank: int, local: bool = False):
    ev = report.get_evaluation(local)
    if rank == 0:
        print("rounds evaluated: %d" % len(ev))
        if ev:
            print("last evaluation:", {k: round(v, 4) for k, v in ev[-1][1].items()})
        print("sent=%d failed=%d size=%d" % (report._sent_messages, report._failed_messages, report._total_size))
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    return ev


def regular_graph(n: int, d: int, seed: int = 42):
    """Adjacency (dense 0/1) of a random d-regular graph; networkx when installed, else a circulant."""
    import numpy as np
    try:
        from networkx import to_numpy_array
        from networkx.generators.random_graphs import random_regular_graph
        return to_numpy_array(random_regular_graph(d, n, seed=seed)).astype(int)
    except Exception:
        A = np.zeros((n, n), dtype=int)
        for i in range(n):
            for k in range(1, d // 2 + 1):
                A[i, (i + k) % n] = A[(i + k) % n, i] = 1
        return A
