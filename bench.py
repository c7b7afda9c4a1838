#!/usr/bin/env python
"""Headline benchmark: gossip rounds/s of the 8-node MLP push-pull experiment (BASELINE.json).

Config (BASELINE.md §2 row 1): 8 nodes, ``TorchMLP(784, 10, (100,))`` (P = 79 510), SGD lr 0.1,
batch 32, 1 local epoch, MERGE_UPDATE, PUSH_PULL, sync nodes, delta = 100 ticks per round,
MNIST-shaped synthetic data 60 000 / 10 000 split into 8 non-IID shards of 7 500 samples
(McMahan pathological label skew, 2 shards per node), every node evaluated on the global test set
every round.  One "step" = one gossip round = 16 merge+local-epoch updates (3 760 SGD steps)
+ 8 evaluations.

    python bench.py --gpus N --steps K --warmup W            # this framework
    python bench.py --impl reference --gpus N ...            # unmodified reference (baseline/_ref)

Rank 0 prints one JSON line (contract in the task statement).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_NODES, D_IN, D_H, D_OUT = 8, 784, 100, 10
N_TRAIN, N_TEST, BATCH, DELTA, LR = 60000, 10000, 32, 100, 0.1
BASELINE_ROUNDS_PER_S = 0.44   # BASELINE.md: reference as-is on the survey box (CPU); no published GPU number
METRIC = "gossip rounds/sec (8-node MLP 784-100-10, push-pull, synthetic MNIST-shape non-IID)"


def common_config(world: int):
    """The benchmark configuration, identical in both arms (arm-specific notes go to "details")."""
    return {"model": "TorchMLP(784,10,(100,)) P=79510", "nodes": N_NODES, "global_batch": BATCH * N_NODES,
            "batch_per_node": BATCH, "seq_len": None, "samples_per_node": N_TRAIN // N_NODES, "local_epochs": 1,
            "optimizer": "SGD lr 0.1", "protocol": "PUSH_PULL", "mode": "MERGE_UPDATE", "delta": DELTA,
            "eval": "all 8 nodes on the 10000-sample global test set every round",
            "sgd_steps_per_round": 16 * ((N_TRAIN // N_NODES + BATCH - 1) // BATCH),
            "parallelism": "gossip-dp8 (8 nodes over %d GPU(s))" % world,
            "l2": "inputs (219 MB of shards + 31 MB test set) exceed the 126 MB L2"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--train-impl", default="", help="training kernel: '' = fp32-equivalent default (tc8, 3xTF32), "
                    "cluster (fp32 CUDA cores), tc8-tf32 | tc3 (plain tf32)")
    ap.add_argument("--engine", default="native", choices=["native", "python"],
                    help="control plane of the round loop: C++ scheduler or the Python loop")
    ap.add_argument("--executor", default="native", choices=["native", "python"],
                    help="native engine only: C++ executor (csrc/exec) or the per-event Python executor")
    ap.add_argument("--transport", default="p2p", choices=["p2p", "nccl"],
                    help="several GPUs: p2p = fused kernels read peer memory over NVLink (default); nccl = the same engine "
                         "with ncclSend/ncclRecv of every model into a staging row (the NCCL-only baseline)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-tf32", action="store_true", help="skip the secondary plain-tf32 measurement")
    ap.add_argument("--curve", action="store_true", help="(kept for compatibility: the curve is always printed)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed rounds, write what the last one computed (every node's model, the round's "
                         "evaluation) to DIR/<name>.npy, to compare two builds output for output")
    return ap.parse_args()


# --------------------------------------------------------------------------------------------
# helpers shared by both arms (data generation and clocks only -- no framework code)
# --------------------------------------------------------------------------------------------
def make_data(seed: int = 0):
    import torch
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(N_TRAIN + N_TEST, D_IN, generator=g)
    teacher = torch.randn(D_IN, D_OUT, generator=g) / D_IN ** 0.5
    y = (X @ teacher + 0.3 * torch.randn(N_TRAIN + N_TEST, D_OUT, generator=g)).argmax(1)
    return X[:N_TRAIN], y[:N_TRAIN], X[N_TRAIN:], y[N_TRAIN:]


def make_split(y, n_nodes: int = N_NODES, shards_per_client: int = 2, seed: int = 42):
    """McMahan's pathological non-IID split, computed HERE (NumPy only) so that both arms train on identical shards:
    samples sorted by label, cut into n_nodes * shards_per_client contiguous shards, shards dealt to the nodes at
    random.  (Each framework's own AssignmentHandler draws from a different random stream: with only 16 shards of 10
    classes the particular deal moves the accuracy curve by several points, which is not what a comparison of the two
    implementations should measure.)"""
    import numpy as np
    yy = np.asarray(y)
    order = np.argsort(yy, kind="stable")
    shards = np.array_split(order, n_nodes * shards_per_client)
    deal = np.random.RandomState(seed).permutation(len(shards))
    return [np.sort(np.concatenate([shards[k] for k in deal[i * shards_per_client:(i + 1) * shards_per_client]]))
            for i in range(n_nodes)]


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int = 0):
        self.gpu_index = gpu_index
        self.rows = []
        self._stop = threading.Event()
        self._thr = None

    def _loop(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu_index),
                                      "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._thr = threading.Thread(target=self._loop, daemon=True)
        self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thr.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


def dist_setup(n_gpus: int):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if torch.cuda.is_available():
        torch.cuda.set_device(local % max(1, torch.cuda.device_count()))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl" if torch.cuda.is_available() else "gloo")
    return rank, world, local


def max_over_ranks(value: float, world: int) -> float:
    if world == 1:
        return value
    import torch
    import torch.distributed as dist
    t = torch.tensor([value], dtype=torch.float64,
                     device="cuda" if torch.cuda.is_available() else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(value: float, world: int) -> float:
    if world == 1:
        return value
    import torch
    import torch.distributed as dist
    t = torch.tensor([value], dtype=torch.float64,
                     device="cuda" if torch.cuda.is_available() else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


def barrier(world: int):
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    if torch.cuda.is_available():
        torch.cuda.synchronize()


# --------------------------------------------------------------------------------------------
# this framework
# --------------------------------------------------------------------------------------------
def build_native(world: int, rank: int, train_impl: str, engine: str = "native", executor: str = "python", transport: str = "p2p"):
    import torch
    import gossipy_b200 as g
    from gossipy_b200.core import AntiEntropyProtocol, CreateModelMode, StaticP2PNetwork
    from gossipy_b200.data import AssignmentHandler, DataDispatcher
    from gossipy_b200.data.handler import ClassificationDataHandler
    from gossipy_b200.model.handler import TorchModelHandler
    from gossipy_b200.model.nn import TorchMLP
    from gossipy_b200.node import GossipNode
    from gossipy_b200.simul import GossipSimulator, SimulationReport
    from gossipy_b200 import ops

    dev = "cuda:%d" % torch.cuda.current_device() if torch.cuda.is_available() else "cpu"
    g.GlobalSettings().set_device(dev)
    if world > 1:
        from gossipy_b200.parallel import runtime as prt
        prt.init(rank, world, transport=transport)
    g.set_seed(98765)
    Xtr, ytr, Xte, yte = make_data()
    dh = ClassificationDataHandler(Xtr, ytr, Xte, yte)
    disp = DataDispatcher(dh, n=N_NODES, eval_on_user=False, auto_assign=False)
    disp.set_assignments(make_split(ytr), None)
    ops.set_train_impl(train_impl or "")
    proto = TorchModelHandler(net=TorchMLP(D_IN, D_OUT, (D_H,)), optimizer=torch.optim.SGD,
                              optimizer_params={"lr": LR}, criterion=torch.nn.CrossEntropyLoss(),
                              local_epochs=1, batch_size=BATCH,
                              create_model_mode=CreateModelMode.MERGE_UPDATE)
    nodes = GossipNode.generate(disp, StaticP2PNetwork(N_NODES), proto, round_len=DELTA, sync=True)
    sim = GossipSimulator(nodes, disp, DELTA, AntiEntropyProtocol.PUSH_PULL)
    sim.progress = False
    sim.engine = engine          # "native": C++ scheduler (csrc/sched) drives the round loop
    sim.native_executor = executor == "native"   # ... and the C++ executor (csrc/exec) enqueues it (one rank)
    rep = SimulationReport()
    sim.add_receiver(rep)
    if torch.cuda.is_available():
        sim.add_receiver(L2Flusher())
    sim.init_nodes(seed=42)
    return sim, rep


class L2Flusher:
    """Once per round (between timed iterations) overwrite a buffer larger than the 126 MB L2, so no
    round finds its inputs cached by the previous one -- matters at N=8 where a GPU holds one 23.5 MB
    shard + the 31 MB test set.  Runs on the current stream inside the timed region."""

    def __init__(self):
        import torch
        self.buf = torch.empty(192 << 20, dtype=torch.uint8, device="cuda")

    def update_message(self, failed, msg=None): pass
    def update_timestep(self, t): pass
    def update_end(self): pass

    def update_evaluation(self, round, on_user, evaluation):
        self.buf.zero_()


def time_rounds(sim, rounds: int, world: int, resume: bool = True):
    """Device time (CUDA events on the current stream, all node streams joined) of ``rounds``."""
    import torch
    from gossipy_b200.engine import arena
    barrier(world)
    if not torch.cuda.is_available():
        t0 = time.perf_counter()
        sim.start(rounds, resume=resume)
        return (time.perf_counter() - t0) * 1e3
    dev = torch.device("cuda", torch.cuda.current_device())
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    arena.fork_from_current(dev)          # node streams start after `start`
    sim.start(rounds, resume=resume)
    arena.sync_all_streams(dev)           # ... and `stop` waits for all of them
    from gossipy_b200.model.handler import join_copy_streams
    join_copy_streams(dev)                # ... and for the input prefetch issued in the last round
    stop.record()
    barrier(world)
    return start.elapsed_time(stop)


def dump_outputs(sim, rep, out_dir: str, rank: int, world: int):
    """What the timed rounds hand back to a caller, as of the last one: every node's model (its parameters, flattened
    in module order; with several GPUs each rank writes the nodes it holds) and that round's evaluation (mean over
    the nodes)."""
    import numpy as np
    import torch
    from gossipy_b200.parallel import runtime as prt
    os.makedirs(out_dir, exist_ok=True)
    ids = [i for i in sorted(sim.nodes) if world == 1 or prt.is_mine(i)]
    rows = torch.stack([torch.cat([p.detach().reshape(-1) for p in sim.nodes[i].model_handler.model.parameters()])
                        for i in ids]).float().cpu()
    np.save(os.path.join(out_dir, "models%s.npy" % ("" if world == 1 else "_rank%d" % rank)), rows.numpy())
    if rank == 0:
        for name, v in rep.get_evaluation(False)[-1][1].items():
            np.save(os.path.join(out_dir, "eval_%s.npy" % name), np.array([float(v)], dtype=np.float64))


def run_native(args, rank, world):
    import torch
    from gossipy_b200 import ops
    K = args.steps if args.steps is not None else 100
    W = args.warmup if args.warmup is not None else 3
    W = max(W, 3)
    sim, rep = build_native(world, rank, args.train_impl, args.engine, args.executor, args.transport)
    time_rounds(sim, W, world, resume=False)
    launches0 = ops.launch_count
    with ClockSampler(torch.cuda.current_device() if torch.cuda.is_available() else 0) as clk:
        ms = time_rounds(sim, K, world)
    if args.dump_outputs:
        dump_outputs(sim, rep, args.dump_outputs, rank, world)
    launches = int(sum_over_ranks(ops.launch_count - launches0, world))
    ms = max_over_ranks(ms, world)
    value = K / (ms / 1e3)
    acc = [round(e["accuracy"], 4) for _, e in rep.get_evaluation(False)]

    e2e = None
    if not args.no_e2e:
        sim.stream_inputs = True       # re-upload every node's shard from pinned host memory per round
        time_rounds(sim, 1, world)     # allocate pinned staging outside the timed region
        ms_e = max_over_ranks(time_rounds(sim, K, world), world)
        sim.stream_inputs = False
        h2d = sum(int(n.data[0][0].numel()) * 4 + int(n.data[0][1].numel()) * 8 for n in sim.nodes.values())
        e2e = {"value": K / (ms_e / 1e3), "unit": "rounds/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": N_NODES * D_OUT * D_OUT * 4, "ms_per_step": ms_e / K}
    dtype = ops.train_dtype() if torch.cuda.is_available() else \
        "fp32 (no GPU: the PyTorch reference implementations of the fused operations, ops/torch_ref.py)"
    n_main = len(acc)
    tf32 = None
    if not args.no_tf32 and torch.cuda.is_available() and ops.TRAIN_IMPL in ("", "tc8"):
        # secondary number: the same rounds with plain tf32 tensor-core products (GlobalSettings().allow_tf32)
        import gossipy_b200 as g
        g.GlobalSettings().allow_tf32 = True
        K2 = max(10, K // 4)
        time_rounds(sim, 2, world)
        ms_t = max_over_ranks(time_rounds(sim, K2, world), world)
        g.GlobalSettings().allow_tf32 = False
        ops.set_train_impl(args.train_impl or "")
        tf32 = {"value": K2 / (ms_t / 1e3), "unit": "rounds/s", "steps": K2,
                "dtype": "tf32 (operands truncated to 10 mantissa bits; NOT the headline: below the reference's fp32)"}
    if rank == 0:
        out = {"metric": METRIC,
               "value": value, "unit": "rounds/s", "n_gpus": world, "steps": K, "warmup": W,
               "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong",
               "vs_baseline": value / BASELINE_ROUNDS_PER_S, "dtype": dtype,
               "data": "synthetic", "impl": "native", "config": common_config(world),
               "details": {"l2_flush": "192 MB buffer rewritten every round inside the timed region",
                           "placement": "block (node i on rank i*N//8), peer rows pulled over NVLink by the fused merge+train kernel",
                           "train_kernel": args.train_impl or "auto (tc8: 3xTF32 tcgen05, 8-CTA cluster)",
                           "engine": args.engine, "transport": args.transport if world > 1 else "none",
                           "executor": ("c++ (csrc/exec)" if "_stream_exec" in sim.__dict__ else "python (per event)")},
               "clocks": clk.summary(), "gpu_launches": launches,
               "test_acc_by_round_tail": acc[n_main - 5:n_main], "test_acc_by_round": acc[:n_main], "e2e": e2e,
               "tf32": tf32}
        print(json.dumps(out))


# --------------------------------------------------------------------------------------------
# the unmodified reference (baseline/_ref), stock code path, device = cuda
# --------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    import types
    import numpy as np
    K = args.steps if args.steps is not None else 3
    W = args.warmup if args.warmup is not None else 3
    W = max(W, 3)
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "gossipy")):
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref/gossipy not installed "
                              "(run baseline/install_reference.sh)"}))
        return
    # environment shims for modules missing in this image (not modifications of the reference)
    for name in ("matplotlib", "matplotlib.pyplot", "pyparsing"):
        try:
            __import__(name)
        except Exception:
            m = types.ModuleType(name)
            if name == "pyparsing":
                m.ParseSyntaxException = Exception
            sys.modules[name] = m
    if not hasattr(sys.modules["matplotlib"], "pyplot"):
        sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.path.insert(0, ref_dir)
    import torch
    try:
        import gossipy
        from gossipy import GlobalSettings, set_seed
        from gossipy.core import AntiEntropyProtocol, CreateModelMode, StaticP2PNetwork
        from gossipy.data import AssignmentHandler, DataDispatcher
        from gossipy.data.handler import ClassificationDataHandler
        from gossipy.model.handler import TorchModelHandler
        from gossipy.model.nn import TorchMLP
        from gossipy.node import GossipNode
        from gossipy.simul import GossipSimulator, SimulationReport
        import gossipy.simul as S
    except Exception as exc:  # noqa: BLE001
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": "import failed: %r" % (exc,)}))
        return

    class _It:
        def __init__(self, it): self.it = it
        def __iter__(self): return iter(self.it)
        def close(self): pass
    S.track = lambda it, description="": _It(it)      # silence the progress bar only
    gossipy.LOG.setLevel(50)

    ms = 0.0
    acc = []
    clocks = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    if rank == 0:   # the reference is single-process / single-device: extra ranks only wait
        GlobalSettings().set_device("cuda" if torch.cuda.is_available() else "cpu")
        set_seed(98765)
        Xtr, ytr, Xte, yte = make_data()
        dh = ClassificationDataHandler(Xtr, ytr, Xte, yte)
        disp = DataDispatcher(dh, n=N_NODES, eval_on_user=False, auto_assign=False)
        disp.set_assignments(make_split(ytr), None)
        proto = TorchModelHandler(net=TorchMLP(D_IN, D_OUT, (D_H,)), optimizer=torch.optim.SGD,
                                  optimizer_params={"lr": LR}, criterion=torch.nn.CrossEntropyLoss(),
                                  local_epochs=1, batch_size=BATCH,
                                  create_model_mode=CreateModelMode.MERGE_UPDATE)
        nodes = GossipNode.generate(data_dispatcher=disp, p2p_net=StaticP2PNetwork(N_NODES),
                                    model_proto=proto, round_len=DELTA, sync=True)
        sim = GossipSimulator(nodes=nodes, data_dispatcher=disp, delta=DELTA,
                              protocol=AntiEntropyProtocol.PUSH_PULL)
        rep = SimulationReport()
        sim.add_receiver(rep)
        sim.init_nodes(seed=42)
        sim.start(n_rounds=W)
        cuda = torch.cuda.is_available()
        if cuda:
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(torch.cuda.current_device() if cuda else 0) as clk:
            t0 = time.perf_counter()
            if cuda:
                ev0.record()
            sim.start(n_rounds=K)
            if cuda:
                ev1.record()
                torch.cuda.synchronize()
                ms = ev0.elapsed_time(ev1)
            else:
                ms = (time.perf_counter() - t0) * 1e3
        clocks = clk.summary()
        acc = [round(float(e["accuracy"]), 4) for _, e in rep.get_evaluation(False)]
        gossipy.CACHE.clear()
    barrier(world)
    ms = max_over_ranks(ms, world)
    if rank == 0:
        value = K / (ms / 1e3)
        steps_round = 16 * ((N_TRAIN // N_NODES + BATCH - 1) // BATCH)
        p_bytes = (D_H * D_IN + D_H + D_OUT * D_H + D_OUT) * 4
        h2d = steps_round * (BATCH * D_IN * 4 + BATCH * 8) + 16 * p_bytes + 8 * (N_TEST * D_IN * 4 + p_bytes)
        d2h = 16 * p_bytes + 8 * (p_bytes + N_TEST * 8 * 2)
        print(json.dumps({
            "metric": METRIC,
            "value": value, "unit": "rounds/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": value / BASELINE_ROUNDS_PER_S, "dtype": "fp32", "data": "synthetic",
            "impl": "reference",
            "config": common_config(world),
            "details": {"parallelism": "single process, single device (the reference has no multi-GPU mode; ranks > 0 idle)"},
            "clocks": clocks, "gpu_launches": 0, "test_acc_by_round_tail": acc[-5:], "test_acc_by_round": acc,
            "e2e": {"value": value, "unit": "rounds/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "note": "the reference's stock path already moves every mini-batch and the model "
                            "host<->device inside the timed region"}}))


def main():
    args = parse()
    if args.dump_outputs and args.impl != "native":
        sys.exit("--dump-outputs writes the outputs of this framework's rounds (--impl native)")
    rank, world, _ = dist_setup(args.gpus)
    try:
        if args.impl == "reference":
            run_reference(args, rank, world)
        else:
            run_native(args, rank, world)
    finally:
        if world > 1:
            import torch.distributed as dist
            if dist.is_initialized():
                dist.destroy_process_group()


if __name__ == "__main__":
    main()
