#!/usr/bin/env python
"""The banked engine against the per-event executor for the k-means and matrix-factorisation experiments, at the
reference scripts' full size by default:

* ``--model kmeans``: main_berta_2014 -- 4 601 nodes (one spambase-shaped sample each), k = 2 centroids of 57 floats,
  "hungarian" matching, MERGE_UPDATE, round_len = delta = 1000, PUSH, drop .1, 1 % of the nodes evaluated per round;
* ``--model mf``: main_hegedus_2020 -- the synthetic ml-1m shape (6 040 users, 3 706 items, ~165 ratings each), rank 5,
  MERGE_UPDATE, a 20-regular graph, round_len = delta = 100, PUSH, UniformDelay(0, 10), 10 % evaluated per round.

Both implementations run the native scheduler on the same seed: ``--impl banked`` executes a round with one launch
per phase of a tick (``engine/bank.py``), ``--impl events`` node by node.  Prints one JSON line (rounds/s and ms per
round from device events after the warm-up rounds, kernel launches per round, the GPU's name and power limit) and
writes the final rows, ages and last-round metrics under ``--out`` as .npy files; ``--check DIR`` compares them with
another run's outputs.

    python benchmarks/bank_families.py --model kmeans|mf --impl banked|events [--nodes N] [--rounds R] --out DIR
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))


def build(a):
    import gossipy_b200 as g
    from gossipy_b200.core import AntiEntropyProtocol, CreateModelMode, StaticP2PNetwork, UniformDelay
    from gossipy_b200.node import GossipNode
    from gossipy_b200.simul import GossipSimulator
    g.set_seed(98765)
    if a.model == "kmeans":
        from gossipy_b200.data import DataDispatcher, load_classification_dataset
        from gossipy_b200.data.handler import ClusteringDataHandler
        from gossipy_b200.model.handler import KMeansHandler
        X, y = load_classification_dataset("spambase", as_tensor=True, synthetic_fallback=True)
        n = min(a.nodes or X.shape[0], X.shape[0])
        dh = ClusteringDataHandler(X[:n], y[:n])
        disp = DataDispatcher(dh, eval_on_user=False, auto_assign=True)
        proto = KMeansHandler(k=2, dim=dh.size(1), alpha=.1, matching="hungarian",
                              create_model_mode=CreateModelMode.MERGE_UPDATE)
        nodes = GossipNode.generate(data_dispatcher=disp, p2p_net=StaticP2PNetwork(disp.size(), None),
                                    model_proto=proto, round_len=1000, sync=True)
        sim = GossipSimulator(nodes=nodes, data_dispatcher=disp, delta=1000, protocol=AntiEntropyProtocol.PUSH,
                              drop_prob=.1, sampling_eval=.01)
    else:
        from _common import regular_graph
        from gossipy_b200.data import RecSysDataDispatcher, synthetic
        from gossipy_b200.data.handler import RecSysDataHandler
        from gossipy_b200.model.handler import MFModelHandler
        ratings, n_users, n_items = synthetic.ratings_like("ml-1m")
        n = min(a.nodes or n_users, n_users)
        ratings = {u: r for u, r in ratings.items() if u < n}
        disp = RecSysDataDispatcher(RecSysDataHandler(ratings, n, n_items, test_size=.1, seed=42))
        topo = StaticP2PNetwork(n, regular_graph(n, min(20, n - 1 - (n - 1) % 2)))
        proto = MFModelHandler(dim=5, n_items=n_items, lam_reg=.1, learning_rate=.001,
                               create_model_mode=CreateModelMode.MERGE_UPDATE)
        nodes = GossipNode.generate(data_dispatcher=disp, p2p_net=topo, model_proto=proto, round_len=100, sync=True)
        sim = GossipSimulator(nodes=nodes, data_dispatcher=disp, delta=100, protocol=AntiEntropyProtocol.PUSH,
                              delay=UniformDelay(0, 10), sampling_eval=.1)
    sim.progress = False
    sim.engine = "native"
    sim.batched = a.impl == "banked"
    return sim


def gpu_info(device):
    if device.type != "cuda":
        return {"gpu": "none (CPU rehearsal)", "power_limit_w": None}
    info = {"gpu": torch.cuda.get_device_name(device), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits",
                              "-i", str(device.index or 0)], capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(out.stdout.strip().splitlines()[0])
    except Exception:
        pass
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", choices=["kmeans", "mf"], required=True)
    ap.add_argument("--impl", choices=["banked", "events"], required=True)
    ap.add_argument("--nodes", type=int, default=0, help="cap on the number of nodes (0: the full data set)")
    ap.add_argument("--rounds", type=int, default=5, help="timed rounds")
    ap.add_argument("--warmup", type=int, default=1, help="rounds before the timed window")
    ap.add_argument("--device", default="cuda:0", help="a CUDA device (cpu only to rehearse at a small size)")
    ap.add_argument("--out", required=True)
    ap.add_argument("--check", default="", help="directory with the other implementation's outputs to compare with")
    a = ap.parse_args()
    device = torch.device(a.device)
    if device.type == "cuda" and not torch.cuda.is_available():
        sys.exit("bank_families.py: no GPU (pass --device cpu to rehearse)")
    import gossipy_b200 as g
    from gossipy_b200 import ops
    from gossipy_b200.simul import SimulationReport
    g.LOG.setLevel(50)
    g.GlobalSettings().set_device(str(device))
    sim = build(a)
    rep = SimulationReport()
    sim.add_receiver(rep)
    t0 = time.perf_counter()
    sim.init_nodes(seed=42)
    sim.start(n_rounds=a.warmup)
    init_s = time.perf_counter() - t0
    on_user = a.model == "mf"
    n_ev0 = len(rep.get_evaluation(on_user))
    cuda = device.type == "cuda"
    if cuda:
        torch.cuda.synchronize(device)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
    h0 = time.perf_counter()
    l0 = ops.launch_count
    sim.start(n_rounds=a.rounds, resume=True)
    launches = ops.launch_count - l0
    if cuda:
        torch.cuda.synchronize(device)          # every stream (the per-event path runs one per node)
        ev1.record()
        ev1.synchronize()
        secs = ev0.elapsed_time(ev1) / 1e3
    else:
        secs = time.perf_counter() - h0
    assert ("_bank" in sim.__dict__) == (a.impl == "banked"), "the banked engine did not take the run"
    ids = sorted(sim.nodes)
    rows = np.stack([sim.nodes[i].model_handler.row.detach().cpu().numpy() for i in ids]).astype(np.float32)
    ages = np.asarray([int(sim.nodes[i].model_handler.n_updates) for i in ids], dtype=np.int64)
    evs = rep.get_evaluation(on_user)
    metric = "rmse" if on_user else "nmi"
    last = evs[-1][0] if len(evs) > n_ev0 else None
    metrics = np.asarray([m[metric] for t, m in evs if t == last], dtype=np.float64)
    os.makedirs(a.out, exist_ok=True)
    np.save(os.path.join(a.out, "rows.npy"), rows)
    np.save(os.path.join(a.out, "ages.npy"), ages)
    np.save(os.path.join(a.out, "metrics.npy"), metrics)
    res = {"model": a.model, "impl": a.impl, "nodes": len(ids), "row_floats": int(rows.shape[1]),
           "timed_rounds": a.rounds, "warmup_rounds": a.warmup, "rounds_per_s": a.rounds / secs,
           "ms_per_round": 1e3 * secs / a.rounds, "launches_per_round": launches / a.rounds,
           "messages_sent": rep._sent_messages, "init_and_warmup_s": round(init_s, 2),
           "last_round_mean_%s" % metric: float(np.mean(metrics)) if metrics.size else None}
    res.update(gpu_info(device))
    if a.check:
        o_rows, o_ages, o_met = (np.load(os.path.join(a.check, f)) for f in ("rows.npy", "ages.npy", "metrics.npy"))
        res["check"] = {"ages_equal": bool(np.array_equal(o_ages, ages)),
                        "rows_max_abs_diff": float(np.max(np.abs(o_rows - rows))),
                        "metrics_max_abs_diff": float(np.max(np.abs(o_met - metrics))) if metrics.size else None,
                        "metrics_max_rel_diff": float(np.max(np.abs(o_met - metrics) / np.maximum(np.abs(o_met), 1e-12)))
                        if metrics.size else None}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
