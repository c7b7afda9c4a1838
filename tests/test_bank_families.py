"""The banked engine for k-means (KMeansBank) and matrix factorisation (MFBank): same native schedule, same results as
the per-event executor; checkpoints resume exactly; set-ups outside its scope fall back with a reason."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

from gossipy_b200.ops.native import native_available

pytestmark = pytest.mark.skipif(not native_available(), reason="extension not built")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cuda():
    return torch.cuda.is_available()


# ---------------------------------------------------------------------------------------------
# set-ups
# ---------------------------------------------------------------------------------------------
def _kmeans_sim(batched, protocol, mode, matching="naive", n=60, rounds=5, device="cpu", k=3, dim=6, faults=True,
                node_cls=None, mixed=False, start=True):
    import gossipy_b200 as g
    from gossipy_b200.core import AntiEntropyProtocol, CreateModelMode, StaticP2PNetwork, UniformDelay
    from gossipy_b200.data import DataDispatcher
    from gossipy_b200.data.handler import ClusteringDataHandler
    from gossipy_b200.model.handler import KMeansHandler
    from gossipy_b200.node import GossipNode
    from gossipy_b200.simul import GossipSimulator, SimulationReport
    g.GlobalSettings().set_device(device)
    g.CACHE.clear()
    g.set_seed(11)
    sizes = [1 + i % 3 for i in range(n)]                 # 1 to 3 samples per node: the last-sample-wins rule matters
    rng = np.random.default_rng(4)
    centers = rng.normal(size=(3, dim)) * 3
    y = rng.integers(0, 3, size=sum(sizes))
    X = (centers[y] + rng.normal(size=(len(y), dim))).astype(np.float32)
    disp = DataDispatcher(ClusteringDataHandler(torch.tensor(X), torch.tensor(y)), n=n, eval_on_user=False,
                          auto_assign=False)
    bounds = np.cumsum([0] + sizes)
    disp.set_assignments([np.arange(bounds[i], bounds[i + 1]) for i in range(n)], None)
    proto = KMeansHandler(k=k, dim=dim, alpha=.1, matching=matching, create_model_mode=getattr(CreateModelMode, mode))
    nodes = (node_cls or GossipNode).generate(disp, StaticP2PNetwork(n), proto, 10, True)
    if mixed:
        nodes[1].model_handler.alpha = .2
    kw = dict(drop_prob=.1, online_prob=.8, delay=UniformDelay(0, 3), sampling_eval=.2) if faults else {}
    sim = GossipSimulator(nodes, disp, 10, getattr(AntiEntropyProtocol, protocol), **kw)
    sim.progress = False
    sim.engine = "native"
    sim.batched = batched
    rep = SimulationReport(); sim.add_receiver(rep)
    sim.init_nodes(seed=9)
    if start:
        sim.start(rounds)
    return rep, sim


def _mf_sim(batched, protocol, mode, n=40, n_items=50, k=3, per_user=8, rounds=5, device="cpu", start=True):
    import gossipy_b200 as g
    from gossipy_b200.core import AntiEntropyProtocol, CreateModelMode, StaticP2PNetwork, UniformDelay
    from gossipy_b200.data import RecSysDataDispatcher
    from gossipy_b200.data.handler import RecSysDataHandler
    from gossipy_b200.model.handler import MFModelHandler
    from gossipy_b200.node import GossipNode
    from gossipy_b200.simul import GossipSimulator, SimulationReport
    g.GlobalSettings().set_device(device)
    g.CACHE.clear()
    g.set_seed(12)
    rng = np.random.default_rng(5)
    ratings = {u: [(int(i), float(rng.integers(1, 6))) for i in rng.choice(n_items, per_user, replace=False)]
               for u in range(n)}
    disp = RecSysDataDispatcher(RecSysDataHandler(ratings, n, n_items, test_size=.25, seed=42))
    proto = MFModelHandler(dim=k, n_items=n_items, lam_reg=.1, learning_rate=.05,
                           create_model_mode=getattr(CreateModelMode, mode))
    nodes = GossipNode.generate(disp, StaticP2PNetwork(n), proto, 10, True)
    sim = GossipSimulator(nodes, disp, 10, getattr(AntiEntropyProtocol, protocol), delay=UniformDelay(0, 3),
                          sampling_eval=.25)
    sim.progress = False
    sim.engine = "native"
    sim.batched = batched
    rep = SimulationReport(); sim.add_receiver(rep)
    sim.init_nodes(seed=9)
    if start:
        sim.start(rounds)
    return rep, sim


def _state(sim):
    n = len(sim.nodes)
    rows = torch.stack([sim.nodes[i].model_handler.row.detach().cpu().clone() for i in range(n)])
    ages = [int(sim.nodes[i].model_handler.n_updates) for i in range(n)]
    return rows, ages


def _counters(rep):
    return rep._sent_messages, rep._failed_messages, rep._total_size


def _compare(rep_a, sim_a, rep_b, sim_b, rtol, atol, metric, metric_tol, on_user):
    assert "_bank" not in sim_a.__dict__ and "_bank" in sim_b.__dict__
    assert _counters(rep_a) == _counters(rep_b)
    rows_a, ages_a = _state(sim_a)
    rows_b, ages_b = _state(sim_b)
    assert ages_a == ages_b
    torch.testing.assert_close(rows_a, rows_b, rtol=rtol, atol=atol)
    ev_a, ev_b = rep_a.get_evaluation(on_user), rep_b.get_evaluation(on_user)
    assert rep_a.get_evaluation(not on_user) == [] and rep_b.get_evaluation(not on_user) == []
    assert len(ev_a) == len(ev_b) > 0
    for (t1, m1), (t2, m2) in zip(ev_a, ev_b):
        assert t1 == t2
        if metric_tol[0] == "abs":
            assert m1[metric] == pytest.approx(m2[metric], abs=metric_tol[1])
        else:
            assert m1[metric] == pytest.approx(m2[metric], rel=metric_tol[1])


KMEANS_CASES = [("PUSH", "MERGE_UPDATE", "hungarian"), ("PUSH_PULL", "UPDATE_MERGE", "naive"),
                ("PULL", "UPDATE", "hungarian"), ("PUSH", "PASS", "naive")]
MF_CASES = [("PUSH", "MERGE_UPDATE"), ("PUSH_PULL", "UPDATE"), ("PULL", "UPDATE_MERGE")]


# ---------------------------------------------------------------------------------------------
# CPU: the bank's vectorised torch path against the per-event executor
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("protocol,mode,matching", KMEANS_CASES)
def test_kmeans_banked_equals_per_event(protocol, mode, matching):
    import gossipy_b200 as g
    rep_a, sim_a = _kmeans_sim(False, protocol, mode, matching)
    rep_b, sim_b = _kmeans_sim(True, protocol, mode, matching)
    _compare(rep_a, sim_a, rep_b, sim_b, 1e-4, 1e-5, "nmi", ("abs", 1e-4), on_user=False)
    g.CACHE.clear()


@pytest.mark.parametrize("protocol,mode", MF_CASES)
def test_mf_banked_equals_per_event(protocol, mode):
    import gossipy_b200 as g
    rep_a, sim_a = _mf_sim(False, protocol, mode)
    rep_b, sim_b = _mf_sim(True, protocol, mode)
    _compare(rep_a, sim_a, rep_b, sim_b, 1e-4, 1e-5, "rmse", ("rel", 1e-5), on_user=True)
    g.CACHE.clear()


def test_mf_wide_rows_banked_equals_per_event():
    """ml-1m's item count: rows of 3 706 x 5 + 3 706 + 6 floats, far wider than the warp-per-item kernels cover."""
    import gossipy_b200 as g
    rep_a, sim_a = _mf_sim(False, "PUSH", "MERGE_UPDATE", n=6, n_items=3706, k=5, per_user=12, rounds=3)
    rep_b, sim_b = _mf_sim(True, "PUSH", "MERGE_UPDATE", n=6, n_items=3706, k=5, per_user=12, rounds=3)
    assert sim_b._bank.Dp > 1024
    _compare(rep_a, sim_a, rep_b, sim_b, 1e-4, 1e-5, "rmse", ("rel", 1e-5), on_user=True)
    g.CACHE.clear()


def test_family_banks_size_the_first_slot_pool_by_row_width():
    import gossipy_b200 as g
    from gossipy_b200.engine.bank import _SLOT_BYTES
    _, sim = _mf_sim(True, "PUSH", "MERGE_UPDATE", n=6, n_items=3706, k=5, per_user=12, rounds=1)
    bank = sim._bank
    assert bank.S.shape[1] == bank.Dp and bank.cap * bank.Dp * 4 <= max(_SLOT_BYTES, 64 * bank.Dp * 4)
    g.CACHE.clear()


@pytest.mark.parametrize("family", ["kmeans", "mf"])
def test_family_checkpoint_resume_is_exact(family, tmp_path):
    import gossipy_b200 as g
    from gossipy_b200.simul import GossipSimulator
    make = (lambda r: _kmeans_sim(True, "PUSH_PULL", "MERGE_UPDATE", "hungarian", rounds=r)) if family == "kmeans" else \
        (lambda r: _mf_sim(True, "PUSH", "MERGE_UPDATE", rounds=r))
    rep_full, sim_full = make(6)
    rows_full, ages_full = _state(sim_full)
    g.CACHE.clear()
    _, sim = make(3)
    assert sim._scheduler.pending > 0              # delays up to 3 ticks: messages are on the wire at the cut
    path = str(tmp_path / "ckpt.pkl")
    sim.save(path)
    g.CACHE.clear()
    del sim
    sim2 = GossipSimulator.load(path)
    rep_b = [r for r in sim2._receivers if type(r).__name__ == "SimulationReport"][0]
    sim2.start(3, resume=True)
    assert "_bank" in sim2.__dict__
    rows, ages = _state(sim2)
    assert ages == ages_full
    torch.testing.assert_close(rows, rows_full, rtol=0, atol=1e-6)
    assert _counters(rep_b) == _counters(rep_full)
    g.CACHE.clear()


@pytest.mark.parametrize("variant", ["hungarian_k9", "mixed", "passthrough"])
def test_bankable_declines_with_a_reason_and_per_event_runs(variant):
    import gossipy_b200 as g
    from gossipy_b200.engine.bank import bankable
    from gossipy_b200.node import PassThroughNode
    kw = {"hungarian_k9": dict(matching="hungarian", k=9), "mixed": dict(mixed=True),
          "passthrough": dict(node_cls=PassThroughNode)}[variant]
    rep, sim = _kmeans_sim(True, "PUSH", "MERGE_UPDATE", rounds=2, n=20, start=False, **kw)
    why = bankable(sim)
    assert isinstance(why, str) and why
    sim.start(2)
    assert "_bank" not in sim.__dict__
    assert rep._sent_messages > 0 and len(rep.get_evaluation(False)) == 2
    g.CACHE.clear()


def _run_example(script, batched, nodes):
    env = dict(os.environ, GOSSIPY_ENGINE="native", GOSSIPY_BATCHED=batched, GOSSIPY_NODES=str(nodes),
               GOSSIPY_ROUNDS="3", GOSSIPY_DEVICE="cpu", PYTHONPATH=ROOT)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "examples", script)], env=env, capture_output=True,
                         text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("last evaluation")]
    assert lines, out.stdout
    return lines[-1]


@pytest.mark.parametrize("script,nodes", [("main_berta_2014.py", 300), ("main_hegedus_2020.py", 40)])
def test_examples_print_the_same_last_evaluation_banked_and_per_event(script, nodes):
    assert _run_example(script, "1", nodes) == _run_example(script, "0", nodes)


# ---------------------------------------------------------------------------------------------
# the kernels are in the binary (SASS census, no GPU needed)
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def census():
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import sass_census
    k = sass_census.census()
    if k is None:
        pytest.skip("extension not built")
    return k


def test_family_bank_kernels_are_in_the_binary(census):
    names = " ".join(census)
    for fam in ("bank_snapshot_wide_kernel", "kmeans_bank_deliver_kernel", "kmeans_bank_eval_kernel",
                "mf_bank_deliver_kernel", "mf_bank_eval_kernel"):
        assert fam in names, fam


# ---------------------------------------------------------------------------------------------
# GPU: the bank kernels against the per-event kernels
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.skipif(not _cuda(), reason="needs a GPU")
@pytest.mark.parametrize("protocol,mode,matching", KMEANS_CASES)
def test_kmeans_bank_kernels_equal_per_event_kernels(protocol, mode, matching):
    import gossipy_b200 as g
    try:
        rep_a, sim_a = _kmeans_sim(False, protocol, mode, matching, device="cuda:0")
        rep_b, sim_b = _kmeans_sim(True, protocol, mode, matching, device="cuda:0")
        _compare(rep_a, sim_a, rep_b, sim_b, 1e-3, 1e-4, "nmi", ("abs", 2e-2), on_user=False)
    finally:
        g.GlobalSettings().set_device("cpu")
        g.CACHE.clear()


@pytest.mark.gpu
@pytest.mark.skipif(not _cuda(), reason="needs a GPU")
@pytest.mark.parametrize("protocol,mode,wide", [c + (False,) for c in MF_CASES] + [("PUSH", "MERGE_UPDATE", True)])
def test_mf_bank_kernels_equal_per_event_kernels(protocol, mode, wide):
    import gossipy_b200 as g
    kw = dict(n=6, n_items=3706, k=5, per_user=12, rounds=3) if wide else {}
    try:
        rep_a, sim_a = _mf_sim(False, protocol, mode, device="cuda:0", **kw)
        rep_b, sim_b = _mf_sim(True, protocol, mode, device="cuda:0", **kw)
        assert (sim_b._bank.Dp > 1024) == wide
        _compare(rep_a, sim_a, rep_b, sim_b, 1e-3, 1e-4, "rmse", ("rel", 1e-3), on_user=True)
    finally:
        g.GlobalSettings().set_device("cpu")
        g.CACHE.clear()


@pytest.mark.gpu
@pytest.mark.skipif(not _cuda(), reason="needs a GPU")
def test_mf_bank_launch_count_does_not_follow_the_node_count():
    import gossipy_b200 as g
    from gossipy_b200 import ops
    per_round = {}
    try:
        for n in (40, 80):
            _, sim = _mf_sim(True, "PUSH", "MERGE_UPDATE", n=n, rounds=1, device="cuda:0")
            c0 = ops.launch_count
            sim.start(4)
            per_round[n] = (ops.launch_count - c0) / 4
            assert "_bank" in sim.__dict__
            g.CACHE.clear()
    finally:
        g.GlobalSettings().set_device("cpu")
        g.CACHE.clear()
    assert per_round[80] < 1.5 * per_round[40], per_round
