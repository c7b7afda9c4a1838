"""Discrete-time gossip simulators and their observability layer.

Behavioural reference: ``gossipy/simul.py`` (cited per class).  The reference has three almost
identical copies of the timestep loop; here one engine (:meth:`GossipSimulator._run`) implements
the four phases of a tick and the variants override two hooks:

* ``_tick_node(i, t)``        what a node does when examined in phase A (fire / earn a token /
                              merge the cached neighbourhood and broadcast);
* ``_after_delivery(msg, reply, t)``  reaction to a delivered message (token accounts).

Ordering facts preserved from the reference (SURVEY §3.2): within a tick all sends (snapshots)
precede all deliveries; deliveries happen in queue order; replies after first-leg messages; a
delay-0 PUSH_PULL completes inside its tick; sent counters tick at send time for first-leg
messages and at delivery time for replies; the drop test is ``>=`` for sends and ``>`` for
replies.  The host loop never waits for the GPU: device work is enqueued on per-node streams and
only the per-round metrics (a few integers per node) are read back, once per round.
"""
from __future__ import annotations

import json
import pickle
from abc import ABC, abstractmethod
from collections import defaultdict
from copy import deepcopy
from typing import Any, Callable, DefaultDict, Dict, Iterable, List, Optional, Tuple

import numpy as np

from . import CACHE, LOG, CacheKey, GlobalSettings
from .core import (AntiEntropyProtocol, ConstantDelay, Delay, Message, MessageType, MixingMatrix,
                   StaticP2PNetwork, UniformMixing)
from .data import DataDispatcher
from .flow_control import TokenAccount
from .model.handler import ModelHandler, PendingEval
from .node import All2AllGossipNode, GossipNode, PENSNode
from .utils import StringEncoder
from .utils.profiling import nvtx_range

try:
    import dill as _pickler
except Exception:  # pragma: no cover
    _pickler = pickle

__all__ = ["SimulationEventReceiver", "SimulationEventSender", "SimulationReport",
           "GossipSimulator", "TokenizedGossipSimulator", "All2AllGossipSimulator"]


# --------------------------------------------------------------------------------------
# observers
# --------------------------------------------------------------------------------------
class SimulationEventReceiver(ABC):
    """Observer interface (ref ``simul.py:37-88``)."""

    @abstractmethod
    def update_message(self, failed: bool, msg: Optional[Message] = None) -> None: ...

    def update_evaluation(self, round: int, on_user: bool,
                          evaluation: List[Dict[str, float]]) -> None:
        pass

    @abstractmethod
    def update_end(self) -> None: ...

    @abstractmethod
    def update_timestep(self, t: int) -> None: ...


class SimulationEventSender(ABC):
    """Observable side.  FIX(B8): the receiver list is per instance, not class-wide."""

    @property
    def _receivers(self) -> List[SimulationEventReceiver]:
        lst = self.__dict__.get("_receiver_list")
        if lst is None:
            lst = self.__dict__["_receiver_list"] = []
        return lst

    def add_receiver(self, receiver: SimulationEventReceiver) -> None:
        if receiver not in self._receivers:
            self._receivers.append(receiver)

    def remove_receiver(self, receiver: SimulationEventReceiver) -> None:
        if receiver in self._receivers:
            self._receivers.remove(receiver)

    def notify_message(self, falied: bool, msg: Optional[Message] = None) -> None:
        for r in self._receivers:
            r.update_message(falied, msg)

    def notify_evaluation(self, round: int, on_user: bool,
                          evaluation: List[Dict[str, float]]) -> None:
        for r in self._receivers:
            r.update_evaluation(round, on_user, evaluation)

    def notify_timestep(self, t: int) -> None:
        for r in self._receivers:
            r.update_timestep(t)

    def notify_end(self) -> None:
        for r in self._receivers:
            r.update_end()


def _check_device_fault() -> None:
    """Bounded device-side waits (cross-GPU ``ready`` flags, all-reduce epochs) report a timeout in a per-device
    fault word instead of hanging the GPU; surface it where the host synchronises anyway."""
    if GlobalSettings().get_device().type != "cuda":
        return
    from .ops.native import native_available, native
    if not native_available():
        return
    bits = int(native().device_fault(True))
    if bits:
        raise RuntimeError("gossipy_b200: device fault word = %d (1: a wait for a peer's model timed out, 2: an "
                           "all-reduce epoch timed out, 4: handshake ticket shared by two launches, 8: a rank barrier of the "
                           "banked engine timed out, 16: a wait for the acknowledgements of a row's remote readers timed "
                           "out) -- results "
                           "of this round are invalid" % bits)


class SimulationReport(SimulationEventReceiver):
    """Message counters and per-round mean metrics (ref ``simul.py:180-270``)."""

    def __init__(self) -> None:
        self.clear()

    def clear(self) -> None:
        self._sent_messages = 0
        self._total_size = 0
        self._failed_messages = 0
        self._global_evaluations: List[Tuple[int, Dict[str, float]]] = []
        self._local_evaluations: List[Tuple[int, Dict[str, float]]] = []

    def update_message(self, failed: bool, msg: Optional[Message] = None) -> None:
        if failed:
            self._failed_messages += 1
            return
        assert msg is not None, "msg is not set"
        self._sent_messages += 1
        self._total_size += msg.get_size()

    def update_evaluation(self, round: int, on_user: bool,
                          evaluation: List[Dict[str, float]]) -> None:
        target = self._local_evaluations if on_user else self._global_evaluations
        target.append((round, self._collect_results(evaluation)))

    def update_end(self) -> None:
        LOG.info("# Sent messages: %d" % self._sent_messages)
        LOG.info("# Failed messages: %d" % self._failed_messages)
        LOG.info("Total size: %d" % self._total_size)

    @staticmethod
    def _collect_results(results: List[Dict[str, float]]) -> Dict[str, float]:
        if not results:
            return {}
        return {k: float(np.mean([r[k] for r in results])) for k in results[0]}

    def get_evaluation(self, local: bool = False) -> List[Tuple[int, Dict[str, float]]]:
        return self._local_evaluations if local else self._global_evaluations

    def update_timestep(self, t: int) -> None:
        pass


# --------------------------------------------------------------------------------------
# the engine
# --------------------------------------------------------------------------------------
def _model_key(msg: Optional[Message]) -> Optional[CacheKey]:
    if msg is not None and msg.value and isinstance(msg.value[0], CacheKey):
        return msg.value[0]
    return None


class GossipSimulator(SimulationEventSender):
    """Vanilla gossip learning simulator (ref ``simul.py:273-503``).

    Parameters as in the reference: ``nodes, data_dispatcher, delta, protocol, drop_prob=0,
    online_prob=1, delay=ConstantDelay(0), sampling_eval=0``.
    """

    def __init__(self, nodes: Dict[int, GossipNode], data_dispatcher: DataDispatcher, delta: int,
                 protocol: AntiEntropyProtocol, drop_prob: float = 0., online_prob: float = 1.,
                 delay: Delay = ConstantDelay(0), sampling_eval: float = 0.) -> None:
        assert 0 <= drop_prob <= 1, "drop_prob must be in the range [0,1]."
        assert 0 <= online_prob <= 1, "online_prob must be in the range [0,1]."
        assert 0 <= sampling_eval <= 1, "sampling_eval must be in the range [0,1]."
        self.data_dispatcher = data_dispatcher
        self.n_nodes = len(nodes)
        self.delta = delta
        self.protocol = protocol
        self.drop_prob = drop_prob
        self.online_prob = online_prob
        self.delay = delay
        self.sampling_eval = sampling_eval
        self.initialized = False
        self.nodes = nodes
        self.progress = True
        self.stream_inputs = False  # True: re-upload every node's shard from pinned memory each round
        self._clock = 0  # next tick to simulate (kept for checkpoint/resume)
        self._msg_queues: DefaultDict[int, List[Message]] = defaultdict(list)
        self._rep_queues: DefaultDict[int, List[Message]] = defaultdict(list)

    # -- set-up -------------------------------------------------------------------------------
    def init_nodes(self, seed: int = 98765) -> None:
        """Initialise every node's model (one local update each).

        FIX(B7): ``seed`` is honoured (the reference ignores it): it seeds the engine's
        counter-based RNG used for model init / shuffles, leaving the host RNG streams alone.
        """
        from .engine import rng as _rng
        if seed is not None:
            _rng.set_base_seed(seed)
        self.initialized = True
        from .parallel import runtime as _prt
        if _prt.active():
            _prt.set_num_nodes(self.n_nodes)
        for node in self.nodes.values():
            node.init_model()
        self._prime_device_paths()

    def _prime_device_paths(self) -> None:
        """Run every node's evaluation once, before any cross-GPU dependency exists, and discard the
        result: first-use costs (pre-tiling of the test set, scratch buffers, allocator growth --
        ``cudaMalloc`` is an implicit device-wide barrier) are paid here instead of in the middle of
        round 1, when kernels of other nodes may be waiting on flags of other GPUs."""
        if GlobalSettings().get_device().type != "cuda":
            return
        try:
            eval_set = self.data_dispatcher.get_eval_set() if self.data_dispatcher.has_test() else None
        except Exception:
            eval_set = None
        # generic (autograd) models also use library kernels on their snapshot / merge path (integer-buffer max, clones,
        # gathers) that CUDA would otherwise load lazily at the first exchange -- loading a module can need a device-wide
        # synchronisation, which must not happen while kernels wait on other GPUs' flags: exercise that path once here
        # (a snapshot merged back into its own model with weights 1/2 + 1/2 leaves every value unchanged)
        for node in self.nodes.values():
            h = node.model_handler
            if getattr(h, "_fused", True) or not hasattr(h, "_snapshot") or not hasattr(h, "layout"):
                continue
            try:
                snap = h._snapshot()
                h._weighted_merge(snap, 0.5, 0.5)
                h._merge_int_buffers(snap)
                snap.release()
            except Exception as err:           # priming is best effort
                LOG.debug("priming the exchange path of node %s failed: %s" % (getattr(node, "idx", "?"), err))
        pend = []
        for node in self.nodes.values():
            fn = getattr(node, "evaluate_async", None)
            if fn is None:
                continue
            if node.has_test():
                pend.append(fn())
            if eval_set is not None:
                pend.append(fn(eval_set))
        for p in pend:
            p.result()

    # -- message plumbing ---------------------------------------------------------------------
    def _forget_messages_on_the_wire(self) -> None:
        """A fresh ``start`` (no ``resume``) restarts the clock with the models as they are; what the previous run left on the
        wire is gone, like in the reference where the queues are locals of ``start`` (ref ``simul.py:385-386``) -- but its
        snapshots go back to the arenas / the executor's slot pools (same leak class as B10)."""
        pending: List[Message] = []
        for queues in (self.__dict__.get("_msg_queues"), self.__dict__.get("_rep_queues")):
            for msgs in (queues or {}).values():
                pending.extend(msgs)
        pending.extend((self.__dict__.get("_native_msgs") or {}).values())
        for msg in pending:
            key = _model_key(msg)
            if key is not None:
                CACHE.drop(key)
        if self.__dict__.get("_native_msgs"):
            self._native_msgs.clear()
        sx = self.__dict__.get("_stream_exec")
        if sx is not None:
            sx.drop_inflight()
        bank = self.__dict__.get("_bank")
        if bank is not None:
            bank.drop_inflight()
        self.__dict__.pop("_exec_inflight", None)
        self.__dict__.pop("_bank_inflight", None)

    def _lost(self, msg: Optional[Message]) -> None:
        """Account a lost message and free its in-flight snapshot (FIX B10)."""
        self.notify_message(True)
        key = _model_key(msg)
        if key is not None:
            CACHE.drop(key)

    def _dispatch(self, msg: Optional[Message], t: int) -> None:
        """Send-side bookkeeping of a first-leg message: count, drop test, delay, enqueue."""
        self.notify_message(False, msg)
        if not msg:
            return
        if np.random.random() >= self.drop_prob:
            self._msg_queues[t + self.delay.get(msg)].append(msg)
        else:
            self._lost(msg)

    def _fire(self, node: GossipNode, t: int) -> bool:
        """Let ``node`` gossip with one random peer.  Returns False when it has no peer."""
        peer = node.get_peer()
        if peer is None:
            return False  # FIX(B6): skip this node instead of aborting the whole node loop
        self._dispatch(node.send(t, peer, self.protocol), t)
        return True

    # -- hooks ------------------------------------------------------------------------------------
    def _tick_node(self, i: int, t: int) -> None:
        node = self.nodes[i]
        if node.timed_out(t):
            self._fire(node, t)

    def _after_delivery(self, msg: Message, reply: Optional[Message], sender_mh: Any,
                        t: int) -> None:
        pass

    def _peek_sender(self, msg: Message) -> Any:
        return None

    # -- the four phases of a tick -----------------------------------------------------------
    def _deliver_messages(self, t: int, is_online: np.ndarray) -> None:
        queue = self._msg_queues.get(t)
        if not queue:
            self._msg_queues.pop(t, None)
            return
        i = 0
        while i < len(queue):  # the queue may grow while we walk it (reactive delay-0 sends)
            msg = queue[i]
            i += 1
            if not is_online[msg.receiver]:
                self._lost(msg)
                continue
            sender_mh = self._peek_sender(msg)
            reply = self.nodes[msg.receiver].receive(t, msg)
            if reply:
                if np.random.random() > self.drop_prob:
                    self._rep_queues[t + self.delay.get(reply)].append(reply)
                else:
                    self._lost(reply)
            self._after_delivery(msg, reply, sender_mh, t)
        del self._msg_queues[t]

    def _deliver_replies(self, t: int, is_online: np.ndarray) -> None:
        queue = self._rep_queues.pop(t, None)
        if not queue:
            return
        for reply in queue:
            if is_online[reply.receiver]:
                self.notify_message(False, reply)
                self.nodes[reply.receiver].receive(t, reply)
            else:
                self._lost(reply)

    def _eval_sample(self) -> List[GossipNode]:
        if self.sampling_eval > 0:
            k = max(int(self.n_nodes * self.sampling_eval), 1)
            return [self.nodes[int(i)] for i in np.random.choice(list(self.nodes.keys()), k)]
        return list(self.nodes.values())

    def _evaluate_round(self, t: int) -> None:
        self._evaluate_nodes(t, self._eval_sample())

    def _evaluate_nodes(self, t: int, sample: List[GossipNode], defer: bool = False):
        """Enqueue the evaluation of ``sample`` and report it.  With ``defer`` the (blocking)
        device->host read is returned as a callable instead, so the caller can enqueue the next
        round's device work first and keep the GPUs busy while the host waits."""
        local: List[PendingEval] = [n.evaluate_async() for n in sample if n.has_test()]
        glob: List[PendingEval] = []
        if self.data_dispatcher.has_test():
            eval_set = self.data_dispatcher.get_eval_set()
            glob = [n.evaluate_async(eval_set) for n in sample]

        def finish() -> None:
            # everything is enqueued; only now touch the host (one wait per round, not per node)
            from .parallel import runtime as _prt
            if _prt.active() and int(self.metrics_sync_every) > 1:
                # several ranks: keep this rank's results and exchange them every k rounds (one all-reduce for k rounds
                # instead of one per round; the receivers see the same evaluations in the same order, k rounds later)
                backlog = self.__dict__.setdefault("_metric_backlog", [])
                backlog.append((t, [p.result() for p in local], [p.result() for p in glob]))
                if len(backlog) >= int(self.metrics_sync_every):
                    self._flush_metrics()
                return
            if local:
                self.notify_evaluation(t, True, _prt.share_metrics([p.result() for p in local]))
            if glob:
                self.notify_evaluation(t, False, _prt.share_metrics([p.result() for p in glob]))
            if (local or glob) and _prt.active():
                _check_device_fault()
        if defer:
            return finish
        finish()
        return None

    metrics_sync_every = 1      # several ranks: rounds between two exchanges of the evaluation results (1 = every round)

    def _flush_metrics(self) -> None:
        """Share the evaluation results kept back by ``metrics_sync_every`` and report them in order."""
        backlog = self.__dict__.pop("_metric_backlog", None)
        if not backlog:
            return
        from .parallel import runtime as _prt
        flat = [d for _, loc, glob in backlog for d in loc + glob]
        shared = _prt.share_metrics(flat)
        pos = 0
        for t, loc, glob in backlog:
            if loc:
                self.notify_evaluation(t, True, shared[pos:pos + len(loc)])
                pos += len(loc)
            if glob:
                self.notify_evaluation(t, False, shared[pos:pos + len(glob)])
                pos += len(glob)
        _check_device_fault()

    def notify_end(self) -> None:
        self._flush_metrics()
        super().notify_end()

    def _stream_round_inputs(self) -> None:
        """Fresh inputs for the coming round: host (pinned) -> device, async on each node's stream."""
        for node in self.nodes.values():
            refresh = getattr(node.model_handler, "refresh_inputs", None)
            if refresh is not None:
                refresh(node.data[0])

    def _run(self, n_rounds: int, resume: bool = False) -> None:
        assert self.initialized, \
            "The simulator is not inizialized. Please, call the method 'init_nodes'."
        LOG.info("Simulation started.")
        if not resume:
            self._forget_messages_on_the_wire()
            self._clock = 0
            self._msg_queues = defaultdict(list)
            self._rep_queues = defaultdict(list)
            self._node_order = np.arange(self.n_nodes)
        first, last = self._clock, self._clock + n_rounds * self.delta
        ticks: Iterable[int] = range(first, last)
        bar = None
        if self.progress:
            try:
                from rich.progress import track
                bar = track(ticks, description="Simulating...")
                ticks = bar
            except Exception:
                bar = None
        try:
            for t in ticks:
                if t % self.delta == 0:
                    np.random.shuffle(self._node_order)
                    if self.stream_inputs:
                        self._stream_round_inputs()
                for i in self._node_order:
                    self._tick_node(int(i), t)
                is_online = np.random.random(self.n_nodes) <= self.online_prob
                if self._msg_queues.get(t) or self._rep_queues.get(t):
                    with nvtx_range("deliver"):
                        self._deliver_messages(t, is_online)
                        self._deliver_replies(t, is_online)
                else:
                    self._msg_queues.pop(t, None)
                    self._rep_queues.pop(t, None)
                if (t + 1) % self.delta == 0:
                    with nvtx_range("evaluate"):
                        self._evaluate_round(t)
                self.notify_timestep(t)
                self._clock = t + 1
        except KeyboardInterrupt:
            LOG.warning("Simulation interrupted by user.")
        if bar is not None and hasattr(bar, "close"):
            bar.close()
        self.notify_end()

    def start(self, n_rounds: int = 100, resume: bool = False) -> None:
        """Run ``n_rounds`` rounds of ``delta`` ticks.  ``resume=True`` continues the clock and
        the pending message queues of a previous (possibly checkpointed) run.

        ``self.engine`` selects the control plane: ``"python"`` (default; consumes the host RNGs
        exactly like the reference, used by the differential tests) or ``"native"`` (the C++
        scheduler of ``csrc/sched``: one call per round instead of ``N x delta`` Python iterations,
        its own counter-based random streams)."""
        if self._use_native_engine():
            self._run_native(n_rounds, resume)
        else:
            self._run(n_rounds, resume)

    # -- native control plane ---------------------------------------------------------------------
    engine = "python"
    pipeline_eval = True                   # native engine: read round r's metrics after enqueuing round r+1
    native_utility: Optional[int] = None   # tokenized runs: constant utility evaluated natively

    def _native_supported(self) -> Optional[str]:
        """``None`` when the C++ scheduler can drive this simulation, else the reason it cannot."""
        from .ops.native import native_available
        if not native_available():
            return "extension not built"
        for node in self.nodes.values():
            cls = type(node)
            if cls is PENSNode:          # its step switch and peer choice are driven from _run_native
                if self.protocol != AntiEntropyProtocol.PUSH:
                    return "PENSNode sends PUSH messages whatever the protocol"
                continue
            if cls.timed_out is not GossipNode.timed_out and not isinstance(node, All2AllGossipNode):
                return "node class overrides timed_out"
            if cls.get_peer is not GossipNode.get_peer:
                return "node class overrides get_peer"
        from .core import LinearDelay, UniformDelay
        if type(self.delay) not in (ConstantDelay, UniformDelay, LinearDelay):
            return "custom delay model"
        return None

    def _use_native_engine(self) -> bool:
        if self.engine != "native":
            return False
        why = self._native_supported()
        if why is not None:
            LOG.warning("native scheduler unavailable (%s); using the Python loop" % why)
            return False
        return True

    def _make_scheduler(self):
        from .core import AntiEntropyProtocol as AEP, LinearDelay, UniformDelay
        from .engine import rng as _rng
        from .ops.native import _try_import
        C = _try_import()
        proto = {AEP.PUSH: 1, AEP.PULL: 2, AEP.PUSH_PULL: 3}[self.protocol]
        sch = C.GossipScheduler(self.n_nodes, self.delta, proto, float(self.drop_prob),
                                float(self.online_prob), float(self.sampling_eval),
                                _rng.derive(0x5C4ED))
        ids = sorted(self.nodes)
        assert ids == list(range(self.n_nodes)), "node ids must be 0..N-1"
        sch.set_nodes([1 if self.nodes[i].sync else 0 for i in ids], [int(self.nodes[i].delta) for i in ids],
                      [int(self.nodes[i].round_len) for i in ids])
        net = self.nodes[0].p2p_net
        if not (type(net) is StaticP2PNetwork and net.__dict__.get("_clique", False)):
            # (an implicit clique needs no peer table: the scheduler's default enumerates "everybody but me" in the order of
            # StaticP2PNetwork's lists -- at 4 141 nodes the table would have 17 M entries and take seconds to hand over)
            indptr, indices = net.as_csr()
            sch.set_topology(indptr.tolist(), indices.tolist())
        if isinstance(self.delay, UniformDelay):
            sch.set_delay(1, float(self.delay._min_delay), float(self.delay._max_delay))
        elif isinstance(self.delay, LinearDelay):
            sch.set_delay(2, float(self.delay._timexunit), float(self.delay._overhead))
        else:
            sch.set_delay(0, float(self.delay._delay), 0.0)
        self._configure_scheduler(sch)
        return sch

    def _configure_scheduler(self, sch) -> None:
        node = self.nodes[0]
        counters = {k: node.__dict__.get(k) for k in ("_model_msgs", "_pt_draws", "_cn_draws")}
        extras = len(node._payload_extras())        # only the NUMBER of extras matters here ...
        for k, v in counters.items():               # ... a keyed draw it may have made must not count (exact resume)
            if v is None:
                node.__dict__.pop(k, None)
            else:
                node.__dict__[k] = v
        sch.set_message_sizes(int(node.model_handler.get_size()) + extras, 1)

    def _run_native(self, n_rounds: int, resume: bool = False) -> None:
        assert self.initialized, \
            "The simulator is not inizialized. Please, call the method 'init_nodes'."
        LOG.info("Simulation started (native scheduler).")
        from .ops.native import _try_import
        C = _try_import()
        if not GlobalSettings().reference_compat:
            for node in self.nodes.values():      # node-side random draws (partition ids) come from keyed streams that
                node._keyed_draws = True          # the C++ executor reproduces, not from the host NumPy generator
        sch = self.__dict__.get("_scheduler")
        saved = self.__dict__.pop("_scheduler_state", None)
        if resume and sch is None and saved is not None:
            # a checkpoint taken under the native engine: same configuration + the saved dynamic
            # state (stream counters, queues, balances) continue the exact schedule
            sch = self.__dict__["_scheduler"] = self._make_scheduler()
            sch.set_state(saved)
            self.__dict__.setdefault("_native_msgs", {})
        elif sch is None or not resume:
            if not resume:
                self._forget_messages_on_the_wire()
            sch = self.__dict__["_scheduler"] = self._make_scheduler()
            self._native_msgs: Dict[int, Message] = {}
            self.__dict__.pop("_bank_inflight", None)
            if resume and getattr(self, "_clock", 0):
                # checkpoint taken under the Python engine: keep the clock (and the evaluation phase
                # of sync nodes) but the pending Python queues are not transferable: their messages are
                # lost (like drops) and the snapshots they reference are returned to the arenas
                sch.clock = int(self._clock)
                lost = 0
                for queues in (self._msg_queues, self._rep_queues):
                    for msgs in queues.values():
                        for msg in msgs:
                            lost += 1
                            if msg.value and isinstance(msg.value[0], CacheKey):
                                CACHE.drop(msg.value[0])
                    queues.clear()
                if lost:
                    LOG.warning("Resuming a Python-engine checkpoint under the native engine: %d pending messages "
                                "were discarded." % lost)
            else:
                self._clock = 0
        pens = [n for n in self.nodes.values() if type(n) is PENSNode]
        for node in pens:                  # resumed run: the restricted peer lists are configuration, not scheduler state
            if node.step == 2 and node.best_nodes:
                sch.set_peer_list(node.idx, [int(p) for p in node.best_nodes])
        use_bank = self.batched is True or (self.batched == "auto" and (
            GlobalSettings().get_device().type == "cuda" or self.n_nodes >= 512))
        if use_bank and type(self) is GossipSimulator:
            from .engine import bank as _bank
            why = _bank.bankable(self)
            if why is None:
                self._run_native_banked(sch, n_rounds, C)
                return
        if self.native_executor and type(self) in (GossipSimulator, TokenizedGossipSimulator, All2AllGossipSimulator):
            from .engine import stream_exec as _sx
            if _sx.eligible(self) is None and self._handover_to_executor():
                self._run_native_streamed(sch, n_rounds)
                return
        sx_prev = self.__dict__.get("_stream_exec")
        if ((self.__dict__.get("_exec_inflight") and self.__dict__["_exec_inflight"].get("ids"))
                or (resume and sx_prev is not None and len(sx_prev.ex.inflight()) > 0)):
            # messages on the wire are snapshot slots of the C++ executor (a checkpoint taken under it): the per-event
            # executor cannot deliver them
            raise RuntimeError("messages on the wire are snapshot slots of the C++ executor (this run, or the checkpoint it was "
                               "loaded from, used it); resume with native_executor = True and the same handlers")
        msgs = self._native_msgs
        prev_finish = None
        try:
            for rnd in range(n_rounds):
                if self.stream_inputs:
                    self._stream_round_inputs()
                eval_nodes: List[GossipNode] = []
                if not pens:
                    with nvtx_range("schedule"):
                        events = sch.run(1).tolist()
                    eval_nodes = self._native_execute(events, msgs)
                else:
                    # PENS (ref node.py:716-741): a node leaves step 1 at the first tick of round `step1_rounds`.  The
                    # round is simulated in pieces so that the switch (peer list of the scheduler, `step` of the node,
                    # which decides how a delivery is consumed) falls between two pieces, each executed before the next
                    t_end = int(sch.clock) + self.delta
                    while int(sch.clock) < t_end:
                        t0, nxt = int(sch.clock), t_end
                        for node in pens:
                            if node.step == 1:
                                t_sw = int(node.step1_rounds) * int(node.round_len)
                                if t_sw <= t0:
                                    node.step = 2
                                    node._select_neighbors()
                                    sch.set_peer_list(node.idx, [int(p) for p in node.best_nodes])
                                elif t_sw < nxt:
                                    nxt = t_sw
                        with nvtx_range("schedule"):
                            events = sch.run_ticks(nxt - t0).tolist()
                        eval_nodes += self._native_execute(events, msgs)
                t_last = int(sch.clock) - 1
                # software pipelining of the host: the metrics of round r are read back only after
                # round r+1 has been enqueued (evaluation snapshots the statistics on the device)
                finish = self._evaluate_nodes(t_last, eval_nodes, defer=self.pipeline_eval)
                if prev_finish is not None:
                    prev_finish()
                prev_finish = finish
                self._clock = int(sch.clock)
                self.notify_timestep(t_last)
                if pens and self.native_executor and rnd + 1 < n_rounds and all(n.step == 2 for n in pens):
                    # every PENS node has left its selection phase: from here on a delivery is a plain merge + update,
                    # the rest of the run is enqueued from C++ (messages on the wire move into the executor's slots)
                    from .engine import stream_exec as _sx
                    if _sx.eligible(self) is None and self._handover_to_executor():
                        if prev_finish is not None:
                            prev_finish()
                        self._run_native_streamed(sch, n_rounds - rnd - 1)
                        return
                    pens = []               # not eligible (generic model, ...): no need to ask again
        except KeyboardInterrupt:
            LOG.warning("Simulation interrupted by user.")
        if prev_finish is not None:
            prev_finish()
        self.notify_end()

    def _handover_to_executor(self) -> bool:
        """Messages the per-event executor left on the wire (``_native_msgs``: snapshot handlers in ``CACHE``) become
        in-flight snapshot slots of the C++ executor.  ``False`` = they carry something the conversion does not cover
        (partition ids, degrees, ...) and the per-event executor keeps the run."""
        msgs = self.__dict__.get("_native_msgs") or {}
        if not msgs:
            return True
        if "_stream_exec" in self.__dict__ or "_exec_inflight" in self.__dict__:
            return False
        from .core import CreateModelMode
        mode = self.nodes[0].model_handler.mode
        if mode == CreateModelMode.UPDATE_MERGE or any(m.value is not None and len(m.value) != 1 for m in msgs.values()):
            return False
        from .parallel import runtime as _prt
        ids, ranks, ages, rows = [], [], [], []
        for mid in sorted(msgs):
            msg = msgs[mid]
            if msg.value is None:            # a PULL request carries no model
                continue
            snap = CACHE[msg.value[0]]
            ids.append(int(mid))
            ranks.append(int(_prt.rank_of(msg.sender)) if _prt.active() else 0)
            ages.append(int(snap.n_updates))
            rows.append(snap.row.detach().cpu().clone())    # (several ranks: only the sender's rank holds the values, and
            CACHE.drop(msg.value[0])                        #  only that rank fills the slot)
        msgs.clear()
        if ids:
            import torch
            self.__dict__["_exec_inflight"] = {"ids": ids, "ranks": ranks, "ages": ages, "extra": [[] for _ in ids],
                                               "rows": torch.stack(rows)}
        return True

    # native engine: execute bankable set-ups (linear learners, k-means, MF) many nodes per launch.  "auto" = on a GPU, or from
    # 512 nodes on the CPU (where the bank's vectorised-over-nodes update loses to per-node calls for a few big shards)
    batched: Any = "auto"
    native_executor = True    # native engine: eligible set-ups are enqueued from C++ (engine/stream_exec.py);
                              # everything else (other node / handler types) goes through the per-event Python executor

    def _run_native_streamed(self, sch, n_rounds: int) -> None:
        """Rounds of an eligible simulation (``engine.stream_exec.eligible``): the scheduler's event list
        goes straight to the C++ executor, which enqueues snapshots and fused merge+update kernels on the
        nodes' streams; Python only evaluates (on the same streams) and keeps the books per ROUND."""
        from .engine.stream_exec import StreamExec
        sx = self.__dict__.get("_stream_exec")
        if sx is None:
            sx = self.__dict__["_stream_exec"] = StreamExec(self)
            inflight = self.__dict__.pop("_exec_inflight", None)
            if inflight is not None:
                sx.import_inflight(inflight)
        else:
            sx.bind_nodes()
        reports = [r for r in self._receivers if type(r) is SimulationReport]
        others = [r for r in self._receivers if type(r) is not SimulationReport]
        size_model = int(self.nodes[0].model_handler.get_size())
        prev_finish = None
        try:
            for _ in range(n_rounds):
                if self.stream_inputs:
                    self._stream_round_inputs()
                    sx.refresh_data()
                sent0, failed0, size0 = int(sch.sent), int(sch.failed), int(sch.total_size)
                with nvtx_range("schedule"):
                    events = sch.run(1)
                t_last = int(sch.clock) - 1
                with nvtx_range("execute"):
                    evals = sx.run_round(events)
                sent, failed, size = int(sch.sent) - sent0, int(sch.failed) - failed0, int(sch.total_size) - size0
                for r in reports:                      # bulk accounting (same totals as per-message calls)
                    r._sent_messages += sent
                    r._total_size += size
                    r._failed_messages += failed
                if others:
                    n_model = (size - sent) // (size_model - 1) if size_model > 1 else sent
                    stub_model = _SizedMessage(Message(t_last, 0, 0, MessageType.PUSH, None), size_model)
                    stub_small = _SizedMessage(Message(t_last, 0, 0, MessageType.PULL, None), 1)
                    for r in others:
                        for _i in range(n_model):
                            r.update_message(False, stub_model)
                        for _i in range(sent - n_model):
                            r.update_message(False, stub_small)
                        for _i in range(failed):
                            r.update_message(True)
                finish = self._evaluate_nodes(t_last, [self.nodes[i] for i in evals], defer=self.pipeline_eval)
                if prev_finish is not None:
                    prev_finish()
                prev_finish = finish
                self._clock = int(sch.clock)
                self.notify_timestep(t_last)
        except KeyboardInterrupt:
            LOG.warning("Simulation interrupted by user.")
        if prev_finish is not None:
            prev_finish()
        sx.sync_back()
        self.notify_end()

    def _run_native_banked(self, sch, n_rounds: int, C) -> None:
        """Rounds of a bankable simulation: the scheduler's event list of a round is executed by a bank
        (``engine.bank.make_bank``: linear learners, k-means or matrix factorisation) with one kernel launch per
        phase of a tick."""
        from .engine.bank import make_bank
        bank = self.__dict__.get("_bank")
        if bank is None:
            bank = self.__dict__["_bank"] = make_bank(self)
            inflight = self.__dict__.pop("_bank_inflight", None)
            if inflight is not None:
                bank.import_inflight(inflight)
        reports = [r for r in self._receivers if type(r) is SimulationReport]
        others = [r for r in self._receivers if type(r) is not SimulationReport]
        try:
            for _ in range(n_rounds):
                with nvtx_range("schedule"):
                    events = sch.run(1)
                t_last = int(sch.clock) - 1
                with nvtx_range("bank"):
                    evals, cnt = bank.run_round(events, C)
                for r in reports:                      # bulk accounting (same totals as per-message calls)
                    r._sent_messages += cnt["sent"]
                    r._total_size += cnt["sent_size"]
                    r._failed_messages += cnt["failed"]
                if others:
                    n_model = (cnt["sent_size"] - cnt["sent"]) // max(1, bank.size_model - 1) if bank.size_model > 1 else cnt["sent"]
                    stub_model = _SizedMessage(Message(t_last, 0, 0, MessageType.PUSH, None), bank.size_model)
                    stub_small = _SizedMessage(Message(t_last, 0, 0, MessageType.PULL, None), 1)
                    for r in others:
                        for _i in range(n_model):
                            r.update_message(False, stub_model)
                        for _i in range(cnt["sent"] - n_model):
                            r.update_message(False, stub_small)
                        for _i in range(cnt["failed"]):
                            r.update_message(True)
                if evals:
                    with nvtx_range("evaluate"):
                        # per-node test sets (matrix factorisation) are per-user results, as in _evaluate_nodes
                        self.notify_evaluation(t_last, bank.eval_on_user, bank.evaluate(evals))
                self._clock = int(sch.clock)
                self.notify_timestep(t_last)
        except KeyboardInterrupt:
            LOG.warning("Simulation interrupted by user.")
        bank.writeback()
        self.notify_end()

    def _native_execute(self, events: List[List[int]], msgs: Dict[int, Message]) -> List[GossipNode]:
        """Per-event executor of the native control plane: turns the scheduler's events (rows of
        ``kind, tick, a, b, slot, aux``) into node calls; returns the nodes to evaluate."""
        from .ops.native import _try_import
        C = _try_import()
        SEND, DROP, DELIVER, RSEND, RDELIVER, EVAL, TIMEOUT = (C.EV_SEND, C.EV_DROP, C.EV_DELIVER,
                                                              C.EV_REPLY_SEND, C.EV_REPLY_DELIVER, C.EV_EVAL,
                                                              C.EV_TIMEOUT)
        pending_reply: Optional[Message] = None
        eval_nodes: List[GossipNode] = []
        for kind, t, a, b, slot, aux in events:
            if kind == SEND:
                msg = self._native_send(self.nodes[a], t, b)
                msgs[slot] = msg
                self.notify_message(False, msg)
            elif kind == DROP:
                self._lost(msgs.pop(slot, None))
            elif kind == DELIVER:
                pending_reply = self.nodes[b].receive(t, msgs.pop(slot))
            elif kind == RSEND:
                msgs[aux] = pending_reply
                pending_reply = None
            elif kind == RDELIVER:
                reply = msgs.pop(slot)
                self.notify_message(False, reply)
                self.nodes[a].receive(t, reply)
            elif kind == EVAL:
                eval_nodes.append(self.nodes[a])
            elif kind == TIMEOUT:
                self._native_timeout(self.nodes[a], t)
        return eval_nodes

    def _native_send(self, node: GossipNode, t: int, peer: int) -> Message:
        if type(node) is PENSNode and node.step == 1:      # what PENSNode.get_peer counts (ref node.py:733-737)
            node.selected[peer] += 1
        return node.send(t, peer, self.protocol)

    def _native_timeout(self, node: GossipNode, t: int) -> None:
        pass

    # -- checkpointing ---------------------------------------------------------------------------
    def save(self, filename: str) -> None:
        """Serialise simulator + in-flight models (ref ``simul.py:460-474``).

        Model rows are pulled off the device as CPU tensors; the clock and the pending message
        queues are part of the state, so ``load(...).start(n, resume=True)`` continues the run.
        """
        self._flush_metrics()                # (several ranks save collectively: results held back are exchanged first)
        with open(filename, "wb") as f:
            _pickler.dump({"simul": self, "cache": CACHE.get_cache()}, f)

    @classmethod
    def load(cls, filename: str) -> "GossipSimulator":
        with open(filename, "rb") as f:
            loaded = _pickler.load(f)
        CACHE.load(loaded["cache"])
        from .parallel import runtime as _prt
        if _prt.active():                   # every owner has restored its rows before any rank reads a peer's
            if GlobalSettings().get_device().type == "cuda":
                import torch
                torch.cuda.synchronize()
            _prt.barrier()
        return loaded["simul"]

    def __getstate__(self) -> Dict[str, Any]:
        st = dict(self.__dict__)
        st["_receiver_list"] = list(self._receivers)
        st.pop("_collective", None)
        bank = st.pop("_bank", None)
        sx = st.pop("_stream_exec", None)
        sch = st.pop("_scheduler", None)
        if sch is not None:
            # native engine: the scheduler's dynamic state + the in-flight messages (their models are
            # snapshot handlers in CACHE, or snapshot slots of the bank) -> an exact resume
            state = dict(sch.get_state())
            st["_scheduler_state"] = state
            if bank is not None:
                rows = [r for r in state["msg_q"] if int(r[4]) != 2] + list(state["rep_q"])     # (due, id, sender, receiver, ..)
                st["_bank_inflight"] = bank.export_inflight([int(r[1]) for r in rows], [int(r[3]) for r in rows])
            if sx is not None:                       # (several ranks: the owners' slots are gathered, every rank saves all)
                st["_exec_inflight"] = sx.export_inflight()
        return st

    def __repr__(self) -> str:
        return str(self)

    def __str__(self) -> str:
        skip = {"nodes", "model_handler_params", "gossip_node_params", "_msg_queues",
                "_rep_queues", "_receiver_list", "_node_order", "accounts"}
        attrs = {k: v for k, v in self.__dict__.items() if k not in skip}
        return "%s %s" % (self.__class__.__name__,
                          json.dumps(attrs, indent=4, sort_keys=True, cls=StringEncoder))


class TokenizedGossipSimulator(GossipSimulator):
    """Token-account flow control on top of the vanilla loop (ref ``simul.py:506-689``).

    On timeout a node sends with probability ``proactive()`` and otherwise banks a token; when
    a model message is delivered (and no reply is due) the *receiver* reacts with
    ``reactive(utility)`` extra sends.  FIX(B4/B5): the reference issues the reactive sends from
    a stale loop variable and may read an unbound ``sender_mh``; here the receiver reacts and the
    sender's handler is looked up per message.
    """

    def __init__(self, nodes: Dict[int, GossipNode], data_dispatcher: DataDispatcher,
                 token_account: TokenAccount,
                 utility_fun: Callable[[ModelHandler, ModelHandler, Message], int], delta: int,
                 protocol: AntiEntropyProtocol, drop_prob: float = 0., online_prob: float = 1.,
                 delay: Delay = ConstantDelay(0), sampling_eval: float = 0.) -> None:
        super().__init__(nodes, data_dispatcher, delta, protocol, drop_prob, online_prob, delay,
                         sampling_eval)
        self.utility_fun = utility_fun
        self.token_account_proto = token_account
        self.accounts: Dict[int, TokenAccount] = {}

    def init_nodes(self, seed: int = 98765) -> None:
        super().init_nodes(seed)
        self.accounts = {i: deepcopy(self.token_account_proto) for i in range(self.n_nodes)}

    def _tick_node(self, i: int, t: int) -> None:
        node = self.nodes[i]
        if not node.timed_out(t):
            return
        if np.random.random() < self.accounts[i].proactive():
            self._fire(node, t)
        else:
            self.accounts[i].add(1)

    def _peek_sender(self, msg: Message) -> Any:
        key = _model_key(msg)
        return CACHE[key] if key is not None else None

    def _after_delivery(self, msg: Message, reply: Optional[Message], sender_mh: Any,
                        t: int) -> None:
        if reply:
            return
        receiver = self.nodes[msg.receiver]
        utility = self.utility_fun(receiver.model_handler, sender_mh, msg)
        account = self.accounts[msg.receiver]
        reaction = account.reactive(utility)
        if reaction:
            account.sub(reaction)
            actor = receiver
            if GlobalSettings().reference_compat:
                # B4 mimicked: the reference issues the reactive sends from its stale loop variable `node`,
                # i.e. the LAST node of this round's shuffled order, whoever received the message
                actor = self.nodes[int(self._node_order[-1])]
            for _ in range(int(reaction)):
                if not self._fire(actor, t):
                    break

    def __getstate__(self) -> Dict[str, Any]:
        return super().__getstate__()

    def _constant_utility(self) -> Optional[int]:
        """The utility the C++ scheduler evaluates the token accounts with: ``native_utility`` if set, else the constant
        ``utility_fun`` returns when its body is nothing but ``return <int>`` (the reference scripts' ``lambda mh1, mh2,
        msg: 1``) -- decided from the byte code, the function is never called for it."""
        if self.native_utility is not None:
            return int(self.native_utility)
        import dis
        try:
            ops = [i for i in dis.get_instructions(self.utility_fun) if i.opname not in ("RESUME", "NOP", "CACHE")]
        except TypeError:
            return None
        value: Any = None
        if len(ops) == 1 and ops[0].opname == "RETURN_CONST":
            value = ops[0].argval
        elif len(ops) == 2 and ops[0].opname == "LOAD_CONST" and ops[1].opname == "RETURN_VALUE":
            value = ops[0].argval
        if isinstance(value, (int, np.integer)) and not isinstance(value, bool):
            return int(value)
        return None

    def _native_supported(self) -> Optional[str]:
        if self._constant_utility() is None:
            return "utility_fun is a Python callback (set native_utility to a constant to go native)"
        if GlobalSettings().reference_compat:
            return "reference_compat mimics B4 in the Python loop only"
        return super()._native_supported()

    def _configure_scheduler(self, sch) -> None:
        super()._configure_scheduler(sch)
        kind, C, A, k = self.token_account_proto.spec()
        sch.set_token_account(int(kind) + 1, int(C), int(A), max(1, int(k)), int(self._constant_utility()))


class All2AllGossipSimulator(GossipSimulator):
    """Decentralised SGD with neighbourhood averaging (ref ``simul.py:720-852``).

    ``start(W_matrix, n_rounds)``: on timeout a node first merges the models cached from its
    neighbours with row ``W[i]`` and trains, then pushes its model to *every* peer.
    """

    def _tick_node(self, i: int, t: int) -> None:
        node: All2AllGossipNode = self.nodes[i]  # type: ignore[assignment]
        if node.timed_out(t, self._W[i]):
            for peer in node.get_peers():
                self._dispatch(node.send(t, peer, self.protocol), t)

    def start(self, W_matrix: MixingMatrix, n_rounds: int = 100,  # type: ignore[override]
              resume: bool = False, synchronous: bool = False) -> None:
        """``synchronous=True`` runs textbook D-PSGD rounds (Koloskova 2020): every round ALL nodes
        average simultaneously and then train, instead of the reference's tick-by-tick simulation
        in which nodes fire at different offsets inside a round.  On a clique with uniform mixing
        this is one all-reduce per round -- executed by the one-shot NVLS kernel
        (``parallel.collectives.SymmetricAllReduce``) -- followed by the fused local update."""
        self._W = W_matrix
        if synchronous:
            self._run_synchronous(n_rounds)
            return
        if self._use_native_engine():
            self._run_native(n_rounds, resume)
        else:
            self._run(n_rounds, resume)

    def _configure_scheduler(self, sch) -> None:
        super()._configure_scheduler(sch)
        sch.set_broadcast(True)

    def _native_timeout(self, node: GossipNode, t: int) -> None:
        node.on_timeout(self._W[node.idx])     # type: ignore[attr-defined]

    # -- synchronous D-PSGD rounds: all-reduce + local update ------------------------------------------
    def _run_synchronous(self, n_rounds: int) -> None:
        assert self.initialized, \
            "The simulator is not inizialized. Please, call the method 'init_nodes'."
        import torch
        from . import ops
        from .engine import arena as _arena
        from .parallel import runtime as _prt
        from .parallel.collectives import SymmetricAllReduce
        ids = sorted(self.nodes)
        n = len(ids)
        net = self.nodes[ids[0]].p2p_net
        for i in ids:
            if sorted(net.get_peers(i)) != [j for j in ids if j != i]:
                raise ValueError("synchronous all-to-all rounds need a clique")
            w = np.asarray(self._W[i], dtype=float)
            if not np.allclose(w, 1.0 / n):
                raise ValueError("synchronous all-to-all rounds need uniform mixing weights 1/N")
        if self.drop_prob or self.online_prob < 1 or self.delay.get(None) != 0:  # type: ignore[arg-type]
            raise ValueError("synchronous all-to-all rounds model a fault-free network")
        handlers = {i: self.nodes[i].model_handler for i in ids}
        mine = [i for i in ids if handlers[i]._mine()]
        h0 = handlers[ids[0]]
        dev = h0.device
        numel = h0._row_numel
        coll = self.__dict__.get("_collective")
        if coll is None or coll.numel != numel:
            coll = self.__dict__["_collective"] = SymmetricAllReduce(numel, dev)
        mean = None if len(mine) == 1 else torch.zeros(numel, dtype=torch.float32, device=dev)
        size = int(h0.get_size())
        LOG.info("Synchronous all-to-all rounds (%s all-reduce)." % coll.kind)
        prev_finish = None
        try:
            for r in range(n_rounds):
                t = self._clock + self.delta - 1
                if self.stream_inputs:
                    self._stream_round_inputs()
                # message accounting of the equivalent push round: every node pushes to N-1 peers
                msg = Message(t, ids[0], ids[0], MessageType.PUSH, None)
                for _ in range(n * (n - 1)):
                    self.notify_message(False, _SizedMessage(msg, size))
                cur = _arena.current(dev)
                # 1. this rank's contribution = sum of its nodes' rows (work joins the current stream)
                for i in mine:
                    s_i = handlers[i]._stream()
                    if s_i is not None:
                        ev = torch.cuda.Event(); ev.record(s_i); cur.wait_event(ev)
                rows = [handlers[i].row for i in mine]
                if rows:
                    ops.merge_pair(coll.contribution, rows[0], 0.0, 1.0, 0, numel)
                    if len(rows) > 1:
                        ops.merge_kway(coll.contribution, rows[1:], [1.0] * len(rows))
                else:
                    coll.contribution.zero_()
                # 2. one-shot all-reduce (NVLS multicast / P2P pull) -> mean model
                target = handlers[mine[0]].row if len(mine) == 1 else mean
                coll.mean_into(target, n)
                if cur is not None:
                    done = torch.cuda.Event(); done.record(cur)
                age = max(int(np.max(handlers[i].n_updates)) for i in ids)
                # 3. every node adopts the mean and trains (adopt fused into the training kernel)
                for i in ids:
                    h = handlers[i]
                    h.n_updates = age if np.ndim(h.n_updates) == 0 else np.maximum(h.n_updates, age)
                    if h._mine():
                        s_i = h._stream()
                        if s_i is not None:
                            s_i.wait_event(done)
                        if len(mine) > 1:
                            if getattr(h, "_fused", False):
                                h._update(self.nodes[i].data[0], merge_from=(mean, 0.0, 1.0, None))
                                continue
                            with _arena.on_stream(s_i):
                                ops.merge_pair(h.row, mean, 0.0, 1.0, 0, numel)
                    h._update(self.nodes[i].data[0])
                self._clock += self.delta
                # read round r's metrics after round r+1 is enqueued (the host-side read blocks; the GPUs stay busy)
                finish = self._evaluate_nodes(t, self._eval_sample(), defer=self.pipeline_eval)
                if prev_finish is not None:
                    prev_finish()
                prev_finish = finish
                self.notify_timestep(t)
        except KeyboardInterrupt:
            LOG.warning("Simulation interrupted by user.")
        if prev_finish is not None:
            prev_finish()
        self.notify_end()


class _SizedMessage:
    """Accounting stand-in for a model message of known size (synchronous rounds)."""

    def __init__(self, msg: Message, size: int) -> None:
        self._msg, self._size = msg, size

    def get_size(self) -> int:
        return self._size

    def __getattr__(self, name: str) -> Any:
        return getattr(self._msg, name)
