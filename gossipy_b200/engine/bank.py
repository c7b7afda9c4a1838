"""Batched execution of the linear learners: many gossip nodes per kernel launch.

The reference's experiments with AdaLine / Pegasos models run one node per training sample
(4 141 nodes, ``main_ormandi_2013.py`` / ``main_giaretta_2019.py``); a model is 57 floats.  Executing
such a simulation event by event -- one snapshot object and one launch per message -- is pure
overhead.  :class:`LinearBank` keeps ALL nodes' models in one device tensor ``W[N, Dp]`` (ages in
``age[N]``), in-flight snapshots in ``S[slots, Dp]``, and turns the event list of a whole round
(produced by the native scheduler, ``csrc/sched``) into one launch per *phase of a tick*
(``csrc/kernels/bank.cu``; vectorised torch ops on CPU):

    phase A  all sends of the tick            -> one snapshot launch
    phase B  deliveries, in conflict-free waves (the k-th delivery of every receiver), each followed
             by the snapshot of the replies it triggers (PULL / PUSH_PULL)
    phase C  deliveries of replies, in waves
    phase D  end of round: one launch computes the scores of all sampled nodes on the test set

Ordering inside a tick is exactly the per-event order of the reference for every single node;
only events that touch *different* nodes are executed together.  Used by
``GossipSimulator`` when ``engine="native"`` and the set-up is bankable (plain ``GossipNode``s, one
shared AdaLine/Pegasos handler configuration, global evaluation set); the handlers' rows and ages
are written back when the run ends, so the object API sees the same final state.

The model-agnostic part (slot pool, waves, the phases of ``run_round``, checkpoint export / import) is
:class:`_SlotBank`.  Two more families share it on one rank (``csrc/kernels/bank_families.cu``, one CTA per work
item): :class:`KMeansBank` (``KMeansHandler``, ``main_berta_2014.py``: 4 601 nodes) and :class:`MFBank`
(``MFModelHandler``, ``main_hegedus_2020.py``: 6 040 users, rows of ~22 k floats, per-user evaluation).
:func:`make_bank` picks the bank of a simulation.
"""
from __future__ import annotations

import os
from typing import Any, Dict, List, Optional, Tuple

import numpy as np
import torch

from .. import ops
from ..core import CreateModelMode
from . import arena as _arena

_RING = 1 << 22     # in-flight message ids are far younger than this

_MODE = {CreateModelMode.UPDATE: 1, CreateModelMode.MERGE_UPDATE: 2, CreateModelMode.UPDATE_MERGE: 3,
         CreateModelMode.PASS: 4}


_OPEN: List["LinearBank"] = []      # banks holding shared-memory segments (closed by parallel.runtime.shutdown)
_PINNED_IDX = os.environ.get("GOSSIPY_BANK_PINNED_IDX", "") == "1"
_BANK_SEQ = 0                        # banks created in this session (names their shared-memory segments)


def close_all() -> None:
    while _OPEN:
        _OPEN.pop().close()


def bankable(sim) -> Optional[str]:
    """``None`` if a bank (:func:`make_bank`) can execute ``sim``; otherwise the reason it cannot."""
    from ..model.handler import AdaLineHandler, KMeansHandler, MFModelHandler
    from ..node import CacheNeighNode, GossipNode, PassThroughNode
    from ..parallel import runtime as prt
    if isinstance(list(sim.nodes.values())[0].model_handler, (KMeansHandler, MFModelHandler)):
        return _family_bankable(sim)
    if prt.active() and prt.transport() != "p2p":
        return "several ranks without shared memory"
    if prt.active() and prt.world() > 16:
        return "more than 16 ranks"
    nodes = list(sim.nodes.values())
    h0 = nodes[0].model_handler
    if not isinstance(h0, AdaLineHandler):
        return "handler is not AdaLine/Pegasos/KMeans/MF"
    cls = type(nodes[0])
    if cls in (PassThroughNode, CacheNeighNode) and not getattr(nodes[0], "_keyed_draws", False):
        return "node-side draws from the host stream"
    if cls is CacheNeighNode and "_bank" not in sim.__dict__ and any(n.local_cache for n in nodes):
        return "neighbour caches filled by another executor"
    for n in nodes:
        h = n.model_handler
        if type(n) is not cls or cls not in (GossipNode, PassThroughNode, CacheNeighNode):
            return "node subclass"
        if type(h) is not type(h0) or h.learning_rate != h0.learning_rate or h.dim != h0.dim or h.mode != h0.mode:
            return "heterogeneous handlers"
        if n.has_test():
            return "per-node test sets"
    if h0.mode not in _MODE:
        return "unsupported mode"
    if type(sim).__name__ != "GossipSimulator":
        return "simulator variant"
    return None


class _SlotBank:
    """What every bank shares, whatever its model: the snapshot slot pool (``S[slots, Dp]``, ``slot_age``, a stack of
    free slots, ``slot_map`` from message id to slot), the grouping of a tick's deliveries into conflict-free waves,
    the phase structure of ``run_round`` and the export / import / drop of the messages on the wire (checkpoints).
    A subclass owns its row layout and data and implements ``_snapshot``, ``_deliver``, ``evaluate`` and
    ``writeback``."""

    multi = False               # several ranks (LinearBank only)
    world, rank = 1, 0
    passthrough = cacheneigh = False
    eval_on_user = False        # evaluations are reported as per-node (True) or global (False) results

    def _init_slots(self, cap: int) -> None:
        """Single-rank slot pool of ``cap`` rows (grows on demand, see ``_alloc``)."""
        self.cap = cap
        self.S = torch.zeros(self.cap, self.Dp, dtype=torch.float32, device=self.device)
        self.slot_age = torch.zeros(self.cap, dtype=torch.int64, device=self.device)
        self.free = np.arange(self.cap - 1, -1, -1, dtype=np.int64)   # stack of free slots
        self.n_free = self.cap

    def _item_modes(self, recvs: np.ndarray, senders: np.ndarray, slots: np.ndarray) -> Optional[np.ndarray]:
        return None

    def _idx(self, a) -> torch.Tensor:
        arr = np.asarray(a, dtype=np.int32)
        if _PINNED_IDX and self.device.type == "cuda" and arr.size:
            # a pageable host -> device copy blocks the host until the stream has drained, i.e. it serialises host and device
            # once per launch; through pinned memory the copy is asynchronous (the caching host allocator keeps the staging
            # block alive until the copy has run).  Written after the last GPU session: opt-in (GOSSIPY_BANK_PINNED_IDX=1)
            return torch.from_numpy(np.ascontiguousarray(arr)).pin_memory().to(self.device, non_blocking=True)
        return torch.as_tensor(arr, device=self.device)

    # -- one round ----------------------------------------------------------------------------------
    def _alloc(self, k: int) -> np.ndarray:
        if self.n_free < k:
            grow = max(self.cap, k)
            self.S = torch.cat([self.S, torch.zeros(grow, self.Dp, dtype=torch.float32, device=self.device)])
            self.slot_age = torch.cat([self.slot_age, torch.zeros(grow, dtype=torch.int64, device=self.device)])
            self.free = np.concatenate([self.free[:self.n_free], np.arange(self.cap, self.cap + grow, dtype=np.int64)])
            self.n_free += grow
            self.cap += grow
        out = self.free[self.n_free - k:self.n_free].copy()
        self.n_free -= k
        return out

    def _release(self, slots: np.ndarray) -> None:
        slots = slots[slots >= 0]
        k = slots.size
        if k:
            if self.n_free + k > self.free.size:
                self.free = np.concatenate([self.free, np.empty(self.n_free + k - self.free.size, dtype=np.int64)])
            self.free[self.n_free:self.n_free + k] = slots
            self.n_free += k

    @staticmethod
    def _waves(recv: np.ndarray) -> List[np.ndarray]:
        """Indices of ``recv`` grouped so that wave k holds the k-th occurrence of every receiver."""
        if recv.size == 0:
            return []
        order = np.argsort(recv, kind="stable")
        sorted_r = recv[order]
        first = np.r_[True, sorted_r[1:] != sorted_r[:-1]]
        start = np.maximum.accumulate(np.where(first, np.arange(recv.size), 0))
        rank = np.empty(recv.size, dtype=np.int64)
        rank[order] = np.arange(recv.size) - start
        return [np.flatnonzero(rank == k) for k in range(int(rank.max()) + 1)]

    def run_round(self, events: np.ndarray, C: Any) -> Tuple[List[int], Dict[str, int]]:
        """Execute one round's event list; returns (nodes to evaluate, message counters)."""
        if self.multi:
            return self._run_round_multi(events, C)
        kind, tick, a, b, slot, aux = (events[:, i] for i in range(6))
        counters = {"sent": 0, "sent_size": 0, "failed": 0}
        evals: List[int] = []
        if events.shape[0] == 0:
            return evals, counters
        bounds = np.flatnonzero(np.r_[True, tick[1:] != tick[:-1], True])
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            k, ea, eb, es, ex = kind[lo:hi], a[lo:hi], b[lo:hi], slot[lo:hi], aux[lo:hi]
            # ---- phase A: sends (a snapshot per model-carrying message) -------------------------------
            m = k == C.EV_SEND
            if m.any():
                senders, mids, mtypes = ea[m], es[m], ex[m]
                carries = mtypes != 2                                   # 2 = PULL request
                if self.cacheneigh:                                     # consume one cached model before the snapshot
                    cn_nodes, cn_slots = self._cn_pick(senders, mtypes)
                    self._deliver(cn_nodes, cn_slots)
                    self._release(cn_slots)
                slots = np.full(senders.size, -1, dtype=np.int64)
                slots[carries] = self._alloc(int(carries.sum()))
                self.slot_map[mids % _RING] = slots
                self._snapshot(senders, slots)
                counters["sent"] += int(senders.size)
                counters["sent_size"] += int(carries.sum()) * self.size_model + int((~carries).sum())
            # ---- phase B: deliveries (+ the replies they trigger), conflict-free waves ---------------
            m = k == C.EV_DELIVER
            if m.any():
                origin, recv, mids = ea[m], eb[m], es[m]
                # replies: EV_REPLY_SEND(slot = request id, aux = reply id) follows its delivery
                rs = k == C.EV_REPLY_SEND
                req_ids, rep_ids = es[rs], ex[rs]
                has_reply = np.isin(mids, req_ids) if req_ids.size else np.zeros(mids.size, dtype=bool)
                rep_of = None
                if req_ids.size:
                    srt = np.argsort(req_ids)
                    pos_in = np.searchsorted(req_ids[srt], mids[has_reply])
                    rep_of = np.full(mids.size, -1, dtype=np.int64)
                    rep_of[has_reply] = rep_ids[srt][pos_in]
                for idx in ([np.arange(recv.size)] if self.cacheneigh else self._waves(recv)):
                    r_w, mid_w = recv[idx], mids[idx]
                    s_w = self.slot_map[mid_w % _RING].copy()
                    if self.cacheneigh:                                 # only stored (newest per sender)
                        self._release(self._cn_store(r_w, origin[idx], s_w))
                    else:
                        self._deliver(r_w, s_w, self._item_modes(r_w, origin[idx], s_w))
                        self._release(s_w)
                    if rep_of is not None:
                        sel = has_reply[idx]
                        if sel.any():
                            rslots = self._alloc(int(sel.sum()))
                            self.slot_map[rep_of[idx][sel] % _RING] = rslots
                            self._snapshot(r_w[sel], rslots)
            # ---- phase C: replies delivered ------------------------------------------------------------
            m = k == C.EV_REPLY_DELIVER
            if m.any():
                recv, repl, mids = ea[m], eb[m], es[m]
                counters["sent"] += int(recv.size)
                counters["sent_size"] += int(recv.size) * self.size_model
                for idx in ([np.arange(recv.size)] if self.cacheneigh else self._waves(recv)):
                    s_w = self.slot_map[mids[idx] % _RING].copy()
                    if self.cacheneigh:
                        self._release(self._cn_store(recv[idx], repl[idx], s_w))
                    else:
                        self._deliver(recv[idx], s_w, self._item_modes(recv[idx], repl[idx], s_w))
                        self._release(s_w)
            # ---- losses: free the snapshot -------------------------------------------------------------
            m = k == C.EV_DROP
            if m.any():
                counters["failed"] += int(m.sum())
                dropped = self.slot_map[es[m] % _RING].copy()
                self.slot_map[es[m] % _RING] = -1
                self._release(dropped)
            m = k == C.EV_EVAL
            if m.any():
                evals.extend(ea[m].tolist())
        return evals, counters

    # -- checkpointing -----------------------------------------------------------------------------
    def export_inflight(self, message_ids: List[int], receivers: Optional[List[int]] = None) -> Dict[str, Any]:
        """Snapshots of the messages that are still on the wire (ids from the scheduler's queues; ``receivers`` = the
        node each of them travels to).  Several ranks: a snapshot lives in the bank of its receiver's rank, so every
        rank contributes its part and all ranks end up with the complete set (every rank writes a full checkpoint)."""
        ids = np.asarray(message_ids, dtype=np.int64)
        recv = np.asarray(receivers if receivers is not None else np.zeros(ids.size), dtype=np.int64)
        slots = self.slot_map[ids % _RING] if ids.size else np.zeros(0, dtype=np.int64)
        keep = slots >= 0
        ids, slots, recv = ids[keep], slots[keep], recv[keep]
        ent = []
        if self.cacheneigh:                 # models waiting in the neighbour caches are state as well
            ent = [(n, s, sl) for n, cache in enumerate(self.cn_cache) for s, sl in sorted(cache.items())]
        if self.multi:
            return self._export_inflight_multi(ids, slots, recv, ent)
        idx = torch.as_tensor(slots, dtype=torch.int64, device=self.device)
        out = {"ids": ids, "receivers": recv, "rows": self.S[idx].cpu(), "ages": self.slot_age[idx].cpu()}
        if self.cacheneigh:
            cidx = torch.as_tensor([e[2] for e in ent], dtype=torch.int64, device=self.device)
            out["cn"] = {"nodes": [e[0] for e in ent], "senders": [e[1] for e in ent],
                         "rows": self.S[cidx].cpu(), "ages": self.slot_age[cidx].cpu()}
        return out

    def _place(self, dst_nodes: np.ndarray, rows: torch.Tensor, ages: torch.Tensor) -> Tuple[np.ndarray, np.ndarray]:
        """Slots for restored snapshots that travel to / are cached at ``dst_nodes``; returns (slots, ranks)."""
        k = int(dst_nodes.size)
        if not self.multi:
            slots = self._alloc(k)
            idx = torch.as_tensor(slots, dtype=torch.int64, device=self.device)
            self.S[idx] = rows.to(self.device)
            self.slot_age[idx] = ages.to(self.device)
            return slots, np.zeros(k, dtype=np.int64)
        ranks = self.owner[dst_nodes]
        slots = self._alloc_multi(ranks)            # replicated bookkeeping; every rank fills the slots of its own bank
        mine = ranks == self.rank
        if mine.any():
            idx = torch.as_tensor(slots[mine], dtype=torch.int64, device=self.device)
            sel = torch.as_tensor(np.flatnonzero(mine), dtype=torch.int64)
            self.S[idx] = rows[sel].to(self.device)
            self.slot_age[idx] = ages[sel].to(self.device)
        return slots, ranks

    def import_inflight(self, st: Dict[str, Any]) -> None:
        cn = st.get("cn")
        if cn is not None and len(cn["nodes"]):
            slots, _ = self._place(np.asarray(cn["nodes"], dtype=np.int64), cn["rows"], cn["ages"])
            for n, s, sl in zip(cn["nodes"], cn["senders"], slots.tolist()):
                self.cn_cache[n][s] = sl
        ids = np.asarray(st["ids"], dtype=np.int64)
        if ids.size == 0:
            return
        recv = np.asarray(st.get("receivers", np.zeros(ids.size)), dtype=np.int64)
        slots, ranks = self._place(recv, st["rows"], st["ages"])
        self.slot_map[ids % _RING] = slots
        if self.multi:
            self.slot_rank[ids % _RING] = ranks

    def drop_inflight(self) -> None:
        """A fresh ``start`` forgets the messages on the wire: every slot that is not a cached model (cache-neighbour nodes:
        node state) goes back to its pool.  Replicated bookkeeping, no device work."""
        cached = [dict() for _ in range(self.world)]
        if self.cacheneigh:
            for node, cache in enumerate(self.cn_cache):
                for sl in cache.values():
                    cached[int(self.owner[node]) if self.multi else 0][int(sl)] = True
        self.slot_map[:] = -1
        if self.multi:
            for r in range(self.world):
                free = np.asarray([s for s in range(self.cap - 1, -1, -1) if s not in cached[r]], dtype=np.int64)
                self.free_r[r], self.n_free_r[r], self.pending_r[r] = free, int(free.size), []
        else:
            self.free = np.asarray([s for s in range(self.cap - 1, -1, -1) if s not in cached[0]], dtype=np.int64)
            self.n_free = int(self.free.size)

class LinearBank(_SlotBank):
    def __init__(self, sim) -> None:
        from ..model.handler import PegasosHandler
        self.sim = sim
        ids = sorted(sim.nodes)
        self.n = len(ids)
        h0 = sim.nodes[ids[0]].model_handler
        self.device = h0.device
        self.D = int(h0.dim)
        self.Dp = (self.D + 31) // 32 * 32
        self.kind = 1 if isinstance(h0, PegasosHandler) else 0
        self.mode = _MODE[h0.mode]
        self.lr = float(h0.learning_rate)
        dev = self.device
        from ..parallel import runtime as prt
        self.multi = prt.active()
        self.world = prt.world() if self.multi else 1
        self.rank = prt.rank() if self.multi else 0
        # several ranks: every rank keeps the whole index space (N x Dp floats is small) but only the rows of ITS nodes
        # are live; the event list and all slot bookkeeping are replicated, the launches cover the own nodes
        self.owner = np.asarray([prt.rank_of(i) if self.multi else 0 for i in ids], dtype=np.int64)
        # models and ages
        self.W = torch.zeros(self.n, self.Dp, dtype=torch.float32, device=dev)
        self.age = torch.zeros(self.n, dtype=torch.int64, device=dev)
        for i in ids:
            h = sim.nodes[i].model_handler
            if self.owner[i] == self.rank:
                self.W[i, :self.D].copy_(h.row[:self.D])
            self.age[i] = int(h.n_updates)
        # data: all shards concatenated
        xs, ys, off, cnt = [], [], [], []
        pos = 0
        for i in ids:
            x, y = sim.nodes[i].data[0]
            x = torch.as_tensor(np.asarray(x) if not isinstance(x, torch.Tensor) else x, dtype=torch.float32)
            y = torch.as_tensor(np.asarray(y) if not isinstance(y, torch.Tensor) else y, dtype=torch.float32)
            x = x.reshape(-1, self.D)
            xs.append(x); ys.append(y.reshape(-1))
            off.append(pos); cnt.append(x.shape[0]); pos += x.shape[0]
        self.X = torch.cat(xs).contiguous().to(dev)
        self.y = torch.cat(ys).contiguous().to(dev)
        self.off = torch.tensor(off, dtype=torch.int64, device=dev)
        self.cnt = torch.tensor(cnt, dtype=torch.int32, device=dev)
        self.max_cnt = int(max(cnt)) if cnt else 0
        # snapshot slots
        self.cap = max(64, 4 * self.n)
        self.slot_map = np.full(_RING, -1, dtype=np.int64)            # message id (mod ring) -> slot
        if self.multi:
            self._init_shared_slots()
        else:
            self._init_slots(self.cap)
        # evaluation set
        self.Xte = self.yte = None
        if sim.data_dispatcher.has_test():
            Xte, yte = sim.data_dispatcher.get_eval_set()
            self.Xte = torch.as_tensor(Xte, dtype=torch.float32).reshape(-1, self.D).contiguous().to(dev)
            self.yte = torch.as_tensor(yte).reshape(-1).to(dev)
        self.size_model = int(h0.get_size())
        # PassThroughNode (Giaretta 2019): the sender's degree rides along; the receiver merges with probability
        # min(1, deg_sender / deg_self), else adopts the model untouched -- a keyed draw per delivery (node.py::_accepts)
        from ..node import PassThroughNode
        self.passthrough = type(sim.nodes[ids[0]]) is PassThroughNode
        if self.passthrough:
            self.deg = np.asarray([int(sim.nodes[i].n_neighs) for i in ids], dtype=np.uint64)
            self.pt_count = np.asarray([int(getattr(sim.nodes[i], "_pt_draws", 0)) for i in ids], dtype=np.uint64)
            self.size_model += 1                    # the degree is one more atom on the wire
        # CacheNeighNode (Giaretta 2019): received models are only stored, newest per sender; at a PUSH / PUSH_PULL send one
        # cached model (keyed choice among the senders in the cache) is consumed before the snapshot (node.py::CacheNeighNode)
        from ..node import CacheNeighNode
        self.cacheneigh = type(sim.nodes[ids[0]]) is CacheNeighNode
        if self.cacheneigh:
            self.cn_cache: List[Dict[int, int]] = [dict() for _ in ids]      # node -> {sender: slot}
            self.cn_count = [int(getattr(sim.nodes[i], "_cn_draws", 0)) for i in ids]

    def _cn_store(self, recvs: np.ndarray, senders: np.ndarray, slots: np.ndarray) -> np.ndarray:
        """Deliveries to cache-neighbour nodes: remember the slot, return the slots of the models they replace."""
        stale, owners = [], []
        for r, s, sl in zip(recvs.tolist(), senders.tolist(), slots.tolist()):
            if sl < 0:
                continue
            old = self.cn_cache[r].get(s)
            if old is not None:
                stale.append(old)
                owners.append(r)
            self.cn_cache[r][s] = sl
        self._cn_stale_nodes = np.asarray(owners, dtype=np.int64)      # (several ranks: a slot lives on its receiver's rank)
        return np.asarray(stale, dtype=np.int64)

    def _cn_pick(self, senders: np.ndarray, mtypes: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
        """Sends of cache-neighbour nodes: (nodes, slots) of the cached models consumed before the snapshots."""
        from . import rng as _rng
        nodes, slots = [], []
        for a, mt in zip(senders.tolist(), mtypes.tolist()):
            cache = self.cn_cache[a]
            if mt == 2 or not cache:            # PULL requests do not consume
                continue
            keys = sorted(cache)
            k = keys[_rng.derive(0x9A59, a, self.cn_count[a]) % len(keys)]
            self.cn_count[a] += 1
            nodes.append(a)
            slots.append(cache.pop(k))
        return np.asarray(nodes, dtype=np.int64), np.asarray(slots, dtype=np.int64)

    def _item_modes(self, recvs: np.ndarray, senders: np.ndarray, slots: np.ndarray) -> Optional[np.ndarray]:
        """Per delivered message: the bank's mode (merge) or 4 (PASS), from the receivers' keyed draws."""
        if not self.passthrough:
            return None
        from ..ops.torch_ref import _mix64_np
        from . import rng as _rng
        carries = slots >= 0
        r = recvs.astype(np.int64)
        k = self.pt_count[r]
        h = np.uint64(_rng.mix64(_rng.mix64(_rng.base_seed()) ^ 0x9A55))
        u = _mix64_np(_mix64_np(h ^ r.astype(np.uint64)) ^ k)
        u = (u & np.uint64((1 << 63) - 1)) >> np.uint64(20)
        accept = u * self.deg[r] < (self.deg[senders.astype(np.int64)] << np.uint64(43))
        self.pt_count[r[carries]] += np.uint64(1)   # (a receiver appears once per wave)
        return np.where(accept, self.mode, 4).astype(np.int32)

    # -- several ranks: slot banks in shared memory, snapshots pushed to the receiver's rank ----------------------
    def _init_shared_slots(self) -> None:
        """One allocation per rank, mapped into every process (CUDA IPC; POSIX shared memory on CPU):
        ``S[cap][Dp]`` fp32 | ``slot_age[cap]`` int64 | barrier generations ``[16]`` uint32.  A message's snapshot lives in
        the bank of the RECEIVER's rank: the sender's rank pushes it there (stores over NVLink), deliveries read local
        memory only.  Slots are allocated from per-rank pools by replicated bookkeeping (identical on every rank)."""
        import torch.distributed as dist
        from ..parallel import runtime as prt
        cap, Dp, W = self.cap, self.Dp, self.world
        off_age = cap * Dp * 4
        off_flag = off_age + cap * 8
        total = off_flag + 64
        self._gen = 0
        self.slot_rank = np.zeros(_RING, dtype=np.int64)              # message id (mod ring) -> rank of its slot
        self.free_r = [np.arange(cap - 1, -1, -1, dtype=np.int64) for _ in range(W)]
        self.n_free_r = [cap] * W
        self.pending_r: List[List[np.ndarray]] = [[] for _ in range(W)]   # released, reusable after the next barrier
        if self.device.type == "cuda":
            from ..ops.native import native
            nat = native()
            torch.cuda.set_device(self.device)
            base = nat.ipc_alloc(total)
            dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
            nat.tensor_from_ptr(base, [total // 4], dev_index, True).zero_()
            torch.cuda.synchronize(self.device)
            handles: List = [None] * W
            dist.all_gather_object(handles, nat.ipc_get_handle(base))
            bases = [base if r == self.rank else nat.ipc_open_handle(handles[r]) for r in range(W)]
            dist.barrier()
            self._peer_S = [int(bptr) for bptr in bases]
            self._peer_age = [int(bptr) + off_age for bptr in bases]
            self._peer_flags = [int(bptr) + off_flag for bptr in bases]
            self.S = nat.tensor_from_ptr(base, [cap, Dp], dev_index, False)
            self.slot_age = nat.tensor_from_ptr(base + off_age, [2 * cap], dev_index, True).view(torch.int64)
        else:
            from multiprocessing import shared_memory
            global _BANK_SEQ                  # (a resumed checkpoint builds a second bank in the same session)
            _BANK_SEQ += 1
            names = ["gb200_bank_%s_%d_%d" % (prt.session_tag(), _BANK_SEQ, r) for r in range(W)]
            mine = shared_memory.SharedMemory(name=names[self.rank], create=True, size=total)
            _arena._unlink_at_exit()
            np.frombuffer(mine.buf, dtype=np.uint8)[:] = 0
            dist.barrier()
            self._shm = [mine if r == self.rank else _arena.attach_shm(names[r]) for r in range(W)]
            dist.barrier()
            _OPEN.append(self)
            self._S_of = [torch.frombuffer(sh.buf, dtype=torch.float32, count=cap * Dp).view(cap, Dp) for sh in self._shm]
            self._age_of = [torch.frombuffer(sh.buf, dtype=torch.int64, count=cap, offset=off_age) for sh in self._shm]
            self.S, self.slot_age = self._S_of[self.rank], self._age_of[self.rank]

    def close(self) -> None:
        """Release the shared-memory mappings (CPU runs; CUDA IPC allocations live until the process ends)."""
        shm = self.__dict__.pop("_shm", None)
        if shm is None:
            return
        self.__dict__.pop("_S_of", None)
        self.__dict__.pop("_age_of", None)
        self.S = self.slot_age = None
        for r, sh in enumerate(shm):
            if r == self.rank:
                try:
                    sh.unlink()
                except Exception:
                    pass
            try:
                sh.close()
            except Exception:      # tensors created with torch.frombuffer may still reference the mapping
                pass

    def _barrier(self) -> None:
        """All ranks: what was pushed before is visible, what was read before may be overwritten.  On a GPU a
        stream-ordered flag barrier over NVLink (one small kernel, no host synchronisation)."""
        if self.device.type == "cuda":
            from ..ops.native import native
            self._gen += 1
            native().rank_barrier(self._peer_flags, self.rank, self._gen)
            ops._count()
        else:
            import torch.distributed as dist
            dist.barrier()
        for r in range(self.world):                       # slots released before the barrier may be written again
            for sl in self.pending_r[r]:
                k = sl.size
                if self.n_free_r[r] + k > self.free_r[r].size:
                    self.free_r[r] = np.concatenate([self.free_r[r], np.empty(self.n_free_r[r] + k - self.free_r[r].size, dtype=np.int64)])
                self.free_r[r][self.n_free_r[r]:self.n_free_r[r] + k] = sl
                self.n_free_r[r] += k
            self.pending_r[r] = []

    def _alloc_multi(self, dst: np.ndarray) -> np.ndarray:
        out = np.empty(dst.size, dtype=np.int64)
        for r in np.unique(dst):
            sel = dst == r
            k = int(sel.sum())
            if self.n_free_r[r] < k:
                self._barrier()                           # (replicated decision) recycle what was released since
            if self.n_free_r[r] < k:
                raise RuntimeError("banked engine: more than %d messages in flight towards rank %d" % (self.cap, r))
            out[sel] = self.free_r[r][self.n_free_r[r] - k:self.n_free_r[r]]
            self.n_free_r[r] -= k
        return out

    def _release_multi(self, slots: np.ndarray, ranks: np.ndarray) -> None:
        keep = slots >= 0
        slots, ranks = slots[keep], ranks[keep]
        for r in np.unique(ranks):
            self.pending_r[r].append(slots[ranks == r].copy())

    def _snapshot_multi(self, senders: np.ndarray, slots: np.ndarray, dst: np.ndarray) -> bool:
        """Push the snapshots of MY senders into the banks of their receivers' ranks; returns whether the phase has
        cross-rank traffic (a replicated fact: then every rank runs the barrier)."""
        carries = slots >= 0
        cross = bool(np.any(carries & (self.owner[senders] != dst)))
        mine = carries & (self.owner[senders] == self.rank)
        if mine.any():
            s, d, r = senders[mine], slots[mine], dst[mine]
            if self.device.type == "cuda":
                from ..ops.native import native
                native().bank_snapshot_push(*self._args(), self._peer_S, self._peer_age, self._idx(s), self._idx(d), self._idx(r))
                ops._count()
            else:
                st = torch.as_tensor(s, dtype=torch.int64)
                for q in np.unique(r):
                    sel = r == q
                    dd = torch.as_tensor(d[sel], dtype=torch.int64)
                    self._S_of[q][dd] = self.W[st[torch.as_tensor(sel)]]
                    self._age_of[q][dd] = self.age[st[torch.as_tensor(sel)]]
        return cross

    def _deliver_multi(self, recvs: np.ndarray, slots: np.ndarray, modes=None) -> None:
        mine = self.owner[recvs] == self.rank
        if mine.any():
            self._deliver(recvs[mine], slots[mine], None if modes is None else modes[mine])

    # -- low level ops (CUDA kernels / torch on CPU) ---------------------------------------------
    def _args(self):
        return (self.W, self.age, self.S, self.slot_age, self.X, self.y, self.off, self.cnt, self.D, self.kind,
                self.mode, self.lr)

    def _snapshot(self, senders, slots) -> None:
        if len(senders) == 0:
            return
        if self.device.type == "cuda":
            from ..ops.native import native
            native().bank_snapshot(*self._args(), self._idx(senders), self._idx(slots))
            ops._count()
            return
        s = torch.as_tensor(np.asarray(senders), dtype=torch.int64)
        d = torch.as_tensor(np.asarray(slots), dtype=torch.int64)
        keep = d >= 0
        self.S[d[keep]] = self.W[s[keep]]
        self.slot_age[d[keep]] = self.age[s[keep]]

    def _update_cpu(self, w: torch.Tensor, age: torch.Tensor, nodes: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """Vectorised over nodes: step i of every node's sequential pass happens at once."""
        cnt = self.cnt[nodes].long()
        off = self.off[nodes]
        for i in range(int(cnt.max()) if cnt.numel() else 0):
            live = cnt > i
            if not bool(live.any()):
                break
            rows = (off + i)[live]
            x = torch.zeros(int(live.sum()), self.Dp)
            x[:, :self.D] = self.X[rows]
            ys = self.y[rows]
            wl = w[live]
            yhat = (wl * x).sum(1)
            if self.kind == 0:
                wl = wl + (self.lr * (ys - yhat))[:, None] * x
                age[live] += 1
            else:
                age[live] += 1
                eta = 1.0 / (age[live].float() * self.lr)
                wl = wl * (1.0 - eta * self.lr)[:, None]
                hit = (yhat * ys - 1.0) < 0
                wl = wl + (hit.float() * eta * ys)[:, None] * x
            w[live] = wl
        return w, age

    def _deliver(self, recvs, slots, modes=None) -> None:
        if len(recvs) == 0:
            return
        if self.device.type == "cuda":
            from ..ops.native import native
            native().bank_deliver(*self._args(), self._idx(recvs), self._idx(slots),
                                  None if modes is None else self._idx(modes))
            ops._count()
            return
        if modes is not None:                       # per-message modes: one vectorised pass per mode
            modes = np.asarray(modes)
            saved = self.mode
            try:
                for m in np.unique(modes):
                    sel = modes == m
                    self.mode = int(m)
                    self._deliver(np.asarray(recvs)[sel], np.asarray(slots)[sel])
            finally:
                self.mode = saved
            return
        r = torch.as_tensor(np.asarray(recvs), dtype=torch.int64)
        s = torch.as_tensor(np.asarray(slots), dtype=torch.int64)
        keep = s >= 0
        r, s = r[keep], s[keep]
        if r.numel() == 0:
            return
        w, sv = self.W[r].clone(), self.S[s].clone()
        aw, asn = self.age[r].clone(), self.slot_age[s].clone()
        if self.mode == 1:
            w, aw = sv, asn
            w, aw = self._update_cpu(w, aw, r)
        elif self.mode == 2:
            w = 0.5 * (w + sv)
            aw = torch.maximum(aw, asn)
            w, aw = self._update_cpu(w, aw, r)
        elif self.mode == 3:
            w, aw = self._update_cpu(w, aw, r)
            sv, asn = self._update_cpu(sv, asn, r)
            w = 0.5 * (w + sv)
            aw = torch.maximum(aw, asn)
        else:
            w = sv
        self.W[r] = w
        self.age[r] = aw

    def _scores(self, nodes) -> torch.Tensor:
        if self.device.type == "cuda":
            from ..ops.native import native
            out = native().bank_scores(*self._args(), self._idx(nodes), self.Xte)
            ops._count()
            return out
        idx = torch.as_tensor(np.asarray(nodes), dtype=torch.int64)
        return self.W[idx, :self.D] @ self.Xte.t()

    # -- one round, several ranks -----------------------------------------------------------------------
    def _run_round_multi(self, events: np.ndarray, C: Any) -> Tuple[List[int], Dict[str, int]]:
        """``run_round`` with the nodes spread over several ranks: same phases, every rank launches the work of its own
        nodes; a phase that pushed snapshots across ranks ends with a barrier."""
        kind, tick, a, b, slot, aux = (events[:, i] for i in range(6))
        counters = {"sent": 0, "sent_size": 0, "failed": 0}
        evals: List[int] = []
        if events.shape[0] == 0:
            return evals, counters
        own = self.owner
        bounds = np.flatnonzero(np.r_[True, tick[1:] != tick[:-1], True])
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            k, ea, eb, es, ex = kind[lo:hi], a[lo:hi], b[lo:hi], slot[lo:hi], aux[lo:hi]
            m = k == C.EV_SEND
            if m.any():
                senders, recvs, mids, mtypes = ea[m], eb[m], es[m], ex[m]
                carries = mtypes != 2
                if self.cacheneigh:
                    cn_nodes, cn_slots = self._cn_pick(senders, mtypes)
                    if cn_nodes.size:
                        self._deliver_multi(cn_nodes, cn_slots)
                        self._release_multi(cn_slots, own[cn_nodes])
                dst = own[recvs]
                slots = np.full(senders.size, -1, dtype=np.int64)
                if carries.any():
                    slots[carries] = self._alloc_multi(dst[carries])
                self.slot_map[mids % _RING] = slots
                self.slot_rank[mids % _RING] = dst
                if self._snapshot_multi(senders, slots, dst):
                    self._barrier()
                counters["sent"] += int(senders.size)
                counters["sent_size"] += int(carries.sum()) * self.size_model + int((~carries).sum())
            m = k == C.EV_DELIVER
            if m.any():
                origin, recv, mids = ea[m], eb[m], es[m]
                rs = k == C.EV_REPLY_SEND
                req_ids, rep_ids = es[rs], ex[rs]
                has_reply = np.isin(mids, req_ids) if req_ids.size else np.zeros(mids.size, dtype=bool)
                rep_of = None
                if req_ids.size:
                    srt = np.argsort(req_ids)
                    pos_in = np.searchsorted(req_ids[srt], mids[has_reply])
                    rep_of = np.full(mids.size, -1, dtype=np.int64)
                    rep_of[has_reply] = rep_ids[srt][pos_in]
                for idx in ([np.arange(recv.size)] if self.cacheneigh else self._waves(recv)):
                    r_w, mid_w = recv[idx], mids[idx]
                    s_w = self.slot_map[mid_w % _RING].copy()
                    if self.cacheneigh:
                        stale = self._cn_store(r_w, origin[idx], s_w)
                        self._release_multi(stale, own[self._cn_stale_nodes])
                    else:
                        self._deliver_multi(r_w, s_w, self._item_modes(r_w, origin[idx], s_w))
                        self._release_multi(s_w, own[r_w])
                    if rep_of is not None:
                        sel = has_reply[idx]
                        if sel.any():
                            dst = own[origin[idx][sel]]
                            rslots = self._alloc_multi(dst)
                            self.slot_map[rep_of[idx][sel] % _RING] = rslots
                            self.slot_rank[rep_of[idx][sel] % _RING] = dst
                            if self._snapshot_multi(r_w[sel], rslots, dst):
                                self._barrier()
            m = k == C.EV_REPLY_DELIVER
            if m.any():
                recv, repl, mids = ea[m], eb[m], es[m]
                counters["sent"] += int(recv.size)
                counters["sent_size"] += int(recv.size) * self.size_model
                for idx in ([np.arange(recv.size)] if self.cacheneigh else self._waves(recv)):
                    s_w = self.slot_map[mids[idx] % _RING].copy()
                    if self.cacheneigh:
                        stale = self._cn_store(recv[idx], repl[idx], s_w)
                        self._release_multi(stale, own[self._cn_stale_nodes])
                    else:
                        self._deliver_multi(recv[idx], s_w, self._item_modes(recv[idx], repl[idx], s_w))
                        self._release_multi(s_w, own[recv[idx]])
            m = k == C.EV_DROP
            if m.any():
                counters["failed"] += int(m.sum())
                dropped = self.slot_map[es[m] % _RING].copy()
                self.slot_map[es[m] % _RING] = -1
                self._release_multi(dropped, self.slot_rank[es[m] % _RING])
            m = k == C.EV_EVAL
            if m.any():
                evals.extend(ea[m].tolist())
        return evals, counters

    # -- evaluation ------------------------------------------------------------------------------------
    def evaluate(self, nodes: List[int]) -> List[Dict[str, float]]:
        """Metric dicts of ``nodes`` on the global evaluation set: one scores launch, metrics (incl. the
        rank-based AUC with average ranks for ties) vectorised over the nodes on the device, one read-back."""
        if not nodes or self.Xte is None:
            return []
        if self.multi:                      # every rank scores its own nodes; one small all-reduce merges the dicts
            from ..parallel import runtime as prt
            mine = [i for i in nodes if self.owner[i] == self.rank]
            part = dict(zip(mine, self._evaluate_local(mine))) if mine else {}
            return prt.share_metrics([part.get(i) for i in nodes])
        return self._evaluate_local(nodes)

    def _evaluate_local(self, nodes: List[int]) -> List[Dict[str, float]]:
        scores = self._scores(nodes)                                   # [E, T]
        E, T = scores.shape
        pos = (self.yte > 0)
        pred = scores >= 0
        tp = (pred & pos[None, :]).sum(1).double()
        fp = (pred & ~pos[None, :]).sum(1).double()
        fn = (~pred & pos[None, :]).sum(1).double()
        tn = (~pred & ~pos[None, :]).sum(1).double()
        # AUC = (rank sum of positives - n+(n+ + 1)/2) / (n+ n-), average ranks inside tie groups
        srt, order = torch.sort(scores.double(), dim=1)
        pos_sorted = pos[order].double()
        idx = torch.arange(T, device=scores.device).expand(E, T)
        first = torch.ones(E, T, dtype=torch.bool, device=scores.device)
        first[:, 1:] = srt[:, 1:] != srt[:, :-1]
        last = torch.ones(E, T, dtype=torch.bool, device=scores.device)
        last[:, :-1] = srt[:, :-1] != srt[:, 1:]
        start = torch.cummax(torch.where(first, idx, torch.zeros_like(idx)), dim=1).values
        end = torch.flip(torch.cummin(torch.flip(torch.where(last, idx, torch.full_like(idx, T - 1)), [1]), dim=1).values, [1])
        rank = (start + end).double() / 2.0 + 1.0
        n_pos = float(pos.sum())
        n_neg = float(T) - n_pos
        if n_pos == 0 or n_neg == 0:
            auc = torch.full((E,), 0.5, dtype=torch.float64, device=scores.device)
        else:
            auc = ((rank * pos_sorted).sum(1) - n_pos * (n_pos + 1) / 2.0) / (n_pos * n_neg)
        stats = torch.stack([tn, fp, fn, tp, auc], 1).cpu().numpy()
        tn, fp, fn, tp, auc = (stats[:, i] for i in range(5))
        total = tn + fp + fn + tp
        with np.errstate(divide="ignore", invalid="ignore"):
            # class 0 = negative, class 1 = positive; macro average over the classes that occur (sklearn)
            p1 = np.where(tp + fp > 0, tp / (tp + fp), 0.0); r1 = np.where(tp + fn > 0, tp / (tp + fn), 0.0)
            p0 = np.where(tn + fn > 0, tn / (tn + fn), 0.0); r0 = np.where(tn + fp > 0, tn / (tn + fp), 0.0)
            f1_1 = np.where(p1 + r1 > 0, 2 * p1 * r1 / (p1 + r1), 0.0)
            f1_0 = np.where(p0 + r0 > 0, 2 * p0 * r0 / (p0 + r0), 0.0)
            pres1 = ((tp + fp) + (tp + fn)) > 0
            pres0 = ((tn + fn) + (tn + fp)) > 0
            kk = np.maximum(pres1.astype(float) + pres0.astype(float), 1.0)
            acc = np.where(total > 0, (tp + tn) / total, 0.0)
            prec = (p1 * pres1 + p0 * pres0) / kk
            recl = (r1 * pres1 + r0 * pres0) / kk
            f1 = (f1_1 * pres1 + f1_0 * pres0) / kk
        return [{"accuracy": float(acc[e]), "precision": float(prec[e]), "recall": float(recl[e]),
                 "f1_score": float(f1[e]), "auc": float(auc[e])} for e in range(E)]

    # -- checkpointing, several ranks --------------------------------------------------------------------
    def _export_inflight_multi(self, ids: np.ndarray, slots: np.ndarray, recv: np.ndarray, ent: List) -> Dict[str, Any]:
        import torch.distributed as dist
        self._barrier()                     # everything pushed towards this rank has landed
        if self.device.type == "cuda":
            torch.cuda.synchronize(self.device)

        def local(sl: np.ndarray):
            idx = torch.as_tensor(sl, dtype=torch.int64, device=self.device)
            return self.S[idx].cpu().clone(), self.slot_age[idx].cpu().clone()
        mine = self.slot_rank[ids % _RING] == self.rank
        part: Dict[str, Any] = {"ids": ids[mine], "receivers": recv[mine]}
        part["rows"], part["ages"] = local(slots[mine])
        own_ent = [e for e in ent if self.owner[e[0]] == self.rank]       # a cached model sits on its holder's rank
        part["cn_nodes"], part["cn_senders"] = [e[0] for e in own_ent], [e[1] for e in own_ent]
        part["cn_rows"], part["cn_ages"] = local(np.asarray([e[2] for e in own_ent], dtype=np.int64))
        parts: List[Any] = [None] * self.world
        dist.all_gather_object(parts, part)
        out = {"ids": np.concatenate([q["ids"] for q in parts]), "receivers": np.concatenate([q["receivers"] for q in parts]),
               "rows": torch.cat([q["rows"] for q in parts]), "ages": torch.cat([q["ages"] for q in parts])}
        if self.cacheneigh:
            out["cn"] = {"nodes": [n for q in parts for n in q["cn_nodes"]], "senders": [x for q in parts for x in q["cn_senders"]],
                         "rows": torch.cat([q["cn_rows"] for q in parts]), "ages": torch.cat([q["cn_ages"] for q in parts])}
        return out

    def writeback(self) -> None:
        W = self.W[:, :self.D]
        age = self.age
        if self.multi:                      # ages of the other ranks' nodes (device results): one all-reduce per run
            import torch.distributed as dist
            mask = torch.as_tensor(self.owner == self.rank, device=age.device)
            age = torch.where(mask, age, torch.zeros_like(age))
            dist.all_reduce(age)
        ages = age.cpu().tolist()
        for i, node in self.sim.nodes.items():
            h = node.model_handler
            if self.owner[i] == self.rank:
                h.row[:self.D].copy_(W[i])
            h.n_updates = int(ages[i])
            h._version += 1
            if self.passthrough:
                node._pt_draws = int(self.pt_count[i])
            if self.cacheneigh:
                node._cn_draws = int(self.cn_count[i])
        if self.multi:
            self.age.copy_(age)


# -- k-means and matrix factorisation ------------------------------------------------------------------------------
_SLOT_BYTES = 256 << 20     # first slot-pool allocation of the family banks (the pool grows on demand)


def _family_bankable(sim) -> Optional[str]:
    """:class:`KMeansBank` / :class:`MFBank`: plain ``GossipNode``s on a ``GossipSimulator``, one rank, one handler
    configuration.  Under ``reference_compat`` k-means "hungarian" merges like "naive", as ``KMeansHandler`` does then."""
    from ..model.handler import KMeansHandler, MFModelHandler
    from ..node import GossipNode
    from ..parallel import runtime as prt
    if prt.active():
        return "several ranks (k-means / MF banks run on one rank)"
    if type(sim).__name__ != "GossipSimulator":
        return "simulator variant"
    nodes = list(sim.nodes.values())
    h0 = nodes[0].model_handler
    if isinstance(h0, KMeansHandler):
        key = lambda h: (type(h), h.k, h.dim, h.alpha, h.matching, h.mode)     # noqa: E731
        if h0.matching == "hungarian" and h0.k > 8:
            return "hungarian matching with k > 8"
        if h0.k > 64:
            return "k-means with k > 64"
    else:
        key = lambda h: (type(h), h.k, h.n_items, h.reg, h.lr, h.mode)         # noqa: E731
        if h0.k > 128:
            return "matrix factorisation with k > 128"
    if type(h0) not in (KMeansHandler, MFModelHandler):
        return "handler subclass"
    k0 = key(h0)
    for n in nodes:
        if type(n) is not GossipNode:
            return "node class %s" % type(n).__name__
        if key(n.model_handler) != k0:
            return "heterogeneous handlers"
        if isinstance(h0, KMeansHandler) and n.has_test():
            return "per-node test sets"
    if h0.mode not in _MODE:
        return "unsupported mode"
    if isinstance(h0, KMeansHandler) and not sim.data_dispatcher.has_test():
        return "no evaluation set"
    return None


def make_bank(sim) -> _SlotBank:
    """The bank that executes ``sim`` (which :func:`bankable` accepted)."""
    from ..model.handler import KMeansHandler, MFModelHandler
    h0 = sim.nodes[min(sim.nodes)].model_handler
    if isinstance(h0, KMeansHandler):
        return KMeansBank(sim)
    if isinstance(h0, MFModelHandler):
        return MFBank(sim)
    return LinearBank(sim)


def _np(a: Any) -> np.ndarray:
    return a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


class _FamilyBank(_SlotBank):
    """A bank whose rows are exactly the handlers' arena rows (``h._row_numel`` floats), one CTA per work item on a
    GPU.  Subclasses set up ``data`` / ``off`` / ``cnt`` and implement the delivery and the evaluation."""

    def __init__(self, sim) -> None:
        self.sim = sim
        ids = sorted(sim.nodes)
        self.n = len(ids)
        h0 = sim.nodes[ids[0]].model_handler
        self.device = h0.device
        self.Dp = int(h0._row_numel)
        self.mode = _MODE[h0.mode]
        if self.device.type == "cuda":            # the handlers' rows were written on the nodes' streams
            torch.cuda.synchronize(self.device)
        self.W = torch.stack([sim.nodes[i].model_handler.row for i in ids]).to(self.device).contiguous()
        self.age = torch.tensor([int(sim.nodes[i].model_handler.n_updates) for i in ids], dtype=torch.int64,
                                device=self.device)
        self.slot_map = np.full(_RING, -1, dtype=np.int64)            # message id (mod ring) -> slot
        self._init_slots(max(64, min(4 * self.n, _SLOT_BYTES // (4 * self.Dp))))
        self.size_model = int(h0.get_size())

    @staticmethod
    def _concat(parts: List[np.ndarray], width: int, device) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """Per-node arrays [n_i, width] -> (concatenation as fp32, offsets int64, counts int32) on ``device``."""
        cnt = [int(p.shape[0]) for p in parts]
        off = np.concatenate([[0], np.cumsum(cnt)[:-1]]).astype(np.int64) if cnt else np.zeros(0, np.int64)
        flat = np.concatenate(parts).astype(np.float32) if parts else np.zeros((0, width), np.float32)
        if flat.shape[0] == 0:
            flat = np.zeros((1, width), np.float32)                     # (a valid pointer for the kernels)
        return (torch.from_numpy(np.ascontiguousarray(flat.reshape(-1, width))).to(device),
                torch.from_numpy(off).to(device), torch.tensor(cnt, dtype=torch.int32, device=device))

    def _args(self):
        return (self.W, self.age, self.S, self.slot_age, self.data, self.off, self.cnt, self.k, self.dim, self.mode,
                self.hungarian, self.alpha, self.reg, self.lr)

    def _snapshot(self, senders, slots) -> None:
        if len(senders) == 0:
            return
        if self.device.type == "cuda":
            from ..ops.native import native
            native().family_snapshot(*self._args(), self._idx(senders), self._idx(slots))
            ops._count()
            return
        s = torch.as_tensor(np.asarray(senders), dtype=torch.int64)
        d = torch.as_tensor(np.asarray(slots), dtype=torch.int64)
        keep = d >= 0
        self.S[d[keep]] = self.W[s[keep]]
        self.slot_age[d[keep]] = self.age[s[keep]]

    def _deliver(self, recvs, slots, modes=None) -> None:
        if len(recvs) == 0:
            return
        if self.device.type == "cuda":
            self._deliver_cuda(self._idx(recvs), self._idx(slots))
            ops._count()
            return
        r = torch.as_tensor(np.asarray(recvs), dtype=torch.int64)
        s = torch.as_tensor(np.asarray(slots), dtype=torch.int64)
        keep = s >= 0
        r, s = r[keep], s[keep]
        if r.numel() == 0:
            return
        w, sv = self.W[r].clone(), self.S[s].clone()
        aw, asn = self.age[r].clone(), self.slot_age[s].clone()
        if self.mode == 1:                      # UPDATE: adopt the received model (and its age), train it
            w, aw = sv, asn
            aw = aw + self._update_cpu(w, r)
        elif self.mode == 2:                    # MERGE_UPDATE
            self._merge_cpu(w, sv, aw, asn)
            aw = aw + self._update_cpu(w, r)
        elif self.mode == 3:                    # UPDATE_MERGE: both models train on the local data, then merge
            aw = aw + self._update_cpu(w, r)
            asn = asn + self._update_cpu(sv, r)
            self._merge_cpu(w, sv, aw, asn)
        else:                                   # PASS: adopt untouched, age unchanged
            w = sv
        self.W[r] = w
        self.age[r] = aw

    def evaluate(self, nodes: List[int]) -> List[Dict[str, float]]:
        if not nodes:
            return []
        return self._evaluate(nodes)

    def writeback(self) -> None:
        W = self.W.cpu() if self.device.type == "cpu" else self.W
        ages = self.age.cpu().tolist()
        for i, node in self.sim.nodes.items():
            h = node.model_handler
            h.row.copy_(W[i])
            h.n_updates = int(ages[i])
            h._version += 1
        if self.device.type == "cuda":            # the rows are read next on the nodes' own streams
            torch.cuda.synchronize(self.device)


class KMeansBank(_FamilyBank):
    """Online k-means (``KMeansHandler``): row = the ``k x dim`` centroids, padded; data = every node's local samples,
    concatenated.  Deliveries: merge 0.5 / 0.5 (naive, or after the optimal centroid matching for "hungarian",
    k <= 8), local update = the batched EMA step with the last sample per centroid winning.  Evaluation: the NMI of
    the cluster assignment on the shared evaluation set, one contingency table per node from one launch."""

    def __init__(self, sim) -> None:
        from .. import GlobalSettings
        super().__init__(sim)
        h0 = sim.nodes[min(sim.nodes)].model_handler
        self.k, self.dim, self.alpha = int(h0.k), int(h0.dim), float(h0.alpha)
        # (reference_compat: the reference's "hungarian" is the identity assignment, KMeansHandler._merge)
        self.hungarian = h0.matching == "hungarian" and not GlobalSettings().reference_compat
        self.reg = self.lr = 0.0
        parts = [_np(sim.nodes[i].data[0][0]).reshape(-1, self.dim) for i in sorted(sim.nodes)]
        self.data, self.off, self.cnt = self._concat(parts, self.dim, self.device)
        Xte, yte = sim.data_dispatcher.get_eval_set()
        y_host = _np(yte).reshape(-1).astype(np.int64)
        self.n_true = int(y_host.max()) + 1 if y_host.size else 1
        self.Xte = torch.as_tensor(_np(Xte), dtype=torch.float32).reshape(-1, self.dim).contiguous().to(self.device)
        self.yte = torch.from_numpy(y_host).to(self.device)

    def _deliver_cuda(self, recvs: torch.Tensor, slots: torch.Tensor) -> None:
        from ..ops.native import native
        native().kmeans_bank_deliver(*self._args(), recvs, slots)

    def _update_cpu(self, w: torch.Tensor, nodes: torch.Tensor) -> torch.Tensor:
        """In place on the rows ``w`` [B, Dp], vectorised over the nodes (``torch_ref.kmeans_update``); returns the
        age increments."""
        B, k, d = w.shape[0], self.k, self.dim
        C = w[:, :k * d].view(B, k, d)
        cnt, off = self.cnt[nodes].long(), self.off[nodes]
        m = int(cnt.max())
        if m > 0:
            ar = torch.arange(m)
            valid = ar[None, :] < cnt[:, None]
            X = self.data[(off[:, None] + ar[None, :]).clamp(max=self.data.shape[0] - 1)]        # [B, m, d]
            asg = torch.cdist(X, C, p=2).argmin(dim=2)                                          # [B, m]
            hit = (asg[:, :, None] == torch.arange(k)[None, None, :]) & valid[:, :, None]       # [B, m, k]
            winner = torch.where(hit, ar[None, :, None].expand(B, m, k), torch.full_like(hit, -1, dtype=torch.long)).amax(1)
            sel = winner >= 0
            xw = X[torch.arange(B)[:, None], winner.clamp(min=0)]                                 # [B, k, d]
            C.copy_(torch.where(sel[:, :, None], C * (1 - self.alpha) + self.alpha * xw, C))
        return torch.ones(B, dtype=torch.int64)

    def _merge_cpu(self, w: torch.Tensor, sv: torch.Tensor, aw: torch.Tensor, asn: torch.Tensor) -> None:
        k, d = self.k, self.dim
        if not self.hungarian:
            w.mul_(0.5).add_(sv, alpha=0.5)
            return
        from scipy.optimize import linear_sum_assignment
        for b in range(w.shape[0]):
            own, theirs = w[b, :k * d].view(k, d), sv[b, :k * d].view(k, d)
            cols = linear_sum_assignment(torch.cdist(own, theirs).numpy())[1]
            own.copy_(0.5 * own + 0.5 * theirs[torch.as_tensor(cols)])

    def _evaluate(self, nodes: List[int]) -> List[Dict[str, float]]:
        from ..ops import metrics
        k = self.k
        if self.device.type == "cuda":
            from ..ops.native import native
            ct = native().kmeans_bank_eval(*self._args(), self._idx(nodes), self.Xte, self.yte, self.n_true)
            ops._count()
            cts = ct.cpu().numpy()
        else:
            from ..ops import torch_ref
            cts = []
            for i in nodes:
                pred = torch_ref.kmeans_assign(self.W[i, :k * self.dim].view(k, self.dim), self.Xte)
                cts.append(torch.bincount(self.yte * k + pred.long(), minlength=self.n_true * k)
                           .view(self.n_true, k).numpy())
        return [{"nmi": metrics.nmi_from_contingency(c)} for c in cts]


class MFBank(_FamilyBank):
    """Matrix factorisation (``MFModelHandler``): row = ``[Y (n_items*k) | c (n_items) | X (k) | b (1)]``, padded;
    data = every node's train ratings (item, rating), concatenated, and its own test ratings likewise.  Deliveries:
    the item side ``[Y | c]`` merged with the age weights ``a/(2(a+b))``, ``b/(2(a+b))``, then the sequential SGD over
    the node's ratings.  Evaluation: the RMSE of every evaluated node on its own test ratings (per-node results)."""

    eval_on_user = True

    def __init__(self, sim) -> None:
        super().__init__(sim)
        h0 = sim.nodes[min(sim.nodes)].model_handler
        self.k, self.dim = int(h0.k), int(h0.n_items)
        self.reg, self.lr = float(h0.reg), float(h0.lr)
        self.hungarian, self.alpha = False, 0.0
        self.n_shared = self.dim * self.k + self.dim
        ids = sorted(sim.nodes)
        self.data, self.off, self.cnt = self._concat([_np(sim.nodes[i].data[0]).reshape(-1, 2) for i in ids], 2, self.device)
        self.te, self.te_off, self.te_cnt = self._concat(
            [_np(sim.nodes[i].data[1]).reshape(-1, 2) if sim.nodes[i].data[1] is not None else np.zeros((0, 2))
             for i in ids], 2, self.device)
        self.te_cnt_host = self.te_cnt.cpu().numpy()

    def _deliver_cuda(self, recvs: torch.Tensor, slots: torch.Tensor) -> None:
        from ..ops.native import native
        native().mf_bank_deliver(*self._args(), recvs, slots)

    def _parts(self, w: torch.Tensor):
        m, k = self.dim, self.k
        return (w[:, :m * k].view(-1, m, k), w[:, m * k:m * k + m], w[:, m * k + m:m * k + m + k],
                w[:, m * k + m + k])

    def _update_cpu(self, w: torch.Tensor, nodes: torch.Tensor) -> torch.Tensor:
        """In place on the rows ``w`` [B, Dp]: step i of every node's sequential pass at once (``torch_ref.mf_update``:
        fp32 arithmetic, the step ``lr * err`` rounded to fp32); returns the age increments."""
        Y, c, X, b = self._parts(w)
        cnt, off = self.cnt[nodes].long(), self.off[nodes]
        dec = float(np.float32(1.0 - self.reg * self.lr))
        for i in range(int(cnt.max()) if cnt.numel() else 0):
            L = torch.nonzero(cnt > i).squeeze(1)
            rat = self.data[off[L] + i]
            items, r = rat[:, 0].long(), rat[:, 1]
            yi, xl = Y[L, items], X[L]
            err = r - (xl * yi).sum(1) - b[L] - c[L, items]
            step = (err.double() * self.lr).float()
            yn = yi * dec + step[:, None] * xl
            X[L] = xl * dec + step[:, None] * yn
            Y[L, items] = yn
            b[L] += step
            c[L, items] += step
        return cnt

    def _merge_cpu(self, w: torch.Tensor, sv: torch.Tensor, aw: torch.Tensor, asn: torch.Tensor) -> None:
        den = 2.0 * (aw + asn).double()
        wa, wb = (aw.double() / den).float()[:, None], (asn.double() / den).float()[:, None]
        ns = self.n_shared
        w[:, :ns] = w[:, :ns] * wa + sv[:, :ns] * wb

    def _evaluate(self, nodes: List[int]) -> List[Dict[str, float]]:
        cnt = self.te_cnt_host
        if self.device.type == "cuda":
            from ..ops.native import native
            sse = native().mf_bank_eval(*self._args(), self._idx(nodes), self.te, self.te_off, self.te_cnt)
            ops._count()
            sse = sse.cpu().numpy().astype(np.float64)
            with np.errstate(divide="ignore", invalid="ignore"):
                return [{"rmse": float(np.sqrt(s / cnt[i]))} for s, i in zip(sse, nodes)]
        out = []
        for i in nodes:                                       # MFModelHandler.evaluate_async, node by node
            Y, c, X, b = self._parts(self.W[i:i + 1])
            o = int(self.te_off[i])
            r = self.te[o:o + int(cnt[i])]
            idx = r[:, 0].long()
            pred = Y[0][idx] @ X[0] + b[0:1] + c[0][idx]
            out.append({"rmse": float(torch.sqrt(torch.mean((r[:, 1] - pred) ** 2)))})
        return out
