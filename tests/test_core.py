"""Core vocabulary: differential tests against the reference (SURVEY §4 level 1)."""
import numpy as np
import pytest
import torch

import gossipy_b200 as g
from gossipy_b200 import CACHE, CacheKey, GlobalSettings
from gossipy_b200.core import (AntiEntropyProtocol, ConstantDelay, CreateModelMode, LinearDelay,
                               Message, MessageType, MetropolisHastingsMixing, StaticP2PNetwork,
                               UniformDelay, UniformMixing)


def _ring(n):
    A = np.zeros((n, n))
    for i in range(n):
        A[i, (i + 1) % n] = A[i, (i - 1) % n] = 1
    return A


def _enums(core):
    return {name: {m.name: m.value for m in getattr(core, name)}
            for name in ("CreateModelMode", "AntiEntropyProtocol", "MessageType")}


def test_enums_match_reference(ref):
    assert _enums(g.core) == ref(lambda rg: _enums(rg.core))


def test_message_size_rules():
    class Five(g.Sizeable):
        def get_size(self): return 5
    assert Message(0, 0, 1, MessageType.PULL, None).get_size() == 1
    assert Message(0, 0, 1, MessageType.PUSH, (Five(), 3, 2.5, None)).get_size() == 7
    assert Message(0, 0, 1, MessageType.PUSH, (None,)).get_size() == 1
    with pytest.raises(TypeError):
        Message(0, 0, 1, MessageType.PUSH, ("str",)).get_size()
    key = CacheKey(3, 7)
    CACHE.push(key, Five())
    assert Message(0, 3, 1, MessageType.PUSH, (key, 4)).get_size() == 6
    assert CACHE.pop(key).get_size() == 5 and len(CACHE) == 0


def test_cache_refcount_semantics():
    k = CacheKey(0, 1)
    CACHE.push(k, 1.5)
    CACHE.push(k, 2.5)          # same key: first value kept, refcount 2
    assert CACHE[k] == 1.5 and len(CACHE) == 1
    assert CACHE.pop(k) == 1.5 and len(CACHE) == 1
    assert CACHE.pop(k) == 1.5 and len(CACHE) == 0
    assert CACHE.pop(k) is None


def test_delays():
    m = Message(0, 0, 1, MessageType.PULL, None)
    assert ConstantDelay(3).get(m) == 3
    d = [UniformDelay(2, 5).get(m) for _ in range(300)]
    assert min(d) == 2 and max(d) == 5
    assert LinearDelay(2.5, 4).get(m) == 6
    with pytest.raises(AssertionError):
        ConstantDelay(-1)


def test_topology_degrees_fix_and_compat(ref):
    A = _ring(6)

    def theirs(rg):
        net = rg.core.StaticP2PNetwork(6, A)
        return [[int(x) for x in net.get_peers(i)] for i in range(6)], net.size(0)
    peers, size0 = ref(theirs)
    ours = StaticP2PNetwork(6, A)
    for i in range(6):
        assert list(ours.get_peers(i)) == peers[i]
    assert ours.size() == 6
    assert [ours.size(i) for i in range(6)] == [2] * 6          # fixed B1
    assert size0 == 6                                            # the reference bug
    GlobalSettings().reference_compat = True
    assert ours.size(0) == 6
    GlobalSettings().reference_compat = False
    clique = StaticP2PNetwork(4)
    assert clique.get_peers(2) == [0, 1, 3]
    indptr, idx = clique.as_csr()
    assert indptr.tolist() == [0, 3, 6, 9, 12] and idx[:3].tolist() == [1, 2, 3]


def test_sparse_and_networkx_topologies():
    from scipy.sparse import csr_matrix
    import networkx as nx
    A = _ring(5)
    assert StaticP2PNetwork(5, csr_matrix(A)).get_peers(0) == [1, 4]
    assert StaticP2PNetwork(5, nx.cycle_graph(5)).get_peers(0) == [1, 4]
    with pytest.raises(AssertionError):
        StaticP2PNetwork(4, A)                                    # B2: shape check is real


def test_mixing_matches_reference(ref):
    A = _ring(6); A[1, 3] = A[3, 1] = 1

    def theirs(rg):
        net = rg.core.StaticP2PNetwork(6, A)
        return [(np.asarray(rg.core.UniformMixing(net)[i]), np.asarray(rg.core.MetropolisHastingsMixing(net)[i]))
                for i in range(6)]
    weights = ref(theirs)
    ours = StaticP2PNetwork(6, A)
    GlobalSettings().reference_compat = True      # node-0 degree quirk (B1) leaks into MH weights
    for i in range(6):
        np.testing.assert_allclose(UniformMixing(ours)[i], weights[i][0])
        np.testing.assert_allclose(MetropolisHastingsMixing(ours)[i], weights[i][1])
    GlobalSettings().reference_compat = False
    assert len(UniformMixing(ours)[0]) == 3       # fixed: deg(0)+1, not num_nodes+1
    w = MetropolisHastingsMixing(ours, normalized=True)[1]
    assert abs(w.sum() - 1) < 1e-12
