"""Handler math vs the reference: merges (C1-C7), local updates (K1-K6), evaluation."""
import copy

import numpy as np
import pytest
import torch

import gossipy_b200 as g
from gossipy_b200 import CACHE
from gossipy_b200.core import CreateModelMode as M
from gossipy_b200.model import handler as H
from gossipy_b200.model.nn import AdaLine, LogisticRegression, TorchMLP
from gossipy_b200.model.sampling import TorchModelPartition, TorchModelSampling
from gossipy_b200.models import ResNet20

CE = torch.nn.CrossEntropyLoss()


def _data(n=96, d=12, c=3, seed=0):
    gen = torch.Generator().manual_seed(seed)
    X = torch.randn(n, d, generator=gen)
    return X, (X @ torch.randn(d, c, generator=gen)).argmax(1)


def _common(kw):
    common = dict(optimizer=torch.optim.SGD, optimizer_params={"lr": .1, "weight_decay": .01},
                  criterion=CE, batch_size=0, local_epochs=1)
    common.update(kw)
    return common


def _ours(cls_name, net_fn, **kw):
    return getattr(H, cls_name)(net=net_fn(g.model.nn), **_common(kw))


def _theirs(cls_name, net_fn, **kw):
    """The original gossipy's handler with the same arguments."""
    import gossipy.model.handler as RH
    import gossipy.model.nn as RN
    okw = _common(kw)
    if "create_model_mode" in okw:
        okw["create_model_mode"] = getattr(RH.CreateModelMode, okw["create_model_mode"].name)
    return getattr(RH, cls_name)(net=net_fn(RN), **okw)


def _flat(module):
    return torch.cat([p.detach().reshape(-1) for p in module.parameters()])


def _randn_params(module, seed):
    gen = torch.Generator().manual_seed(seed)
    return [torch.randn(p.shape, generator=gen) for p in module.parameters()]


def _set_random(ours, seed):
    names = [n for n, _ in ours.model.named_parameters()]
    ours.model.load_state_dict(dict(zip(names, _randn_params(ours.model, seed))))
    ours.model = ours.model  # re-gather into the row


def _set_random_theirs(theirs, seed):
    for p, v in zip(list(theirs.model.parameters()), _randn_params(theirs.model, seed)):
        p.data = v


def test_fullbatch_update_and_uniform_merge_match_reference(ref):
    X, y = _data()
    mk = lambda ns: ns.TorchMLP(12, 3, (8,))

    def theirs(rg):
        ra, rb = _theirs("TorchModelHandler", mk), _theirs("TorchModelHandler", mk)
        _set_random_theirs(ra, 1); _set_random_theirs(rb, 2)
        for h in (ra, rb):
            h._update((X, y))
        out = [ra.n_updates, _flat(ra.model)]
        ra._merge(rb)
        out.append(_flat(ra.model))
        ra._merge([rb, rb])
        return out + [_flat(ra.model), ra.evaluate((X, y))]
    r_updates, r_upd, r_merge, r_merge2, rev = ref(theirs)
    a, b = _ours("TorchModelHandler", mk), _ours("TorchModelHandler", mk)
    _set_random(a, 1); _set_random(b, 2)
    for h in (a, b):
        h._update((X, y))
    assert a.n_updates == r_updates == 1
    torch.testing.assert_close(_flat(a.model), r_upd, rtol=1e-5, atol=1e-6)
    a._merge(b)
    torch.testing.assert_close(_flat(a.model), r_merge, rtol=1e-5, atol=1e-6)
    a._merge([b, b])
    torch.testing.assert_close(_flat(a.model), r_merge2, rtol=1e-5, atol=1e-6)
    ev = a.evaluate((X, y))
    for k in rev:
        assert ev[k] == pytest.approx(float(rev[k]), abs=1e-6), k


def test_generic_path_matches_fused_path():
    """Same seed/key -> the autograd path and the explicit fused math give the same weights."""
    X, y = _data(100, 12, 3)
    net = TorchMLP(12, 3, (8,)); net.init_weights()
    fused = H.TorchModelHandler(net, torch.optim.SGD, {"lr": .05, "weight_decay": .001}, CE,
                                local_epochs=2, batch_size=32)
    generic = fused.copy()
    generic._fused = False
    assert fused._fused
    fused.owner = generic.owner = 3
    fused._update((X, y)); generic._update((X, y))
    assert fused.n_updates == generic.n_updates == 8
    torch.testing.assert_close(fused.row, generic.row, rtol=1e-4, atol=1e-6)


def test_grad_views_stay_bound():
    X, y = _data()
    h = H.TorchModelHandler(TorchMLP(12, 3, (8, 8)), torch.optim.SGD, {"lr": .1, "momentum": .9}, CE)
    assert not h._fused
    h._update((X, y))
    ptrs = [p.grad.data_ptr() for p in h.model.parameters()]
    h._update((X, y))
    assert ptrs == [p.grad.data_ptr() for p in h.model.parameters()]
    base = h._grad_row.data_ptr()
    assert all(base <= q < base + h._grad_row.numel() * 4 for q in ptrs)


@pytest.mark.parametrize("opt,params", [(torch.optim.SGD, {"lr": .1, "momentum": .9, "nesterov": True}),
                                        (torch.optim.SGD, {"lr": .1, "momentum": .5, "dampening": .1,
                                                           "weight_decay": .01}),
                                        (torch.optim.Adam, {"lr": .01, "weight_decay": .01}),
                                        (torch.optim.AdamW, {"lr": .01}),
                                        (torch.optim.RMSprop, {"lr": .01})])
def test_flat_optimizers_match_torch(opt, params):
    X, y = _data()
    net = TorchMLP(12, 3, (8,)); net.init_weights()
    h = H.TorchModelHandler(net, opt, params, CE, batch_size=0, local_epochs=3)
    twin = copy.deepcopy(net)
    topt = opt(twin.parameters(), **params)
    for _ in range(3):
        topt.zero_grad(); CE(twin(X), y).backward(); topt.step()
    h._update((X, y))
    torch.testing.assert_close(_flat(h.model), _flat(twin), rtol=2e-4, atol=1e-6)


def test_modes_match_reference(ref):
    X, y = _data()
    mk = lambda ns: ns.LogisticRegression(12, 3)
    modes = (M.UPDATE, M.MERGE_UPDATE, M.UPDATE_MERGE, M.PASS)

    def theirs(rg):
        out = []
        for mode in modes:
            ra, rb = _theirs("TorchModelHandler", mk, create_model_mode=mode), \
                _theirs("TorchModelHandler", mk, create_model_mode=mode)
            _set_random_theirs(ra, 3); _set_random_theirs(rb, 4)
            rb.n_updates = 5
            ra(rb.copy(), (X, y))
            out.append((ra.n_updates, _flat(ra.model)))
        return out
    for mode, (r_updates, r_flat) in zip(modes, ref(theirs)):
        a, b = _ours("TorchModelHandler", mk, create_model_mode=mode), _ours("TorchModelHandler", mk, create_model_mode=mode)
        _set_random(a, 3); _set_random(b, 4)
        b.n_updates = 5
        a(b.copy(), (X, y))
        assert a.n_updates == r_updates, mode
        torch.testing.assert_close(_flat(a.model), r_flat, rtol=1e-5, atol=1e-6, msg=str(mode))


def test_limited_merge_branches(ref):
    mk = lambda ns: ns.LogisticRegression(12, 3)
    ages = ((10, 2), (2, 10), (4, 5))   # the reference divides by zero for two fresh models: (0, 0) is ours only

    def theirs(rg):
        out = []
        for na, nb in ages:
            ra, rb = _theirs("LimitedMergeTMH", mk, age_diff_threshold=1), _theirs("LimitedMergeTMH", mk, age_diff_threshold=1)
            _set_random_theirs(ra, 5); _set_random_theirs(rb, 6)
            ra.n_updates, rb.n_updates = na, nb
            ra._merge(rb)
            out.append((_flat(ra.model), ra.n_updates))
        return out
    want = ref(theirs)
    for i, (na, nb) in enumerate(ages + ((0, 0),)):
        a, b = _ours("LimitedMergeTMH", mk, age_diff_threshold=1), _ours("LimitedMergeTMH", mk, age_diff_threshold=1)
        _set_random(a, 5); _set_random(b, 6)
        a.n_updates, b.n_updates = na, nb
        a._merge(b)
        if i < len(ages):
            torch.testing.assert_close(_flat(a.model), want[i][0], rtol=1e-5, atol=1e-6)
            assert a.n_updates == want[i][1]
        else:
            assert torch.isfinite(a.row).all()


def test_weighted_kway_merge(ref):
    mk = lambda ns: ns.LogisticRegression(12, 3)
    w = np.array([.4, .3, .2, .1])

    def theirs(rg):
        hs = [_theirs("WeightedTMH", mk) for _ in range(4)]
        for i, h in enumerate(hs):
            _set_random_theirs(h, 10 + i)
        hs[0]._merge(hs[1:], w)
        return _flat(hs[0].model)
    want = ref(theirs)
    hs = [_ours("WeightedTMH", mk) for _ in range(4)]
    for i, h in enumerate(hs):
        _set_random(h, 10 + i)
    hs[0]._merge(hs[1:], w)
    torch.testing.assert_close(_flat(hs[0].model), want, rtol=1e-5, atol=1e-6)


def test_partition_index_sets_and_merge_match_reference(ref):
    setups = ((lambda ns: ns.LogisticRegression(5, 2), 4), (lambda ns: ns.TorchMLP(7, 3, (5,)), 3),
              (lambda ns: ns.TorchMLP(7, 3, (5,)), 7))

    def theirs(rg):
        import gossipy.model.nn as RN
        import gossipy.model.sampling as RS
        out = []
        for mk, parts in setups:
            pr = RS.TorchModelPartition(mk(RN), parts)
            out.append((pr.n_parts, [[(ti, None if ids is None else [x.tolist() for x in ids])
                                      for ti, ids in pr.partitions[p].items()] for p in range(pr.n_parts)]))
        return out
    for (mk, parts), (n_parts, partitions) in zip(setups, ref(theirs)):
        po = TorchModelPartition(mk(g.model.nn), parts)
        assert po.n_parts == n_parts
        flat_all = []
        for p in range(po.n_parts):
            for ti, ids in partitions[p]:
                mine = po.partitions[p][ti]
                if ids is None:
                    assert mine is None
                    continue
                a = sorted(zip(*ids))
                b = sorted(zip(*[x.tolist() for x in mine]))
                assert a == b, (p, ti)
            # segments cover exactly the flat index set
            cover = []
            for st, nr, rl, sd in po.segments(p).tolist():
                cover += [st + r * sd + c for r in range(nr) for c in range(rl)]
            assert sorted(cover) == po.flat_index(p).tolist()
            flat_all += cover
        assert sorted(flat_all) == list(range(po.n_params))


def test_partitioned_handler_matches_reference(ref):
    X, y = _data()
    mk = lambda ns: ns.TorchMLP(12, 3, (6,))

    def theirs(rg):
        import gossipy.model.nn as RN
        import gossipy.model.sampling as RS
        ra, rb = (_theirs("PartitionedTMH", mk, tm_partition=RS.TorchModelPartition(mk(RN), 4)) for _ in range(2))
        _set_random_theirs(ra, 7); _set_random_theirs(rb, 8)
        ra._update((X, y)); ra._update((X, y))
        rb._update((X, y))
        out = [ra.n_updates.tolist(), _flat(ra.model)]
        ra._merge(rb, 2)
        ra._merge(rb, 1)
        return out + [_flat(ra.model), ra.n_updates.tolist()]
    r_updates, r_upd, r_merge, r_updates2 = ref(theirs)
    a = _ours("PartitionedTMH", mk, tm_partition=TorchModelPartition(mk(g.model.nn), 4))
    b = _ours("PartitionedTMH", mk, tm_partition=TorchModelPartition(mk(g.model.nn), 4))
    _set_random(a, 7); _set_random(b, 8)
    a._update((X, y)); a._update((X, y))
    b._update((X, y))
    assert a.n_updates.tolist() == r_updates == [2] * 4
    torch.testing.assert_close(_flat(a.model), r_upd, rtol=1e-5, atol=1e-6)
    a._merge(b, 2)
    a._merge(b, 5)      # ours wraps the id modulo n_parts (the reference is given 1)
    torch.testing.assert_close(_flat(a.model), r_merge, rtol=1e-5, atol=1e-6)
    assert a.n_updates.tolist() == r_updates2
    assert a.caching(0).key[1] == str(a.n_updates)
    CACHE.clear()


def test_sampled_merge_matches_reference(ref):
    mk = lambda ns: ns.TorchMLP(12, 3, (6,))

    def theirs(rg):
        import gossipy.model.sampling as RS
        ra, rb = _theirs("SamplingTMH", mk, sample_size=.3), _theirs("SamplingTMH", mk, sample_size=.3)
        _set_random_theirs(ra, 9); _set_random_theirs(rb, 10)
        sample = RS.TorchModelSampling.sample(.3, ra.model)
        ra._merge(rb, sample)
        return sample, _flat(ra.model)
    sample, want = ref(theirs)
    sample = {k: None if v is None else tuple(v) for k, v in sample.items()}
    a, b = _ours("SamplingTMH", mk, sample_size=.3), _ours("SamplingTMH", mk, sample_size=.3)
    _set_random(a, 9); _set_random(b, 10)
    a._merge(b, sample)
    torch.testing.assert_close(_flat(a.model), want, rtol=1e-6, atol=1e-7)
    flat = a.draw_sample()
    assert flat.numel() == round(.3 * a.get_size()) and int(flat.max()) < a.get_size()
    d = TorchModelSampling.sample(.5, a.model)
    assert sum(v[0].numel() for v in d.values() if v is not None) == round(.5 * a.get_size())


def test_adaline_and_pegasos_match_reference(ref):
    gen = torch.Generator().manual_seed(0)
    X = torch.randn(40, 9, generator=gen)
    y = torch.sign(X @ torch.randn(9, generator=gen))
    learners = (("AdaLineHandler", .01), ("PegasosHandler", .01))

    def theirs(rg):
        import gossipy.model.handler as RH
        import gossipy.model.nn as RN
        out = []
        for name, lr in learners:
            r = getattr(RH, name)(RN.AdaLine(9), lr)
            r.init()
            r._update((X, y)); r._update((X[:7], y[:7]))
            res = [r.n_updates, r.model.model.detach().clone()]
            r2 = copy.deepcopy(r); r2._update((X[:3], y[:3]))
            r._merge(r2)
            out.append(res + [r.model.model.detach().clone(), r.evaluate((X, y))])
        return out
    for (name, lr), (r_updates, r_upd, r_merge, er) in zip(learners, ref(theirs)):
        o = getattr(H, name)(AdaLine(9), lr)
        o.init()
        o._update((X, y)); o._update((X[:7], y[:7]))
        assert o.n_updates == r_updates == 47
        torch.testing.assert_close(o.model.model.detach(), r_upd, rtol=1e-4, atol=1e-5)
        o2 = o.copy(); o2._update((X[:3], y[:3]))
        o._merge(o2)
        torch.testing.assert_close(o.model.model.detach(), r_merge, rtol=1e-4, atol=1e-5)
        eo = o.evaluate((X, y))
        for k in er:
            assert eo[k] == pytest.approx(float(er[k]), abs=1e-6)


def test_kmeans_and_mf_match_reference(ref):
    gen = torch.Generator().manual_seed(0)
    X = torch.randn(60, 5, generator=gen); yl = (X[:, 0] > 0).long()
    ratings = np.array([(1, 4.), (3, 2.), (0, 5.), (1, 1.)])

    def theirs(rg):
        import gossipy.model.handler as RH
        r = RH.KMeansHandler(3, 5, alpha=.2)
        r.init()
        init = r.model.clone()
        r._update((X[:1], None)); r._update((X[1:9], None))
        km = [init, r.model.clone(), r.evaluate((X, yl))["nmi"]]
        mr = RH.MFModelHandler(4, 6)
        mr.init()
        mf = [copy.deepcopy(mr.model)]
        mr._update(ratings)
        mf += [mr.model[1][0].copy(), mr.model[0][0].copy(), mr.n_updates]
        r2 = copy.deepcopy(mr)
        r2._update(ratings[:2])
        mr._merge(r2)
        return km + mf + [mr.model[1][0].copy(), mr.model[1][1].copy(), mr.evaluate(ratings)["rmse"], mr.get_size()]
    (k_init, k_upd, nmi, mf_init, mf_y, mf_x, mf_updates,
     mf_y_merged, mf_c_merged, rmse, mf_size) = ref(theirs)
    o = H.KMeansHandler(3, 5, alpha=.2)
    o.init()
    o.model = k_init.clone()
    o._update((X[:1], None)); o._update((X[1:9], None))
    torch.testing.assert_close(o.model, k_upd)
    assert o.evaluate((X, yl))["nmi"] == pytest.approx(nmi)
    o2 = o.copy(); o2.model = o.model.flip(0)
    hung = H.KMeansHandler(3, 5, matching="hungarian"); hung.init(); hung.model = o.model.clone()
    hung._merge(o2)                       # optimal matching undoes the flip (B16 fixed)
    torch.testing.assert_close(hung.model, o.model)
    # matrix factorisation
    mo = H.MFModelHandler(4, 6)
    mo.init()
    (Xu, b), (Y, c) = mf_init
    mo.model = ((Xu, b), (Y, c))
    mo._update(ratings)
    np.testing.assert_allclose(mo.model[1][0], mf_y, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(mo.model[0][0], mf_x, rtol=1e-5, atol=1e-6)
    assert mo.n_updates == mf_updates == 5
    m2 = mo.copy()
    m2._update(ratings[:2])
    mo._merge(m2)
    np.testing.assert_allclose(mo.model[1][0], mf_y_merged, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(mo.model[1][1], mf_c_merged, rtol=1e-5, atol=1e-6)
    assert mo.evaluate(ratings)["rmse"] == pytest.approx(rmse, rel=1e-5)
    assert mo.get_size() == mf_size == 4 * 7
def test_batchnorm_model_merges():
    """B12: the reference crashes merging BN models; here float buffers average, counters max."""
    gen = torch.Generator().manual_seed(0)
    X = torch.rand(16, 3, 16, 16, generator=gen); y = torch.randint(0, 10, (16,), generator=gen)
    net = ResNet20(width=4); net.init_weights()
    a = H.TorchModelHandler(net, torch.optim.SGD, {"lr": .05}, CE, batch_size=8)
    b = a.copy()
    a._update((X, y)); a._update((X, y)); b._update((X, y))
    snap_key = b.caching(1)
    snap = CACHE.pop(snap_key)
    ra, rb = a.row.clone(), snap.row.clone()
    a._merge(snap)
    torch.testing.assert_close(a.row, (ra + rb) / 2)
    cnt = dict(a.model.named_buffers())["stem.1.num_batches_tracked"]
    assert int(cnt) == 4    # max(2 updates * 2 batches, 1 * 2)
    assert a.layout.numel > a.layout.n_params == net.get_size()


def test_snapshot_dedupe_and_release():
    X, y = _data()
    h = H.TorchModelHandler(TorchMLP(12, 3, (8,)), torch.optim.SGD, {"lr": .1}, CE)
    h.owner = 0
    h._update((X, y))
    k1, k2 = h.caching(0), h.caching(0)
    assert k1 == k2 and len(CACHE) == 1          # identical version: one snapshot, two refs
    s1 = CACHE.pop(k1); s1.release()
    assert s1._row is not None                   # still referenced by the second message
    s2 = CACHE.pop(k2); s2.release()
    assert s2._row is None and len(CACHE) == 0
    h._update((X, y))
    assert h.caching(0) != k1
    CACHE.clear()


def test_momentum_oracle_equals_torch_optim_sgd():
    """The explicit momentum update of the fused-path oracle (ops.torch_ref.mlp1_train) is torch.optim.SGD's."""
    import torch
    from gossipy_b200.ops import torch_ref as ref
    from gossipy_b200.model.nn import TorchMLP
    torch.manual_seed(3)
    dims = (20, 7, 3)
    net = TorchMLP(20, 3, (7,)).double()
    X = torch.randn(48, 20, dtype=torch.float64); y = torch.randint(0, 3, (48,))
    for kw in (dict(momentum=.9), dict(momentum=.9, nesterov=True), dict(momentum=.5, dampening=.2, weight_decay=.01)):
        m = __import__("copy").deepcopy(net)
        row = torch.cat([p.detach().reshape(-1) for p in m.parameters()]).clone()
        buf = torch.zeros_like(row)
        opt = torch.optim.SGD(m.parameters(), lr=.1, **kw)
        idx_all = list(ref._batches(48, 16, 2, 99))
        for idx in idx_all:
            loss = torch.nn.functional.cross_entropy(m(X[idx]), y[idx])
            opt.zero_grad(); loss.backward(); opt.step()
        ref.mlp1_train(row, X, y, dims, 16, 2, .1, kw.get("weight_decay", 0.), 99, None,
                       (kw["momentum"], kw.get("dampening", 0.), kw.get("nesterov", False), buf, True))
        want = torch.cat([p.detach().reshape(-1) for p in m.parameters()])
        torch.testing.assert_close(row, want, rtol=1e-10, atol=1e-12)


def test_channels_last_rows_are_a_private_layout_choice():
    """``GlobalSettings().channels_last``: conv filters live in the row as [O, kh, kw, I] and are bound as channels-last
    views, mini-batches are gathered as NHWC -- training, merging, evaluation, pickling and the model setter give the
    results of the plain layout."""
    import copy
    import pickle
    import gossipy_b200 as g
    from gossipy_b200.model.handler import PartitionedTMH, TorchModelHandler
    from gossipy_b200.model.nn import CIFAR10Net
    from gossipy_b200.model.sampling import TorchModelPartition

    def run(cl):
        g.GlobalSettings().channels_last = cl
        g.set_seed(3)
        torch.manual_seed(3)
        X, y = torch.rand(96, 3, 32, 32), torch.randint(0, 10, (96,))
        h = TorchModelHandler(CIFAR10Net(), torch.optim.SGD, {"lr": .05, "momentum": .9}, torch.nn.CrossEntropyLoss(), batch_size=32)
        h.init()
        h2 = h.copy()
        for _ in range(2):
            h._update((X, y))
        h2._update((X[:64], y[:64]))
        h._merge(h2)
        ev = h.evaluate((X, y))
        sd = {k: v.detach().clone() for k, v in h.model.state_dict().items()}
        h3 = pickle.loads(pickle.dumps(h))
        assert all(torch.equal(sd[k], v) for k, v in h3.model.state_dict().items())
        h4 = h.copy()
        h4.model = copy.deepcopy(h.model)
        assert all(torch.equal(a, b) for a, b in zip(h4.model.state_dict().values(), sd.values()))
        return h, sd, ev
    try:
        h0, sd0, ev0 = run(False)
        h1, sd1, ev1 = run(True)
        assert not h0.layout.channels_last and h1.layout.channels_last
        w = next(v for v in h1.model.parameters() if v.dim() == 4)
        assert w.is_contiguous(memory_format=torch.channels_last) and not w.is_contiguous()
        for k in sd0:
            torch.testing.assert_close(sd0[k].float(), sd1[k].float(), rtol=1e-5, atol=1e-6)
        assert ev0 == pytest.approx(ev1, abs=1e-6)
        # handlers that address parameters by flat index keep the plain order
        net = CIFAR10Net()
        hp = PartitionedTMH(net, TorchModelPartition(net, 4), torch.optim.SGD, {"lr": .1}, torch.nn.CrossEntropyLoss())
        assert not hp.layout.channels_last
    finally:
        g.GlobalSettings().channels_last = "auto"
