"""Data layer: split properties of the assignment strategies (SURVEY §2.9 [verified] facts)."""
import numpy as np
import pytest
import torch

from gossipy_b200.data import (AssignmentHandler, DataDispatcher, RecSysDataDispatcher,
                               load_classification_dataset, load_recsys_dataset, get_CIFAR10)
from gossipy_b200.data import synthetic
from gossipy_b200.data.handler import (ClassificationDataHandler, ClusteringDataHandler,
                                       RecSysDataHandler, RegressionDataHandler)


@pytest.fixture
def labels():
    return torch.from_numpy(np.random.RandomState(0).randint(0, 10, 2000))


def _disjoint_cover(parts, n, exact=True):
    allidx = np.concatenate(parts)
    assert len(set(allidx.tolist())) == len(allidx)
    if exact:
        assert len(allidx) == n


def test_uniform_drops_remainder(labels):
    parts = AssignmentHandler(1).uniform(labels[:1999], 8)
    assert all(len(p) == 249 for p in parts)
    _disjoint_cover(parts, 1999, exact=False)


def test_quantity_skews(labels):
    ah = AssignmentHandler(2)
    parts = ah.quantity_skew(labels, 8, min_quantity=3)
    _disjoint_cover(parts, 2000)
    sizes = sorted(len(p) for p in parts)
    assert sizes[0] >= 3 and sizes[-1] > 3 * sizes[0]
    parts = ah.classwise_quantity_skew(labels, 8)
    _disjoint_cover(parts, 2000)
    for p in parts:
        assert len(np.unique(labels[p].numpy())) == 10


def test_label_skews(labels):
    ah = AssignmentHandler(3)
    parts = ah.label_quantity_skew(labels, 8, class_per_client=2)
    _disjoint_cover(parts, 2000)
    assert all(len(np.unique(labels[p].numpy())) <= 2 for p in parts)
    assert len(np.unique(np.concatenate([labels[p].numpy() for p in parts]))) == 10
    parts = ah.label_dirichlet_skew(labels, 8, beta=.1)
    _disjoint_cover(parts, 2000)
    sizes = [len(p) for p in parts]
    assert max(sizes) > 2 * min(sizes)
    parts = ah.label_pathological_skew(labels, 8, shards_per_client=2)
    _disjoint_cover(parts, 2000)
    assert all(len(p) == 250 for p in parts)
    assert all(len(np.unique(labels[p].numpy())) <= 4 for p in parts)


def test_assignment_is_seeded_and_private():
    y = torch.arange(100) % 5
    np.random.seed(7); before = np.random.random()
    np.random.seed(7)
    a = AssignmentHandler(11).uniform(y, 4)
    assert np.random.random() == before         # global RNG untouched
    b = AssignmentHandler(11).uniform(y, 4)
    assert all(np.array_equal(x, z) for x, z in zip(a, b))


def test_handlers_and_dispatcher():
    X, y = synthetic.teacher_classification(500, 6, 3)
    dh = ClassificationDataHandler(X, y, test_size=.2)
    assert (dh.size(), dh.eval_size(), dh.size(1), dh.n_classes) == (400, 100, 6, 3)
    assert dh.at([], True) is None and dh.at([1, 2])[0].shape == (2, 6)
    dn = ClassificationDataHandler(X.numpy(), y.numpy(), test_size=.1)
    assert dn.size() == 450 and isinstance(dn.Xtr, np.ndarray)
    cl = ClusteringDataHandler(X, y)
    assert cl.size() == 500 == cl.eval_size()                       # B18 fixed
    rg = RegressionDataHandler(X, X[:, 0], test_size=.2)
    assert rg.at([0, 1])[0].shape == (2, 6)                         # B19 fixed
    disp = DataDispatcher(dh, n=7, eval_on_user=True)
    (xtr, ytr), (xte, yte) = disp[3]
    assert xtr.shape == (57, 6) and xte.shape == (14, 6) and disp.has_test()
    d2 = DataDispatcher(dh, n=4, eval_on_user=False)
    assert d2[0][1] is None
    assert DataDispatcher(dh, eval_on_user=False).size() == 400     # one sample per client
    with pytest.raises(AssertionError):
        d2.set_assignments([[0]] * 3, None)


def test_recsys_and_loaders_offline():
    ratings, nu, ni = load_recsys_dataset("synthetic:tiny")
    dh = RecSysDataHandler(ratings, nu, ni, test_size=.2)
    disp = RecSysDataDispatcher(dh); disp.assign(1)
    tr, te = disp[0]
    assert tr.shape[1] == 2 and len(tr) + len(te) == 30 and not disp.has_test()
    X, y = load_classification_dataset("iris")
    assert X.shape == (150, 4) and abs(float(X.mean())) < 1e-5
    with pytest.raises(Exception):                                 # no network: the default is to fail loudly, like the reference
        load_classification_dataset("spambase")
    Xs, ys = load_classification_dataset("spambase", synthetic_fallback=True)   # explicit opt-in -> synthetic data of that shape
    assert Xs.shape == (4601, 57) and set(ys.tolist()) == {0, 1}
    (xtr, ytr), (xte, yte) = synthetic.images_like("cifar10", n_train=64, n_test=16)
    assert xtr.shape == (64, 3, 32, 32) and float(xtr.min()) >= 0 and float(xtr.max()) <= 1
    (mtr, _), (mte, _) = synthetic.mnist_like(100, 20)
    assert mtr.shape == (100, 784) and mte.shape == (20, 784)


@pytest.mark.parametrize("name,kw", [("uniform", {}), ("quantity_skew", dict(min_quantity=2, alpha=4.)),
                                     ("classwise_quantity_skew", dict(min_quantity=2, alpha=4.)),
                                     ("label_quantity_skew", dict(class_per_client=2)),
                                     ("label_dirichlet_skew", dict(beta=.5)),
                                     ("label_pathological_skew", dict(shards_per_client=2))])
@pytest.mark.parametrize("n,seed", [(7, 42), (10, 42), (10, 7)])
def test_assignment_strategies_reproduce_the_reference_splits_in_compat_mode(ref, name, kw, n, seed):
    """``reference_compat``: same seed -> the reference's index sets, element for element (and the same side effect
    on the global streams); the default draws from a private generator instead."""
    import gossipy_b200 as g
    import gossipy_b200.data as OD
    y = torch.randint(0, 10, (1000,), generator=torch.Generator().manual_seed(0))
    g.GlobalSettings().reference_compat = True
    ours = getattr(OD.AssignmentHandler(seed), name)(y, n, **kw)
    probe_o = (float(np.random.rand()), float(torch.rand(1)))

    def theirs(rg):
        split = getattr(rg.data.AssignmentHandler(seed), name)(y, n, **kw)
        return [np.asarray(a) for a in split], (float(np.random.rand()), float(torch.rand(1)))
    theirs, probe_r = ref(theirs)
    probe_r = tuple(probe_r)
    assert len(ours) == len(theirs) == n
    for a, b in zip(ours, theirs):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    assert probe_o == probe_r                      # the global streams end in the same state
    g.GlobalSettings().reference_compat = False
    other = getattr(OD.AssignmentHandler(seed), name)(y, n, **kw)
    assert sorted(len(a) for a in other) != [] and sum(len(a) for a in other) <= 1000


def test_train_test_split_and_auto_assignment_reproduce_the_reference_in_compat_mode(ref):
    import gossipy_b200 as g
    import gossipy_b200.data as OD
    import gossipy_b200.data.handler as OH
    gen = torch.Generator().manual_seed(0)
    X = torch.randn(200, 5, generator=gen)
    y = torch.randint(0, 3, (200,), generator=gen)
    splits = ((.2, 42), (.3, 7))

    def rows(Xs):        # the rows of X (all distinct) that a split holds, in its order
        pos = (torch.as_tensor(Xs)[:, None, :] == X[None]).all(-1).nonzero()
        assert pos[:, 0].tolist() == list(range(len(Xs)))
        return pos[:, 1]

    def theirs(rg):
        import gossipy.data.handler as RH
        out = []
        for ts, seed in splits:
            b = RH.ClassificationDataHandler(X, y, test_size=ts, seed=seed)
            out.append((rows(b.Xtr), b.ytr, rows(b.Xte), b.yte))
        b = RH.ClassificationDataHandler(X.numpy(), y.numpy(), test_size=.25, seed=3)
        out.append((rows(b.Xtr), b.yte))
        b = rg.data.DataDispatcher(RH.ClassificationDataHandler(X, y, X[:40], y[:40]), n=7, eval_on_user=True,
                                   auto_assign=True)
        out.append(([np.asarray(p) for p in b.tr_assignments], [np.asarray(p) for p in b.te_assignments]))
        return out
    want = ref(theirs)
    g.GlobalSettings().reference_compat = True
    for (ts, seed), (tr, ytr, te, yte) in zip(splits, want):
        a = OH.ClassificationDataHandler(X, y, test_size=ts, seed=seed)
        for p, q in ((a.Xtr, X[tr]), (a.ytr, ytr), (a.Xte, X[te]), (a.yte, yte)):
            assert torch.equal(p, q)
    a = OH.ClassificationDataHandler(X.numpy(), y.numpy(), test_size=.25, seed=3)
    assert np.array_equal(a.Xtr, X.numpy()[want[2][0].numpy()]) and np.array_equal(a.yte, want[2][1])
    a = OD.DataDispatcher(OH.ClassificationDataHandler(X, y, X[:40], y[:40]), n=7, eval_on_user=True, auto_assign=True)
    tr, te = want[3]
    assert len(a.tr_assignments) == len(tr) and len(a.te_assignments) == len(te)
    for p, q in list(zip(a.tr_assignments, tr)) + list(zip(a.te_assignments, te)):
        assert np.array_equal(np.asarray(p), q)
