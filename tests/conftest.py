"""Test configuration: the ``gpu`` marker, state isolation, and the original gossipy's side of the comparisons
(recorded results, or the original itself with its import shims)."""
import json
import os
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with `pytest -m gpu` on a B200)")


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(autouse=True)
def _fresh_state():
    import gossipy_b200 as g
    from gossipy_b200.engine import arena
    g.CACHE.clear()
    g.GlobalSettings().reference_compat = False
    g.GlobalSettings().set_device("cpu")
    g.set_seed(1234)
    yield
    g.CACHE.clear()
    g.GlobalSettings().set_device("cpu")


def _import_reference():
    """Import the read-only reference with the three environment shims of SURVEY §0."""
    ref_root = os.environ.get("GOSSIPY_REFERENCE", "")
    if not ref_root or not os.path.isdir(os.path.join(ref_root, "gossipy")):
        return None
    for name in ("matplotlib", "matplotlib.pyplot", "pyparsing"):
        if name not in sys.modules:
            try:
                __import__(name)
            except Exception:
                mod = types.ModuleType(name)
                if name == "pyparsing":
                    mod.ParseSyntaxException = Exception
                sys.modules[name] = mod
    if "matplotlib" in sys.modules and not hasattr(sys.modules["matplotlib"], "pyplot"):
        sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    if ref_root not in sys.path:
        sys.path.append(ref_root)
    try:
        import gossipy  # noqa: F401
        import gossipy.model.handler as H
        _auc = H.roc_auc_score
        if not getattr(H, "_b200_patched", False):
            H.roc_auc_score = lambda *a, **k: np.float64(_auc(*a, **k))
            H._b200_patched = True
        import gossipy.simul as S

        class _It:
            def __init__(self, it): self.it = it
            def __iter__(self): return iter(self.it)
            def close(self): pass
        S.track = lambda it, description="": _It(it)
        return gossipy
    except Exception:
        return None


GOLDEN = os.path.join(ROOT, "tests", "golden", "reference")
_golden = {}        # test module file name -> {result key: encoded value}
_recorded = set()   # files holding results recorded in this session


def _encode(v):
    import torch
    if isinstance(v, torch.Tensor):
        t = v.detach().cpu()
        return {"__tensor__": str(t.dtype).replace("torch.", ""), "shape": list(t.shape), "data": t.reshape(-1).tolist()}
    if isinstance(v, np.ndarray):
        return {"__ndarray__": v.dtype.str, "shape": list(v.shape), "data": v.reshape(-1).tolist()}
    if isinstance(v, np.generic):
        return v.item()
    if isinstance(v, dict):
        return {"__dict__": [[_encode(k), _encode(x)] for k, x in v.items()]}
    if isinstance(v, (list, tuple)):
        return [_encode(x) for x in v]
    assert v is None or isinstance(v, (bool, int, float, str)), type(v)
    return v


def _decode(v):
    import torch
    if isinstance(v, list):
        return [_decode(x) for x in v]
    if isinstance(v, dict):
        if "__tensor__" in v:
            return torch.tensor(v["data"], dtype=getattr(torch, v["__tensor__"])).reshape(v["shape"])
        if "__ndarray__" in v:
            return np.array(v["data"], dtype=np.dtype(v["__ndarray__"])).reshape(v["shape"])
        return {_decode_key(k): _decode(x) for k, x in v["__dict__"]}
    return v


def _decode_key(k):
    return tuple(_decode_key(x) for x in k) if isinstance(k, list) else k


class Reference:
    """Results of the original gossipy for one test.

    ``ref(fn)`` returns ``fn(gossipy)``.  With ``GOSSIPY_REFERENCE`` naming a checkout of the original project the
    function runs against it and its result is recorded under ``tests/golden/reference/``; without it, the result
    recorded there is returned, so every comparison with the original runs on any machine.  Results are keyed by the
    test id and the order of the calls within the test; values are numbers, strings, lists, tuples (read back as
    lists), dicts, tensors and arrays (read back with their dtype, exactly)."""

    def __init__(self, module, nodeid):
        path, _, name = nodeid.partition("::")
        self.module, self.file, self.name, self.calls = module, os.path.basename(path)[:-3] + ".json", name, 0
        if self.file not in _golden:
            try:
                with open(os.path.join(GOLDEN, self.file)) as f:
                    _golden[self.file] = json.load(f)
            except FileNotFoundError:
                _golden[self.file] = {}

    def __call__(self, fn):
        key = "%s#%d" % (self.name, self.calls)
        self.calls += 1
        store = _golden[self.file]
        if self.module is not None:
            store[key] = _encode(fn(self.module))
            _recorded.add(self.file)
        elif key not in store:
            pytest.fail("no recorded result of the original gossipy for %s in %s (record it: GOSSIPY_REFERENCE=<checkout> "
                        "pytest ...)" % (key, os.path.join(GOLDEN, self.file)))
        return _decode(store[key])


def pytest_sessionfinish(session):
    for name in sorted(_recorded):
        os.makedirs(GOLDEN, exist_ok=True)
        with open(os.path.join(GOLDEN, name), "w") as f:
            json.dump(_golden[name], f, sort_keys=True, separators=(",", ":"))
            f.write("\n")


@pytest.fixture
def ref(request):
    return Reference(_import_reference(), request.node.nodeid)
