"""Public-API parity with the reference (SURVEY.md Appendix A), checked mechanically.

For every module of the reference: each name in its ``__all__`` (plus the unexported classes user scripts
import) must exist here, classes must keep their public methods, and constructors / methods must accept the
reference's parameter names in the reference's order (extra trailing keyword parameters are allowed)."""
import importlib
import inspect

import pytest

MODULES = {            # reference module -> ours, extra (unexported but used) names
    "gossipy": ("gossipy_b200", ["LOG", "CACHE", "set_seed", "CacheKey", "CacheItem", "Sizeable", "Cache",
                                 "GlobalSettings"]),
    "gossipy.core": ("gossipy_b200.core", ["Delay", "MixingMatrix", "Message", "MessageType"]),
    "gossipy.node": ("gossipy_b200.node", ["All2AllGossipNode"]),
    "gossipy.model": ("gossipy_b200.model", []),
    "gossipy.model.nn": ("gossipy_b200.model.nn", []),
    "gossipy.model.sampling": ("gossipy_b200.model.sampling", []),
    "gossipy.model.handler": ("gossipy_b200.model.handler", ["ModelHandler", "WeightedTMH", "LimitedMergeTMH",
                                                              "LimitedMergeMixin"]),
    "gossipy.flow_control": ("gossipy_b200.flow_control", []),
    "gossipy.data": ("gossipy_b200.data", ["RecSysDataDispatcher", "get_FEMNIST"]),
    "gossipy.data.handler": ("gossipy_b200.data.handler", []),
    "gossipy.simul": ("gossipy_b200.simul", ["All2AllGossipSimulator", "SimulationEventSender"]),
    "gossipy.utils": ("gossipy_b200.utils", []),
}


def _params(fn):
    try:
        sig = inspect.signature(fn)
    except (TypeError, ValueError):
        return None
    return [p for p in sig.parameters.values() if p.name != "self"]


def _describe_callable(fn):
    params = _params(fn)
    return None if params is None else [(p.name, p.kind.name, p.default is not p.empty) for p in params]


def _describe_module(rmod, extra):
    """The reference module's public API as plain data: names, kinds, parameters, class members."""
    names = list(getattr(rmod, "__all__", [])) + [n for n in extra if hasattr(rmod, n)]
    out = []
    for name in dict.fromkeys(names):
        robj = getattr(rmod, name)
        if inspect.isclass(robj):
            d = {"kind": "class", "skip": issubclass(robj, BaseException) or name in ("LOG",), "members": []}
            if "__init__" in vars(robj):
                d["init"] = _describe_callable(robj.__init__)
            for attr, member in vars(robj).items():
                if attr.startswith("_") or inspect.isclass(member) or inspect.ismodule(member):
                    continue       # (the reference imports a class inside one class body)
                d["members"].append((attr, _describe_callable(member) if inspect.isfunction(member) else False))
        elif inspect.isfunction(robj):
            d = {"kind": "function", "params": _describe_callable(robj)}
        else:
            d = {"kind": "other"}
        out.append((name, d))
    return out


def _check_callable(rp, our_fn, where):
    op = _params(our_fn)
    if rp is None or op is None:
        return
    if any(p.kind in (p.VAR_POSITIONAL, p.VAR_KEYWORD) for p in op):
        return      # we forward *args/**kwargs (e.g. handler subclasses): accepted by construction
    ours = [p.name for p in op]
    for i, (name, kind, has_default) in enumerate(rp):
        if kind in ("VAR_POSITIONAL", "VAR_KEYWORD"):
            continue
        assert name in ours, "%s: parameter %r missing (ours: %s)" % (where, name, ours)
        if kind == "POSITIONAL_OR_KEYWORD" and not has_default:
            assert ours.index(name) == i, "%s: positional parameter %r moved" % (where, name)
    for p in op:      # anything we added must be optional
        if p.name not in [q[0] for q in rp]:
            assert p.default is not p.empty or p.kind == p.KEYWORD_ONLY and p.default is not p.empty, \
                "%s: new required parameter %r" % (where, p.name)


@pytest.mark.parametrize("ref_name", sorted(MODULES))
def test_module_api_parity(ref, ref_name):
    ours_name, extra = MODULES[ref_name]
    api = ref(lambda rg: _describe_module(importlib.import_module(ref_name), extra))
    omod = importlib.import_module(ours_name)
    assert api, ref_name
    for name, d in api:
        assert hasattr(omod, name), "%s.%s is missing" % (ours_name, name)
        oobj = getattr(omod, name)
        if d["kind"] == "class":
            assert inspect.isclass(oobj), name
            if d["skip"]:
                continue
            if "init" in d:
                _check_callable(d["init"], oobj.__init__, "%s.%s.__init__" % (ours_name, name))
            for attr, params in d["members"]:
                assert hasattr(oobj, attr), "%s.%s.%s is missing" % (ours_name, name, attr)
                if params is not False:
                    _check_callable(params, getattr(oobj, attr), "%s.%s.%s" % (ours_name, name, attr))
        elif d["kind"] == "function":
            _check_callable(d["params"], oobj, "%s.%s" % (ours_name, name))


def _enum_members(core):
    return [[(m.name, m.value) for m in getattr(core, name)] for name in ("CreateModelMode", "AntiEntropyProtocol", "MessageType")]


def test_enum_members_match(ref):
    import gossipy_b200.core as oc
    assert [[tuple(m) for m in e] for e in ref(lambda rg: _enum_members(rg.core))] == _enum_members(oc)
