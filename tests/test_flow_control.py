"""Token accounts: exhaustive table comparison with the reference."""
import numpy as np
import pytest

from gossipy_b200 import flow_control as fc


@pytest.mark.parametrize("name,args", [("PurelyReactiveTokenAccount", (2,)),
                                        ("SimpleTokenAccount", (3,)),
                                        ("GeneralizedTokenAccount", (8, 3)),
                                        ("RandomizedTokenAccount", (20, 10))])
def test_tables_match_reference(ref, name, args):
    def table(module):
        acc = getattr(module, name)(*args)
        rows = []
        for a in range(0, 45):
            acc.n_tokens = a
            row = [acc.proactive()]
            for u in (0, 1, 2):
                if name == "RandomizedTokenAccount":
                    np.random.seed(a * 7 + u)
                row.append(acc.reactive(u))
            rows.append(row)
        return rows
    ours, theirs = table(fc), ref(lambda rg: table(rg.flow_control))
    assert len(ours) == len(theirs) == 45
    for a, (o, t) in enumerate(zip(ours, theirs)):
        assert o[0] == pytest.approx(t[0]), a
        assert o[1:] == t[1:], a


def test_add_sub_and_proactive_account():
    acc = fc.PurelyProactiveTokenAccount()
    assert acc.n_tokens == 0 and acc.proactive() == 1 and acc.reactive(5) == 0   # B21 fixed
    acc.add(3); acc.sub(5)
    assert acc.n_tokens == 0
    with pytest.raises(AssertionError):
        fc.GeneralizedTokenAccount(2, 3)
    assert fc.RandomizedTokenAccount(20, 10).spec() == (4, 20, 10, 0)
