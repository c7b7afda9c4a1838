"""BASELINE.json's metric is "rounds/sec AND test-acc-vs-round": the accuracy curve of the native engine + fused
fp32-equivalent kernels must lie inside the seed band of the UNMODIFIED reference on identical shards (its curves are
recorded under tests/golden/reference/)."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def test_accuracy_curve_inside_reference_band(ref):
    sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
    import acc_band
    import gossipy_b200 as g
    seeds, rounds = 3, 12
    try:
        ours = [acc_band.run_ours(s, rounds, True) for s in range(seeds)]
        theirs = ref(lambda rg: [acc_band.run_reference(s, rounds, True) for s in range(seeds)])
    finally:
        g.GlobalSettings().set_device("cpu")
    out = acc_band.band(ours, theirs)
    assert out["inside_band"], out
    assert out["ours_mean"][-1] > out["ours_mean"][0] + 0.03          # and it learns
