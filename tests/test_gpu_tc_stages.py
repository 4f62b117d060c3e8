"""Stage-by-stage check of the tensor-core network against the oracle's intermediates."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.parametrize("name,C", [("cfg1_ont_drna", 18), ("phased_noisy", 30)])
def test_tc_intermediates(name, C):
    from clair3_rna_b200 import weights
    from clair3_rna_b200.engine import Engine
    from oracle import model
    g = np.load(os.path.join(HERE, "golden", name + ".npz"))
    x = g["tensor"][:300]
    w = weights.synthetic(C, sharpen=8.0)
    eng = Engine(0, C, nn_impl=1)
    eng.set_weights(w)
    p, ms = eng.forward(x)
    inter = {}
    ref = model.forward(w, x, intermediates=inter)
    n = x.shape[0]
    report = {}
    for which, key in ((0, "h1"), (2, "h2"), (3, "l4")):
        report[key] = float(np.abs(eng.debug_fetch(which, n) - inter[key]).max())
    report["probs"] = float(np.abs(p - ref).max())
    print(name, report, "ms", ms)
    eng.close()
    assert report["h1"] < 2e-3, report
    assert report["h2"] < 3e-3, report
    assert report["l4"] < 2e-2, report
    assert report["probs"] <= 1e-3, report
