"""The two-group pass plan of the tensor-core network (nn_sched.h) against the rounds plan (C3R_PASS_SCHEDULE=rounds).

A site's result does not depend on which SMs or which launch ran its tile, so every batch size must give the same
bits under both plans and as the same sites sent in batches of 256.  Sizes where the planner splits a pass into two
groups (a partly filled last round: 45, 58 and 90 tile pairs on 148 SMs) and where it does not (one and two whole
rounds) are both covered, and so are passes of both plans in flight at once."""
import os
from contextlib import contextmanager

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# in tile pairs of 256 sites, R = sm_count // 4; "-40" leaves the last tile pair partly filled
SIZES = ["256*R", "512*R", "14617", "256*(R+8)-40", "256*(2*R+16)-40"]


def resolve(size):
    import torch
    R = torch.cuda.get_device_properties(0).multi_processor_count // 4
    return int(eval(size, {"R": R}))


@contextmanager
def rounds_schedule():
    old = os.environ.get("C3R_PASS_SCHEDULE")
    os.environ["C3R_PASS_SCHEDULE"] = "rounds"
    try:
        yield
    finally:
        if old is None:
            del os.environ["C3R_PASS_SCHEDULE"]
        else:
            os.environ["C3R_PASS_SCHEDULE"] = old


@pytest.fixture(scope="module")
def net():
    from clair3_rna_b200 import weights
    from clair3_rna_b200.engine import Engine
    from tests.test_gpu_network_large import _tensor
    x = _tensor(max(resolve(s) for s in SIZES), 18)
    eng = Engine(0, 18, nn_impl=1)
    eng.set_weights(weights.adversarial(18, recurrent_scale=1.0, forget_bias=1.5))
    p256 = np.concatenate([eng.forward(x[o:o + 256])[0] for o in range(0, len(x), 256)])
    yield eng, x, p256
    eng.close()


@pytest.mark.parametrize("size", SIZES)
def test_same_bits_as_rounds_and_as_batches_of_256(net, size):
    eng, x, p256 = net
    n = resolve(size)
    p, _ = eng.forward(x[:n])
    with rounds_schedule():
        r, _ = eng.forward(x[:n])
    assert np.array_equal(p.view(np.uint32), p256[:n].view(np.uint32))
    assert np.array_equal(p.view(np.uint32), r.view(np.uint32))


def test_tickets_in_flight_equal_rounds_alone():
    """three tickets in flight (config 2 at full size, a one-pair golden, config 2 again ...) under the default plan,
    each equal bit for bit to its call made alone under the rounds plan"""
    from collections import deque
    from clair3_rna_b200 import weights
    from clair3_rna_b200.engine import Engine
    from tests.golden import cases as golden_cases
    from tests.test_gpu_fullsize import make
    from tests.test_gpu_fused_window import assert_same_candidates
    _, batch2, ref2, clen = make(2)
    jobs = [(batch2, ref2, 1, 1, clen + 33, None)]
    b, r, _ = golden_cases.build("cfg2_ont_cdna")
    jobs.append((b, np.frombuffer(r, np.uint8), 1, 1, len(r) + 33, None))
    eng = Engine(0, 18)
    eng.set_weights(weights.synthetic(18, sharpen=8.0))
    with rounds_schedule():
        alone = [eng.call_chunk(*j) for j in jobs]
    q = deque()
    for i in [0, 0, 1, 0, 0, 1, 0, 0, 0]:
        q.append((i, eng.submit(*jobs[i])))
        if len(q) == 3:
            k, t = q.popleft()
            got = eng.wait(t)
            assert_same_candidates(got, alone[k])
            assert np.array_equal(got.probs.view(np.uint32), alone[k].probs.view(np.uint32)), k
    while q:
        k, t = q.popleft()
        got = eng.wait(t)
        assert_same_candidates(got, alone[k])
        assert np.array_equal(got.probs.view(np.uint32), alone[k].probs.view(np.uint32)), k
    eng.close()
