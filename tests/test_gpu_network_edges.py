"""The tensor-core network at the edges of its schedule and of its input range.

Batch shapes: tc_forward runs LSTM2 in rounds of R = sm // 4 tile pairs (S = 256 R sites), launches the full rounds
and the remainder separately, and cuts a batch into sub-passes of Q = 128 (320 // 2R) 2R sites.  Sizes on each side
of these boundaries are compared with the fp32 oracle and with the same sites sent in batches of 256.

Deep inputs: a window's 33 rows can be far deeper than its centre (the fp64 rescale divides by the centre depth
only), so counts of 2 049 - 8 000 reach the network, where fp16 holds only every 2nd / 4th integer.

Tickets: passes of different sizes in flight at once, each equal to its call made alone."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
PROB_TOL = 1e-3

SIZES_18 = ["1", "2", "127", "128", "129", "255", "256", "257", "S-1", "S", "S+1", "2*S", "2*S+1", "Q", "Q+1"]
SIZES_30 = ["1", "129", "256", "S", "S+1", "Q+1"]


def schedule():
    """(R tile pairs per LSTM2 round, S sites per round, Q sites per sub-pass) of this device (nn_tc.cuh)"""
    import torch
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    R = sm // 4
    return R, 256 * R, 128 * (320 // (2 * R)) * 2 * R


def resolve(size):
    _, S, Q = schedule()
    return int(eval(size, {"S": S, "Q": Q}))


def make_weights(kind, C):
    from clair3_rna_b200 import weights
    if kind == "keras_init":
        return weights.synthetic(C, sharpen=8.0)
    return weights.adversarial(C, recurrent_scale=1.0, forget_bias=1.5)


def assert_close_to_oracle(probs, ref, tol=PROB_TOL):
    err = float(np.abs(probs - ref).max()) if ref.size else 0.0
    assert err <= tol, err
    for lo, hi in ((0, 21), (21, 24)):
        top2 = np.sort(ref[:, lo:hi], axis=1)[:, -2:]
        clear = (top2[:, 1] - top2[:, 0]) > 2 * tol
        assert np.array_equal(probs[:, lo:hi].argmax(1)[clear], ref[:, lo:hi].argmax(1)[clear])
    return err


def oracle(w, x):
    import torch
    from oracle import model
    torch.set_num_threads(max(1, (os.cpu_count() or 2) - 1))
    return np.concatenate([model.forward(w, x[o:o + 2048]) for o in range(0, len(x), 2048)]) if len(x) else \
        np.zeros((0, 24), np.float32)


# ------------------------------------------------------------------------------------------------ batch shapes
_shape_cache = {}


def _shape_setup(kind, C):
    """per (weights, C): the engine, real windows for the largest size, and their probabilities in batches of 256"""
    key = (kind, C)
    if key not in _shape_cache:
        from clair3_rna_b200.engine import Engine
        from tests.test_gpu_network_large import _tensor
        w = make_weights(kind, C)
        x = _tensor(max(resolve(s) for s in (SIZES_18 if C == 18 else SIZES_30)), C)
        eng = Engine(0, C, nn_impl=1)
        eng.set_weights(w)
        p256 = np.concatenate([eng.forward(x[o:o + 256])[0] for o in range(0, len(x), 256)])
        _shape_cache[key] = dict(w=w, x=x, eng=eng, p256=p256, oracle={})
    return _shape_cache[key]


@pytest.fixture(scope="module", autouse=True)
def _close_engines():
    yield
    for v in _shape_cache.values():
        v["eng"].close()
    _shape_cache.clear()


def checked_sites(n):
    """every site up to 2 048; beyond, the first 256, 256 on each side of every round and sub-pass boundary, the
    last 300"""
    if n <= 2048:
        return np.arange(n)
    _, S, Q = schedule()
    bounds = set(range(S, n, S)) | set(range(Q, n, Q))
    parts = [np.arange(256), np.arange(n - 300, n)] + [np.arange(max(0, b - 256), min(n, b + 256)) for b in bounds]
    return np.unique(np.concatenate(parts))


@pytest.mark.parametrize("kind,C,size", [(k, 18, s) for k in ("keras_init", "stress") for s in SIZES_18] +
                         [(k, 30, s) for k in ("keras_init", "stress") for s in SIZES_30])
def test_batch_shape_edges(kind, C, size):
    st = _shape_setup(kind, C)
    n = resolve(size)
    p, _ = st["eng"].forward(st["x"][:n])
    assert p.shape == (n, 24)
    # same bits as the same sites in batches of 256 (a site's result does not depend on the batch around it)
    assert np.array_equal(p.view(np.uint32), st["p256"][:n].view(np.uint32))
    idx = checked_sites(n)
    cache = st["oracle"]
    todo = np.array([i for i in idx if i not in cache], np.int64)
    if todo.size:
        for i, row in zip(todo, oracle(st["w"], st["x"][todo])):
            cache[int(i)] = row
    ref = np.stack([cache[int(i)] for i in idx])
    err = assert_close_to_oracle(p[idx], ref)
    print(kind, C, size, n, "checked %d sites, max |dp| %.3e" % (idx.size, err))


# ------------------------------------------------------------------------------------------------ deep inputs
def deep_windows(C, n=3000, seed=23):
    """real windows whose 32 non-centre rows are scaled by 60-190 plus an offset, so most counts fall in
    2 049 - 8 000 (positive counts, negative reference channels), then made odd or 2 mod 4: values fp16 cannot
    hold.  The centre row keeps its depth, as the rescale leaves it."""
    name = "cfg1_ont_drna" if C == 18 else "phased_noisy"
    g = np.load(os.path.join(HERE, "golden", name + ".npz"))["tensor"].astype(np.int64)
    rng = np.random.default_rng(seed)
    x = g[rng.integers(0, len(g), n)]
    mag = np.abs(x) * rng.uniform(60, 190, (n, 1, 1)) + rng.integers(1500, 4500, x.shape) * (x != 0)
    mag = np.minimum(np.rint(mag).astype(np.int64), 7999)
    two_mod4 = (mag > 4096) & (rng.random(mag.shape) < 0.5)
    mag = np.where(mag > 2048, np.where(two_mod4, (mag & ~3) | 2, mag | 1), mag)
    out = (np.sign(x) * mag).astype(np.int32)
    out[:, 16, :] = x[:, 16, :]
    return out


def fp16_rounded(x):
    return x.astype(np.float16).astype(np.int32)


@pytest.mark.parametrize("kind", ["keras_init", "stress"])
@pytest.mark.parametrize("C", [18, 30])
def test_deep_input_counts(kind, C):
    from clair3_rna_b200.engine import Engine
    x = deep_windows(C)
    x16 = fp16_rounded(x)
    side = np.ones(33, bool)
    side[16] = False
    big = np.abs(x[:, side]) > 2048
    assert big.sum() > 0.5 * (x[:, side] != 0).sum() and np.all(x[:, side][big] != x16[:, side][big])
    assert np.abs(x).max() <= 8000
    w = make_weights(kind, C)
    eng = Engine(0, C, nn_impl=1)
    eng.set_weights(w)
    p, _ = eng.forward(x)
    p16, _ = eng.forward(x16)
    eng.close()
    ref, ref16 = oracle(w, x), oracle(w, x16)
    total = float(np.abs(p - ref).max())
    rest = float(np.abs(p16 - ref16).max())            # the network's own error on inputs fp16 holds exactly
    inp = float(np.abs(ref - ref16).max())             # what rounding the input to fp16 alone moves
    print("deep inputs", kind, C, "GPU vs oracle(x) %.3e | GPU vs oracle(x16) on x16 %.3e | oracle(x) vs oracle(x16) %.3e"
          % (total, rest, inp))
    assert_close_to_oracle(p, ref)


def _junction_batch(seed=5150):
    """two splice junctions: ~6 000 (and ~7 000) reads, three in four on the forward strand, cover an exon and
    splice out with an N op; ~150 (~220) continue into the intron and carry mismatches there.  The intron candidates have depth 150-300, below the rescale
    threshold, and their windows hold the exon's rows of thousands of reads."""
    from clair3_rna_b200.reads import ReadBatch
    rng = np.random.default_rng(seed)
    L = 9000
    ref_codes = rng.integers(0, 4, L)
    nt16 = np.array([1, 2, 4, 8], np.uint8)
    records = []

    def read(p0, ops, codes):
        err = rng.random(codes.size) < 0.01
        codes[err] = (codes[err] + rng.integers(1, 4, int(err.sum()))) % 4
        records.append((p0, 16 if rng.random() < 0.25 else 0, 60, 0, ops, nt16[codes]))

    for ex0, ex1, n_spliced, n_retained in ((1000, 1300, 6000, 150), (5000, 5300, 7000, 220)):
        intron = 1000
        for _ in range(n_spliced):
            p0 = int(rng.integers(ex0, ex0 + 150))
            m1 = ex1 - p0
            codes = np.concatenate([ref_codes[p0:ex1], ref_codes[ex1 + intron:ex1 + intron + 100]])
            read(p0, [(m1, 0), (intron, 3), (100, 0)], codes)
        sites = np.concatenate([np.arange(ex1 + 1, ex1 + 16), np.arange(ex1 + 18, ex1 + 60, 3)])
        alt = (ref_codes[sites] + rng.integers(1, 4, sites.size)) % 4
        af = rng.uniform(0.3, 1.0, sites.size)
        for _ in range(n_retained):
            p0 = int(rng.integers(ex0 + 150, ex1 - 20))
            ln = ex1 + 80 - p0
            codes = ref_codes[p0:p0 + ln].copy()
            carry = rng.random(sites.size) < af
            codes[sites[carry] - p0] = alt[carry]
            read(p0, [(ln, 0)], codes)
    records.sort(key=lambda r: r[0])
    ref = np.frombuffer(b"ACGT", np.uint8)[ref_codes].copy()
    return ReadBatch.from_records("chr1", records), ref


def test_deep_rows_beside_a_shallow_centre_end_to_end():
    """call_chunk on the default path (fused window) against the unfused run and the oracle on its tensor"""
    from clair3_rna_b200 import weights
    from clair3_rna_b200.engine import Engine
    from tests.test_gpu_fused_window import assert_same_candidates, window_reference
    batch, ref = _junction_batch()
    w = weights.synthetic(18, sharpen=8.0)
    res = {}
    for keep in (False, True):
        eng = Engine(0, 18, keep_tensor=keep, keep_rows=keep)
        eng.set_weights(w)
        res[keep] = eng.call_chunk(batch, ref, 1, 1, ref.size + 33)
        eng.close()
    fused, unfused = res[False], res[True]
    want, deep = window_reference(unfused, 18)
    assert np.array_equal(unfused.tensor, want)
    x = unfused.tensor
    shallow = (unfused.depth >= 100) & (unfused.depth <= 300)
    assert shallow.sum() >= 20
    unrepresentable = (np.abs(x) > 2048) & (x != fp16_rounded(x))
    assert unrepresentable[shallow].any(axis=(1, 2)).sum() >= 20
    assert_same_candidates(fused, unfused)
    assert np.array_equal(fused.probs.view(np.uint32), unfused.probs.view(np.uint32))
    ref_p = oracle(w, x)
    err = assert_close_to_oracle(fused.probs, ref_p)
    inp = float(np.abs(ref_p - oracle(w, fp16_rounded(x))).max())
    print("junction: %d sites (%d of depth 100-300 with rows fp16 cannot hold), max |dp| %.3e, input share %.3e" % (
        fused.n_cand, int(unrepresentable[shallow].any(axis=(1, 2)).sum()), err, inp))


# ------------------------------------------------------------------------------------------------ tickets
def test_tickets_of_different_sizes_in_flight():
    """three tickets in flight from a rotation of config 2 at full size (a full LSTM2 round + a remainder), a
    one-pair golden and the two chunks of cfg5_two_chunks: LSTM1 of a pass is queued beside a previous pass whose
    last LSTM2 launch had a different number of tile pairs.  Every ticket equals its call made alone, bit for bit."""
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
    b, r, _ = golden_cases.build("cfg5_two_chunks")
    r = np.frombuffer(r, np.uint8)
    for plan in golden_cases.chunk_plans("cfg5_two_chunks"):
        jobs.append((b.fetch(plan.start1, plan.end1), r[plan.ref_start1 - 1:plan.ref_end1], plan.ref_start1,
                     plan.start1, plan.end1, plan.site_filter()))
    eng = Engine(0, 18)
    eng.set_weights(weights.synthetic(18, sharpen=8.0))
    alone = [eng.call_chunk(*j) for j in jobs]
    assert alone[0].n_cand > 2 * 128 * schedule()[0] and 0 < alone[1].n_cand <= 256
    order = [i % len(jobs) for i in range(14)]
    q = deque()
    for i in order:
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
