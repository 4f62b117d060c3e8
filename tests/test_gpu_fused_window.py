"""The production input path of the tensor-core network: with nn_impl = 1, no keep_tensor and no padding rule, K4
writes LSTM1's fp16 operand images directly (k_window_xop, csrc/pileup.cuh) and the int32 tensor is never built.

Every run here is made twice, fused (keep_tensor=False) and unfused (keep_tensor=True: k_window, then k_xop in
tc_forward).  Both images come from the same round-to-nearest conversion of the same (rescaled) counts, so the
probabilities must be bit-identical; the unfused tensor is the reference the fused probabilities are compared with
through the fp32 oracle (|dp| <= 1e-3, BASELINE.json north_star)."""
import os

import numpy as np
import pytest

from tests.golden import cases as golden_cases

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
PROB_TOL = 1e-3
MAX_DEPTH = 144
# allele-frequency thresholds that take config 2 at full size past two sub-passes of tc_forward
SUBPASS_AF = 0.03

# every golden case the fused path serves (padding=False), C = 18 and C = 30, region modes and head/tail calling
FUSED_CASES = ["cfg1_ont_drna", "cfg2_ont_cdna", "ties_lowdepth", "cfg5_two_chunks", "af_zero",
               "cfg4_hifi_phased", "phased_noisy", "bed_regions", "known_sites", "range_mode",
               "headtail_ont", "headtail_known", "headtail_phased_bed"]


def assert_same_candidates(a, b):
    for k in ("pos", "depth", "alt_off", "alt_n"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    # the allele-table entries of every candidate (slots between them are never written)
    n = a.alt_n.astype(np.int64)
    idx = np.repeat(a.alt_off - (np.cumsum(n) - n), n) + np.arange(int(n.sum()))
    assert a.alt[idx].tobytes() == b.alt[idx].tobytes()


def assert_close_to_oracle(probs, ref, tol=PROB_TOL):
    """|dp| <= tol, and the argmax of both heads agrees wherever the oracle's top two are further apart than 2 tol"""
    assert probs.shape == ref.shape
    err = float(np.abs(probs - ref).max()) if ref.size else 0.0
    assert err <= tol, err
    for lo, hi in ((0, 21), (21, 24)):
        top2 = np.sort(ref[:, lo:hi], axis=1)[:, -2:]
        clear = (top2[:, 1] - top2[:, 0]) > 2 * tol
        assert np.array_equal(probs[:, lo:hi].argmax(1)[clear], ref[:, lo:hi].argmax(1)[clear])
    return err


def window_reference(res, C):
    """the K4 windows of res (keep_rows=True) gathered from its count rows with numpy, deep centres divided by
    depth / 144 in fp64 and truncated (clair3_rna/utils.py:85-92,120)"""
    rows = res.row_counts.reshape(-1, C).astype(np.int64)
    row_of = np.searchsorted(res.row_pos, res.pos)
    win = rows[row_of[:, None] + np.arange(-16, 17)[None, :]]
    deep = res.depth.astype(np.float64) > MAX_DEPTH * 1.5
    want = win.astype(np.int32)
    sf = res.depth[deep].astype(np.float64) / MAX_DEPTH
    want[deep] = (win[deep].astype(np.float64) / sf[:, None, None]).astype(np.int32)
    return want, deep


def run_pair(make_engine, call):
    """(fused result, unfused result) of the same call on two engines that differ only in keep_tensor"""
    out = []
    for keep in (False, True):
        eng = make_engine(keep)
        try:
            out.append(call(eng))
        finally:
            eng.close()
    return out


def _golden_runs(name, eng):
    """one ChunkResult per producer call, with the chunk plans of test_gpu_parity.run_chunked"""
    batch, ref_bytes, _ = golden_cases.build(name)
    ref = np.frombuffer(ref_bytes, np.uint8)
    plans = golden_cases.chunk_plans(name)
    whole = len(plans) == 1 and plans[0].site_filter() is None and \
        (plans[0].start1, plans[0].end1, plans[0].ref_start1) == (1, len(ref_bytes) + 33, 1)
    if whole:
        return [eng.call_chunk(batch, ref, 1, 1, len(ref_bytes) + 33)]
    out = []
    for plan in plans:
        if plan is None:
            continue
        s1, e1, rs1, re1 = plan.start1, plan.end1, plan.ref_start1, plan.ref_end1
        out.append(eng.call_chunk(batch.fetch(s1, e1), ref[rs1 - 1:re1], rs1, s1, e1, plan.site_filter()))
    return out


@pytest.mark.parametrize("name", FUSED_CASES)
def test_fused_window_matches_unfused_and_oracle(name):
    from clair3_rna_b200 import weights
    from clair3_rna_b200.engine import Engine
    from oracle import model
    case = golden_cases.CASES[name]
    assert not case["padding"]
    C = 30 if case["phased"] else 18
    w = weights.synthetic(C, sharpen=8.0)

    def make_engine(keep):
        eng = Engine(0, C, snp_min_af=case["snp_af"], indel_min_af=case["indel_af"], min_coverage=case["min_cov"],
                     min_mq=case["min_mq"], enable_padding=False, nn_impl=1, keep_tensor=keep,
                     enable_head_tail=case.get("head_tail", False))
        eng.set_weights(w)
        return eng

    fused, unfused = run_pair(make_engine, lambda eng: _golden_runs(name, eng))
    assert len(fused) == len(unfused)
    for f, u in zip(fused, unfused):
        assert f.tensor is None and u.tensor is not None        # the fused run never built the int32 tensor
        assert_same_candidates(f, u)
        assert np.array_equal(f.probs.view(np.uint32), u.probs.view(np.uint32))
    g = np.load(os.path.join(HERE, "golden", name + ".npz"))
    assert np.array_equal(np.concatenate([u.tensor for u in unfused]), g["tensor"])
    probs = np.concatenate([f.probs for f in fused])
    assert probs.shape[0] == g["tensor"].shape[0] > 0
    err = assert_close_to_oracle(probs, model.forward(w, g["tensor"]))
    print(name, "sites", probs.shape[0], "max |dp| fused vs oracle %.3e" % err)


def _deep_exon_batch(seed=4101):
    """three exons at about 300x, 1200x and 3000x with a mismatch site every 7 bp (alt fraction 0.1-0.9) and 1 %
    random substitutions, reads on both strands: most candidates are deeper than 1.5 x 144, so k_window_xop divides
    their windows in fp64"""
    from clair3_rna_b200.reads import ReadBatch
    rng = np.random.default_rng(seed)
    L = 3600
    ref_codes = rng.integers(0, 4, L)
    nt16 = np.array([1, 2, 4, 8], np.uint8)                         # A C G T
    records = []
    for a, b, depth in ((500, 900, 300), (1500, 1900, 1200), (2600, 3000, 3000)):
        sites = np.arange(a + 20, b - 20, 7)
        alt = (ref_codes[sites] + rng.integers(1, 4, sites.size)) % 4
        af = rng.uniform(0.1, 0.9, sites.size)
        n = int(depth * (b - a - 140) / 140)
        for _ in range(n):
            ln = int(rng.integers(80, 201))
            p0 = int(rng.integers(a, b - ln + 1))
            codes = ref_codes[p0:p0 + ln].copy()
            m = (sites >= p0) & (sites < p0 + ln)
            carry = m & (rng.random(sites.size) < af)
            codes[sites[carry] - p0] = alt[carry]
            err = rng.random(ln) < 0.01
            codes[err] = (codes[err] + rng.integers(1, 4, int(err.sum()))) % 4
            records.append((p0, 16 if rng.random() < 0.5 else 0, 60, 0, [(ln, 0)], nt16[codes]))
    records.sort(key=lambda r: r[0])
    ref = np.frombuffer(b"ACGT", np.uint8)[ref_codes].copy()
    return ReadBatch.from_records("chr1", records), ref


def test_deep_centre_windows_rescaled_in_the_fused_path():
    from clair3_rna_b200 import weights
    from clair3_rna_b200.engine import Engine
    from oracle import model
    batch, ref = _deep_exon_batch()
    w = weights.synthetic(18, sharpen=8.0)

    def make_engine(keep):
        eng = Engine(0, 18, nn_impl=1, keep_tensor=keep, keep_rows=keep)
        eng.set_weights(w)
        return eng

    fused, unfused = run_pair(make_engine, lambda eng: eng.call_chunk(batch, ref, 1, 1, ref.size + 33))
    assert unfused.n_cand > 100
    want, deep = window_reference(unfused, 18)
    assert deep.sum() > 50 and (~deep).sum() > 0        # both the rescaled and the plain branch of k_window_xop
    assert unfused.depth.max() > 2000
    assert np.array_equal(unfused.tensor, want)
    assert_same_candidates(fused, unfused)
    assert np.array_equal(fused.probs.view(np.uint32), unfused.probs.view(np.uint32))
    err = assert_close_to_oracle(fused.probs, model.forward(w, unfused.tensor))
    print("deep centre: %d sites (%d rescaled), max depth %d, max |dp| %.3e" % (
        fused.n_cand, int(deep.sum()), int(fused.depth.max()), err))


def test_fused_window_across_sub_passes():
    """config 2 at full size with lowered thresholds: more than two sub-passes of tc_forward, where LSTM1 reads the
    fused image at the sub-pass's offset (xop_ready + o / 128 tiles)"""
    import torch
    from clair3_rna_b200 import weights
    from clair3_rna_b200.engine import Engine
    from oracle import model
    from tests.test_gpu_fullsize import make
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    R = sm // 4
    Q = 128 * (320 // (2 * R)) * 2 * R                     # sites per sub-pass (TC_SUB_TILES in nn_tc.cuh)
    cfg, batch, ref, clen = make(2)
    w = weights.synthetic(18, sharpen=8.0)

    def make_engine(keep):
        eng = Engine(0, 18, snp_min_af=SUBPASS_AF, indel_min_af=SUBPASS_AF, min_coverage=2, nn_impl=1,
                     keep_tensor=keep)
        eng.set_weights(w)
        return eng

    fused, unfused = run_pair(make_engine, lambda eng: eng.call_chunk(batch, ref, 1, 1, clen + 33))
    n = fused.n_cand
    print("sub-pass test: %d candidates, %d sites per sub-pass" % (n, Q))
    assert n > 2 * Q
    assert_same_candidates(fused, unfused)
    assert np.array_equal(fused.probs.view(np.uint32), unfused.probs.view(np.uint32))
    rng = np.random.default_rng(3)
    idx = []
    for o in range(0, n, Q):
        e = min(n, o + Q)
        idx += [np.arange(o, min(e, o + 128)), np.arange(max(o, e - 128), e), rng.choice(np.arange(o, e), 256)]
    idx = np.unique(np.concatenate(idx))
    err = assert_close_to_oracle(fused.probs[idx], model.forward(w, unfused.tensor[idx]))
    print("sub-pass test: %d sampled sites, max |dp| %.3e" % (idx.size, err))

