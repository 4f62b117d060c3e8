"""Call records made on the GPU (k_call, csrc/call.cuh): for every golden case, at full size across sub-passes, with
several tickets in flight, without candidates and over a resident reference, the device records equal the host
instantiation of the same code (c3r_debug_decide_calls) bit for bit, and the rows c3r_format_vcf prints from them
equal c3r_decode_vcf's.  With records off a ticket is exactly what it was before they existed."""
import ctypes as C
import os

import numpy as np
import pytest

from tests.golden import cases as golden_cases

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
SUBPASS_AF = 0.03                                   # config 2 at full size: several sub-passes of the network


def _engine(case, **kw):
    from clair3_rna_b200 import weights
    from clair3_rna_b200.engine import Engine
    C_ = 30 if case["phased"] else 18
    eng = Engine(0, C_, snp_min_af=case["snp_af"], indel_min_af=case["indel_af"], min_coverage=case["min_cov"],
                 min_mq=case["min_mq"], enable_padding=case["padding"], enable_head_tail=case.get("head_tail", False),
                 **kw)
    eng.set_weights(weights.synthetic(C_, sharpen=8.0))          # sharpened: the non-RefCall families occur
    return eng


def _chunks(name):
    """(reads, reference window, ref_start1, region start1, region end1, site filter) of every producer call"""
    batch, ref_bytes, _ = golden_cases.build(name)
    ref = np.frombuffer(ref_bytes, np.uint8)
    out = []
    for plan in golden_cases.chunk_plans(name):
        if plan is None:
            continue
        out.append((batch.fetch(plan.start1, plan.end1), ref[plan.ref_start1 - 1:plan.ref_end1], plan.ref_start1,
                    plan.start1, plan.end1, plan.site_filter()))
    return out


def assert_records_match(res, batch, ref, rs1, contig="chr1"):
    """device records == host records (bytes); format(records) == decode; returns the records"""
    from clair3_rna_b200 import lib as L
    from clair3_rna_b200.engine import decode_vcf_rows, format_vcf_rows, decide_calls
    assert res.calls is not None and res.calls.dtype == L.CALL_DTYPE and res.calls.shape[0] == res.n_cand
    host = decide_calls(res, batch, ref, rs1)
    if res.calls.tobytes() != host.tobytes():
        i = int(np.nonzero((res.calls.view(np.uint8).reshape(res.n_cand, -1) !=
                            host.view(np.uint8).reshape(res.n_cand, -1)).any(1))[0][0])
        raise AssertionError("record %d: device %s host %s" % (i, res.calls[i], host[i]))
    for show_ref in (True, False):
        want = decode_vcf_rows(res, batch, ref, rs1, contig, show_ref=show_ref)
        assert format_vcf_rows(res, batch, ref, rs1, contig, show_ref=show_ref) == want
    return res.calls


@pytest.mark.parametrize("name", sorted(golden_cases.CASES))
def test_device_records_on_goldens(name):
    case = golden_cases.CASES[name]
    eng = _engine(case, device_calls=True)
    fams = set()
    try:
        for sub, r, rs1, s1, e1, flt in _chunks(name):
            res = eng.call_chunk(sub, r, rs1, s1, e1, flt)
            fams |= set(assert_records_match(res, sub, r, rs1)["family"].tolist())
            assert res.call_ms >= 0.0
    finally:
        eng.close()
    print(name, "families", sorted(fams))
    assert fams - {0, 0xFF}, "only reference calls: the weights are not sharp enough to test the decision"


def test_device_records_at_full_size():
    """config 2 at full size with thresholds lowered to 0.03: > 200 k candidates over several network sub-passes"""
    from clair3_rna_b200 import weights
    from clair3_rna_b200.engine import Engine
    from tests.test_gpu_fullsize import make
    cfg, batch, ref, clen = make(2)
    eng = Engine(0, 18, snp_min_af=SUBPASS_AF, indel_min_af=SUBPASS_AF, min_coverage=2, device_calls=True)
    eng.set_weights(weights.synthetic(18, sharpen=8.0))
    try:
        res = eng.call_chunk(batch, ref, 1, 1, clen + 33)
    finally:
        eng.close()
    assert res.n_cand > 200_000
    calls = assert_records_match(res, batch, ref, 1)
    print("full size: %d candidates, k_call %.3f ms, families %s" % (res.n_cand, res.call_ms,
                                                                      np.bincount(calls["family"], minlength=256)[[*range(10), 255]]))


def test_records_off_changes_nothing():
    from clair3_rna_b200 import lib as L
    name = "cfg1_ont_drna"
    case = golden_cases.CASES[name]
    (sub, r, rs1, s1, e1, flt), = _chunks(name)
    off, on = _engine(case), _engine(case, device_calls=True)
    try:
        a = off.call_chunk(sub, r, rs1, s1, e1, flt)
        b = on.call_chunk(sub, r, rs1, s1, e1, flt)
        assert a.calls is None and b.calls is not None and a.n_cand > 0
        assert b.launches == a.launches + 1                         # k_call, and nothing else
        for k in ("pos", "depth", "alt_off", "alt_n"):
            assert np.array_equal(getattr(a, k), getattr(b, k)), k
        assert a.probs.tobytes() == b.probs.tobytes() and a.alt.tobytes() == b.alt.tobytes()
        # a ticket submitted with records off has none
        t = off.submit(sub, r, rs1, s1, e1, flt)
        res = L.Result()
        assert off.lib.c3r_wait(off.ctx, t, C.byref(res)) == 0
        cp, cn = C.c_void_p(), C.c_int64(0)
        assert off.lib.c3r_wait_calls(off.ctx, t, C.byref(cp), C.byref(cn), None) == -3
        off.release(t)
        # switched off again: the next ticket is an ordinary one
        on.set_device_calls(False)
        c = on.call_chunk(sub, r, rs1, s1, e1, flt)
        assert c.calls is None and c.launches == a.launches and c.probs.tobytes() == a.probs.tobytes()
    finally:
        off.close()
        on.close()


def test_three_tickets_in_flight_zero_candidates_and_resident_reference():
    name = "cfg5_two_chunks"
    case = golden_cases.CASES[name]
    chunks = _chunks(name)
    batch, ref_bytes, _ = golden_cases.build(name)
    ref = np.frombuffer(ref_bytes, np.uint8)
    # a chunk without candidates: no reads
    from clair3_rna_b200.reads import ReadBatch
    z32, z8 = np.zeros(0, np.int32), np.zeros(0, np.uint8)
    nothing = ReadBatch("chr1", z32, np.zeros(0, np.uint16), z8, z8, np.zeros(1, np.int32), np.zeros(0, np.uint32),
                        np.zeros(1, np.int64), z8)
    empty = (nothing, ref, 1, 1, 400, None)
    jobs = [chunks[0], empty, chunks[-1]]
    eng = _engine(case, device_calls=True)
    try:
        alone = [eng.call_chunk(*j) for j in jobs]
        tickets = [eng.submit(*j) for j in jobs]
        together = [eng.wait(t) for t in tickets]
        for j, a, b in zip(jobs, alone, together):
            assert a.calls.tobytes() == b.calls.tobytes() and a.probs.tobytes() == b.probs.tobytes()
            assert_records_match(b, j[0], j[1], j[2])
        assert alone[1].n_cand == 0 and alone[1].calls.shape == (0,)
        assert alone[0].n_cand > 0 and alone[2].n_cand > 0
        # ref = None over the resident reference (the whole contig): same records as the chunk's own window
        eng.set_reference(ref, 1)
        sub, r, rs1, s1, e1, flt = chunks[-1]
        res = eng.call_chunk(sub, None, 1, s1, e1, flt)
        assert res.n_cand == alone[2].n_cand
        assert_records_match(res, sub, ref, 1)
        assert format_rows(res, sub, ref, 1) == format_rows(alone[2], sub, r, rs1)
    finally:
        eng.close()


def format_rows(res, batch, ref, rs1):
    from clair3_rna_b200.engine import format_vcf_rows
    return format_vcf_rows(res, batch, ref, rs1, "chr1")


def test_run_chunks_device_calls_writes_the_same_vcf(tmp_path):
    from clair3_rna_b200 import run_chunks
    from tests.test_gpu_run_chunks import make_inputs
    cfg, ref, batches, fa, bam_fn, w_fn = make_inputs(str(tmp_path))
    outs, stats = [], []
    for on in (False, True):
        out = os.path.join(str(tmp_path), "merged_%d.vcf" % on)
        st = {}
        run_chunks.run(bam_fn, fa, w_fn, out, stats=st, device_calls=on)
        outs.append(open(out).read())
        stats.append(st)
    assert outs[0] == outs[1] and outs[0].count("\n") > 50
    assert stats[0]["call_device_ms"] == 0.0 and stats[1]["call_device_ms"] > 0.0
    # a caller's engine: records for this run only, its own setting back afterwards
    from clair3_rna_b200 import weights
    from clair3_rna_b200.engine import Engine
    eng = Engine(0, 18)
    eng.set_weights(weights.load(w_fn))
    try:
        out = os.path.join(str(tmp_path), "merged_engine.vcf")
        st = {}
        run_chunks.run(bam_fn, fa, w_fn, out, stats=st, device_calls=True, engine=eng)
        assert open(out).read() == outs[0] and st["call_device_ms"] > 0.0
        assert eng.device_calls is False
    finally:
        eng.close()
    # the command line
    out = os.path.join(str(tmp_path), "cli.vcf")
    assert run_chunks.main(["--bam_fn", bam_fn, "--ref_fn", fa, "--chkpnt_fn", w_fn, "--output", out,
                            "--include_all_ctgs", "--device_calls"]) == 0
    base = os.path.join(str(tmp_path), "cli0.vcf")
    assert run_chunks.main(["--bam_fn", bam_fn, "--ref_fn", fa, "--chkpnt_fn", w_fn, "--output", base,
                            "--include_all_ctgs"]) == 0
    data = lambda path: [l for l in open(path).read().splitlines() if not l.startswith("#")]
    assert data(out) == data(base) and len(data(out)) > 50


@pytest.mark.parametrize("name", ["bed_regions", "known_sites"])
def test_run_chunks_device_calls_in_region_modes(tmp_path, name):
    from clair3_rna_b200 import run_chunks
    from tests.test_gpu_regions import _write_case_files
    f = _write_case_files(str(tmp_path), name)
    kw = dict(bed_fn=f["bed"]) if "bed" in f else dict(vcf_fn=f["vcf"])
    texts = []
    for on in (False, True):
        out = os.path.join(str(tmp_path), "all_%d.vcf" % on)
        rows = run_chunks.run(f["bam"], f["fa"], f["w"], out, device_calls=on, **kw)
        assert rows
        texts.append(open(out).read())
    assert texts[0] == texts[1]
