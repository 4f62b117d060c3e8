"""VCF rows printed on the GPU (c3r_set_vcf; k_vcf_len, the offsets scan and k_vcf_write of csrc/vcf_row.cuh): for every
golden case and every show_ref / QUAL cut-off, at full size across network sub-passes, with several tickets in flight
under different contig names, without candidates, over a resident reference and from a device-parsed BAM, the text a
ticket returns equals what c3r_format_vcf prints from the device's call records, byte for byte.  With text off a ticket
is exactly what it was before; run_chunks --device_vcf writes the same merged VCF as the host decoder."""
import ctypes as C
import dataclasses
import os

import numpy as np
import pytest

from tests.golden import cases as golden_cases
from tests.test_gpu_device_calls import SUBPASS_AF, _chunks, _engine

pytestmark = pytest.mark.gpu
SETTINGS = [(show_ref, qual) for show_ref in (True, False) for qual in (None, 2, 8)]


def assert_text_matches(res, batch, ref, rs1, contig, qual=2, show_ref=True):
    """the ticket's text == c3r_format_vcf over its device records (same contig, qual, show_ref); -> the rows"""
    from clair3_rna_b200.engine import device_vcf_rows, format_vcf_rows
    want = format_vcf_rows(res, batch, ref, rs1, contig, qual=qual, show_ref=show_ref)
    assert res.vcf_text == "".join(r + "\n" for r in want)
    assert res.vcf_rows == len(want) and device_vcf_rows(res) == want
    return want


@pytest.mark.parametrize("name", sorted(golden_cases.CASES))
def test_device_text_on_goldens(name):
    case = golden_cases.CASES[name]
    eng = _engine(case, device_calls=True, device_vcf=True)
    n_rows = 0
    try:
        for sub, r, rs1, s1, e1, flt in _chunks(name):
            for show_ref, qual in SETTINGS:
                eng.set_device_vcf(True, qual=qual, show_ref=show_ref)
                res = eng.call_chunk(sub, r, rs1, s1, e1, flt)
                n_rows += len(assert_text_matches(res, sub, r, rs1, sub.contig, qual, show_ref))
                assert res.vcf_ms >= 0.0
    finally:
        eng.close()
    assert n_rows > 0


def test_device_text_at_full_size():
    """config 2 at full size with thresholds lowered to 0.03: > 200 k candidates over several network sub-passes"""
    from clair3_rna_b200 import weights
    from clair3_rna_b200.engine import Engine
    from tests.test_gpu_fullsize import make
    cfg, batch, ref, clen = make(2)
    eng = Engine(0, 18, snp_min_af=SUBPASS_AF, indel_min_af=SUBPASS_AF, min_coverage=2, device_calls=True,
                 device_vcf=True)
    eng.set_weights(weights.synthetic(18, sharpen=8.0))
    try:
        res = eng.call_chunk(batch, ref, 1, 1, clen + 33)
    finally:
        eng.close()
    assert res.n_cand > 200_000
    rows = assert_text_matches(res, batch, ref, 1, batch.contig)
    print("full size: %d candidates, %d rows, %d bytes, text kernels %.3f ms, D2H %.3f ms" % (
        res.n_cand, len(rows), len(res.vcf_text), res.vcf_ms, res.stage_ms[7]))


def test_text_off_changes_nothing():
    name = "cfg1_ont_drna"
    case = golden_cases.CASES[name]
    (sub, r, rs1, s1, e1, flt), = _chunks(name)
    off, on = _engine(case), _engine(case, device_vcf=True)
    try:
        a = off.call_chunk(sub, r, rs1, s1, e1, flt)
        b = on.call_chunk(sub, r, rs1, s1, e1, flt)
        assert a.vcf_text is None and b.calls is None and a.n_cand > 0
        assert b.launches == a.launches + 4                         # k_call, k_vcf_len, the scan, k_vcf_write
        for k in ("pos", "depth", "alt_off", "alt_n"):
            assert np.array_equal(getattr(a, k), getattr(b, k)), k
        assert a.probs.tobytes() == b.probs.tobytes() and a.alt.tobytes() == b.alt.tobytes()
        from clair3_rna_b200.engine import decode_vcf_rows
        assert b.vcf_text == "".join(x + "\n" for x in decode_vcf_rows(a, sub, r, rs1, sub.contig))
        # text on without records: c3r_wait_calls still refuses; a ticket with text off has no text
        from clair3_rna_b200 import lib as L
        t = on.submit(sub, r, rs1, s1, e1, flt)
        res = L.Result()
        assert on.lib.c3r_wait(on.ctx, t, C.byref(res)) == 0
        cp, cn = C.c_void_p(), C.c_int64(0)
        assert on.lib.c3r_wait_calls(on.ctx, t, C.byref(cp), C.byref(cn), None) == -3
        on.release(t)
        t = off.submit(sub, r, rs1, s1, e1, flt)
        assert off.lib.c3r_wait(off.ctx, t, C.byref(res)) == 0
        tp, nb, nr = C.c_void_p(), C.c_int64(0), C.c_int64(0)
        assert off.lib.c3r_wait_vcf(off.ctx, t, C.byref(tp), C.byref(nb), C.byref(nr), None) == -3
        off.release(t)
        on.set_device_vcf(False)
        c = on.call_chunk(sub, r, rs1, s1, e1, flt)
        assert c.vcf_text is None and c.launches == a.launches and c.probs.tobytes() == a.probs.tobytes()
    finally:
        off.close()
        on.close()


def test_three_tickets_two_contigs_empty_chunk_and_resident_reference():
    from clair3_rna_b200.reads import ReadBatch
    name = "cfg5_two_chunks"
    case = golden_cases.CASES[name]
    chunks = _chunks(name)
    batch, ref_bytes, _ = golden_cases.build(name)
    ref = np.frombuffer(ref_bytes, np.uint8)
    z32, z8 = np.zeros(0, np.int32), np.zeros(0, np.uint8)
    nothing = ReadBatch("chrE", z32, np.zeros(0, np.uint16), z8, z8, np.zeros(1, np.int32), np.zeros(0, np.uint32),
                        np.zeros(1, np.int64), z8)
    last = chunks[-1]
    renamed = (dataclasses.replace(last[0], contig="chrOther_name"),) + last[1:]
    jobs = [chunks[0], (nothing, ref, 1, 1, 400, None), renamed]
    eng = _engine(case, device_calls=True, device_vcf=True)
    try:
        alone = [eng.call_chunk(*j) for j in jobs]
        tickets = [eng.submit(*j) for j in jobs]
        together = [eng.wait(t) for t in tickets]
        for j, a, b in zip(jobs, alone, together):
            assert a.vcf_text == b.vcf_text
            assert_text_matches(b, j[0], j[1], j[2], j[0].contig)
        assert alone[1].n_cand == 0 and alone[1].vcf_text == "" and alone[1].vcf_rows == 0
        assert alone[0].vcf_rows > 0 and alone[2].vcf_text.startswith("chrOther_name\t")
        eng.set_reference(ref, 1)
        sub, r, rs1, s1, e1, flt = last
        res = eng.call_chunk(sub, None, 1, s1, e1, flt)
        assert_text_matches(res, sub, ref, 1, sub.contig)
        assert res.vcf_text == eng.call_chunk(*last).vcf_text
    finally:
        eng.close()


def test_device_text_of_a_device_parsed_bam(tmp_path):
    from clair3_rna_b200 import bam
    batch, ref_bytes, contig = golden_cases.build("cfg2_ont_cdna")
    n = len(ref_bytes)
    ref = np.frombuffer(ref_bytes, np.uint8)
    p = str(tmp_path / "t.bam")
    bam.write_bam(p, [(contig, n)], {contig: batch}, level=1)
    eng = _engine(golden_cases.CASES["cfg2_ont_cdna"], device_calls=True, device_vcf=True)
    try:
        with bam.BamFile(p) as bf:
            res = eng.wait(eng.submit_bam(bf.fetch_raw(contig, 1, n), ref, 1, 1, n))
            host = eng.call_chunk(bf.fetch(contig, 1, n), ref, 1, 1, n)
        assert res.vcf_rows > 0 and res.vcf_text == host.vcf_text
        assert_text_matches(res, res.reads, ref, 1, contig)
    finally:
        eng.close()


@pytest.mark.parametrize("mode", ["plain", "device_bam", "bed", "vcf"])
def test_run_chunks_device_vcf_writes_the_same_vcf(tmp_path, mode):
    from clair3_rna_b200 import run_chunks
    from tests.test_gpu_device_bam import write_inputs
    bam_fn, fa, w_fn, bed, vcf = write_inputs(str(tmp_path))
    kw = dict(device_bam=mode == "device_bam", bed_fn=bed if mode == "bed" else None,
              vcf_fn=vcf if mode == "vcf" else None)
    outs = []
    for dev in (False, True):
        out = str(tmp_path / ("m%d.vcf" % dev))
        st = {}
        run_chunks.run(bam_fn, fa, w_fn, out, device_vcf=dev, stats=st, **kw)
        outs.append(open(out, "rb").read())
        assert (st["vcf_device_ms"] > 0) == dev
    assert outs[0] == outs[1] and outs[0].count(b"\n") > 30
    if mode != "plain":
        return
    # a caller's engine: text for this run only, its own setting back afterwards
    from clair3_rna_b200 import weights
    from clair3_rna_b200.engine import Engine
    eng = Engine(0, 18)
    eng.set_weights(weights.load(w_fn))
    try:
        out = str(tmp_path / "engine.vcf")
        run_chunks.run(bam_fn, fa, w_fn, out, device_vcf=True, engine=eng)
        assert open(out, "rb").read() == outs[0] and eng.device_vcf is False
    finally:
        eng.close()
    # the command line
    cli = [str(tmp_path / ("cli%d.vcf" % k)) for k in range(2)]
    for path, extra in zip(cli, ([], ["--device_vcf"])):
        assert run_chunks.main(["--bam_fn", bam_fn, "--ref_fn", fa, "--chkpnt_fn", w_fn, "--output", path,
                                "--include_all_ctgs"] + extra) == 0
    data = lambda path: [l for l in open(path).read().splitlines() if not l.startswith("#")]
    assert data(cli[0]) == data(cli[1]) and len(data(cli[0])) > 30
