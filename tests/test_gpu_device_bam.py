"""Device BAM reading (c3r_submit_bam_chunk, csrc/bgzf.cuh) on the GPU: the records the GPU inflates and parses
equal c3r_bam_fetch's bit for bit, and everything computed from them equals the host-read path - on the fixtures
of the CPU tests, with tickets of both kinds in flight, a corrupt block, and through run_chunks --device_bam."""
import os

import numpy as np
import pytest

from tests.golden import cases as golden_cases
from tests.test_bam_cpu import batch_records, py_write_bam
from tests.test_bgzf_cpu import special_records, write_aligned_bam

pytestmark = pytest.mark.gpu
READ_FIELDS = ("pos", "flag", "mapq", "hp", "cigar_off", "cigar", "seq_off", "seq")


@pytest.fixture(scope="module")
def eng():
    from clair3_rna_b200 import weights
    from clair3_rna_b200.engine import Engine
    e = Engine(0, 18, device_calls=True)
    e.set_weights(weights.synthetic(18, sharpen=8.0))
    yield e
    e.close()


def assert_reads_equal(got, want):
    for k in READ_FIELDS:
        assert np.array_equal(getattr(got, k), getattr(want, k)), k


def assert_results_equal(a, b):
    assert a.n_rows == b.n_rows
    for k in ("pos", "depth", "probs", "alt_off", "alt_n"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    # each candidate's alleles (the table has unused entries between candidates)
    used = np.concatenate([np.arange(o, o + n) for o, n in zip(a.alt_off, a.alt_n)]) if a.n_cand else np.zeros(0, int)
    assert np.array_equal(a.alt[used], b.alt[used])
    assert a.calls.tobytes() == b.calls.tobytes()


def both_paths(eng, bf, contig, s, e, ref, rs1):
    """(host-read result, device-read result, host fetch) of one chunk"""
    batch = bf.fetch(contig, s, e)
    host = eng.call_chunk(batch, ref, rs1, s, e)
    dev = eng.wait(eng.submit_bam(bf.fetch_raw(contig, s, e), ref, rs1, s, e))
    return host, dev, batch


def fixtures(tmp):
    """(path, contig, contig length, reference) of every BAM layout the CPU tests cover"""
    from clair3_rna_b200 import bam
    out = []
    batch, ref_bytes, contig = golden_cases.build("cfg1_ont_drna")
    n = len(ref_bytes)
    p = os.path.join(tmp, "lib.bam")
    bam.write_bam(p, [("chr0", 5000), (contig, n), ("chrZ", 100)], {contig: batch}, level=1)
    out.append((p, contig, n, np.frombuffer(ref_bytes, np.uint8)))
    batch, ref_bytes, contig = golden_cases.build("cfg2_ont_cdna")
    n = len(ref_bytes)
    recs = batch_records(batch)
    p = os.path.join(tmp, "small.bam")
    py_write_bam(p, [(contig, n)], recs)
    out.append((p, contig, n, np.frombuffer(ref_bytes, np.uint8)))
    p = os.path.join(tmp, "aligned.bam")
    write_aligned_bam(p, [(contig, n)], recs)
    out.append((p, contig, n, np.frombuffer(ref_bytes, np.uint8)))
    p = os.path.join(tmp, "special.bam")
    py_write_bam(p, [("c", 200000)], special_records(), payload=5000)
    out.append((p, "c", 200000, np.frombuffer(b"ACGT" * 50000, np.uint8)))
    return out


def test_same_reads_and_results(eng, tmp_path):
    from clair3_rna_b200 import bam
    rng = np.random.default_rng(2)
    for path, contig, n, ref in fixtures(str(tmp_path)):
        with bam.BamFile(path) as bf:
            regions = [(1, n), (1, 1), (n, n), (max(1, n - 50), n)]
            for _ in range(4):
                s = int(rng.integers(1, n))
                regions.append((s, min(n, s + int(rng.integers(1, 40000)))))
            for s, e in regions:
                host, dev, batch = both_paths(eng, bf, contig, s, e, ref, 1)
                assert_reads_equal(dev.reads, batch)
                assert_results_equal(dev, host)
                assert dev.bam_ms >= 0.0 and host.reads is None
            if "chr0" in bf.references:              # a contig without records: an empty chunk
                empty = eng.wait(eng.submit_bam(bf.fetch_raw("chr0", 1, 5000), ref, 1, 1, 5000))
                assert empty.reads.n_reads == 0 and empty.n_cand == 0


def test_tickets_in_flight_and_resident_reference(eng, tmp_path):
    from clair3_rna_b200 import bam
    batch, ref_bytes, contig = golden_cases.build("cfg2_ont_cdna")
    n = len(ref_bytes)
    ref = np.frombuffer(ref_bytes, np.uint8)
    p = str(tmp_path / "t.bam")
    bam.write_bam(p, [(contig, n)], {contig: batch}, level=1)
    cuts = [(1, n // 3), (n // 3 + 1, 2 * n // 3), (2 * n // 3 + 1, n)]
    with bam.BamFile(p) as bf:
        want = [eng.call_chunk(bf.fetch(contig, s, e), ref, 1, s, e) for s, e in cuts]
        for kinds in (("bam", "host", "bam"), ("host", "bam", "bam"), ("bam", "bam", "bam")):
            tickets = []
            for (s, e), k in zip(cuts, kinds):
                if k == "bam":
                    tickets.append(eng.submit_bam(bf.fetch_raw(contig, s, e), ref, 1, s, e))
                else:
                    tickets.append(eng.submit(bf.fetch(contig, s, e), ref, 1, s, e))
            for t, w, k in zip(tickets, want, kinds):
                r = eng.wait(t)
                assert_results_equal(r, w)
                assert (r.reads is not None) == (k == "bam")
        eng.set_reference(ref, 1)
        for (s, e), w in zip(cuts, want):
            assert_results_equal(eng.wait(eng.submit_bam(bf.fetch_raw(contig, s, e), None, 1, s, e)), w)


def test_corrupt_block_is_a_status(eng, tmp_path):
    from clair3_rna_b200 import bam
    from clair3_rna_b200.engine import C3RError
    batch, ref_bytes, contig = golden_cases.build("cfg2_ont_cdna")
    n = len(ref_bytes)
    ref = np.frombuffer(ref_bytes, np.uint8)
    p = str(tmp_path / "x.bam")
    bam.write_bam(p, [(contig, n)], {contig: batch}, level=1)
    with bam.BamFile(p) as bf:
        good = bf.fetch_raw(contig, 1, n)
        want = eng.call_chunk(bf.fetch(contig, 1, n), ref, 1, 1, n)
    bad = bam.BamFile(p).fetch_raw(contig, 1, n)
    b = bad.blocks[int(bad.raw.n_blocks) // 2]
    bad.data[b.coff + b.csize // 2] ^= 0x5a                 # inside the deflate payload: inflate or CRC fails
    t = eng.submit_bam(bad, ref, 1, 1, n)
    with pytest.raises(C3RError) as e:
        eng.wait(t)
    assert "BGZF" in str(e.value) and "rc=-1" in str(e.value)
    assert_results_equal(eng.wait(eng.submit_bam(good, ref, 1, 1, n)), want)      # the context goes on


def write_inputs(tmp, n_contigs=4):
    from tests.test_gpu_run_chunks import make_inputs
    cfg, ref, batches, fa, bam_fn, w_fn = make_inputs(tmp, n_contigs=n_contigs)
    bed = os.path.join(tmp, "r.bed")
    vcf = os.path.join(tmp, "g.vcf")
    rng = np.random.default_rng(7)
    with open(bed, "w") as fb, open(vcf, "w") as fv:
        fv.write("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n")
        for name, length in cfg.contigs:
            for s in sorted(rng.integers(0, length - 2000, 6).tolist()):
                fb.write("%s\t%d\t%d\n" % (name, s, s + int(rng.integers(100, 2000))))
            for s in sorted(set(rng.integers(1, length, 40).tolist())):
                fv.write("%s\t%d\t.\tA\tC\t.\t.\t.\n" % (name, s))
    return bam_fn, fa, w_fn, bed, vcf


@pytest.mark.parametrize("mode", ["plain", "device_calls", "bed", "vcf"])
def test_run_chunks_device_bam(tmp_path, mode):
    from clair3_rna_b200 import run_chunks
    bam_fn, fa, w_fn, bed, vcf = write_inputs(str(tmp_path))
    kw = dict(device_calls=mode == "device_calls", bed_fn=bed if mode == "bed" else None,
              vcf_fn=vcf if mode == "vcf" else None)
    outs = []
    for dev in (False, True):
        out = str(tmp_path / ("m%d.vcf" % dev))
        st = {}
        run_chunks.run(bam_fn, fa, w_fn, out, device_bam=dev, stats=st, **kw)
        outs.append(open(out, "rb").read())
        if dev:
            assert st["bam_device_ms"] > 0 and st["host_seconds"]["fetch"] > 0
    assert outs[0] == outs[1] and outs[0].count(b"\n") > 30
