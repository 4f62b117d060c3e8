"""VCF rows the device's way, checked without a GPU: QUAL from the threshold table against QUAL from the host formula
for every float32, GQ and FILTER from hundredths, the row printer of k_vcf_len / k_vcf_write (csrc/vcf_row.cuh) run on
the host against c3r_format_vcf, and the row bound the device sizes its text buffers with."""
import ctypes as C
import os

import numpy as np
import pytest

from tests.golden import cases as golden_cases
from tests.test_decode_native_cpu import CASES, build_result
from tests.test_device_calls_cpu import _fuzz, _small_result

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def lib():
    from clair3_rna_b200 import build, lib as L
    build.build()
    return L.load()


def same_rows(res, batch, ref, rs1, contig="chr1", **kw):
    """debug_vcf_rows (table QUAL, counted lengths, rows written at their offsets) == format_vcf_rows; -> the rows"""
    from clair3_rna_b200.engine import debug_vcf_rows, decide_calls, format_vcf_rows
    calls = decide_calls(res, batch, ref, rs1)
    for show_ref in (True, False):
        for qual in (None, 2, 8):
            want = format_vcf_rows(res, batch, ref, rs1, contig, qual=qual, show_ref=show_ref, calls=calls, **kw)
            got = debug_vcf_rows(res, batch, ref, rs1, contig, qual=qual, show_ref=show_ref, calls=calls)
            assert got == want, (show_ref, qual)
    return format_vcf_rows(res, batch, ref, rs1, contig, calls=calls, **kw)


def test_qual_table_equals_the_formula_for_every_float32(lib):
    """all 2^32 bit patterns (NaN, infinities, negatives and values above 1 included): the same q, and on one pattern
    in 4096 the same text as printf("%.2f") of the formula's value"""
    n, bad = C.c_int64(0), C.c_int64(-1)
    assert lib.c3r_debug_vcf_qual_check(0, C.byref(n), C.byref(bad)) == 0
    assert n.value == 1 << 32 and bad.value == 0


@pytest.mark.parametrize("cut", [-1.0, 0.0, 2.0, 8.0, 2.5])
def test_gq_and_filter_from_hundredths(lib, cut):
    """GQ = q // 100 is (int)(q / 100.0); FILTER's q >= q_min is q / 100.0 >= qual_cut (or always PASS below 0)"""
    qm = C.c_int32(-1)
    assert lib.c3r_debug_vcf_q_min(cut, C.byref(qm)) == 0
    q = np.arange(0, 11002)
    qual = q / 100.0
    assert np.array_equal(qual.astype(np.int64), q // 100)
    want = np.ones(q.size, bool) if cut < 0 else qual >= cut
    assert np.array_equal(q >= qm.value, want)


def test_row_bound_and_worst_case_record(lib):
    """the longest row a record k_call makes can print: a 1024-byte contig, a 10-digit position, REF of 51 letters,
    two ALTs of 101, 11-character ints and AFs of 16; its length equals its counted length and fits the bound"""
    from clair3_rna_b200 import lib as L
    from clair3_rna_b200.engine import debug_vcf_rows, format_vcf_rows
    assert [lib.c3r_vcf_row_max(k) for k in (0, 4, 1024)] == [394, 398, 1418]
    rs1, pos = 2147483600, 2147483647
    ref = np.frombuffer(b"ACGT" * 30, np.uint8)
    res, batch = _small_result(ref, [pos], np.zeros((1, 24), np.float32), [1], [(ord('R'), ord('A'), 0, 1, 0, 0)], [1])
    batch.seq = np.full(64, 0x12, np.uint8)          # 128 nibbles for two 50-base insertions
    c = np.zeros(1, L.CALL_DTYPE)
    c["prob"], c["family"], c["gt"], c["n_alt"], c["n_ad"], c["ref_len"] = 1.0, 9, 4, 2, 2, 51
    c["ref_first"] = ord('A')
    c["ref_count"], c["ad"] = -2147483648, [[-2147483648, -2147483647]]
    for a in range(2):
        c["alt"][0, a] = (ord('C'), 0, 50, 10 * a, 1, 0)
    contig = "c" * 1024
    rows = debug_vcf_rows(res, batch, ref, rs1, contig, qual=1000.0, calls=c)
    assert rows == format_vcf_rows(res, batch, ref, rs1, contig, qual=1000.0, calls=c)
    f = rows[0].split("\t")
    assert len(f[3]) == 51 and [len(x) for x in f[4].split(",")] == [101, 101] and f[6] == "LowQual"
    assert f[9] == "None:110:1:-2147483648,-2147483648,-2147483647:-2147483648.0000,-2147483647.0000"
    assert len(rows[0]) + 1 <= lib.c3r_vcf_row_max(len(contig))
    assert len(rows[0]) + 1 >= lib.c3r_vcf_row_max(len(contig)) - 12


@pytest.mark.parametrize("name", CASES)
def test_printer_on_goldens(lib, name):
    g = np.load(os.path.join(HERE, "golden", name + ".npz"))
    d = np.load(os.path.join(HERE, "golden", "decoder_" + name + ".npz"))
    _, ref_bytes, _ = golden_cases.build(name)
    res, batch = build_result(name, d["probs"], g["pos"], [str(s) for s in g["alt_info"]], ref_bytes)
    assert same_rows(res, batch, np.frombuffer(ref_bytes, np.uint8), 1)


def test_printer_on_windows(lib):
    """the windows of test_device_calls_cpu.py: one starting at 1001 with deletions cut at its end, and candidates on
    both sides of a window 101..110"""
    ref = np.frombuffer(b"CGTACGTTAGCATGCATGACCGTAGCTAGCTAGGATCCATG", np.uint8)
    rs1, n = 1001, ref.size
    end = rs1 + n - 1
    probs = np.zeros((6, 24), np.float32)
    probs[0, 2] = 0.9; probs[0, 23] = 0.8
    probs[1, 10] = 0.7; probs[1, 22] = 0.9
    probs[2, 10] = 0.7; probs[2, 22] = 0.9
    probs[3, 10] = 0.8; probs[3, 23] = 0.9
    probs[4, 20] = 0.8; probs[4, 23] = 0.9
    probs[5, 10] = 0.7; probs[5, 22] = 0.9
    b = lambda p: ord(chr(ref[p - rs1]))
    D = lambda p, ln, c: (ord('D'), b(p), ln, c, 0, 0)
    entries = [(ord('X'), ord('G'), 0, 7, 0, 0), (ord('R'), b(1005), 0, 9, 0, 1),
               D(1020, 3, 11), (ord('R'), b(1020), 0, 2, 0, 1),
               D(end - 2, 5, 6), (ord('R'), b(end - 2), 0, 3, 0, 1),
               D(end - 3, 1, 4), D(end - 3, 7, 5), D(end - 3, 9, 6),
               (ord('I'), b(end - 4), 3, 8, 1, 0), D(end - 4, 2, 5), (ord('R'), b(end - 4), 0, -1, 0, 1),
               D(end, 2, 9), (ord('R'), b(end), 0, 1, 0, 1)]
    res, batch = _small_result(ref, [1005, 1020, end - 2, end - 3, end - 4, end], probs, [16, 13, 20, 18, 17, 12],
                               entries, [2, 2, 2, 3, 3, 2])
    assert len(same_rows(res, batch, ref, rs1, "chrT")) == 6
    ref = np.frombuffer(b"ACGTTGCAAC", np.uint8)
    probs = np.zeros((4, 24), np.float32)
    probs[0, 4] = 0.9; probs[0, 21] = 0.9
    probs[1, 0] = 0.9; probs[1, 21] = 0.9
    probs[2, 7] = 0.9; probs[2, 22] = 0.9
    probs[3, 10] = 0.8; probs[3, 22] = 0.9
    entries = [(ord('R'), ord('C'), 0, 6, 0, 0), (ord('R'), ord('A'), 0, 4, 0, 0),
               (ord('X'), ord('G'), 0, 7, 0, 0), (ord('R'), ord('A'), 0, 1, 0, 1),
               (ord('D'), ord('A'), 5, 6, 0, 0), (ord('R'), ord('A'), 0, 2, 0, 1)]
    res, batch = _small_result(ref, [110, 111, 113, 98], probs, [6, 4, 8, 8], entries, [1, 1, 2, 2])
    assert len(same_rows(res, batch, ref, 101, "chrT")) == 4


def test_printer_on_the_fuzz(lib):
    """200 000 candidates, rows with a NaN AF (depth 0, two AD counts) and negative counts among them"""
    res, batch, ref, rs1 = _fuzz(200_000, seed=20261021)
    rows = same_rows(res, batch, ref, rs1, threads=8)
    assert len(rows) > 100_000
    af = [r.rsplit(":", 1)[1] for r in rows]
    assert sum("nan" in a for a in af) > 0 and sum(a.startswith("-") for a in af) > 0
