"""Call records (csrc/call.cuh) on the host: c3r_format_vcf over the records of c3r_debug_decide_calls - the code
k_call runs on the GPU - must print exactly the lines c3r_decode_vcf prints, on the decoder goldens, on reference
windows that do not start at 1 or cut a deletion short, and on a seeded fuzz of alt tables and probability vectors
built to reach every outcome family, every reachable retry branch and every reachable GT."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests.golden import cases as golden_cases
from tests.test_decode_native_cpu import CASES, build_result

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

# retry branches that cannot be taken: two distinct insertion keys are never equal, and the two ALTs of HET_DELDEL
# come from deletion keys of different lengths, so they never coincide with each other or with REF
UNREACHABLE_RETRIES = {"HET_INSINS_SAME", "HET_DELDEL_SAME"}
RETRIES = ["HOMO_SNP_NO_X", "HOMO_SNP_IS_REF", "HET_SNP_LT2_X", "HET_SNP_NO_X", "HET_SNP_IS_REF", "HOMO_INS_NO_I",
           "HET_ACGT_INS_NO_I", "HET_ACGT_INS_NO_X", "HET_INSINS_LT2_I", "HET_INSINS_SAME", "HOMO_DEL_NO_D",
           "HET_ACGT_DEL_NO_D", "HET_DELDEL_LT2_D", "HET_DELDEL_SAME", "INSDEL_NO_I_OR_D"]


@pytest.fixture(scope="module")
def lib():
    from clair3_rna_b200 import build, lib as L
    build.build()
    return L.load()


def both(res, batch, ref, ref_start1, contig="chr1", **kw):
    """(c3r_decode_vcf rows, c3r_format_vcf rows over the host records, the records)"""
    from clair3_rna_b200.engine import decode_vcf_rows, format_vcf_rows, decide_calls
    calls = decide_calls(res, batch, ref, ref_start1)
    return (decode_vcf_rows(res, batch, ref, ref_start1, contig, **kw),
            format_vcf_rows(res, batch, ref, ref_start1, contig, calls=calls, **kw), calls)


@pytest.mark.parametrize("threads", [1, 5])
@pytest.mark.parametrize("name", CASES)
def test_records_format_like_decode_on_goldens(lib, name, threads):
    g = np.load(os.path.join(HERE, "golden", name + ".npz"))
    d = np.load(os.path.join(HERE, "golden", "decoder_" + name + ".npz"))
    _, ref_bytes, _ = golden_cases.build(name)
    pos = np.concatenate([g["pos"], g["pos"]])
    alt = [str(s) for s in g["alt_info"]] * 2
    res, batch = build_result(name, d["probs"], pos, alt, ref_bytes)
    ref = np.frombuffer(ref_bytes, np.uint8)
    for show_ref in (True, False):
        for qual in (None, 2, 8):
            want, got, calls = both(res, batch, ref, 1, show_ref=show_ref, qual=qual, threads=threads)
            assert got == want and len(want) > 0, (show_ref, qual)
    assert len(set(calls["family"].tolist()) - {0xFF}) >= 2


def _small_result(ref, pos, probs, depth, entries, alt_n):
    from clair3_rna_b200.engine import ChunkResult, ALT_DTYPE
    from clair3_rna_b200.reads import ReadBatch
    alt_off = np.concatenate([[0], np.cumsum(alt_n)[:-1]]).astype(np.int64)
    z32, z8 = np.zeros(0, np.int32), np.zeros(0, np.uint8)
    batch = ReadBatch("c", z32, np.zeros(0, np.uint16), z8, z8, np.zeros(1, np.int32), np.zeros(0, np.uint32),
                      np.zeros(1, np.int64), np.array([0x12, 0x48, 0xf1], np.uint8))
    res = ChunkResult(0, np.asarray(pos, np.int32), np.asarray(depth, np.int32), np.asarray(probs, np.float32),
                      alt_off, np.asarray(alt_n, np.int32), np.array(entries, dtype=ALT_DTYPE), None, None, None, None)
    return res, batch


def test_window_offset_and_deletions_cut_at_the_window_end(lib):
    """a window starting at 1001, a candidate whose flank is padded, and deletions running past the window end:
    HOMO_DEL, HET_DELDEL (one key cut to the same length as a shorter one) and INSDEL"""
    ref = np.frombuffer(b"CGTACGTTAGCATGCATGACCGTAGCTAGCTAGGATCCATG", np.uint8)
    rs1, n = 1001, ref.size
    end = rs1 + n - 1
    pos = [1005, 1020, end - 2, end - 3, end - 4, end]
    probs = np.zeros((6, 24), np.float32)
    probs[0, 2] = 0.9; probs[0, 23] = 0.8            # AG 0/1
    probs[1, 10] = 0.7; probs[1, 22] = 0.9           # DelDel 1/1
    probs[2, 10] = 0.7; probs[2, 22] = 0.9           # DelDel 1/1, deletion cut at the window end
    probs[3, 10] = 0.8; probs[3, 23] = 0.9           # DelDel 0/1
    probs[4, 20] = 0.8; probs[4, 23] = 0.9           # InsDel
    probs[5, 10] = 0.7; probs[5, 22] = 0.9           # deletion entirely off the window: no key
    b = lambda p: ord(chr(ref[p - rs1]))
    D = lambda p, ln, c: (ord('D'), b(p), ln, c, 0, 0)
    entries = [(ord('X'), ord('G'), 0, 7, 0, 0), (ord('R'), b(1005), 0, 9, 0, 1),
               D(1020, 3, 11), (ord('R'), b(1020), 0, 2, 0, 1),
               D(end - 2, 5, 6), (ord('R'), b(end - 2), 0, 3, 0, 1),
               D(end - 3, 1, 4), D(end - 3, 7, 5), D(end - 3, 9, 6),     # 7 and 9 are both cut to 3 letters
               (ord('I'), b(end - 4), 3, 8, 1, 0), D(end - 4, 2, 5), (ord('R'), b(end - 4), 0, -1, 0, 1),
               D(end, 2, 9), (ord('R'), b(end), 0, 1, 0, 1)]
    res, batch = _small_result(ref, pos, probs, [16, 13, 20, 18, 17, 12], entries, [2, 2, 2, 3, 3, 2])
    for show_ref in (True, False):
        for qual in (None, 2, 8):
            want, got, calls = both(res, batch, ref, rs1, "chrT", show_ref=show_ref, qual=qual)
            assert got == want, (show_ref, qual)
    fams = calls["family"].tolist()
    assert fams[1] == 6 and fams[2] == 6 and fams[4] == 9, fams
    assert calls["ref_len"][2] == 3                      # REF = centre + the 2 bases left in the window
    rows = {int(r.split("\t")[1]): r.split("\t") for r in want}
    assert rows[end - 2][3] == ref[-3:].tobytes().decode()


def test_candidates_off_the_window(lib):
    """window 101..110 with candidates at its last base, after it (111, 113) and before it (98): their 33-base context
    is padded with 'A', so they are called like an 'A' centre - a reference call, a HOMO_SNP A>G and a deletion whose
    key starts at the window's first base - and both decoders print all four rows"""
    ref = np.frombuffer(b"ACGTTGCAAC", np.uint8)
    rs1 = 101
    pos = [110, 111, 113, 98]
    probs = np.zeros((4, 24), np.float32)
    probs[0, 4] = 0.9; probs[0, 21] = 0.9             # CC, 0/0 at the window's last base
    probs[1, 0] = 0.9; probs[1, 21] = 0.9             # AA, 0/0 past the end
    probs[2, 7] = 0.9; probs[2, 22] = 0.9             # GG, 1/1 past the end
    probs[3, 10] = 0.8; probs[3, 22] = 0.9            # DelDel, 1/1 before the start
    entries = [(ord('R'), ord('C'), 0, 6, 0, 0),
               (ord('R'), ord('A'), 0, 4, 0, 0),
               (ord('X'), ord('G'), 0, 7, 0, 0), (ord('R'), ord('A'), 0, 1, 0, 1),
               (ord('D'), ord('A'), 5, 6, 0, 0), (ord('R'), ord('A'), 0, 2, 0, 1)]
    res, batch = _small_result(ref, pos, probs, [6, 4, 8, 8], entries, [1, 1, 2, 2])
    for show_ref in (True, False):
        for qual in (None, 2, 8):
            want, got, calls = both(res, batch, ref, rs1, "chrT", show_ref=show_ref, qual=qual)
            assert got == want, (show_ref, qual)
    want, got, calls = both(res, batch, ref, rs1, "chrT")
    rows = {int(r.split("\t")[1]): r.split("\t") for r in got}
    assert sorted(rows) == [98, 110, 111, 113]
    assert rows[113][3:5] == ["A", "G"] and rows[113][9].startswith("1/1")
    assert rows[98][3:5] == ["AACG", "A"]                  # REF: the padded centre + the 3 bases the key keeps
    assert calls["family"].tolist() == [0, 0, 1, 6]


def _fuzz(n, seed):
    """n candidates over and around one reference window: random alt tables (duplicate insertion keys, keys longer than 50,
    deletions cut at the window end, several X alleles with tied counts, R counts <= 0) and probability vectors
    that are random, sharpened towards one outcome, or tied across outcomes on a dyadic grid (exact float32 ties)"""
    from clair3_rna_b200.engine import ChunkResult, ALT_DTYPE
    from clair3_rna_b200.reads import ReadBatch
    rng = np.random.default_rng(seed)
    L, rs1 = 6000, 2001
    letters = np.frombuffer(b"ACGTACGTACGTACGTACGTNRYKU-E", np.uint8)  # IUPAC codes, N, and two outside the table
    ref = letters[rng.integers(0, letters.size, L)].copy()
    acgt = rng.random(L) < 0.6
    ref[acgt] = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(acgt.sum()))]
    pool_codes = np.array([1, 2, 4, 8, 15, 1, 2, 4, 8, 3, 0], np.uint8)[rng.integers(0, 11, 400000)]
    seq = ((pool_codes[0::2] << 4) | pool_codes[1::2]).astype(np.uint8)
    # mostly inside the window, 10 % in its last 40 bases (deletions cut short), 2 % on either side of it
    u = rng.random(n)
    pos = np.where(u < 0.1, rs1 + L - 1 - rng.integers(0, 40, n), rs1 + rng.integers(0, L, n))
    pos = np.where(u > 0.98, rs1 - 1 - rng.integers(0, 40, n), np.where(u > 0.96, rs1 + L + rng.integers(0, 40, n), pos))
    pos = pos.astype(np.int32)
    HOMO_IX, HET_IX = [0, 4, 7, 9], [1, 2, 3, 5, 6, 8]
    # (gt21 index, genotype index) that make one member of one family the largest product
    targets = [(HOMO_IX[i], 1) for i in range(4)] + [(HET_IX[i], 2) for i in range(6)] + [(15, 1), (15, 2)] + \
              [(16 + i, 2) for i in range(4)] + [(10, 1), (10, 2)] + [(11 + i, 2) for i in range(4)] + [(20, 2), (None, 0)]
    grid = np.float32(1 / 64)
    probs = (rng.integers(0, 65, (n, 24)) * grid).astype(np.float32)
    mode = rng.integers(0, 4, n)
    for i in np.nonzero(mode == 0)[0]:                   # plain random (continuous)
        probs[i] = rng.random(24, dtype=np.float32)
    for i in np.nonzero(mode >= 1)[0]:                   # sharpened towards a target, on the grid
        g21, g3 = targets[rng.integers(0, len(targets))]
        probs[i] = (rng.integers(0, 16, 24) * grid).astype(np.float32)
        if g21 is None:                                  # a reference call by the early exit or by the products
            probs[i, 21] = 0.75
            probs[i, HOMO_IX] = 0.75 if rng.random() < 0.5 else 0.3
        else:
            probs[i, g21] = np.float32(rng.integers(40, 65) * grid)
            probs[i, 21 + g3] = np.float32(rng.integers(40, 65) * grid)
            probs[i, 21] = np.float32(rng.integers(0, 32) * grid)
        if mode[i] == 3:                                 # adversarial ties: copy the target's value elsewhere
            for _ in range(int(rng.integers(1, 4))):
                j = int(rng.integers(0, 21))
                probs[i, j] = probs[i, g21 if g21 is not None else 0]
            if rng.random() < 0.5:
                probs[i, 22] = probs[i, 23]
    entries, alt_n, depth = [], np.zeros(n, np.int32), rng.integers(0, 80, n).astype(np.int32)
    depth[rng.random(n) < 0.01] = 0
    xb = b"ACGTN"
    for i in range(n):
        p0 = int(pos[i]) - rs1
        centre = int(ref[p0]) if 0 <= p0 < L else ord('A')    # off the window: the padded context
        mine = []
        ties = rng.random() < 0.3
        for _ in range(int(rng.choice(5, p=[0.3, 0.25, 0.25, 0.1, 0.1]))):
            base = centre if rng.random() < 0.1 else xb[int(rng.integers(0, 5))]
            mine.append((88, base, 0, 5 if ties else int(rng.integers(-2, 30)), 0, 0))
        for _ in range(int(rng.choice(5, p=[0.3, 0.3, 0.2, 0.1, 0.1]))):
            if mine and rng.random() < 0.25 and any(e[0] == 73 for e in mine):     # the same key again
                e = [e for e in mine if e[0] == 73][0]
                mine.append((73, e[1], e[2], int(rng.integers(0, 30)), e[4], 0))
                continue
            ln = int(rng.choice([0, 1, 1, 2, 3, 5, 8, 49, 50, 55])) if rng.random() < 0.97 else 0
            mine.append((73, xb[int(rng.integers(0, 4))], ln, 4 if ties else int(rng.integers(0, 30)),
                         int(rng.integers(0, 399000)), 0))
        for _ in range(int(rng.choice(4, p=[0.3, 0.3, 0.25, 0.15]))):
            ln = int(rng.choice([1, 1, 2, 3, 4, 7, 12, 50, 51, 60]))
            mine.append((68, centre, ln, 4 if ties else int(rng.integers(0, 30)), 0, 0))
        for _ in range(int(rng.choice(3, p=[0.2, 0.7, 0.1]))):
            mine.append((82, centre, 0, int(rng.integers(-3, 40)), 0, 0))
        order = rng.permutation(len(mine))
        entries += [mine[k] for k in order]
        alt_n[i] = len(mine)
    alt_off = np.concatenate([[0], np.cumsum(alt_n)[:-1]]).astype(np.int64)
    z32, z8 = np.zeros(0, np.int32), np.zeros(0, np.uint8)
    batch = ReadBatch("c", z32, np.zeros(0, np.uint16), z8, z8, np.zeros(1, np.int32), np.zeros(0, np.uint32),
                      np.zeros(1, np.int64), seq)
    res = ChunkResult(0, pos, depth, probs, alt_off, alt_n, np.array(entries, dtype=ALT_DTYPE), None, None, None, None)
    return res, batch, ref, rs1


def test_seeded_fuzz_reaches_every_branch_and_formats_like_decode(lib):
    res, batch, ref, rs1 = _fuzz(200_000, seed=20261021)
    want, got, calls = both(res, batch, ref, rs1, threads=8)
    assert len(want) > 100_000
    assert got == want
    want0, got0, _ = both(res, batch, ref, rs1, show_ref=False, qual=8, threads=3)
    assert got0 == want0 and len(got0) < len(want)
    fam = calls["family"]
    assert set(fam.tolist()) == set(range(10)) | {0xFF}, sorted(set(fam.tolist()))
    gts = set(calls["gt"][fam != 0xFF].tolist())
    # "None" needs a row whose only flag is INSDEL without a ',' in ALT, and INSDEL's ALT always has two alleles
    assert gts == {0, 1, 2, 3}, gts
    seen = np.bitwise_or.reduce(calls["retries"].astype(np.uint32))
    for k, name in enumerate(RETRIES):
        assert bool(seen >> k & 1) == (name not in UNREACHABLE_RETRIES), name
    # the two quirks: a family that fails after setting REF and ALT ends the loop with them (HET_ACGT_INS keeps its
    # insertion) ...
    r = calls[(calls["retries"] >> RETRIES.index("HET_ACGT_INS_NO_X") & 1).astype(bool) & (fam == 4)]
    assert r.size > 0 and (r["n_alt"] == 1).all()
    # ... and a decision whose flags tie across families counts its alleles by the rule of the family output_with
    # tests first: HET_INSINS before HET_ACGT_INS, HET_DELDEL before HET_ACGT_DEL
    flags = calls["flags"].astype(np.uint32)
    assert ((fam == 4) & (flags >> 5 & 1).astype(bool)).sum() > 0
    assert ((fam == 7) & (flags >> 8 & 1).astype(bool)).sum() > 0
    assert ((fam != 0xFF) & (fam != 0) & ((flags >> fam.astype(np.uint32)) & 1 == 0)).sum() == 0   # own family flagged
    # candidates on both sides of the window are called and printed
    off = (res.pos < rs1) | (res.pos >= rs1 + ref.size)
    lo, hi = rs1, rs1 + ref.size
    n_off_rows = sum(1 for r in got if not lo <= int(r.split("\t")[1]) < hi)
    assert off.sum() > 1000 and n_off_rows > 1000


def test_call_record_layout_matches_the_header(lib, tmp_path):
    """CALL_DTYPE and lib.Call against sizeof / offsetof of the C compiler"""
    from clair3_rna_b200 import lib as L
    cc = shutil.which("cc") or shutil.which("gcc") or shutil.which("c++")
    if cc is None:
        pytest.skip("no host C compiler")
    fields = ["prob", "ref_count", "support", "ad", "family", "gt", "n_ad", "n_alt", "ref_first", "ref_len",
              "retries", "flags", "alt"]
    afields = ["first", "ins_len", "ins_seq_off", "suffix_from"]
    src = tmp_path / "layout.c"
    body = ['printf("%zu\\n", sizeof(c3r_call));', 'printf("%zu\\n", sizeof(c3r_call_allele));']
    body += ['printf("%%zu\\n", offsetof(c3r_call, %s));' % f for f in fields]
    body += ['printf("%%zu\\n", offsetof(c3r_call_allele, %s));' % f for f in afields]
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "c3r_b200.h"\nint main(void) {\n%s\nreturn 0;\n}\n'
                   % "\n".join(body))
    exe = tmp_path / "layout"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, stdout=subprocess.PIPE, text=True).stdout.split()]
    size, asize, offs, aoffs = got[0], got[1], got[2:2 + len(fields)], got[2 + len(fields):]
    assert size <= 64
    assert L.CALL_DTYPE.itemsize == size == C.sizeof(L.Call)
    assert L.CALL_DTYPE["alt"].base.itemsize == asize == C.sizeof(L.CallAllele)
    assert [L.CALL_DTYPE.fields[f][1] for f in fields] == offs == [getattr(L.Call, f).offset for f in fields]
    assert [L.CALL_DTYPE["alt"].base.fields[f][1] for f in afields] == aoffs == \
        [getattr(L.CallAllele, f).offset for f in afields]


def test_format_refuses_missing_records(lib):
    from clair3_rna_b200.engine import _result_struct
    ref = np.frombuffer(b"ACGTACGTACGT", np.uint8)
    res, batch = _small_result(ref, [3], np.zeros((1, 24), np.float32), [5], [(ord('R'), ord('G'), 0, 5, 0, 0)], [1])
    keep = []
    r = _result_struct(res, keep)
    text, nb, nr = C.c_void_p(), C.c_int64(0), C.c_int64(0)
    rc = lib.c3r_format_vcf(C.byref(r), None, None, ref.ctypes.data, 1, ref.size, b"c", 2.0, 1, 1,
                            C.byref(text), C.byref(nb), C.byref(nr))
    assert rc == -1 and not text.value
    assert lib.c3r_debug_decide_calls(C.byref(r), None, None, 1, ref.size, None) == -1


def test_format_refuses_records_it_cannot_print(lib):
    """a malformed record, or records made over a longer window than the one given, fail the call: no rows go missing"""
    from clair3_rna_b200.engine import format_vcf_rows, decide_calls, C3RError
    ref = np.frombuffer(b"CGTACGTTAGCATGCATGACCGTAGCTAGCTAGGATCCATG", np.uint8)
    probs = np.zeros((1, 24), np.float32)
    probs[0, 10] = 0.7; probs[0, 22] = 0.9                                  # DelDel 1/1
    res, batch = _small_result(ref, [1020], probs, [13], [(ord('D'), ref[19], 6, 11, 0, 0)], [1])
    calls = decide_calls(res, batch, ref, 1001)
    assert calls["family"][0] == 6 and calls["ref_len"][0] == 7
    assert len(format_vcf_rows(res, batch, ref, 1001, "c", calls=calls)) == 1
    with pytest.raises(C3RError):                                           # the window the records were not made on
        format_vcf_rows(res, batch, ref[:22], 1001, "c", calls=calls)
    for field, value in (("gt", 7), ("n_alt", 3), ("n_ad", 3), ("family", 12), ("ref_len", 0)):
        bad = calls.copy()
        bad[field] = value
        with pytest.raises(C3RError):
            format_vcf_rows(res, batch, ref, 1001, "c", calls=bad)
    bad = calls.copy()
    bad["alt"]["suffix_from"][0, 0] = 9
    with pytest.raises(C3RError):
        format_vcf_rows(res, batch, ref, 1001, "c", calls=bad)


def test_no_candidates(lib):
    from clair3_rna_b200.engine import ChunkResult, ALT_DTYPE
    ref = np.frombuffer(b"ACGTACGTACGT", np.uint8)
    _, batch = _small_result(ref, [3], np.zeros((1, 24), np.float32), [5], [(ord('R'), ord('G'), 0, 5, 0, 0)], [1])
    res = ChunkResult(0, np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 24), np.float32),
                      np.zeros(0, np.int64), np.zeros(0, np.int32), np.zeros(0, ALT_DTYPE), None, None, None, None)
    want, got, calls = both(res, batch, ref, 1)
    assert want == got == [] and calls.shape == (0,)
