"""c3r_decode_vcf (csrc/decode.cpp: the decision of csrc/call.cuh on the host and its row printer, native
multi-threaded A7) against the Python decoder and against the rows the reference's own output_with printed
(tests/golden/decoder_*.npz)."""
import os

import numpy as np
import pytest

from tests.golden import cases as golden_cases

HERE = os.path.dirname(os.path.abspath(__file__))
CASES = ["cfg1_ont_drna", "ties_lowdepth", "pad_dense", "phased_noisy"]


def build_result(name, probs, pos, alt_infos, ref_bytes):
    """ChunkResult + ReadBatch (sequence pool only) equivalent to the golden alt_info strings"""
    from clair3_rna_b200.engine import ChunkResult, ALT_DTYPE
    from clair3_rna_b200.reads import ReadBatch, encode_seq
    codes, entries, alt_off, alt_n, depth = [], [], [], [], []
    n_codes = 0
    for p, s in zip(pos, alt_infos):
        d, rest = s.rstrip("\n").split("-", 1) if "-" in s else (s, "")
        toks = rest.split(" ") if rest else []
        alt_off.append(len(entries))
        depth.append(int(d))
        k = 0
        for key, cnt in zip(toks[::2], toks[1::2]):
            kind = key[0]
            if kind in "XR":
                entries.append((ord(kind), ord(key[1]), 0, int(cnt), 0, k))
            elif kind == "I":
                ins = key[2:]
                c = encode_seq(ins)
                if n_codes & 1:                       # alleles may start on an odd base offset
                    pass
                entries.append((ord(kind), ord(key[1]), len(ins), int(cnt), n_codes, k))
                codes.append(c)
                n_codes += len(ins)
            else:
                entries.append((ord(kind), ord(ref_bytes[p - 1:p]), len(key) - 1, int(cnt), 0, k))
                assert ref_bytes[p:p + len(key) - 1].decode() == key[1:]
            k += 1
        alt_n.append(len(entries) - alt_off[-1])
    allc = np.concatenate(codes) if codes else np.zeros(0, np.uint8)
    if allc.size & 1:
        allc = np.concatenate([allc, np.zeros(1, np.uint8)])
    seq = ((allc[0::2] << 4) | allc[1::2]).astype(np.uint8)
    z32, z8 = np.zeros(0, np.int32), np.zeros(0, np.uint8)
    batch = ReadBatch("c", z32, np.zeros(0, np.uint16), z8, z8, np.zeros(1, np.int32), np.zeros(0, np.uint32),
                      np.zeros(1, np.int64), seq)
    res = ChunkResult(n_rows=0, pos=np.asarray(pos, np.int32), depth=np.asarray(depth, np.int32),
                      probs=np.asarray(probs, np.float32), alt_off=np.asarray(alt_off, np.int64),
                      alt_n=np.asarray(alt_n, np.int32), alt=np.array(entries, dtype=ALT_DTYPE),
                      tensor=None, row_pos=None, row_counts=None, row_depth=None)
    return res, batch


@pytest.mark.parametrize("threads", [1, 5])
@pytest.mark.parametrize("name", CASES)
def test_native_rows_equal_python_decoder_and_reference(name, threads):
    from clair3_rna_b200 import build, decoder
    build.build()
    from clair3_rna_b200.engine import decode_vcf_rows
    g = np.load(os.path.join(HERE, "golden", name + ".npz"))
    d = np.load(os.path.join(HERE, "golden", "decoder_" + name + ".npz"))
    _, ref_bytes, contig = golden_cases.build(name)
    pos = np.concatenate([g["pos"], g["pos"]])
    alt = [str(s) for s in g["alt_info"]] * 2
    ref33 = [str(s) for s in g["ref33"]] * 2
    probs, want_ref = d["probs"], [str(r) for r in d["rows"]]
    res, batch = build_result(name, probs, pos, alt, ref_bytes)
    ref = np.frombuffer(ref_bytes, np.uint8)
    got = decode_vcf_rows(res, batch, ref, 1, "chr1", threads=threads)
    py = [decoder.vcf_row("chr1", int(pos[i]), ref33[i], alt[i], probs[i]) for i in range(len(pos))]
    py = [r for r in py if r is not None]
    assert got == py                                         # identical to the Python restatement, QUAL included
    ref_rows = [r for r in want_ref if r]
    assert len(got) == len(ref_rows)
    exact = sum(1 for a, b in zip(got, ref_rows) if a == b)
    assert exact >= 0.99 * len(got)                          # the rest: QUAL last digit (NumPy 1 vs 2, SURVEY.md §8c)


def test_reference_window_offsets_and_padding():
    """candidate near the start of the loaded window: flank padded with 'A', window not starting at 1"""
    from clair3_rna_b200 import build, decoder
    build.build()
    from clair3_rna_b200.engine import decode_vcf_rows, ChunkResult, ALT_DTYPE
    from clair3_rna_b200.reads import ReadBatch
    ref = np.frombuffer(b"CGTACGTTAGCATGCATGACCGTAGCTAGCTAGGATCCATG", np.uint8)
    ref_start1 = 1001
    pos = np.array([1005, 1020], np.int32)
    probs = np.zeros((2, 24), np.float32)
    probs[0, 2] = 0.9; probs[0, 23] = 0.8            # AG, 0/1
    probs[1, 10] = 0.7; probs[1, 22] = 0.9           # DelDel, 1/1
    entries = [(ord('X'), ord('G'), 0, 7, 0, 0), (ord('R'), ord('C'), 0, 9, 0, 1),
               (ord('D'), ord(chr(ref[19])), 3, 11, 0, 0), (ord('R'), ord(chr(ref[19])), 0, 2, 0, 1)]
    res = ChunkResult(0, pos, np.array([16, 13], np.int32), probs, np.array([0, 2], np.int64), np.array([2, 2], np.int32),
                      np.array(entries, dtype=ALT_DTYPE), None, None, None, None)
    z32, z8 = np.zeros(0, np.int32), np.zeros(0, np.uint8)
    batch = ReadBatch("c", z32, np.zeros(0, np.uint16), z8, z8, np.zeros(1, np.int32), np.zeros(0, np.uint32),
                      np.zeros(1, np.int64), z8)
    got = decode_vcf_rows(res, batch, ref, ref_start1, "chrT")
    refs = ref.tobytes().decode()
    want = []
    for i, (p, ai) in enumerate(zip(pos, ["16-XG 7 RC 9", "13-D%s 11 R%s 2" % (refs[20:23], refs[19])])):
        lo = p - 16 - ref_start1
        r33 = 'A' * max(0, -lo) + refs[max(0, lo):p + 17 - ref_start1]
        r33 += 'A' * (33 - len(r33))
        want.append(decoder.vcf_row("chrT", int(p), r33, ai, probs[i]))
    assert got == want
    assert got[1].split("\t")[3] == refs[19:23] and got[1].split("\t")[4] == refs[19]


def test_fixed_point_formatting_equals_printf():
    """the decoder prints QUAL and AF without libc: every value must read like '%.2f' / '%.4f' (correct rounding of
    the exact binary value, ties to even) - exact ties, near-ties one ulp either side, count ratios, random values"""
    import ctypes as C
    from clair3_rna_b200 import lib as L
    lib = L.load()
    buf = C.create_string_buffer(64)

    def fmt(x, d):
        assert lib.c3r_debug_format_fixed(float(x), d, buf) == 0
        return buf.value.decode()
    rng = np.random.default_rng(11)
    vals = [0.0, 0.005, 0.015, 0.025, 0.125, 0.375, 0.00005, 0.00015, 0.03125, 0.09375, 1.0, 0.5, 2.675, 1.005, 109.99499999,
            99.995, 0.99995, 0.99994999999, 1e-300, 5e-324, 123456.785, 33.335, 8.0, 7.9949999999999, 1e11]
    vals += [k / 2.0 ** m for m in range(1, 20) for k in (1, 3, 5, 7, 9, 11, 13, 15)]            # exactly representable ties and non-ties
    vals += [s / d for d in range(1, 400) for s in range(0, d + 1, max(1, d // 7))]             # allele fractions
    vals += list(rng.uniform(0, 1, 20000)) + list(rng.uniform(0, 120, 20000))
    vals += [(k + 0.5) / 10000.0 for k in range(0, 3000, 7)] + [(k + 0.5) / 100.0 for k in range(0, 12000, 37)]
    more = []
    for v in vals:
        more += [np.nextafter(v, 0.0), np.nextafter(v, 1e300)]
    for v in vals + more:
        v = float(v)
        if not (0 <= v < 1e12):
            continue
        assert fmt(v, 2) == "%.2f" % v, repr(v)
        assert fmt(v, 4) == "%.4f" % v, repr(v)
    assert lib.c3r_debug_format_fixed(-1.0, 2, buf) != 0 and lib.c3r_debug_format_fixed(float("nan"), 4, buf) != 0
