"""Device BAM reading without a GPU: the DEFLATE decoder and CRC check the kernels run (c3r_debug_inflate, the same
C3R_HD code on the host) against Python's zlib, and c3r_bam_fetch_raw's blocks and windows, inflated with zlib and
walked here, against c3r_bam_fetch."""
import ctypes as C
import os
import struct
import zlib

import numpy as np
import pytest

from tests.golden import cases as golden_cases
from tests.test_bam_cpu import batch_records, py_write_bam


@pytest.fixture(scope="module")
def lib():
    from clair3_rna_b200 import build
    build.build()
    from clair3_rna_b200 import lib as L
    return L.load()


def bgzf_block(payload: bytes, deflated: bytes, crc=None, isize=None) -> bytes:
    total = len(deflated) + 26
    head = struct.pack("<BBBBIBBHBBHH", 0x1f, 0x8b, 8, 4, 0, 0, 0xff, 6, 66, 67, 2, total - 1)
    crc = zlib.crc32(payload) & 0xffffffff if crc is None else crc
    return head + deflated + struct.pack("<II", crc, len(payload) if isize is None else isize)


def deflate(data: bytes, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, flush_at=None) -> bytes:
    co = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    if flush_at is None:
        return co.compress(data) + co.flush()
    out = b""
    for k in range(0, len(data), flush_at):
        out += co.compress(data[k:k + flush_at]) + co.flush(zlib.Z_FULL_FLUSH)
    return out + co.flush()


def debug_inflate(lib, block: bytes, cap=0x10000):
    out = np.zeros(max(cap, 1), np.uint8)
    n = C.c_int64(0)
    src = np.frombuffer(block, np.uint8).copy()
    rc = lib.c3r_debug_inflate(src.ctypes.data, src.size, out.ctypes.data, cap, C.byref(n))
    return rc, out[:n.value].tobytes() if rc == 0 else None


def payloads():
    rng = np.random.default_rng(3)
    rand = rng.integers(0, 256, 30000, dtype=np.uint8).tobytes()
    qual = bytes(rng.choice([30, 31, 32, 35], 40000).astype(np.uint8))           # quality-string like runs
    rep = b"A" * 20000 + b"ACGT" * 5000 + b"x" * 300
    far = rng.integers(0, 256, 200, dtype=np.uint8).tobytes()
    dist32k = far + bytes(32768 - len(far)) + far                              # a match 32 768 bytes back
    big = (b"ACGTTGCA" * 4096 + qual)[:65536]
    return {"empty": b"", "one": b"Z", "random": rand, "qual": qual, "repetitive": rep, "dist32k": dist32k,
            "full64k": big, "runs258": b"\x07" * 5000 + b"ab" * 2000}


@pytest.mark.parametrize("name", list(payloads()))
@pytest.mark.parametrize("mode", ["stored", "fixed", "l1", "l6", "l9", "huffman_only", "rle", "full_flush"])
def test_inflate_matches_zlib(lib, name, mode):
    data = payloads()[name]
    if mode == "stored":
        if len(data) > 60000:
            pytest.skip("a stored 64 KiB payload does not fit a BGZF block")
        d = deflate(data, 0)
    elif mode == "fixed":
        d = deflate(data, 6, zlib.Z_FIXED)
    elif mode == "huffman_only":
        d = deflate(data, 6, zlib.Z_HUFFMAN_ONLY)
    elif mode == "rle":
        d = deflate(data, 6, zlib.Z_RLE)
    elif mode == "full_flush":
        d = deflate(data, 6, flush_at=max(1, len(data) // 3 + 1))
    else:
        d = deflate(data, int(mode[1:]))
    if len(d) + 26 > 0x10000:
        pytest.skip("does not compress into one BGZF block")
    rc, out = debug_inflate(lib, bgzf_block(data, d))
    assert rc == 0 and out == data


def test_inflate_rejects_corrupt_blocks(lib):
    data = payloads()["qual"]
    d = deflate(data, 6)
    good = bgzf_block(data, d)
    assert debug_inflate(lib, good)[0] == 0
    crc = zlib.crc32(data) & 0xffffffff
    assert debug_inflate(lib, bgzf_block(data, d, crc=crc ^ 1))[0] != 0                  # flipped CRC
    assert debug_inflate(lib, bgzf_block(data, d, isize=len(data) - 1))[0] != 0           # wrong ISIZE (short)
    assert debug_inflate(lib, bgzf_block(data, d, isize=len(data) + 1))[0] != 0           # wrong ISIZE (long)
    assert debug_inflate(lib, bgzf_block(data, d[:len(d) // 2]))[0] != 0                  # truncated stream
    # invalid code lengths: a dynamic block whose code-length code is over-subscribed (all 19 lengths 1)
    bits = [0, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1]             # BFINAL 0, BTYPE 2, HLIT 0, HDIST 0, HCLEN 15
    bits += [1, 0, 0] * 19
    v = sum(b << i for i, b in enumerate(bits))
    bad = v.to_bytes((len(bits) + 7) // 8 + 4, "little")
    assert debug_inflate(lib, bgzf_block(b"abc", bad))[0] != 0
    # a distance reaching before the output's start: fixed block, literal 'a', then length 3 distance 2
    w = []
    def put(v, n, rev=False):
        for i in range(n):
            w.append((v >> (n - 1 - i)) & 1 if rev else (v >> i) & 1)
    put(1, 1); put(1, 2)                                          # BFINAL, BTYPE 01
    put(0x30 + ord("a"), 8, rev=True)                             # literal 'a' (codes 0x30..0xbf, 8 bits)
    put(1, 7, rev=True)                                           # length symbol 257 = 3 (7-bit code 0000001)
    put(1, 5, rev=True)                                           # distance symbol 1 = distance 2
    put(0, 7, rev=True)                                           # end of block
    v = sum(b << i for i, b in enumerate(w))
    far = v.to_bytes((len(w) + 7) // 8, "little")
    assert debug_inflate(lib, bgzf_block(b"aaaa", far))[0] != 0
    # the same stream with distance 1 is valid: 'a' then three copies
    w.clear()
    put(1, 1); put(1, 2); put(0x30 + ord("a"), 8, rev=True); put(1, 7, rev=True); put(0, 5, rev=True); put(0, 7, rev=True)
    v = sum(b << i for i, b in enumerate(w))
    ok = v.to_bytes((len(w) + 7) // 8, "little")
    assert debug_inflate(lib, bgzf_block(b"aaaa", ok)) == (0, b"aaaa")
    # reserved block type 3, and random garbage: errors, no crash
    assert debug_inflate(lib, bgzf_block(b"x", bytes([0x07, 0, 0, 0])))[0] != 0
    rng = np.random.default_rng(1)
    for _ in range(200):
        g = rng.integers(0, 256, int(rng.integers(1, 400)), dtype=np.uint8).tobytes()
        rc, _ = debug_inflate(lib, bgzf_block(b"q" * 100, g))
        assert rc != 0


# ------------------------------------------------------------------ raw fetch
def raw_fetch(bf, contig, s, e, buf=None):
    return bf.fetch_raw(contig, s, e, buf=buf)


def walk_raw(rc, tid):
    """inflate the windows of a raw fetch with zlib and walk them as c3r_bam_fetch does -> dict of flat arrays"""
    raw = rc.raw
    data = bytes(rc.data[:raw.n_bytes]) if raw.n_bytes else b""
    beg, end = raw.beg, raw.end
    out = dict(pos=[], flag=[], mapq=[], hp=[], cigar=[], cigar_off=[0], seq=bytearray(), seq_off=[0])
    for w in range(raw.n_windows):
        W = rc.windows[w]
        assert W.status == 0
        u = bytearray()
        for k in range(W.first_block, W.first_block + W.n_blocks):
            B = rc.blocks[k]
            blk = data[B.coff:B.coff + B.csize]
            xlen, = struct.unpack_from("<H", blk, 10)
            payload = zlib.decompress(blk[12 + xlen:B.csize - 8], -15) if B.usize else b""
            assert len(payload) == B.usize and B.uoff == W.ubase + len(u)
            u += payload
        assert len(u) == W.usize
        o = W.ubeg
        stop = False
        while o + 4 <= W.uend:
            bs, = struct.unpack_from("<I", u, o)
            assert o + 4 + bs <= len(u)
            t, pos, l_name, mapq, _b, n_cig, flag, l_seq = struct.unpack_from("<iiBBHHHi", u, o + 4)
            p = o + 4 + 32 + l_name
            cig = list(struct.unpack_from("<%dI" % n_cig, u, p))
            seq = bytes(u[p + 4 * n_cig:p + 4 * n_cig + (l_seq + 1) // 2])
            a = p + 4 * n_cig + (l_seq + 1) // 2 + l_seq
            aux = bytes(u[a:o + 4 + bs])
            o += 4 + bs
            if t != tid:
                if t > tid or t < 0:
                    stop = True
                    break
                continue
            if pos >= end:
                stop = True
                break
            hp, cg, q = -1, None, 0
            while q < len(aux):
                tag, ty = aux[q:q + 2], chr(aux[q + 2])
                q += 3
                if ty in "AcC":
                    v = struct.unpack_from({"A": "<B", "c": "<b", "C": "<B"}[ty], aux, q)[0]; q += 1
                elif ty in "sS":
                    v = struct.unpack_from("<" + ty.replace("s", "h").replace("S", "H"), aux, q)[0]; q += 2
                elif ty in "iIf":
                    v = struct.unpack_from("<" + ty, aux, q)[0]; q += 4
                elif ty in "ZH":
                    z = aux.index(b"\0", q); q = z + 1; v = None
                else:
                    sub, cnt = chr(aux[q]), struct.unpack_from("<I", aux, q + 1)[0]
                    sz = {"c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}[sub]
                    if tag == b"CG" and sub == "I":
                        cg = list(struct.unpack_from("<%dI" % cnt, aux, q + 5))
                    q += 5 + cnt * sz; v = None
                if tag == b"HP" and ty in "cCsSiI":
                    hp = v
            if cg is not None and len(cig) == 2 and (cig[0] & 15) == 4 and (cig[0] >> 4) == l_seq and (cig[1] & 15) == 3:
                cig = cg
            rl = sum(c >> 4 for c in cig if (c & 15) in (0, 2, 3, 7, 8))
            if pos + max(rl, 1) <= beg:
                continue
            nb = l_seq if l_seq > 0 else sum(c >> 4 for c in cig if (c & 15) in (0, 1, 4, 7, 8))
            out["pos"].append(pos); out["flag"].append(flag); out["mapq"].append(mapq)
            out["hp"].append(0 if hp <= 0 else min(hp, 255))
            out["cigar"] += cig
            out["cigar_off"].append(len(out["cigar"]))
            if l_seq > 0:
                sb = bytearray(seq)
                if l_seq & 1:
                    sb[-1] &= 0xf0
            else:
                sb = bytearray(b"\xff" * ((nb + 1) // 2))
                if nb & 1:
                    sb[-1] = 0xf0
            out["seq"] += sb
            out["seq_off"].append(out["seq_off"][-1] + ((nb + 1) & ~1))
        if stop:
            break
    return out


def same_as_fetch(bf, contig, s, e):
    b = bf.fetch(contig, s, e)
    w = walk_raw(raw_fetch(bf, contig, s, e), bf.references.index(contig))
    assert w["pos"] == b.pos.tolist()
    assert w["flag"] == b.flag.tolist() and w["mapq"] == b.mapq.tolist() and w["hp"] == b.hp.tolist()
    assert w["cigar"] == b.cigar.tolist() and w["cigar_off"] == b.cigar_off.tolist()
    assert bytes(w["seq"]) == b.seq.tobytes() and w["seq_off"] == b.seq_off.tolist()
    return b


def region_set(n, rng, k=12):
    regs = [(1, n), (1, 1), (n, n), (max(1, n - 50), n), (n + 1, n + 1000)]
    for _ in range(k):
        s = int(rng.integers(1, n))
        regs.append((s, min(n, s + int(rng.integers(1, 40000)))))
    return regs


@pytest.mark.parametrize("name", ["cfg1_ont_drna", "phased_noisy"])
def test_raw_fetch_library_writer(lib, tmp_path, name):
    from clair3_rna_b200 import bam
    batch, ref_bytes, contig = golden_cases.build(name)
    n = len(ref_bytes)
    path = str(tmp_path / "r.bam")
    bam.write_bam(path, [("chr0", 5000), (contig, n), ("chrZ", 100)], {contig: batch}, level=1)
    with bam.BamFile(path) as bf:
        for s, e in region_set(n, np.random.default_rng(4)):
            same_as_fetch(bf, contig, s, e)
        assert raw_fetch(bf, "chr0", 1, 5000).raw.n_windows == 0       # a contig without index entries
        same_as_fetch(bf, "chrZ", 1, 100)


def test_raw_fetch_small_blocks_and_aligned_blocks(lib, tmp_path):
    """700-byte blocks (records cross blocks) and one block per record (block-aligned, as htslib writes)"""
    from clair3_rna_b200 import bam
    batch, ref_bytes, contig = golden_cases.build("cfg2_ont_cdna")
    n = len(ref_bytes)
    recs = batch_records(batch)
    for payload, tag in ((700, "small"), (None, "aligned")):
        path = str(tmp_path / ("%s.bam" % tag))
        if payload is None:
            write_aligned_bam(path, [(contig, n)], recs)
        else:
            py_write_bam(path, [(contig, n)], recs, payload=payload)
        with bam.BamFile(path) as bf:
            for s, e in region_set(n, np.random.default_rng(11), k=8):
                same_as_fetch(bf, contig, s, e)


def write_aligned_bam(path, refs, recs):
    """every record in its own BGZF block (the header in the first): the block-aligned layout of htslib"""
    import tests.test_bam_cpu as T
    # reuse the independent writer with a payload that cuts exactly at record ends
    text = b"@HD\tVN:1.6\tSO:coordinate\n"
    head = b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(refs))
    for nm, ln in refs:
        head += struct.pack("<i", len(nm) + 1) + nm.encode() + b"\0" + struct.pack("<i", ln)
    pieces = [head]
    for i, (tid, pos, flag, mapq, cig, seq, l_seq, aux) in enumerate(recs):
        rl = sum(c >> 4 for c in cig if (c & 15) in (0, 2, 3, 7, 8))
        name = b"q%d\0" % i
        body = struct.pack("<iiBBHHHiiii", tid, pos, len(name), mapq, T.py_reg2bin(pos, pos + max(rl, 1)), len(cig), flag,
                           l_seq, -1, -1, 0) + name + struct.pack("<%dI" % len(cig), *cig) + seq + b"\xff" * l_seq + aux
        pieces.append(struct.pack("<i", len(body)) + body)
    out, voffs = bytearray(), []
    for p in pieces:
        voffs.append(len(out) << 16)
        out += bgzf_block(p, deflate(p, 6))
    eof = len(out)
    out += bgzf_block(b"", deflate(b"", 6))
    open(path, "wb").write(out)
    ix = bytearray(b"BAI\1" + struct.pack("<i", len(refs)))
    for tid in range(len(refs)):
        bins, linear = {}, {}
        for k, (t, pos, flag, mapq, cig, seq, l_seq, aux) in enumerate(recs):
            if t != tid:
                continue
            rl = sum(c >> 4 for c in cig if (c & 15) in (0, 2, 3, 7, 8))
            e = pos + max(rl, 1)
            v0 = voffs[k + 1]
            v1 = voffs[k + 2] if k + 2 < len(voffs) else eof << 16
            bins.setdefault(T.py_reg2bin(pos, e), []).append((v0, v1))
            for w in range(pos >> 14, ((e - 1) >> 14) + 1):
                linear.setdefault(w, v0)
        ix += struct.pack("<i", len(bins))
        for b in sorted(bins):
            ix += struct.pack("<Ii", b, len(bins[b]))
            for cb, ce in bins[b]:
                ix += struct.pack("<QQ", cb, ce)
        n_intv = max(linear) + 1 if linear else 0
        ix += struct.pack("<i", n_intv)
        last = 0
        for w in range(n_intv):
            last = linear.get(w, last)
            ix += struct.pack("<Q", last)
    open(path + ".bai", "wb").write(ix)


def special_records():
    M, I, D, N, S = 0, 1, 2, 3, 4
    def c(l, op): return (l << 4) | op
    seq7 = bytes([0x12, 0x48, 0x84, 0x10])
    long_ops = []
    for k in range(40000):
        long_ops += [c(1, M), c(1, D)] if k % 2 == 0 else [c(1, M), c(1, I)]
    ql = sum(x >> 4 for x in long_ops if (x & 15) in (0, 1, 4))
    rl = sum(x >> 4 for x in long_ops if (x & 15) in (0, 2, 3))
    cg_aux = b"CGBI" + struct.pack("<i", len(long_ops)) + struct.pack("<%dI" % len(long_ops), *long_ops)
    return [
        (0, 100, 0, 60, [c(7, M)], seq7, 7, b"NMC\x01" + b"HPc\x01" + b"XZZabc\0"),
        (0, 110, 0, 60, [c(7, M)], seq7, 7, b"HPc\xff"),                                  # negative HP: 0
        (0, 120, 16, 60, [c(3, M), c(50, N), c(4, M)], seq7, 7, b"XBBs\x02\x00\x00\x00\x01\x00\x02\x00" + b"HPS\x02\x01"),
        (0, 125, 0, 60, [c(7, M)], seq7, 7, b"HPs\x05\x00"),
        (0, 130, 0, 30, [c(7, M)], seq7, 7, b"HPi\x03\x01\x00\x00" + b"XFf\x00\x00\x80\x3f"),   # clamped to 255
        (0, 135, 0, 30, [c(7, M)], seq7, 7, b"HPI\x09\x00\x00\x00"),
        (0, 138, 0, 30, [c(7, M)], seq7, 7, b"HPC\x07" + b"HPA\x41"),                        # 'A' is not an integer
        (0, 140, 0, 30, [c(7, M)], b"", 0, b"XAAq"),                                       # SEQ '*'
        (0, 145, 0, 30, [c(3, S), c(4, M)], b"", 0, b""),                                  # SEQ '*', odd length
        (0, 150, 0, 60, [c(ql, S), c(rl, N)], bytes([0x12] * ((ql + 1) // 2)), ql, cg_aux + b"HPC\x02"),
        (0, 160, 4, 0, [], seq7, 7, b""),
    ]


def test_raw_fetch_special_records(lib, tmp_path):
    from clair3_rna_b200 import bam
    path = str(tmp_path / "s.bam")
    py_write_bam(path, [("c", 200000)], special_records(), payload=5000)
    with bam.BamFile(path) as bf:
        b = same_as_fetch(bf, "c", 1, 200000)
        assert b.hp.tolist() == [1, 0, 255, 5, 255, 9, 7, 0, 0, 2, 0]
        same_as_fetch(bf, "c", 171, 171)
        same_as_fetch(bf, "c", 100000, 100010)


def test_raw_fetch_capacity(lib, tmp_path):
    from clair3_rna_b200 import bam
    from clair3_rna_b200 import lib as L
    batch, ref_bytes, contig = golden_cases.build("cfg2_ont_cdna")
    path = str(tmp_path / "c.bam")
    bam.write_bam(path, [(contig, len(ref_bytes))], {contig: batch})
    with bam.BamFile(path) as bf:
        full = bf.fetch_raw(contig, 1, len(ref_bytes))
        need = full.n_bytes
        assert need > 0
        small = np.zeros(need - 1, np.uint8)
        r = L.BamRaw()
        rc = bf.lib.c3r_bam_fetch_raw(bf.h, 0, 1, len(ref_bytes), small.ctypes.data, small.size, C.byref(r))
        assert rc == -4 and r.n_bytes == need                     # C3R_ERR_CAPACITY and the size needed
        got = bf.fetch_raw(contig, 1, len(ref_bytes), buf=small)  # the binding falls back to a buffer of its own
        assert got.data is not small and got.n_bytes == need
        exact = np.zeros(need, np.uint8)
        assert bf.fetch_raw(contig, 1, len(ref_bytes), buf=exact).data is exact
