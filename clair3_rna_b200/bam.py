"""BAM input through libc3r_b200.so (csrc/bam_io.cpp): index fetch of a region into a ReadBatch.

Replaces the reference's only two uses of the BAM, both through external samtools:
`samtools mpileup BAM -r ctg:s-e` (/root/reference/src/create_tensor_pileup.py:436-451) and
`samtools idxstats BAM` (/root/reference/run_clair3_rna:187)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import lib as L
from .reads import ReadBatch


def reads_struct(batch: ReadBatch, keep: list) -> L.Reads:
    """c3r_reads view of a ReadBatch; `keep` receives the arrays that must outlive the call"""
    arrs = dict(pos=np.ascontiguousarray(batch.pos, np.int32), flag=np.ascontiguousarray(batch.flag, np.uint16),
                mapq=np.ascontiguousarray(batch.mapq, np.uint8), hp=np.ascontiguousarray(batch.hp, np.uint8),
                cigar_off=np.ascontiguousarray(batch.cigar_off, np.int32), cigar=np.ascontiguousarray(batch.cigar, np.uint32),
                seq_off=np.ascontiguousarray(batch.seq_off, np.int64), seq=np.ascontiguousarray(batch.seq, np.uint8))
    keep.append(arrs)
    r = L.Reads()
    r.n_reads, r.n_ops, r.n_seq_bytes = batch.n_reads, batch.n_ops, int(arrs["seq"].size)
    for k, a in arrs.items():
        setattr(r, k, a.ctypes.data)
    return r


class BamFile:
    """An indexed BAM opened for region fetches."""

    def __init__(self, path: str, index_path: str | None = None, threads: int = 0):
        self.lib = L.load()
        self.h = C.c_void_p()
        rc = self.lib.c3r_bam_open(path.encode(), index_path.encode() if index_path else None, threads, C.byref(self.h))
        if rc != 0:
            msg = self.lib.c3r_bam_error(self.h).decode() if self.h else "open failed"
            self.close()
            raise RuntimeError("c3r_bam_open(%s): %s" % (path, msg))
        n = self.lib.c3r_bam_n_ref(self.h)
        self.references = [self.lib.c3r_bam_ref_name(self.h, i).decode() for i in range(n)]
        self.lengths = [int(self.lib.c3r_bam_ref_len(self.h, i)) for i in range(n)]
        self._tid = {name: i for i, name in enumerate(self.references)}

    def close(self):
        if getattr(self, "h", None):
            self.lib.c3r_bam_close(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def header_text(self) -> str:
        return self.lib.c3r_bam_header_text(self.h).decode()

    def idxstats(self):
        """[(name, length, mapped, unmapped)] like `samtools idxstats` (run_clair3_rna:187)"""
        out = []
        for i, (n, l) in enumerate(zip(self.references, self.lengths)):
            m, u = C.c_int64(0), C.c_int64(0)
            rc = self.lib.c3r_bam_idxstats(self.h, i, C.byref(m), C.byref(u))
            if rc != 0:
                # an index without the metadata pseudo-bin carries no counts (samtools idxstats then counts records):
                # treat the contig as having reads when a fetch over it finds any, instead of silently skipping it
                probe = self.fetch(n, 1, int(l)) if l > 0 else None
                m = C.c_int64(probe.n_reads if probe is not None else 0)
            out.append((n, l, int(m.value), int(u.value)))
        return out

    def fetch(self, contig: str, start1: int, end1: int) -> ReadBatch:
        """records overlapping the 1-based inclusive region, file order (what `mpileup -r` reads)"""
        if contig not in self._tid:
            raise KeyError("contig %s not in the BAM header" % contig)
        r = L.Reads()
        rc = self.lib.c3r_bam_fetch(self.h, self._tid[contig], int(start1), int(end1), C.byref(r))
        if rc != 0:
            raise RuntimeError("c3r_bam_fetch: " + self.lib.c3r_bam_error(self.h).decode())
        return reads_from(contig, r)

    def fetch_raw(self, contig: str, start1: int, end1: int, buf=None) -> RawChunk:
        """fetch() without the inflate and the record walk: the index query and the compressed blocks of the region
        read into `buf` (a uint8 array, e.g. from engine.PinnedPool); a new array when buf is None or too small"""
        if contig not in self._tid:
            raise KeyError("contig %s not in the BAM header" % contig)
        r = L.BamRaw()
        tid = self._tid[contig]
        cap = 0 if buf is None else int(buf.size)
        rc = self.lib.c3r_bam_fetch_raw(self.h, tid, int(start1), int(end1), buf.ctypes.data if cap else None, cap, C.byref(r))
        if rc == -4:                                 # C3R_ERR_CAPACITY: r.n_bytes is the size needed
            buf = np.empty(max(1, int(r.n_bytes)), np.uint8)
            rc = self.lib.c3r_bam_fetch_raw(self.h, tid, int(start1), int(end1), buf.ctypes.data, buf.size, C.byref(r))
        if rc != 0:
            raise RuntimeError("c3r_bam_fetch_raw: " + self.lib.c3r_bam_error(self.h).decode())
        blocks = _table(r.blocks, int(r.n_blocks), L.BgzfBlock)
        windows = _table(r.windows, int(r.n_windows), L.BamWindow)
        r.blocks = C.addressof(blocks) if r.n_blocks else None
        r.windows = C.addressof(windows) if r.n_windows else None
        return RawChunk(contig, r, buf, blocks, windows)


def reads_from(contig: str, r: L.Reads, copy: bool = True) -> ReadBatch:
    """ReadBatch over a c3r_reads; copy=False aliases the memory behind it"""
    def arr(ptr, n, dt):
        if n == 0 or not ptr:
            return np.zeros(0, dt)
        a = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(np.ctypeslib.as_ctypes_type(dt))), shape=(n,))
        return a.copy() if copy else a

    R, O, S = int(r.n_reads), int(r.n_ops), int(r.n_seq_bytes)
    return ReadBatch(contig, arr(r.pos, R, np.int32), arr(r.flag, R, np.uint16), arr(r.mapq, R, np.uint8),
                     arr(r.hp, R, np.uint8), arr(r.cigar_off, R + 1, np.int32), arr(r.cigar, O, np.uint32),
                     arr(r.seq_off, R + 1, np.int64), arr(r.seq, S, np.uint8))


class RawChunk:
    """The compressed blocks of a region fetch and their tables (c3r_bam_fetch_raw), ready for Engine.submit_bam:
    `data` holds the bytes (a caller's buffer, possibly page-locked), `blocks` / `windows` are private copies of the
    handle's tables, `raw` the c3r_bam_raw over all three.  Keep it unchanged until the ticket is waited for."""

    def __init__(self, contig, raw, data, blocks, windows):
        self.contig, self.raw, self.data, self.blocks, self.windows = contig, raw, data, blocks, windows

    @property
    def n_bytes(self) -> int:
        return int(self.raw.n_bytes)


def _table(ptr, n, ctype):
    return (ctype * n).from_buffer_copy((ctype * n).from_address(ptr)) if n > 0 and ptr else (ctype * max(n, 0))()


def write_bam(path: str, contigs: list, batches: dict, level: int = -1, header_text: str | None = None) -> None:
    """contigs: [(name, length)]; batches: {name: ReadBatch}.  Writes path and path + '.bai'."""
    lib = L.load()
    n = len(contigs)
    names = (C.c_char_p * n)(*[c[0].encode() for c in contigs])
    lens = (C.c_int64 * n)(*[int(c[1]) for c in contigs])
    keep, structs = [], []
    ptrs = (C.POINTER(L.Reads) * n)()
    for i, (name, _) in enumerate(contigs):
        if name in batches and batches[name].n_reads:
            s = reads_struct(batches[name], keep)
            structs.append(s)
            ptrs[i] = C.pointer(s)
    rc = lib.c3r_bam_write(path.encode(), n, names, lens, ptrs, level, header_text.encode() if header_text else None)
    if rc != 0:
        raise RuntimeError("c3r_bam_write(%s) failed with %d" % (path, rc))
