"""Host side of the C ABI: one `Engine` per GPU.

`Engine.call_chunk()` is the in-process replacement of one reference
`call_var_bam` producer|consumer pipeline up to the 24 probabilities
(/root/reference/clair3_rna/call_var_bam.py:278-295): it packs nothing itself,
it hands the flat records of `reads.ReadBatch` to libc3r_b200.so and copies the
library-owned result buffers into numpy arrays.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
import numpy as np

from . import lib as L
from . import params as P
from .reads import ReadBatch, NT16


class C3RError(RuntimeError):
    pass


@dataclass
class ChunkResult:
    n_rows: int
    pos: np.ndarray            # int32 [n] 1-based
    depth: np.ndarray          # int32 [n]
    probs: np.ndarray          # float32 [n,24]
    alt_off: np.ndarray        # int64 [n]
    alt_n: np.ndarray          # int32 [n]
    alt: np.ndarray            # structured [total]
    tensor: np.ndarray | None  # int32 [n,33,C]
    row_pos: np.ndarray | None
    row_counts: np.ndarray | None
    row_depth: np.ndarray | None
    stage_ms: list = field(default_factory=list)
    launches: int = 0
    calls: np.ndarray | None = None   # lib.CALL_DTYPE [n]: call records (Engine(device_calls=True)), else None
    call_ms: float = 0.0              # device time of k_call

    @property
    def n_cand(self) -> int:
        return int(self.pos.size)


ALT_DTYPE = np.dtype([("kind", "u1"), ("base", "u1"), ("len", "<u2"), ("count", "<i4"),
                      ("seq_off", "<u4"), ("order", "<u4")])


def _view(ptr, n, dtype, copy=True):
    """numpy array over library-owned host memory; copy=False aliases it (valid until the ticket is released)"""
    if not ptr or n <= 0:
        return np.zeros(0, dtype)
    nbytes = int(n) * np.dtype(dtype).itemsize
    buf = (C.c_char * nbytes).from_address(ptr)
    a = np.frombuffer(buf, dtype=dtype, count=int(n))
    return a.copy() if copy else a


class Engine:
    def __init__(self, device: int = 0, channels: int = 18, *, snp_min_af=P.SNP_MIN_AF, indel_min_af=P.INDEL_MIN_AF,
                 min_coverage=P.MIN_COVERAGE, min_mq=P.MIN_MQ, enable_padding=False, nn_impl=1,
                 keep_tensor=False, keep_rows=False, enable_head_tail=False, device_calls=False):
        """device_calls: also decide each candidate's genotype on the GPU (ChunkResult.calls, format_vcf_rows)"""
        self.lib = L.load()
        if self.lib.c3r_abi_version() != 2:
            raise C3RError("ABI version mismatch")
        prm = L.Params()
        self.lib.c3r_default_params(C.byref(prm))
        prm.channels = channels
        prm.snp_min_af = snp_min_af
        prm.indel_min_af = indel_min_af
        prm.min_coverage = min_coverage
        prm.min_mq = min_mq
        prm.enable_padding = int(enable_padding)
        prm.nn_impl = nn_impl
        prm.keep_tensor = int(keep_tensor)
        prm.keep_rows = int(keep_rows)
        prm.enable_head_tail = int(enable_head_tail)
        self.params = prm
        self.channels = channels
        self.ctx = C.c_void_p()
        rc = self.lib.c3r_create(C.byref(self.ctx), device, C.byref(prm))
        if rc != 0:
            msg = self.lib.c3r_last_error(self.ctx).decode() if self.ctx else "c3r_create failed"
            if self.ctx:
                self.lib.c3r_destroy(self.ctx)
                self.ctx = C.c_void_p()
            raise C3RError("c3r_create: %s (rc=%d)" % (msg, rc))
        self._keep = {}
        self._calls_of = {}                          # ticket -> records on when it was submitted
        self.device_calls = False
        self.set_device_calls(device_calls)

    # ------------------------------------------------------------------
    def _check(self, rc, what):
        if rc < 0:
            raise C3RError("%s: %s (rc=%d)" % (what, self.lib.c3r_last_error(self.ctx).decode(), rc))
        return rc

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.c3r_destroy(self.ctx)
            self.ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_device_calls(self, on: bool):
        """call records for the tickets submitted from now on (c3r_enable_calls)"""
        self._check(self.lib.c3r_enable_calls(self.ctx, int(bool(on))), "c3r_enable_calls")
        self.device_calls = bool(on)

    def set_weights(self, weights: dict):
        arrs = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in weights.items()}
        views = (L.WeightView * len(arrs))()
        for i, (k, v) in enumerate(arrs.items()):
            views[i].name = k.encode()
            views[i].data = v.ctypes.data
            views[i].n_elem = v.size
        self._check(self.lib.c3r_set_weights(self.ctx, views, len(arrs)), "c3r_set_weights")

    def set_reference(self, ref: np.ndarray, ref_start1: int = 1):
        """keep a reference window resident on the GPU; later submits may pass ref=None"""
        ref = np.ascontiguousarray(ref, np.uint8)
        self._check(self.lib.c3r_set_reference(self.ctx, ref.ctypes.data, ref_start1, int(ref.size)), "c3r_set_reference")

    # ------------------------------------------------------------------
    def submit(self, batch: ReadBatch, ref, ref_start1: int, region_start1: int, region_end1: int,
               site_filter=None) -> int:
        """site_filter: None or dict(pileup_bed=, confident=, known=) as made by regions.ChunkPlan.site_filter():
        merged int32 interval arrays [n,2] / sorted 1-based sites; a missing or None entry = option not given."""
        rd = L.Reads()
        rd.n_reads, rd.n_ops, rd.n_seq_bytes = batch.n_reads, batch.n_ops, int(batch.seq.size)
        arrs = dict(pos=np.ascontiguousarray(batch.pos, np.int32), flag=np.ascontiguousarray(batch.flag, np.uint16),
                    mapq=np.ascontiguousarray(batch.mapq, np.uint8), hp=np.ascontiguousarray(batch.hp, np.uint8),
                    cigar_off=np.ascontiguousarray(batch.cigar_off, np.int32),
                    cigar=np.ascontiguousarray(batch.cigar, np.uint32),
                    seq_off=np.ascontiguousarray(batch.seq_off, np.int64), seq=np.ascontiguousarray(batch.seq, np.uint8))
        for k, v in arrs.items():
            setattr(rd, k, v.ctypes.data)
        t = C.c_int64(-1)
        if ref is None:
            rp, rn = None, 0
        else:
            ref = np.ascontiguousarray(ref, np.uint8)
            rp, rn = ref.ctypes.data, int(ref.size)
        if site_filter is None:
            self._check(self.lib.c3r_submit_chunk(self.ctx, C.byref(rd), rp, ref_start1, rn,
                                                  region_start1, region_end1, C.byref(t)), "c3r_submit_chunk")
            self._keep[int(t.value)] = (arrs, ref)       # the call only queues the copies: inputs live until wait()
            self._calls_of[int(t.value)] = self.device_calls
            return int(t.value)
        f = L.SiteFilter()
        keep = []
        for key, field, width in (("pileup_bed", "pileup_bed", 2), ("confident", "confident_bed", 2), ("known", "known_sites", 1)):
            a = site_filter.get(key)
            if a is None:
                setattr(f, "n_" + field, -1)
                continue
            a = np.ascontiguousarray(a, np.int32).reshape(-1, width)
            keep.append(a)
            setattr(f, field, a.ctypes.data if a.size else None)
            setattr(f, "n_" + field, a.shape[0])
        self._check(self.lib.c3r_submit_chunk_filtered(self.ctx, C.byref(rd), rp, ref_start1, rn, region_start1,
                                                       region_end1, C.byref(f), C.byref(t)), "c3r_submit_chunk_filtered")
        self._keep[int(t.value)] = (arrs, ref, keep)
        self._calls_of[int(t.value)] = self.device_calls
        return int(t.value)

    def wait(self, ticket: int, release: bool = True, copy: bool = True) -> ChunkResult:
        """Result of a ticket.  copy=True (default) returns private numpy copies and, with release=True, frees the
        ticket.  copy=False returns arrays that alias the library's pinned result buffers - no allocation, no page
        faults (copying 3-4 MB into fresh memory costs ~1.5 ms per chunk, more than half a device pass) - which
        stay valid until release(ticket); the ticket is then NOT released here."""
        r = L.Result()
        calls_on = self._calls_of.pop(ticket, False)
        try:
            self._check(self.lib.c3r_wait(self.ctx, ticket, C.byref(r)), "c3r_wait")
        finally:
            self._keep.pop(ticket, None)
        calls, call_ms = None, 0.0
        if calls_on:
            cp, cn, ms = C.c_void_p(), C.c_int64(0), C.c_float(0)
            self._check(self.lib.c3r_wait_calls(self.ctx, ticket, C.byref(cp), C.byref(cn), C.byref(ms)), "c3r_wait_calls")
            calls, call_ms = _view(cp.value, cn.value, L.CALL_DTYPE, copy), float(ms.value)
        n, Ct = int(r.n_cand), self.channels
        v = lambda ptr, cnt, dt: _view(ptr, cnt, dt, copy)
        alt_off = v(r.alt_off, n, np.int64)
        alt_n = v(r.alt_n, n, np.int32)
        total = int((alt_off + alt_n).max()) if n else 0
        out = ChunkResult(
            n_rows=int(r.n_rows), pos=v(r.pos, n, np.int32), depth=v(r.depth, n, np.int32),
            probs=v(r.probs, n * 24, np.float32).reshape(n, 24), alt_off=alt_off, alt_n=alt_n,
            alt=v(r.alt, total, ALT_DTYPE),
            tensor=v(r.tensor, n * 33 * Ct, np.int32).reshape(n, 33, Ct) if r.tensor else None,
            row_pos=v(r.row_pos, r.n_rows, np.int32) if r.row_pos else None,
            row_counts=v(r.row_counts, r.n_rows * Ct, np.int32).reshape(-1, Ct) if r.row_counts else None,
            row_depth=v(r.row_depth, r.n_rows, np.int32) if r.row_depth else None,
            stage_ms=[float(x) for x in r.stage_ms], launches=int(r.kernel_launches), calls=calls, call_ms=call_ms)
        if release and copy:
            self.lib.c3r_release(self.ctx, ticket)
        return out

    def release(self, ticket: int):
        self._keep.pop(ticket, None)
        self._calls_of.pop(ticket, None)
        self.lib.c3r_release(self.ctx, ticket)

    def call_chunk(self, batch, ref, ref_start1, region_start1, region_end1, site_filter=None) -> ChunkResult:
        return self.wait(self.submit(batch, ref, ref_start1, region_start1, region_end1, site_filter))

    def rerun_resident(self, ticket: int):
        """-> (total_ms, [8 stage ms], kernel launches) of one device-resident pass."""
        tot = C.c_float(0)
        st = (C.c_float * 8)()
        n = self._check(self.lib.c3r_rerun_resident(self.ctx, ticket, C.byref(tot), st), "c3r_rerun_resident")
        return float(tot.value), [float(x) for x in st], n

    def forward(self, tensor: np.ndarray):
        """network alone: int32 [n,33,C] -> (float32 [n,24], device ms)"""
        t = np.ascontiguousarray(tensor, np.int32)
        n = t.shape[0]
        out = np.empty((n, 24), np.float32)
        ms = C.c_float(0)
        self._check(self.lib.c3r_forward(self.ctx, t.ctypes.data, n, out.ctypes.data, C.byref(ms)), "c3r_forward")
        return out, float(ms.value)


    def debug_fetch(self, which: int, n_sites: int):
        """intermediate activations of the last tensor-core forward, unpacked to plain arrays:
        0 -> h1 [n,33,256], 2 -> h2 [n,33,320], 3 -> l4 [n,128]"""
        tiles = (n_sites + 127) // 128
        tiles += tiles & 1
        sizes = {0: tiles * 33 * 4 * 8192 * 2, 2: tiles * 33 * 5 * 8192 * 2, 3: tiles * 128 * 128 * 4}
        buf = np.empty(sizes.get(which, 0), np.uint8)              # other numbers: the library refuses them (C3RError)
        nb = C.c_int64(0)
        self._check(self.lib.c3r_debug_fetch(self.ctx, which, buf.ctypes.data, buf.size, C.byref(nb)), "c3r_debug_fetch")
        if which in (0, 2):
            kb = 4 if which == 0 else 5
            a = buf.view(np.float16).reshape(tiles, 33, kb, 8, 128, 8)        # [tile][t][kb][k8][row][8]
            a = a.transpose(0, 4, 1, 2, 3, 5).reshape(tiles * 128, 33, kb * 64)
            return a[:n_sites].astype(np.float32)
        return buf.view(np.float32).reshape(tiles * 128, 128)[:n_sites]


class PinnedPool:
    """A fixed set of page-locked uint8 host buffers (c3r_host_alloc) handed out and taken back: the reference window
    of a chunk is read from the FASTA straight into one (fasta.fetch_into), given to Engine.submit - which then only
    queues a DMA instead of having the driver stage pageable memory inside the call - and returned once the chunk's
    rows are decoded.  get() returns None when the pool is empty or the request is larger than a buffer (the caller
    falls back to ordinary memory)."""

    def __init__(self, n_buffers: int, n_bytes: int):
        import queue
        self.lib = L.load()
        self.n_bytes = int(n_bytes)
        self.ptrs = []
        self.free = queue.SimpleQueue()
        for _ in range(n_buffers):
            p = C.c_void_p()
            if self.lib.c3r_host_alloc(C.byref(p), self.n_bytes) != 0:
                break
            self.ptrs.append(p)
            self.free.put(np.frombuffer((C.c_char * self.n_bytes).from_address(p.value), dtype=np.uint8))

    def get(self, n_bytes: int):
        if n_bytes > self.n_bytes:
            return None
        try:
            return self.free.get_nowait()
        except Exception:
            return None

    def put(self, buf):
        if buf is not None:
            self.free.put(buf)

    def close(self):
        for p in self.ptrs:
            self.lib.c3r_host_free(p)
        self.ptrs = []


# ---------------------------------------------------------------------- native decode
def _result_struct(res: ChunkResult, keep: list):
    """c3r_result over the arrays of res (kept alive in `keep`)"""
    r = L.Result()
    arrs = dict(pos=np.ascontiguousarray(res.pos, np.int32), depth=np.ascontiguousarray(res.depth, np.int32),
                probs=np.ascontiguousarray(res.probs, np.float32), alt_off=np.ascontiguousarray(res.alt_off, np.int64),
                alt_n=np.ascontiguousarray(res.alt_n, np.int32), alt=np.ascontiguousarray(res.alt))
    keep.append(arrs)
    r.n_rows, r.n_cand = res.n_rows, res.n_cand
    for k, a in arrs.items():
        setattr(r, k, a.ctypes.data if a.size else None)
    return r


def _rows_of(lib, rc, text, nb, nr, what):
    if rc != 0:
        raise C3RError("%s failed (rc=%d)" % (what, rc))
    try:
        s = C.string_at(text, nb.value).decode("ascii") if nb.value else ""
    finally:
        lib.c3r_free_text(text)
    rows = s.split("\n")[:-1] if s else []
    assert len(rows) == nr.value
    return rows


def decode_vcf_rows(res: ChunkResult, batch: ReadBatch, ref: np.ndarray, ref_start1: int, contig: str,
                    qual=P.QUAL_CUT_OFF, show_ref: bool = True, threads: int = 0) -> list:
    """VCF data lines of every candidate through c3r_decode_vcf (csrc/decode.cpp): the native, multi-threaded
    form of decoder.vcf_row over alt_info_strings / flank_strings."""
    from .bam import reads_struct
    lib = L.load()
    keep = []
    r = _result_struct(res, keep)
    rd = reads_struct(batch, keep)
    ref = np.ascontiguousarray(ref, np.uint8)
    text, nb, nr = C.c_void_p(), C.c_int64(0), C.c_int64(0)
    rc = lib.c3r_decode_vcf(C.byref(r), C.byref(rd), ref.ctypes.data, int(ref_start1), int(ref.size), contig.encode(),
                            -1.0 if qual is None else float(qual), int(show_ref), threads,
                            C.byref(text), C.byref(nb), C.byref(nr))
    return _rows_of(lib, rc, text, nb, nr, "c3r_decode_vcf")


def format_vcf_rows(res: ChunkResult, batch: ReadBatch, ref: np.ndarray, ref_start1: int, contig: str,
                    qual=P.QUAL_CUT_OFF, show_ref: bool = True, threads: int = 0, calls=None) -> list:
    """decode_vcf_rows from call records (c3r_format_vcf): the same lines, with the genotype decision taken from
    `calls` (default res.calls, made on the GPU by Engine(device_calls=True)) instead of made on the host."""
    from .bam import reads_struct
    calls = res.calls if calls is None else calls
    if calls is None:
        raise C3RError("format_vcf_rows needs call records: Engine(device_calls=True) or decide_calls()")
    calls = np.ascontiguousarray(calls, L.CALL_DTYPE)
    if calls.shape[0] != res.n_cand:
        raise C3RError("%d call records for %d candidates" % (calls.shape[0], res.n_cand))
    lib = L.load()
    keep = []
    r = _result_struct(res, keep)
    rd = reads_struct(batch, keep)
    ref = np.ascontiguousarray(ref, np.uint8)
    text, nb, nr = C.c_void_p(), C.c_int64(0), C.c_int64(0)
    rc = lib.c3r_format_vcf(C.byref(r), calls.ctypes.data if calls.size else None, C.byref(rd), ref.ctypes.data,
                            int(ref_start1), int(ref.size), contig.encode(), -1.0 if qual is None else float(qual),
                            int(show_ref), threads, C.byref(text), C.byref(nb), C.byref(nr))
    return _rows_of(lib, rc, text, nb, nr, "c3r_format_vcf")


def decide_calls(res: ChunkResult, batch: ReadBatch, ref: np.ndarray, ref_start1: int) -> np.ndarray:
    """the call records k_call makes, by the same code on the host (c3r_debug_decide_calls; no GPU needed)"""
    from .bam import reads_struct
    lib = L.load()
    keep = []
    r = _result_struct(res, keep)
    rd = reads_struct(batch, keep)
    ref = np.ascontiguousarray(ref, np.uint8)
    out = np.zeros(res.n_cand, L.CALL_DTYPE)
    rc = lib.c3r_debug_decide_calls(C.byref(r), C.byref(rd), ref.ctypes.data, int(ref_start1), int(ref.size),
                                    out.ctypes.data if out.size else None)
    if rc != 0:
        raise C3RError("c3r_debug_decide_calls failed (rc=%d)" % rc)
    return out


# ---------------------------------------------------------------------- host formatting
def alt_info_strings(res: ChunkResult, batch: ReadBatch, ref: np.ndarray, ref_start1: int) -> list:
    """alt_info text of each candidate exactly as the reference's producer prints it
    (/root/reference/src/create_tensor_pileup.py:595-596): "<depth>-KEY n KEY n ..."."""
    out = []
    seq = batch.seq
    refb = ref.tobytes() if isinstance(ref, np.ndarray) else bytes(ref)
    for i in range(res.n_cand):
        a, n = int(res.alt_off[i]), int(res.alt_n[i])
        items = []
        p0 = int(res.pos[i]) - ref_start1           # offset of the candidate in ref
        for e in res.alt[a:a + n]:
            kind = chr(int(e["kind"]))
            if kind == 'X' or kind == 'R':
                key = kind + chr(int(e["base"]))
            elif kind == 'I':
                q, ln = int(e["seq_off"]), int(e["len"])
                by = seq[q // 2: (q + ln + 1) // 2 + 1]
                codes = np.empty(by.size * 2, np.uint8)
                codes[0::2] = by >> 4
                codes[1::2] = by & 15
                s = codes[q & 1: (q & 1) + ln]
                key = 'I' + chr(int(e["base"])) + "".join(NT16[c] for c in s)
            else:
                ln = int(e["len"])
                key = 'D' + refb[p0 + 1: p0 + 1 + ln].decode("ascii")
            items.append("%s %d" % (key, int(e["count"])))
        out.append("%d-%s" % (int(res.depth[i]), " ".join(items)))
    return out


def flank_strings(res: ChunkResult, ref: np.ndarray, ref_start1: int) -> list:
    """33-base reference context, padded with 'A' off the loaded reference
    (get_flanked_sequence, create_tensor_pileup.py:313-331)."""
    refs = ref.tobytes().decode("ascii")
    out = []
    for p in res.pos:
        lo = int(p) - P.FLANK - ref_start1
        hi = int(p) + P.FLANK + 1 - ref_start1
        if lo >= 0 and hi <= len(refs):
            out.append(refs[lo:hi])
        else:
            s = 'A' * max(0, -lo) + refs[max(0, lo):hi]
            if hi > len(refs):
                s += 'A' * (hi - len(refs))
            out.append(s)
    return out
