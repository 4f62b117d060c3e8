"""ctypes binding of libc3r_b200.so (include/c3r_b200.h).

Fails loudly when the library is missing: there is no CPU or PyTorch fallback."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("C3R_LIB") or os.path.join(HERE, "libc3r_b200.so")   # C3R_LIB: an experimental build

WINDOW = 33
N_OUT = 24


class Params(C.Structure):
    _fields_ = [("channels", C.c_int32), ("min_coverage", C.c_int32), ("min_mq", C.c_int32),
                ("excl_flags", C.c_uint32), ("snp_min_af", C.c_double), ("indel_min_af", C.c_double),
                ("enable_padding", C.c_int32), ("max_depth", C.c_int32), ("skip_proportion", C.c_double),
                ("nn_impl", C.c_int32), ("keep_tensor", C.c_int32), ("keep_rows", C.c_int32),
                ("enable_head_tail", C.c_int32)]


class Reads(C.Structure):
    _fields_ = [("n_reads", C.c_int64), ("n_ops", C.c_int64), ("n_seq_bytes", C.c_int64),
                ("pos", C.c_void_p), ("flag", C.c_void_p), ("mapq", C.c_void_p), ("hp", C.c_void_p),
                ("cigar_off", C.c_void_p), ("cigar", C.c_void_p), ("seq_off", C.c_void_p), ("seq", C.c_void_p)]


class WeightView(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("n_elem", C.c_int64)]


class AltEntry(C.Structure):
    _fields_ = [("kind", C.c_uint8), ("base", C.c_uint8), ("len", C.c_uint16), ("count", C.c_int32),
                ("seq_off", C.c_uint32), ("order", C.c_uint32)]


class Result(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("n_cand", C.c_int64),
                ("pos", C.c_void_p), ("depth", C.c_void_p), ("probs", C.c_void_p),
                ("alt_off", C.c_void_p), ("alt_n", C.c_void_p), ("alt", C.c_void_p),
                ("tensor", C.c_void_p), ("row_pos", C.c_void_p), ("row_counts", C.c_void_p),
                ("row_depth", C.c_void_p), ("stage_ms", C.c_float * 8), ("kernel_launches", C.c_int32)]


class CallAllele(C.Structure):
    """c3r_call_allele (include/c3r_b200.h)"""
    _fields_ = [("first", C.c_uint8), ("reserved", C.c_uint8), ("ins_len", C.c_uint16), ("ins_seq_off", C.c_uint32),
                ("suffix_from", C.c_uint16), ("reserved2", C.c_uint16)]


class Call(C.Structure):
    """c3r_call (include/c3r_b200.h): the call record of one candidate"""
    _fields_ = [("prob", C.c_float), ("ref_count", C.c_int32), ("support", C.c_int32), ("ad", C.c_int32 * 2),
                ("family", C.c_uint8), ("gt", C.c_uint8), ("n_ad", C.c_uint8), ("n_alt", C.c_uint8),
                ("ref_first", C.c_uint8), ("reserved", C.c_uint8), ("ref_len", C.c_uint16), ("retries", C.c_uint16),
                ("flags", C.c_uint16), ("alt", CallAllele * 2)]


CALL_ALLELE_DTYPE = np.dtype([("first", "u1"), ("reserved", "u1"), ("ins_len", "<u2"), ("ins_seq_off", "<u4"),
                              ("suffix_from", "<u2"), ("reserved2", "<u2")])
# numpy view of an array of c3r_call
CALL_DTYPE = np.dtype([("prob", "<f4"), ("ref_count", "<i4"), ("support", "<i4"), ("ad", "<i4", (2,)),
                       ("family", "u1"), ("gt", "u1"), ("n_ad", "u1"), ("n_alt", "u1"),
                       ("ref_first", "u1"), ("reserved", "u1"), ("ref_len", "<u2"), ("retries", "<u2"),
                       ("flags", "<u2"), ("alt", CALL_ALLELE_DTYPE, (2,))])
CALL_NO_ROW = 0xFF
GT_TEXT = ("0/0", "1/1", "0/1", "1/2", "None")


class VcfOptions(C.Structure):
    """c3r_vcf_options (include/c3r_b200.h)"""
    _fields_ = [("on", C.c_int32), ("show_ref", C.c_int32), ("qual_cut", C.c_double), ("contig", C.c_char_p)]


class SiteFilter(C.Structure):
    """c3r_site_filter (include/c3r_b200.h)"""
    _fields_ = [("pileup_bed", C.c_void_p), ("n_pileup_bed", C.c_int64),
                ("confident_bed", C.c_void_p), ("n_confident_bed", C.c_int64),
                ("known_sites", C.c_void_p), ("n_known_sites", C.c_int64)]


class BgzfBlock(C.Structure):
    """c3r_bgzf_block (include/c3r_b200.h)"""
    _fields_ = [("coff", C.c_int64), ("uoff", C.c_int64), ("csize", C.c_int32), ("usize", C.c_int32),
                ("window", C.c_int32), ("reserved", C.c_int32)]


class BamWindow(C.Structure):
    """c3r_bam_window (include/c3r_b200.h)"""
    _fields_ = [("ubase", C.c_int64), ("usize", C.c_int64), ("ubeg", C.c_int64), ("uend", C.c_int64),
                ("first_block", C.c_int32), ("n_blocks", C.c_int32), ("status", C.c_int32), ("reserved", C.c_int32)]


class BamRaw(C.Structure):
    """c3r_bam_raw (include/c3r_b200.h)"""
    _fields_ = [("tid", C.c_int32), ("n_windows", C.c_int32), ("beg", C.c_int64), ("end", C.c_int64),
                ("n_blocks", C.c_int64), ("n_bytes", C.c_int64), ("n_ubytes", C.c_int64), ("data", C.c_void_p),
                ("blocks", C.c_void_p), ("windows", C.c_void_p)]


EXPORTS = ["c3r_abi_version", "c3r_default_params", "c3r_create", "c3r_destroy", "c3r_last_error",
           "c3r_set_weights", "c3r_set_reference", "c3r_submit_chunk", "c3r_submit_chunk_filtered", "c3r_wait", "c3r_release", "c3r_rerun_resident", "c3r_forward", "c3r_debug_fetch",
           "c3r_bam_open", "c3r_bam_close", "c3r_bam_error", "c3r_bam_n_ref", "c3r_bam_ref_name", "c3r_bam_ref_len",
           "c3r_bam_header_text", "c3r_bam_idxstats", "c3r_bam_fetch", "c3r_bam_write",
           "c3r_decode_vcf", "c3r_free_text", "c3r_debug_format_fixed", "c3r_vcf_write_bgzf",
           "c3r_host_alloc", "c3r_host_free", "c3r_fasta_fetch",
           "c3r_enable_calls", "c3r_wait_calls", "c3r_format_vcf", "c3r_debug_decide_calls",
           "c3r_bam_fetch_raw", "c3r_submit_bam_chunk", "c3r_wait_reads", "c3r_wait_reads_stages", "c3r_debug_inflate",
           "c3r_set_vcf", "c3r_wait_vcf", "c3r_vcf_row_max", "c3r_debug_vcf_rows", "c3r_debug_vcf_qual_check",
           "c3r_debug_vcf_q_min"]

_lib = None


def load():
    """dlopen the in-tree library; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libc3r_b200.so is missing (%s): run `python -m clair3_rna_b200.build`; "
                           "this package has no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.c3r_abi_version.restype = C.c_int
    lib.c3r_default_params.argtypes = [C.POINTER(Params)]
    lib.c3r_default_params.restype = None
    lib.c3r_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(Params)]
    lib.c3r_destroy.argtypes = [C.c_void_p]
    lib.c3r_destroy.restype = None
    lib.c3r_last_error.argtypes = [C.c_void_p]
    lib.c3r_last_error.restype = C.c_char_p
    lib.c3r_set_weights.argtypes = [C.c_void_p, C.POINTER(WeightView), C.c_int]
    lib.c3r_set_reference.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64]
    lib.c3r_submit_chunk.argtypes = [C.c_void_p, C.POINTER(Reads), C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
                                     C.c_int64, C.POINTER(C.c_int64)]
    lib.c3r_submit_chunk_filtered.argtypes = [C.c_void_p, C.POINTER(Reads), C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
                                              C.c_int64, C.POINTER(SiteFilter), C.POINTER(C.c_int64)]
    lib.c3r_wait.argtypes = [C.c_void_p, C.c_int64, C.POINTER(Result)]
    lib.c3r_release.argtypes = [C.c_void_p, C.c_int64]
    lib.c3r_rerun_resident.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    lib.c3r_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(C.c_float)]
    lib.c3r_debug_fetch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    lib.c3r_debug_format_fixed.argtypes = [C.c_double, C.c_int, C.c_char_p]
    lib.c3r_vcf_write_bgzf.argtypes = [C.c_char_p, C.c_char_p, C.c_int64, C.c_int]
    lib.c3r_bam_open.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.POINTER(C.c_void_p)]
    lib.c3r_bam_close.argtypes = [C.c_void_p]
    lib.c3r_bam_close.restype = None
    lib.c3r_bam_error.argtypes = [C.c_void_p]
    lib.c3r_bam_error.restype = C.c_char_p
    lib.c3r_bam_n_ref.argtypes = [C.c_void_p]
    lib.c3r_bam_ref_name.argtypes = [C.c_void_p, C.c_int]
    lib.c3r_bam_ref_name.restype = C.c_char_p
    lib.c3r_bam_ref_len.argtypes = [C.c_void_p, C.c_int]
    lib.c3r_bam_ref_len.restype = C.c_int64
    lib.c3r_bam_header_text.argtypes = [C.c_void_p]
    lib.c3r_bam_header_text.restype = C.c_char_p
    lib.c3r_bam_idxstats.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.c3r_bam_fetch.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.POINTER(Reads)]
    lib.c3r_bam_write.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_int64),
                                  C.POINTER(C.POINTER(Reads)), C.c_int, C.c_char_p]
    lib.c3r_decode_vcf.argtypes = [C.POINTER(Result), C.POINTER(Reads), C.c_void_p, C.c_int64, C.c_int64, C.c_char_p,
                                   C.c_double, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int64),
                                   C.POINTER(C.c_int64)]
    lib.c3r_enable_calls.argtypes = [C.c_void_p, C.c_int]
    lib.c3r_wait_calls.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_void_p), C.POINTER(C.c_int64),
                                   C.POINTER(C.c_float)]
    lib.c3r_format_vcf.argtypes = [C.POINTER(Result), C.c_void_p, C.POINTER(Reads), C.c_void_p, C.c_int64, C.c_int64,
                                   C.c_char_p, C.c_double, C.c_int, C.c_int, C.POINTER(C.c_void_p),
                                   C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.c3r_debug_decide_calls.argtypes = [C.POINTER(Result), C.POINTER(Reads), C.c_void_p, C.c_int64, C.c_int64,
                                           C.c_void_p]
    lib.c3r_set_vcf.argtypes = [C.c_void_p, C.POINTER(VcfOptions)]
    lib.c3r_wait_vcf.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_void_p), C.POINTER(C.c_int64),
                                 C.POINTER(C.c_int64), C.POINTER(C.c_float)]
    lib.c3r_vcf_row_max.argtypes = [C.c_int64]
    lib.c3r_vcf_row_max.restype = C.c_int64
    lib.c3r_debug_vcf_rows.argtypes = [C.POINTER(Result), C.c_void_p, C.POINTER(Reads), C.c_void_p, C.c_int64,
                                       C.c_int64, C.c_char_p, C.c_double, C.c_int, C.POINTER(C.c_void_p),
                                       C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.c3r_debug_vcf_qual_check.argtypes = [C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.c3r_debug_vcf_q_min.argtypes = [C.c_double, C.POINTER(C.c_int32)]
    lib.c3r_bam_fetch_raw.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.c_int64,
                                      C.POINTER(BamRaw)]
    lib.c3r_submit_bam_chunk.argtypes = [C.c_void_p, C.POINTER(BamRaw), C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
                                         C.c_int64, C.POINTER(SiteFilter), C.POINTER(C.c_int64)]
    lib.c3r_wait_reads.argtypes = [C.c_void_p, C.c_int64, C.POINTER(Reads), C.POINTER(C.c_float)]
    lib.c3r_wait_reads_stages.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_float)]
    lib.c3r_debug_inflate.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    lib.c3r_host_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_int64]
    lib.c3r_host_free.argtypes = [C.c_void_p]
    lib.c3r_host_free.restype = None
    lib.c3r_fasta_fetch.argtypes = [C.c_char_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                    C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    lib.c3r_free_text.argtypes = [C.c_void_p]
    lib.c3r_free_text.restype = None
    _lib = lib
    return lib
