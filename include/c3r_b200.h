/*
 * c3r_b200.h — C ABI of libc3r_b200.so: the B200-native pileup calling hot path
 * of Clair3-RNA (candidate tensor generation + pileup-network inference).
 *
 * The reference has no in-process plugin API for this path: it sits behind a
 * process boundary, `python clair3_rna.py call_var_bam ...` per (contig, chunk)
 * (/root/reference/run_clair3_rna:681-706, clair3_rna/call_var_bam.py:88-333),
 * which pipes `create_tensor_pileup` text rows into `call_variants`.  The entry
 * points below are what a binding for that unit of work needs; each one cites
 * the reference code it replaces.  See INTEGRATION.md for the ctypes stub.
 *
 * Conventions: every call returns 0 on success and a negative c3r_status on
 * failure; c3r_last_error(ctx) returns a message for the last failure on that
 * context (valid until the next call on it).  No exceptions cross the boundary.
 * A context is bound to one GPU and is single-producer (not thread safe);
 * distinct contexts are independent.  Inputs are borrowed for the duration of
 * the call only (they are copied to the device before the call returns).
 * Result buffers are owned by the library (pinned host memory) and stay valid
 * until c3r_release() for that ticket or c3r_destroy().
 */
#ifndef C3R_B200_H
#define C3R_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define C3R_ABI_VERSION 2
#define C3R_WINDOW 33        /* shared/param_p.py:34-35  no_of_positions */
#define C3R_N_OUT 24         /* 21 gt21 + 3 genotype, shared/param_p.py:37 */

typedef enum {
    C3R_OK = 0,
    C3R_ERR_ARG = -1,        /* bad argument / unsupported value            */
    C3R_ERR_CUDA = -2,       /* CUDA runtime error, see c3r_last_error      */
    C3R_ERR_STATE = -3,      /* call order violated (no weights, bad ticket)*/
    C3R_ERR_CAPACITY = -4    /* input exceeds a documented limit            */
} c3r_status;

typedef struct c3r_ctx c3r_ctx;

/* Options of the path.  Defaults mirror shared/param_p.py and the argv
 * call_var_bam forwards (clair3_rna/call_var_bam.py:205-245). */
typedef struct {
    int32_t channels;        /* 18, or 30 with --enable_phasing_model (create_tensor_pileup.py:466) */
    int32_t min_coverage;    /* --minCoverage, param_p.py:90 (4)           */
    int32_t min_mq;          /* --minMQ, param_p.py:20 (5)                 */
    uint32_t excl_flags;     /* samtools --excl-flags, param_p.py:41 (2316)*/
    double snp_min_af;       /* --snp_min_af, param_p.py:88 (0.08)         */
    double indel_min_af;     /* --indel_min_af, param_p.py:89 (0.15)       */
    int32_t enable_padding;  /* --enable_padding_in_splice_junction_regions (create_tensor_pileup.py:573-593) */
    int32_t max_depth;       /* param_p.py:14 (144): depth > 1.5*max_depth rescales the window (clair3_rna/utils.py:85-92) */
    double skip_proportion;  /* param_p.py:46 (0.2)                        */
    int32_t nn_impl;         /* 0 = fp32 CUDA-core network, 1 = tcgen05 fp16/fp32-accumulate network */
    int32_t keep_tensor;     /* also return the int32 windows (parity / debug) */
    int32_t keep_rows;       /* also return the per-position count matrix (parity / debug) */
    int32_t enable_head_tail;/* --enable_variant_calling_at_sequence_head_and_tail: zero rows stand in for the columns
                                before a run of pileup columns and after the end of the stream
                                (create_tensor_pileup.py:467, 508-514, 613-637) */
} c3r_params;

/* Flat alignment records of one region, BAM record order (coordinate sorted).
 * This is what `samtools mpileup BAM -r ctg:s-e` reads from the BAM
 * (create_tensor_pileup.py:446-451); layout in clair3_rna_b200/reads.py. */
typedef struct {
    int64_t n_reads;
    int64_t n_ops;
    int64_t n_seq_bytes;
    const int32_t* pos;        /* [n_reads]   0-based leftmost position          */
    const uint16_t* flag;      /* [n_reads]   SAM flag                           */
    const uint8_t* mapq;       /* [n_reads]                                      */
    const uint8_t* hp;         /* [n_reads]   HP:i tag, 0 = absent               */
    const int32_t* cigar_off;  /* [n_reads+1] CSR into cigar                     */
    const uint32_t* cigar;     /* [n_ops]     BAM encoding len<<4|op             */
    const int64_t* seq_off;    /* [n_reads+1] base offsets, each even            */
    const uint8_t* seq;        /* [n_seq_bytes] nt16 nibbles, high nibble first  */
} c3r_reads;

/* Network weights in Keras layout, fp32 (clair3_rna/model.py:126-156):
 *   LSTM{1,2}/{forward,backward}/{kernel[in,4u], recurrent_kernel[u,4u], bias[4u]}   gate order i,f,c,o
 *   L4, L5_1, L5_2, Y_gt21_logits, Y_genotype_logits: {kernel[in,out], bias[out]}
 * Replaces m.load_weights(chkpnt_fn) at clair3_rna/call_variants.py:1472. */
typedef struct {
    const char* name;          /* e.g. "LSTM1/forward/kernel" */
    const float* data;
    int64_t n_elem;
} c3r_weight_view;

/* One allele of a candidate's alt_info (create_tensor_pileup.py:595-596),
 * in the reference's dict insertion order. */
typedef struct {
    uint8_t kind;              /* 'X' base, 'I' insertion, 'D' deletion, 'R' reference */
    uint8_t base;              /* X: alt base letter; R/I: reference base letter       */
    uint16_t len;              /* I: inserted length; D: deleted length                */
    int32_t count;
    uint32_t seq_off;          /* I: base offset of the inserted bases in c3r_reads.seq */
    uint32_t order;            /* first-occurrence key (read ordinal*2 + is_indel)     */
} c3r_alt_entry;

typedef struct {
    int64_t n_rows;            /* pileup rows (covered positions kept on the device)   */
    int64_t n_cand;            /* emitted candidates                                   */
    const int32_t* pos;        /* [n_cand] 1-based candidate position                  */
    const int32_t* depth;      /* [n_cand] depth as in alt_info                        */
    const float* probs;        /* [n_cand*24] network output                           */
    const int64_t* alt_off;    /* [n_cand]   start of each candidate's alleles         */
    const int32_t* alt_n;      /* [n_cand]   number of alleles                         */
    const c3r_alt_entry* alt;
    const int32_t* tensor;     /* [n_cand*33*channels] or NULL (keep_tensor)           */
    const int32_t* row_pos;    /* [n_rows] 1-based, or NULL (keep_rows)                */
    const int32_t* row_counts; /* [n_rows*channels] or NULL (keep_rows)                */
    const int32_t* row_depth;  /* [n_rows] or NULL (keep_rows)                         */
    float stage_ms[8];         /* device time of: 0 H2D, 1 K1 scan+rows, 2 K2 compare + row events, 3 K2 rows, 4 K3 filter,
                                  5 K4 window+alt, 6 K5 network, 7 D2H                  */
    int32_t kernel_launches;   /* kernels launched for this ticket                     */
} c3r_result;

typedef int64_t c3r_ticket;

int c3r_abi_version(void);
void c3r_default_params(c3r_params* p);

int c3r_create(c3r_ctx** out, int device_ordinal, const c3r_params* params);
void c3r_destroy(c3r_ctx* ctx);
const char* c3r_last_error(c3r_ctx* ctx);

int c3r_set_weights(c3r_ctx* ctx, const c3r_weight_view* views, int n_views);

/* Keep the reference bases of a contig (or any window of it) resident on the device, like the
 * weights: later c3r_submit_chunk calls may then pass ref = NULL.  Replaces the per-chunk
 * `samtools faidx` of shared/utils.py:168-194 (the reference re-reads it for every chunk). */
int c3r_set_reference(c3r_ctx* ctx, const uint8_t* ref, int64_t ref_start1, int64_t ref_len);

/* One (contig, chunk): replaces one `call_var_bam` producer|consumer pipeline up
 * to the 24 probabilities (clair3_rna/call_var_bam.py:278-295).
 *   ref / ref_start1 / ref_len: upper-case reference bytes of [ref_start1, ref_start1+ref_len)
 *                               (create_tensor_pileup.py:416-428, expandReferenceRegion)
 *                               ref == NULL: use the window given to c3r_set_reference
 *   region_start1..region_end1: the 1-based inclusive mpileup region (:412-415)
 * The call queues the host-to-device copies and the position / row stages and returns; it does not wait for the
 * device.  `reads` and `ref` must stay valid and unchanged until c3r_wait(ticket) has returned (pinned host memory is
 * read by DMA after the call).  The stages that need the candidate count (windows, allele table, network, result
 * copies) are queued by a later call into the library once the count has reached the host - by the next
 * c3r_submit_chunk if it is in by then, else by c3r_wait - so errors found on the device (capacity, the 8000-read
 * depth cap of mpileup) are returned by c3r_wait, which then also gives the ticket back.          */
int c3r_submit_chunk(c3r_ctx* ctx, const c3r_reads* reads, const uint8_t* ref, int64_t ref_start1,
                     int64_t ref_len, int64_t region_start1, int64_t region_end1, c3r_ticket* ticket);

/* Optional site filters of one chunk: the region modes of the producer.  Intervals are 0-based half-open BED
 * intervals as (start, end) int32 pairs, sorted, non-empty, disjoint and non-touching (merge on the host);
 * a count < 0 means "option not given", 0 means "given but empty for this contig".
 *   pileup_bed     --extend_bed -> `samtools mpileup -l`: pileup columns exist only inside these intervals, so
 *                  a candidate needs its 33 columns inside one of them   (create_tensor_pileup.py:446-451)
 *   confident_bed  --bed_fn: a candidate needs [pos-1, pos+max_del_length+1) to overlap an interval, where
 *                  max_del_length is the longest deletion starting at the site
 *                  (create_tensor_pileup.py:480-481, 551-554; shared/interval_tree.py:80-89)
 *   known_sites    --vcf_fn: strictly increasing 1-based positions; candidates are exactly these sites,
 *                  whatever their allele fractions, depth or reference base    (create_tensor_pileup.py:397-405, 555-556)
 * The arrays are host memory, read during the call.  Chunk geometry in these modes (BED span, site-count
 * chunks) is host logic: clair3_rna_b200/regions.py restates create_tensor_pileup.py:373-418.            */
typedef struct {
    const int32_t* pileup_bed;    int64_t n_pileup_bed;
    const int32_t* confident_bed; int64_t n_confident_bed;
    const int32_t* known_sites;   int64_t n_known_sites;
} c3r_site_filter;

/* c3r_submit_chunk with site filters; filter == NULL is c3r_submit_chunk. */
int c3r_submit_chunk_filtered(c3r_ctx* ctx, const c3r_reads* reads, const uint8_t* ref, int64_t ref_start1,
                              int64_t ref_len, int64_t region_start1, int64_t region_end1,
                              const c3r_site_filter* filter, c3r_ticket* ticket);
/* Blocks until the ticket's results are in the library's pinned host buffers (valid until c3r_release).  Before it
 * blocks it queues the candidate-count dependent stages of EVERY ticket submitted so far, so with two tickets in
 * flight the device goes from one chunk's network pass to the next without waiting for the host. */
int c3r_wait(c3r_ctx* ctx, c3r_ticket ticket, c3r_result* result);
int c3r_release(c3r_ctx* ctx, c3r_ticket ticket);

/* Re-run the device stages of a ticket on the inputs already resident in HBM
 * (no H2D, no D2H).  Used by bench.py for the device-resident throughput and
 * by ncu captures.  total_ms receives the CUDA-event time of the pass. */
int c3r_rerun_resident(c3r_ctx* ctx, c3r_ticket ticket, float* total_ms, float* stage_ms8);

/* Network forward alone on host int32 windows [n,33,channels] -> probs [n,24]
 * (clair3_rna/model.py:175-216 via predict_on_batch, call_variants.py:1505). */
int c3r_forward(c3r_ctx* ctx, const int32_t* tensor, int64_t n, float* probs, float* device_ms);

/* Diagnostics: copy an intermediate activation buffer of the last tensor-core forward to the
 * host (which: 0 = LSTM1 output, packed fp16; 2 = LSTM2 output, packed fp16; 3 = L4 output,
 * fp32 [sites,128]).  Layouts in csrc/nn_tc.cuh. */
int c3r_debug_fetch(c3r_ctx* ctx, int which, void* dst, int64_t max_bytes, int64_t* n_bytes);

/* Page-locked host memory for the arrays handed to c3r_submit_chunk (read by DMA while the call has long returned;
 * pageable memory is staged by the driver inside the call instead: 0.5 ms per 5 MB reference window).  Needs a
 * CUDA device.  Release with c3r_host_free. */
int c3r_host_alloc(void** out, int64_t n_bytes);
void c3r_host_free(void* p);

/* Upper-cased bases of the 1-based inclusive region [start1, end1] (clipped to the contig) of an indexed FASTA into
 * `out` (out_cap bytes; *n_out receives the count).  contig_len / offset / linebases / linewidth are the contig's
 * .fai columns.  Replaces the per-chunk `samtools faidx` of shared/utils.py:168-194 (reference_sequence_from). */
int c3r_fasta_fetch(const char* path, int64_t contig_len, int64_t offset, int64_t linebases, int64_t linewidth,
                    int64_t start1, int64_t end1, uint8_t* out, int64_t out_cap, int64_t* n_out);

/* ------------------------------------------------------------------------------------------
 * Probabilities + allele table -> VCF data lines (host, multi-threaded; csrc/decode.cpp).  Replaces the
 * per-candidate Python of output_with / output_from (clair3_rna/call_variants.py:684-1392, options as
 * forwarded by call_var_bam.py:247-272: --pileup --showRef, add_indel_length False): each candidate's call
 * record is made on the host by the code k_call runs (csrc/call.cuh) and printed like c3r_format_vcf.  One line per
 * candidate of `res` in order ("CHROM POS . REF ALT QUAL FILTER . GT:GQ:DP:AD:AF ..."), candidates whose
 * centre reference base is outside the IUPAC table are skipped (clair3_rna/utils.py:113).
 *   reads: the records `res` was computed from (inserted bases are read from reads->seq)
 *   ref / ref_start1 / ref_len: the reference window given to c3r_submit_chunk
 *   qual_cut: --qual (2); < 0 disables the LowQual filter.  n_threads <= 0: all host cores.
 * *text is malloc'ed, NUL terminated, *n_bytes long; release it with c3r_free_text.               */
int c3r_decode_vcf(const c3r_result* res, const c3r_reads* reads, const uint8_t* ref, int64_t ref_start1,
                   int64_t ref_len, const char* contig, double qual_cut, int show_ref, int n_threads,
                   char** text, int64_t* n_bytes, int64_t* n_rows);
void c3r_free_text(char* text);
/* test hook: the decoder's own "%.2f" / "%.4f" formatting (exact, ties to even on the binary value) of
 * 0 <= x < 1e12 into out (>= 32 bytes) */
int c3r_debug_format_fixed(double x, int decimals, char* out);

/* ------------------------------------------------------------------------------------------
 * Call records: the genotype decision of c3r_decode_vcf (output_from and the allele counts of output_with) made
 * on the GPU, one fixed-size record per candidate (csrc/call.cuh, kernel k_call).  Only QUAL (a log), AF (a
 * division) and the text are left to the host: c3r_format_vcf turns records into the lines c3r_decode_vcf prints.
 *
 * An allele's text is `first`, then ins_len inserted bases from c3r_reads.seq (nt16, base offset ins_seq_off),
 * then REF's letters [suffix_from, ref_len).  REF's letter 0 is ref_first (the centre base; for a reference call
 * the A/C/G/T it stands for), letters 1.. are the reference bases after the candidate, ref[pos - ref_start1 + 1 ..].
 * Every ALT the decision makes has this form: SNP bases, insertion keys, INSDEL's ins + REF[1:], HET_ACGT_DEL's
 * b + REF[1:] and HET_DELDEL's REF[0] + REF[1+len:]. */
typedef struct {
    uint8_t first;
    uint8_t reserved;
    uint16_t ins_len;
    uint32_t ins_seq_off;
    uint16_t suffix_from;
    uint16_t reserved2;
} c3r_call_allele;

#define C3R_CALL_NO_ROW 0xFF   /* c3r_call.family of a candidate that gives no VCF row */

/* c3r_call.gt: 0 "0/0", 1 "1/1", 2 "0/1", 3 "1/2", 4 "None" */
typedef struct {
    float prob;                /* probability of the call, the float32 QUAL is computed from            */
    int32_t ref_count;         /* AD's first number (reads of the reference allele)                     */
    int32_t support;           /* AF's numerator                                                        */
    int32_t ad[2];             /* AD's numbers after ref_count, n_ad of them                            */
    uint8_t family;            /* outcome family the call came from (0 = reference call, 1 HOMO_SNP, 2 HET_SNP,
                                  3 HOMO_INS, 4 HET_ACGT_INS, 5 HET_INSINS, 6 HOMO_DEL, 7 HET_ACGT_DEL,
                                  8 HET_DELDEL, 9 INSDEL), C3R_CALL_NO_ROW: no row                        */
    uint8_t gt;
    uint8_t n_ad;
    uint8_t n_alt;             /* ALT alleles, comma separated; 0: ALT is "."                           */
    uint8_t ref_first;
    uint8_t reserved;
    uint16_t ref_len;
    uint16_t retries;          /* diagnostics: bit C3R_RETRY_* of every retry branch the decision passed */
    uint16_t flags;            /* diagnostics: bit f of every family flagged by the last pass (its best member ties
                                  the call's probability); AD follows the first flagged family in output_with's order,
                                  which may differ from `family`                                              */
    c3r_call_allele alt[2];
} c3r_call;

/* c3r_call.retries: the branches of output_from's retry loop that zero a family member and try again */
enum {
    C3R_RETRY_HOMO_SNP_NO_X = 0,      /* no X allele                                        */
    C3R_RETRY_HOMO_SNP_IS_REF,        /* the chosen base is the centre base                 */
    C3R_RETRY_HET_SNP_LT2_X,          /* neither genotype base is the centre: < 2 X alleles */
    C3R_RETRY_HET_SNP_NO_X,
    C3R_RETRY_HET_SNP_IS_REF,
    C3R_RETRY_HOMO_INS_NO_I,          /* no insertion key of 1..50 letters                  */
    C3R_RETRY_HET_ACGT_INS_NO_I,
    C3R_RETRY_HET_ACGT_INS_NO_X,
    C3R_RETRY_HET_INSINS_LT2_I,
    C3R_RETRY_HET_INSINS_SAME,        /* the two keys are equal (distinct dict keys: never)   */
    C3R_RETRY_HOMO_DEL_NO_D,
    C3R_RETRY_HET_ACGT_DEL_NO_D,
    C3R_RETRY_HET_DELDEL_LT2_D,
    C3R_RETRY_HET_DELDEL_SAME,        /* the two ALTs coincide (distinct lengths: never)    */
    C3R_RETRY_INSDEL_NO_I_OR_D
};

/* Make call records for the tickets submitted after this call (on != 0) or stop (0; the default).  With records
 * off nothing about a ticket changes: the same kernels, copies and results. */
int c3r_enable_calls(c3r_ctx* ctx, int on);
/* The records of a ticket submitted with records on, one per candidate of its c3r_result, in pinned library
 * memory valid until c3r_release.  Call after c3r_wait.  device_ms (may be NULL): device time of k_call.
 * C3R_ERR_STATE when records were off for the ticket or c3r_wait has not returned it. */
int c3r_wait_calls(c3r_ctx* ctx, c3r_ticket ticket, const c3r_call** calls, int64_t* n, float* device_ms);
/* c3r_decode_vcf from call records: the same arguments and the same text, with the decision read from
 * calls[n_cand] instead of made.  C3R_ERR_ARG (and no text) when a record cannot be printed: malformed, or made
 * over another reference window or read pool than the ones given. */
int c3r_format_vcf(const c3r_result* res, const c3r_call* calls, const c3r_reads* reads, const uint8_t* ref,
                   int64_t ref_start1, int64_t ref_len, const char* contig, double qual_cut, int show_ref,
                   int n_threads, char** text, int64_t* n_bytes, int64_t* n_rows);
/* test hook: the records k_call makes, by the same code on the host (no GPU needed), into out[res->n_cand] */
int c3r_debug_decide_calls(const c3r_result* res, const c3r_reads* reads, const uint8_t* ref, int64_t ref_start1,
                           int64_t ref_len, c3r_call* out);

/* ------------------------------------------------------------------------------------------
 * VCF text made on the GPU: after k_call, each candidate's row is printed on the device (csrc/vcf_row.cuh, the same
 * printer c3r_decode_vcf and c3r_format_vcf use on the host) and a ticket returns its data lines as one block of text,
 * byte for byte what c3r_format_vcf prints for the same contig, qual_cut and show_ref.
 * QUAL on the device comes from a table of the host formula's thresholds (built once per process, uploaded once per
 * context); the text of a NaN AF is the host printf's. */
typedef struct {
    int32_t on;
    int32_t show_ref;
    double qual_cut;           /* < 0: no LowQual filter                                                  */
    const char* contig;        /* CHROM of the rows (copied; at most 1024 bytes)                          */
} c3r_vcf_options;

/* VCF text for the tickets submitted after this call (opts->on != 0) or not (the default).  The options are copied
 * into a ticket when it is submitted, so a caller may set the contig before every submit.  Text on implies k_call;
 * its records reach the host only if c3r_enable_calls is on too (else c3r_wait_calls keeps returning C3R_ERR_STATE).
 * With text off nothing about a ticket changes: the same kernels, copies and results. */
int c3r_set_vcf(c3r_ctx* ctx, const c3r_vcf_options* opts);
/* The data lines of a ticket submitted with text on ('\n' after each, not NUL terminated), in pinned library memory
 * valid until c3r_release; call after c3r_wait.  device_ms (may be NULL): device time of the text kernels (row lengths,
 * offsets, rows).  C3R_ERR_STATE for a ticket submitted with text off or not returned by c3r_wait. */
int c3r_wait_vcf(c3r_ctx* ctx, c3r_ticket ticket, const char** text, int64_t* n_bytes, int64_t* n_rows, float* device_ms);
/* The most bytes one row can take with a contig name of contig_len bytes: the device sizes a ticket's text buffers
 * as n_cand times this. */
int64_t c3r_vcf_row_max(int64_t contig_len);
/* test hooks (no GPU): the device's printing on the host - QUAL from the table, lengths counted first, rows written
 * at their offsets, each checked to fill its counted length (else C3R_ERR_STATE) - with c3r_format_vcf's arguments
 * and result (one thread; free with c3r_free_text); QUAL by table against QUAL by formula for all 2^32 float32 bit
 * patterns (n_threads <= 0: all cores); FILTER's threshold q_min (hundredths) of a qual_cut. */
int c3r_debug_vcf_rows(const c3r_result* res, const c3r_call* calls, const c3r_reads* reads, const uint8_t* ref,
                       int64_t ref_start1, int64_t ref_len, const char* contig, double qual_cut, int show_ref,
                       char** text, int64_t* n_bytes, int64_t* n_rows);
int c3r_debug_vcf_qual_check(int n_threads, int64_t* n_checked, int64_t* n_mismatch);
int c3r_debug_vcf_q_min(double qual_cut, int32_t* q_min);

/* ------------------------------------------------------------------------------------------
 * BAM / BGZF / BAI input (host side, zlib; csrc/bam_io.cpp).  The reference reads the BAM only
 * through external samtools: `samtools mpileup BAM -r ctg:s-e ...` (src/create_tensor_pileup.py:
 * 436-451) and `samtools idxstats BAM` (run_clair3_rna:187).  c3r_bam_fetch is the index fetch
 * of that mpileup call: the records overlapping the 1-based inclusive region, in file order,
 * as the flat arrays c3r_submit_chunk takes (flag / MAPQ filtering stays on the device).
 * Buffers behind the returned c3r_reads belong to the handle and are valid until the next
 * c3r_bam_fetch on it or c3r_bam_close.  A handle is not thread safe.                        */
typedef struct c3r_bam c3r_bam;

/* index_path NULL: <path>.bai, then <path minus .bam>.bai.  n_threads <= 0: all host cores
 * (BGZF blocks are inflated in parallel).  *out is set even on failure (for c3r_bam_error). */
int c3r_bam_open(const char* path, const char* index_path, int n_threads, c3r_bam** out);
void c3r_bam_close(c3r_bam* bam);
const char* c3r_bam_error(c3r_bam* bam);
int c3r_bam_n_ref(c3r_bam* bam);
const char* c3r_bam_ref_name(c3r_bam* bam, int tid);
int64_t c3r_bam_ref_len(c3r_bam* bam, int tid);
const char* c3r_bam_header_text(c3r_bam* bam);
/* mapped / unmapped record counts of a reference from the index (samtools idxstats columns 3, 4) */
int c3r_bam_idxstats(c3r_bam* bam, int tid, int64_t* n_mapped, int64_t* n_unmapped);
int c3r_bam_fetch(c3r_bam* bam, int tid, int64_t start1, int64_t end1, c3r_reads* out);

/* ------------------------------------------------------------------------------------------
 * Device BAM reading: the host does c3r_bam_fetch's index query and reads the compressed bytes; the GPU inflates the
 * BGZF blocks, finds and checks the records and writes the flat arrays c3r_bam_fetch would return, bit for bit, with
 * the same status for every input the host fetch rejects (csrc/bgzf.cuh).
 *
 * A window is one merged index chunk: the BGZF blocks c3r_bam_fetch inflates for it, read back to back into the
 * caller's buffer.  Its records start at ubeg of its inflated bytes and continue while a record's length field ends
 * at or before uend; a block shared by two windows is read (and inflated) once for each. */
typedef struct {
    int64_t coff;              /* offset of the block in c3r_bam_raw.data                                  */
    int64_t uoff;              /* offset of its inflated bytes in the fetch's inflated bytes (n_ubytes)     */
    int32_t csize;             /* compressed size (BSIZE + 1)                                              */
    int32_t usize;             /* ISIZE                                                                    */
    int32_t window;            /* window of the block                                                      */
    int32_t reserved;
} c3r_bgzf_block;

typedef struct {
    int64_t ubase;             /* offset of the window's inflated bytes in the fetch's inflated bytes      */
    int64_t usize;             /* inflated bytes of the window                                             */
    int64_t ubeg, uend;        /* record walk bounds within the window                                     */
    int32_t first_block, n_blocks;
    int32_t status;            /* 0, or why the window could not be read (its blocks are then absent):
                                  2 corrupt BGZF header, 3 block larger than 64 KiB, 4 short read; the error
                                  is reported only if the fetch gets that far                               */
    int32_t reserved;
} c3r_bam_window;

typedef struct {
    int32_t tid;
    int32_t n_windows;
    int64_t beg, end;          /* 0-based half-open region of the fetch                                    */
    int64_t n_blocks;
    int64_t n_bytes;           /* compressed bytes in data                                                 */
    int64_t n_ubytes;          /* inflated bytes of all windows                                            */
    const uint8_t* data;
    const c3r_bgzf_block* blocks;    /* [n_blocks], in window order                                        */
    const c3r_bam_window* windows;   /* [n_windows]                                                        */
} c3r_bam_raw;

/* c3r_bam_fetch without the inflate and the record walk: the index query, and the compressed blocks of every
 * window read into buf (cap bytes; page-locked memory from c3r_host_alloc makes the submit a pure DMA).  The block
 * and window tables belong to the handle until its next fetch.  C3R_ERR_CAPACITY with the needed size in
 * out->n_bytes when cap is too small. */
int c3r_bam_fetch_raw(c3r_bam* bam, int tid, int64_t start1, int64_t end1, uint8_t* buf, int64_t cap, c3r_bam_raw* out);

/* c3r_submit_chunk_filtered for the records of a raw fetch, parsed on the device.  raw->data and the tables must
 * stay unchanged until c3r_wait returns.  The parse runs ahead of the chunk's stages: a later call into the library
 * sizes the read buffers from its counts and queues the rest.  A corrupt BAM makes c3r_wait return C3R_ERR_ARG
 * (the host fetch's message in c3r_last_error) and gives the ticket back. */
int c3r_submit_bam_chunk(c3r_ctx* ctx, const c3r_bam_raw* raw, const uint8_t* ref, int64_t ref_start1, int64_t ref_len,
                         int64_t region_start1, int64_t region_end1, const c3r_site_filter* filter, c3r_ticket* ticket);
/* The device-parsed records of a ticket from c3r_submit_bam_chunk, in pinned library memory valid until
 * c3r_release; call after c3r_wait.  device_ms (may be NULL): device time of the parse stages (inflate, record
 * boundaries, parse, offsets, write).  C3R_ERR_STATE for a ticket submitted from host reads. */
int c3r_wait_reads(c3r_ctx* ctx, c3r_ticket ticket, c3r_reads* out, float* device_ms);
/* The same stages split: [0] inflate, [1] record boundaries, [2] parse + offsets + write (ms). */
int c3r_wait_reads_stages(c3r_ctx* ctx, c3r_ticket ticket, float stage_ms[3]);
/* test hook: the device's DEFLATE decoder and CRC check run on the host over one BGZF block of n bytes
 * (header, payload, trailer) into out (cap bytes); *n_out receives ISIZE.  C3R_ERR_ARG on any failure.  No GPU. */
int c3r_debug_inflate(const uint8_t* block, int64_t n, uint8_t* out, int64_t cap, int64_t* n_out);

/* Writes a coordinate-sorted BAM and <path>.bai from flat records, batches[r] = records of
 * reference r (NULL = none): fixtures for the reader and for the drop-in entry point (there is
 * no samtools in the build image).  level: zlib level, -1 = default.  header_text NULL: minimal
 * @HD/@SQ header.                                                                           */
int c3r_bam_write(const char* path, int n_ref, const char* const* names, const int64_t* lens,
                  const c3r_reads* const* batches, int level, const char* header_text);

/* bgzip + tabix of the merged VCF: what `sort_vcf --compress_vcf True` does through the external `bgzip` and
 * `tabix -p vcf` (src/sort_vcf.py:70-76, run_clair3_rna:722).  Writes `path` (BGZF) and `path`.tbi from the VCF
 * text (header lines, then data lines sorted by position within each contig).  level <= 0: zlib default.      */
int c3r_vcf_write_bgzf(const char* path, const char* text, int64_t n_bytes, int level);

#ifdef __cplusplus
}
#endif
#endif /* C3R_B200_H */
