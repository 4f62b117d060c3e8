// libc3r_b200.so — C ABI (include/c3r_b200.h) and host orchestration of the kernels in
// pileup.cuh (integer half) and nn_fp32.cuh / nn_tc.cuh (network forward).
//
// One context = one GPU.  A ticket owns a slot: device input buffers, scratch, pinned
// result buffers and a stream.  submit() queues the copies of the flat records to HBM and
// the position/row-space stages (stage A) and returns; the scalars stage A leaves (rows,
// candidates, error word) travel to the host behind it, and the next call into the library
// that finds them there sizes the candidate-space buffers and queues windows, alt_info, the
// network and the D2H copies (stage B, advance()); wait() does that for every ticket in
// flight, then synchronises the slot's stream.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <chrono>
#include <map>
#include <cuda_runtime.h>

#include "../../include/c3r_b200.h"
#include "pileup.cuh"
#include "nn_fp32.cuh"
#include "nn_tc.cuh"
#include "call.cuh"
#include "vcf_row.cuh"
#include "bgzf.cuh"

using namespace c3r;

namespace {

struct Buf {
    void* p = nullptr;
    size_t cap = 0;
};
struct Pin {
    void* p = nullptr;
    size_t cap = 0;
};

constexpr int N_SLOTS = 4;
constexpr int N_EV = 9;

struct Slot {
    bool in_use = false;
    bool has_result = false;
    cudaStream_t st = nullptr;        // stage B: windows, allele table, network, result copies (high priority)
    cudaStream_t st_a = nullptr;      // H2D copies and stage A (low priority: they fill the SMs the network passes leave idle)
    cudaEvent_t ev[N_EV] = {};
    cudaEvent_t ev_alt = nullptr;
    cudaEvent_t ev_call[2] = {};      // around k_call
    bool calls = false;               // call records for this ticket (c3r_enable_calls when it was submitted)
    // VCF text for this ticket (c3r_set_vcf when it was submitted): k_vcf_len, the offsets scan and k_vcf_write after
    // k_call; the totals (bytes, rows) land in the scalars [8], [9]
    bool vcf = false;
    int32_t vcf_show_ref = 1, vcf_q_min = 0;
    std::string vcf_contig;
    int64_t vcf_row_max = 0;
    cudaEvent_t ev_vcf[2] = {};       // around the text kernels
    Buf d_vlen, d_voff, d_text, d_contig;
    Pin h_text;
    // inputs
    Buf pos, flag, mapq, hp, cigar_off, cigar, seq_off, seq, ref;
    // per read/op
    Buf admit, read_end, op_x, op_y, op_info, blockmax;
    // position space
    Buf covA, covE, rowR, cov_up, ptile, ctile, csuper, word_base;
    // row space
    Buf row_pos, counts, row_depth, row_flag, head_cnt, tail_cnt, skipdiff, max_skip, row_ins, row_del;
    Buf binc, bin_cur, events, raw, cov, cov_tile, refnib;
    Buf pbed, cbed, known, covP;   // site filters of the chunk; printed columns (covA inside the pileup BED)
    Buf cand_row, cand_pos, cand_depth, tensor, alt_off, alt_n, alt, cur_ref, deleted, probs;
    Buf d_calls;          // call records (k_call)
    Buf xop;              // LSTM1 operand images written by k_window_xop (fused K4 -> K5 path)
    bool fused_window = false;
    Buf scalars;          // [0] n_rows (i64) [1] n_cand (i64) [2] alt_total (i64) [3] err (i32) [4] tail columns (2 x i32) [5] raw row events (i64)
    Buf scan_scratch;     // look-back scan state: ticket counters, tile status words, tile aggregates / prefixes
    ScanState scan = {};
    uint32_t scan_epoch = 0;
    size_t zero_bytes = 0;            // bytes of the pool behind covA that every pass starts from zero
    // submit returns once stage A is queued; stage B (windows, alt table, network, result copies) is queued by a later
    // call into the library, when the candidate count has arrived on the host (advance())
    bool pending_b = false;
    cudaEvent_t ev_cnt = nullptr;     // the scalars of stage A are on the host
    uint64_t order = 0;               // submit order
    int64_t n_seq_bytes = 0, n_known_sites = 0;
    bool exact_bounds = false;        // capacity bounds from an exact pass over the CIGARs (retry after a device capacity error)
    int deferred_rc = 0;              // error of the deferred part, reported by c3r_wait
    std::string deferred_err;
    // pinned results
    Pin h_scalars, h_pos, h_depth, h_probs, h_alt_off, h_alt_n, h_alt, h_tensor, h_row_pos, h_counts, h_row_depth, h_calls;
    Dev d;
    int64_t n_rows = 0, n_cand = 0, alt_total = 0;
    int launches = 0;
    c3r_result res;
    // device BAM reading (c3r_submit_bam_chunk): the records are parsed on the device before stage A
    bool bam = false;
    bool pending_parse = false;       // the parse counts have not been taken yet (advance())
    cudaEvent_t ev_parse = nullptr;   // the parse counts are on the host
    cudaEvent_t ev_bam[6] = {};       // [0, 1) inflate, [1, 2) record boundaries, [2, 3) parse + offsets, [4, 5) k_rec_write
    c3rbgzf::Fetch fetch = {};
    Buf b_cdata, b_blk, b_win, b_ubuf, b_nrec, b_soff, b_scls, b_skey, b_snops, b_snb, b_sdst, b_sc;
    Pin h_fsc, h_rpos, h_rflag, h_rmapq, h_rhp, h_rcoff, h_rcig, h_rsoff, h_rseq;
    c3r_reads h_reads = {};           // the parsed records in the pinned buffers above
    // what c3r_submit_bam_chunk was given, for the part queued once the parse counts are in
    const uint8_t* ref_host = nullptr;
    int64_t ref_start1 = 0, ref_len = 0, region_start1 = 0, region_end1 = 0;
    bool has_filter = false;
    std::vector<int32_t> f_pbed, f_cbed, f_known;
    c3r_site_filter flt = {};
};

}  // namespace

struct c3r_ctx {
    int device = 0;
    c3r_params prm;
    std::string err;
    Slot slots[N_SLOTS];
    int sm_count = 148;
    // weights
    bool have_weights = false;
    Buf wbuf;                 // all fp32 weights, Keras-derived layouts
    NetF32 net;
    Buf nn_scratch;
    NetF32Scratch nscr;
    TcNet tc;                 // tensor-core path state (nn_tc.cuh)
    uint64_t submit_seq = 0;
    int prio_hi = 0;
    const c3r_site_filter* filter = nullptr;   // of the submit in progress
    bool tc_dirty = false;    // a tensor-core forward ran since the last device error check
    cudaEvent_t nn_done = nullptr;   // end of the last network pass: the scratch (h1, h2, l4 ...) is shared by all tickets
    Buf thr;                  // allele-frequency threshold tables (k_thr_table)
    Buf ref_res;              // resident reference window (c3r_set_reference)
    Buf refnib_res;           // its one-hot nibble form (k_refnib)
    int64_t ref_res_start0 = 0, ref_res_len = 0;
    double t_phase[8] = {};   // C3R_TIMING: host seconds of submit's phases (printed by c3r_destroy)
    int64_t n_submit = 0;
    bool calls = false;       // c3r_enable_calls: tickets submitted from now on make call records
    // c3r_set_vcf: tickets submitted from now on print their VCF rows on the device
    bool vcf = false;
    int32_t vcf_show_ref = 1, vcf_q_min = 0;
    std::string vcf_contig;
    Buf vcf_qtab;             // QUAL thresholds (c3rvcf::qual_table), uploaded by the first c3r_set_vcf that turns text on
    int32_t vcf_q_n = 0;
    char nan_text[8] = {}, ninf_text[8] = {};
    Buf fwd_in, fwd_out;      // c3r_forward staging
    cudaStream_t fwd_stream = nullptr;
};

namespace {

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            char b__[512];                                                                         \
            snprintf(b__, sizeof b__, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            ctx->err = b__;                                                                        \
            return C3R_ERR_CUDA;                                                                   \
        }                                                                                          \
    } while (0)

int fail(c3r_ctx* ctx, int code, const std::string& msg) {
    ctx->err = msg;
    return code;
}

int ensure(c3r_ctx* ctx, Buf& b, size_t bytes) {
    if (bytes < 256) bytes = 256;
    if (b.cap >= bytes) return 0;
    if (b.p) CK(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    size_t want = bytes + bytes / 4 + 4096;
    CK(cudaMalloc(&b.p, want));
    b.cap = want;
    return 0;
}
int ensure_pin(c3r_ctx* ctx, Pin& b, size_t bytes) {
    if (bytes < 256) bytes = 256;
    if (b.cap >= bytes) return 0;
    if (b.p) CK(cudaFreeHost(b.p));
    b.p = nullptr;
    b.cap = 0;
    size_t want = bytes + bytes / 4 + 4096;
    CK(cudaMallocHost(&b.p, want));
    b.cap = want;
    return 0;
}
void release(Buf& b) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; }
void release(Pin& b) { if (b.p) cudaFreeHost(b.p); b.p = nullptr; b.cap = 0; }

template <class T> T* P(Buf& b) { return (T*)b.p; }

// ------------------------------------------------------------ device stages
// The call record of every candidate (csrc/call.cuh): a thread per candidate, reading the allele table, the
// probabilities, the reference window and the reads' sequence pool where stage B left them.
__global__ void __launch_bounds__(128) k_call(const Dev d, const float* __restrict__ probs, int64_t n, c3r_call* __restrict__ out) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        c3rcall::CallIn c;
        c.e = reinterpret_cast<const c3r_alt_entry*>(d.alt) + d.alt_off[i];
        c.n = d.alt_n[i];
        c.probs = probs + 24 * i;
        c.ref = d.ref;
        c.ref_len = d.ref_len;
        c.p0 = (int64_t)d.cand_pos[i] - (d.ref_start0 + 1);
        c.seq = d.seq;
        c3r_call r;
        c3rcall::decide_call(c, r);
        out[i] = r;
    }
}
static_assert(sizeof(AltEntry) == sizeof(c3r_alt_entry), "AltEntry mirrors c3r_alt_entry");

// Stage A: everything up to the candidate list.  Needs only the resident inputs.
int run_stage_a(c3r_ctx* ctx, Slot& s) {
    Dev& d = s.d;
    cudaStream_t st = s.st_a;
    int& L = s.launches;
    // clear accumulators
    CK(cudaMemsetAsync(s.covA.p, 0, s.zero_bytes, st));      // covA | covE | their summary levels | blockmax: one pool, one memset
    CK(cudaMemsetAsync(s.scalars.p, 0, 64, st));
    CK(cudaEventRecord(s.ev[1], st));
    if (d.n_reads > 0) {
        // a warp per read, 8 lanes when reads carry few ops (the group walks a read's ops G at a time)
        static const int force_g = getenv("C3R_CIGAR_G") ? atoi(getenv("C3R_CIGAR_G")) : 0;
        const int64_t avg = d.n_ops / d.n_reads;
        const int G = force_g ? force_g : avg >= 16 ? 32 : 8;     // measured at config 2 (34 ops per read): 28.5 us with 32 lanes, 32.3 with 8
        if (G == 32) k_cigar<32><<<(unsigned)((d.n_reads * 32 + 255) / 256), 256, 0, st>>>(d);
        else if (G == 16) k_cigar<16><<<(unsigned)((d.n_reads * 16 + 255) / 256), 256, 0, st>>>(d);
        else k_cigar<8><<<(unsigned)((d.n_reads * 8 + 255) / 256), 256, 0, st>>>(d);
        ++L;
    }
    if (d.n_known > 0) { k_mark_known<<<(unsigned)((d.n_known + 255) / 256), 256, 0, st>>>(d); ++L; }
    const unsigned ptiles = (unsigned)((d.NW + PT_WORDS - 1) / PT_WORDS);
    k_row_bits<<<ptiles, 256, 0, st>>>(d); ++L;
    if (d.n_pbed >= 0) { k_bed_mask<<<(unsigned)((d.NW + 4 + 255) / 256), 256, 0, st>>>(d, (uint32_t*)s.covP.p); ++L; }
    if (d.head_tail) {
        k_last_col<<<(unsigned)((d.NW + 255) / 256), 256, 0, st>>>(d);
        k_last_gap<<<(unsigned)((d.NW + 255) / 256), 256, 0, st>>>(d);
        L += 2;
    }
    k_row_rank<<<ptiles, 256, 0, st>>>(d); ++L;
    CK(cudaEventRecord(s.ev[2], st));
    if (d.n_ops > 0) {
        const int64_t chunks = (d.n_ops + CMP_THREADS - 1) / CMP_THREADS;
        const int64_t cap = (int64_t)ctx->sm_count * 6;
        k_cmp<<<(unsigned)(chunks < cap ? chunks : cap), CMP_THREADS, 0, st>>>(d);
        ++L;
    }
    if (d.padding) { OpSkip op; op.d = d; L += device_scan(op, d.L_ub, s.scan, s.scan_epoch, (Int2*)nullptr, st); }
    { OpEvents op; op.d = d; L += device_scan(op, d.L_ub + 1, s.scan, s.scan_epoch, (int32_t*)nullptr, st); }
    if (d.C == 18) k_scatter_aggr<4><<<(unsigned)(ctx->sm_count * 8 + 1), 1024, 0, st>>>(d);
    else k_scatter_aggr<6><<<(unsigned)(ctx->sm_count * 8 + 1), 1024, 0, st>>>(d);
    ++L;
    CK(cudaEventRecord(s.ev[3], st));
    int64_t nb = (d.L_ub + COV_TILE - 1) / COV_TILE;
    {
        const int64_t res = (int64_t)ctx->sm_count * (d.C == 30 ? 4 : 5);      // resident blocks: tiles come from a counter
        const unsigned grid = (unsigned)(nb < res ? nb : res);
        if (d.C == 18) k_rows<18><<<grid, ROWS_WARPS * 32, 0, st>>>(d);
        else k_rows<30><<<grid, ROWS_WARPS * 32, 0, st>>>(d);
        ++L;
    }
    CK(cudaEventRecord(s.ev[4], st));
    k_cand_emit<<<(unsigned)(nb < ctx->sm_count * 16 ? nb : ctx->sm_count * 16), 256, 0, st>>>(d); ++L;
    CK(cudaEventRecord(s.ev[5], st));
    CK(cudaGetLastError());
    return 0;
}

// the scalars of stage A are on the host: check them
int parse_scalars(c3r_ctx* ctx, Slot& s) {
    const int64_t* hs = (const int64_t*)s.h_scalars.p;
    s.n_rows = hs[0];
    s.n_cand = hs[1];
    const int32_t err = ((const int32_t*)s.h_scalars.p)[6];
    if (err == 7)
        return fail(ctx, C3R_ERR_CAPACITY, "a position is covered by more than 8000 reads: samtools mpileup (the reference's "
                                           "column source) caps the depth there and drops reads; this chunk is refused "
                                           "rather than called on different counts");
    if (err) {
        char b[128];
        snprintf(b, sizeof b, "device capacity check failed (code %d): rows=%lld cand=%lld", err, (long long)s.n_rows, (long long)s.n_cand);
        return fail(ctx, C3R_ERR_CAPACITY, b);
    }
    if (s.n_cand > s.d.cand_cap) return fail(ctx, C3R_ERR_CAPACITY, "candidate capacity exceeded");
    return 0;
}

int read_scalars(c3r_ctx* ctx, Slot& s) {
    CK(cudaMemcpyAsync(s.h_scalars.p, s.scalars.p, 64, cudaMemcpyDeviceToHost, s.st_a));
    CK(cudaStreamSynchronize(s.st_a));                // stage A is complete: stage B (on s.st) may be queued without an event
    return parse_scalars(ctx, s);
}

int ensure_stage_b(c3r_ctx* ctx, Slot& s) {
    Dev& d = s.d;
    const int64_t n = s.n_cand > 0 ? s.n_cand : 1;
    const int per = WIN * d.C;
    // the window goes straight into the network's operand images unless the tensor itself is wanted (keep_tensor),
    // the padding pass has to patch it first, or the fp32 network (which reads the int32 tensor) runs
    s.fused_window = ctx->prm.nn_impl == 1 && !ctx->prm.keep_tensor && !d.padding && getenv("C3R_NO_FUSED_WINDOW") == nullptr;
    if (s.fused_window) {
        const size_t tiles = (size_t)((n + 255) / 256) * 2;
        if (ensure(ctx, s.xop, tiles * WIN * (size_t)(lstm1_kx(d.C) * 128) * 2)) return C3R_ERR_CUDA;
    } else if (ensure(ctx, s.tensor, (size_t)n * per * 4)) return C3R_ERR_CUDA;
    if (ensure(ctx, s.alt_off, (size_t)(n + 1) * 8)) return C3R_ERR_CUDA;
    if (ensure(ctx, s.alt_n, (size_t)n * 4)) return C3R_ERR_CUDA;
    d.alt_cap = 4 * n + d.events_ub + 8;
    if (ensure(ctx, s.alt, (size_t)d.alt_cap * sizeof(AltEntry))) return C3R_ERR_CUDA;
    if (ensure(ctx, s.probs, (size_t)n * 24 * 4)) return C3R_ERR_CUDA;
    if ((s.calls || s.vcf) && ensure(ctx, s.d_calls, (size_t)n * sizeof(c3r_call))) return C3R_ERR_CUDA;
    if (s.vcf) {
        s.vcf_row_max = c3rvcf::row_max((int64_t)s.vcf_contig.size());
        if (ensure(ctx, s.d_vlen, (size_t)n * 4) || ensure(ctx, s.d_voff, (size_t)n * 8) ||
            ensure(ctx, s.d_text, (size_t)n * s.vcf_row_max + 16) || ensure(ctx, s.d_contig, s.vcf_contig.size() + 1))
            return C3R_ERR_CUDA;
    }
    d.tensor = P<int32_t>(s.tensor);
    d.alt_off = P<int64_t>(s.alt_off);
    d.alt_n = P<int32_t>(s.alt_n);
    d.alt = P<AltEntry>(s.alt);
    return 0;
}

int nn_forward(c3r_ctx* ctx, const int32_t* tensor_dev, int64_t n, float* probs_dev, cudaStream_t st, int* launches,
               const __half* xop_ready = nullptr);

// Stage B: windows, padding, alt_info, network.  Needs n_cand on the host.
int run_stage_b(c3r_ctx* ctx, Slot& s) {
    Dev& d = s.d;
    cudaStream_t st = s.st;
    int& L = s.launches;
    const int64_t n = s.n_cand;
    if (n > 0) {
        const unsigned grid = (unsigned)(n < ctx->sm_count * 16 ? n : ctx->sm_count * 16);
        if (s.fused_window) {
            const int64_t wb = ((n + 255) / 256) * 2 * WIN;                // (tile, window row) blocks
            const unsigned gx = (unsigned)(wb < (int64_t)ctx->sm_count * 32 ? wb : (int64_t)ctx->sm_count * 32);
            if (d.C == 18) k_window_xop<18, lstm1_kx(18)><<<gx, 128, 0, st>>>(d, P<__half>(s.xop));
            else k_window_xop<30, lstm1_kx(30)><<<gx, 128, 0, st>>>(d, P<__half>(s.xop));
        } else k_window<<<grid, 128, 0, st>>>(d, d.padding ? 0 : 1);
        ++L;
        if (d.padding) {
            k_padding<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(d); ++L;
            k_rescale<<<grid, 128, 0, st>>>(d); ++L;
        }
        { OpAltOff op; op.d = d; L += device_scan(op, n, s.scan, s.scan_epoch, ((long long*)s.scalars.p) + 2, st); }
        k_altinfo<<<(unsigned)((n + 7) / 8), 256, 0, st>>>(d); ++L;
    }
    CK(cudaEventRecord(s.ev[6], st));
    CK(cudaEventRecord(s.ev_alt, st));
    if (n > 0) {
        int nl = 0;
        int rc = nn_forward(ctx, d.tensor, n, P<float>(s.probs), st, &nl, s.fused_window ? P<__half>(s.xop) : nullptr);
        if (rc) return rc;
        L += nl;
    }
    CK(cudaEventRecord(s.ev[7], st));
    if (s.calls || s.vcf) {
        CK(cudaEventRecord(s.ev_call[0], st));
        if (n > 0) {
            const int64_t blocks = (n + 127) / 128;
            k_call<<<(unsigned)(blocks < ctx->sm_count * 16 ? blocks : ctx->sm_count * 16), 128, 0, st>>>(d, P<float>(s.probs), n, P<c3r_call>(s.d_calls));
            ++L;
        }
        CK(cudaEventRecord(s.ev_call[1], st));
    }
    if (s.vcf) {
        CK(cudaEventRecord(s.ev_vcf[0], st));
        if (n > 0) {
            CK(cudaMemcpyAsync(s.d_contig.p, s.vcf_contig.data(), s.vcf_contig.size(), cudaMemcpyHostToDevice, st));
            c3rvcf::DevRows r;
            r.f.contig = P<char>(s.d_contig);
            r.f.contig_len = (int32_t)s.vcf_contig.size();
            r.f.q_min = s.vcf_q_min;
            r.f.ref = d.ref;
            r.f.ref_start1 = d.ref_start0 + 1;
            r.f.seq = d.seq;
            r.f.show_ref = s.vcf_show_ref;
            memcpy(r.f.nan_text, ctx->nan_text, 8);
            memcpy(r.f.ninf_text, ctx->ninf_text, 8);
            r.calls = P<c3r_call>(s.d_calls);
            r.pos = d.cand_pos;
            r.depth = d.cand_depth;
            r.n = n;
            r.qtab = P<float>(ctx->vcf_qtab);
            r.q_n = ctx->vcf_q_n;
            r.len = P<int32_t>(s.d_vlen);
            r.off = P<long long>(s.d_voff);
            r.out = P<char>(s.d_text);
            const int64_t blocks = (n + 127) / 128;
            c3rvcf::k_vcf_len<<<(unsigned)(blocks < ctx->sm_count * 16 ? blocks : ctx->sm_count * 16), 128, 0, st>>>(r);
            c3rvcf::OpVcfOff op;
            op.len = r.len; op.off = r.off; op.n = n;
            L += 1 + device_scan(op, n, s.scan, s.scan_epoch, (c3rvcf::VcfTotals*)(P<long long>(s.scalars) + 8), st);
            const int64_t tiles = (n + c3rvcf::VCF_TILE - 1) / c3rvcf::VCF_TILE;
            c3rvcf::k_vcf_write<<<(unsigned)(tiles < ctx->sm_count * 32 ? tiles : ctx->sm_count * 32), c3rvcf::VCF_TILE,
                                  c3rvcf::vcf_write_smem(s.vcf_row_max), st>>>(r, s.vcf_row_max);
            ++L;
        }
        CK(cudaEventRecord(s.ev_vcf[1], st));
    }
    CK(cudaGetLastError());
    return 0;
}

int queue_d2h(c3r_ctx* ctx, Slot& s) {
    Dev& d = s.d;
    cudaStream_t st = s.st;
    const int64_t n = s.n_cand;
    const int per = WIN * d.C;
    // alt total (and the text totals): a second tiny readback, taken before the network so it overlaps it
    CK(cudaMemcpyAsync(s.h_scalars.p, s.scalars.p, s.vcf ? 80 : 64, cudaMemcpyDeviceToHost, st));
    if (n > 0) {
        if (ensure_pin(ctx, s.h_pos, n * 4) || ensure_pin(ctx, s.h_depth, n * 4) || ensure_pin(ctx, s.h_probs, n * 96) ||
            ensure_pin(ctx, s.h_alt_off, n * 8) || ensure_pin(ctx, s.h_alt_n, n * 4)) return C3R_ERR_CUDA;
        CK(cudaMemcpyAsync(s.h_pos.p, s.cand_pos.p, n * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(s.h_depth.p, s.cand_depth.p, n * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(s.h_probs.p, s.probs.p, n * 96, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(s.h_alt_off.p, s.alt_off.p, n * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(s.h_alt_n.p, s.alt_n.p, n * 4, cudaMemcpyDeviceToHost, st));
        if (s.calls) {
            if (ensure_pin(ctx, s.h_calls, (size_t)n * sizeof(c3r_call))) return C3R_ERR_CUDA;
            CK(cudaMemcpyAsync(s.h_calls.p, s.d_calls.p, (size_t)n * sizeof(c3r_call), cudaMemcpyDeviceToHost, st));
        }
        if (s.vcf) {                                 // the bound: the size of a copy is fixed when it is queued
            const size_t bound = (size_t)n * s.vcf_row_max;
            if (ensure_pin(ctx, s.h_text, bound)) return C3R_ERR_CUDA;
            CK(cudaMemcpyAsync(s.h_text.p, s.d_text.p, bound, cudaMemcpyDeviceToHost, st));
        }
        if (ctx->prm.keep_tensor) {
            if (ensure_pin(ctx, s.h_tensor, (size_t)n * per * 4)) return C3R_ERR_CUDA;
            CK(cudaMemcpyAsync(s.h_tensor.p, s.tensor.p, (size_t)n * per * 4, cudaMemcpyDeviceToHost, st));
        }
    }
    if (ctx->prm.keep_rows && s.n_rows > 0) {
        const int64_t L = s.n_rows;
        if (ensure_pin(ctx, s.h_row_pos, L * 4) || ensure_pin(ctx, s.h_counts, (size_t)L * d.C * 4) ||
            ensure_pin(ctx, s.h_row_depth, L * 4)) return C3R_ERR_CUDA;
        CK(cudaMemcpyAsync(s.h_row_pos.p, s.row_pos.p, L * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(s.h_counts.p, s.counts.p, (size_t)L * d.C * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(s.h_row_depth.p, s.row_depth.p, L * 4, cudaMemcpyDeviceToHost, st));
    }
    return 0;
}

int build_net(c3r_ctx* ctx, const std::map<std::string, std::pair<const float*, int64_t>>& w);

// bounded mbarrier waits in the tensor-core kernels report protocol failures here
int check_tc(c3r_ctx* ctx, cudaStream_t st) {
    if (!ctx->tc_dirty) return 0;
    ctx->tc_dirty = false;
    int code = 0;
    if (tc_check_error(ctx->tc, st, &code)) return fail(ctx, C3R_ERR_CUDA, "could not read the tensor-core error word");
    if (code) {
        char b[96];
        snprintf(b, sizeof b, "tensor-core kernel synchronisation timed out (wait site %d)", code);
        return fail(ctx, C3R_ERR_CUDA, b);
    }
    return 0;
}

}  // namespace

// =============================================================== C ABI
extern "C" {

int c3r_abi_version(void) { return C3R_ABI_VERSION; }

void c3r_default_params(c3r_params* p) {
    memset(p, 0, sizeof *p);
    p->channels = 18;
    p->min_coverage = 4;
    p->min_mq = 5;
    p->excl_flags = 2316;
    p->snp_min_af = 0.08;
    p->indel_min_af = 0.15;
    p->enable_padding = 0;
    p->max_depth = 144;
    p->skip_proportion = 0.2;
    p->nn_impl = 1;
    p->keep_tensor = 0;
    p->keep_rows = 0;
    p->enable_head_tail = 0;
}

int c3r_create(c3r_ctx** out, int device_ordinal, const c3r_params* params) {
    if (!out || !params) return C3R_ERR_ARG;
    *out = nullptr;
    if (params->channels != 18 && params->channels != 30) return C3R_ERR_ARG;
    c3r_ctx* ctx = new c3r_ctx();
    ctx->device = device_ordinal;
    ctx->prm = *params;
    *out = ctx;                       // returned even on failure so the caller can read last_error
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev <= 0)
        return fail(ctx, C3R_ERR_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e) + " (there is no CPU fallback)");
    if (device_ordinal < 0 || device_ordinal >= n_dev) return fail(ctx, C3R_ERR_ARG, "device ordinal out of range");
    CK(cudaSetDevice(device_ordinal));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device_ordinal));
    if (prop.major != 10)
        return fail(ctx, C3R_ERR_CUDA, std::string("built for sm_100a only, device is ") + prop.name);
    ctx->sm_count = prop.multiProcessorCount;
    // Two streams per ticket: the network passes (stage B) on high-priority streams, the H2D copies and integer stages
    // of the tickets ahead (stage A) on low-priority ones - when SMs free up between the network's kernels, the next
    // network kernel goes first and the integer kernels take what is left.  C3R_ONE_STREAM: both on one stream.
    int prio_lo = 0, prio_hi = 0;
    CK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    if (getenv("C3R_FLAT_PRIORITY")) prio_hi = prio_lo;
    ctx->prio_hi = prio_hi;
    for (int i = 0; i < N_SLOTS; ++i) {
        Slot& s = ctx->slots[i];
        CK(cudaStreamCreateWithPriority(&s.st, cudaStreamNonBlocking, prio_hi));
        CK(cudaStreamCreateWithPriority(&s.st_a, cudaStreamNonBlocking, prio_lo));
        for (int k = 0; k < N_EV; ++k) CK(cudaEventCreate(&s.ev[k]));
        CK(cudaEventCreateWithFlags(&s.ev_alt, cudaEventDisableTiming));
        for (int k = 0; k < 2; ++k) CK(cudaEventCreate(&s.ev_call[k]));
        for (int k = 0; k < 2; ++k) CK(cudaEventCreate(&s.ev_vcf[k]));
        // spin-wait by default: a blocking-sync event wakes the waiting thread ~0.3 ms late (measured), which delays
        // stage B by as much; C3R_BLOCKING_COUNTS trades that for an idle core while waiting
        CK(cudaEventCreateWithFlags(&s.ev_cnt, cudaEventDisableTiming | (getenv("C3R_BLOCKING_COUNTS") ? cudaEventBlockingSync : 0)));
        CK(cudaEventCreateWithFlags(&s.ev_parse, cudaEventDisableTiming | (getenv("C3R_BLOCKING_COUNTS") ? cudaEventBlockingSync : 0)));
        for (int k = 0; k < 6; ++k) CK(cudaEventCreate(&s.ev_bam[k]));
        if (ensure(ctx, s.scalars, 256)) return C3R_ERR_CUDA;
        if (ensure_pin(ctx, s.h_scalars, 256)) return C3R_ERR_CUDA;
    }
    CK(cudaStreamCreateWithFlags(&ctx->fwd_stream, cudaStreamNonBlocking));
    if (ensure(ctx, ctx->thr, 2 * THR_N * sizeof(uint16_t))) return C3R_ERR_CUDA;
    k_thr_table<<<(THR_N + 255) / 256, 256>>>((uint16_t*)ctx->thr.p, (uint16_t*)ctx->thr.p + THR_N, params->snp_min_af, params->indel_min_af);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    return C3R_OK;
}

void c3r_destroy(c3r_ctx* ctx) {
    if (!ctx) return;
    if (getenv("C3R_TIMING") && ctx->tc.pipe)
        fprintf(stderr, "[c3r] %ld network passes, %ld with LSTM1 in pieces beside the previous pass\n", ctx->tc.pipe->n_pass, ctx->tc.pipe->n_overlap);
    if (getenv("C3R_TIMING") && ctx->n_submit)
        fprintf(stderr, "[c3r] %lld submits, host ms each: buffers %.3f, h2d calls %.3f, stage A launches %.3f, earlier "
                        "tickets advanced at submit %.3f, deferred part (wait for the counts + stage B + d2h calls) %.3f, - %.3f\n", (long long)ctx->n_submit,
                1e3 * ctx->t_phase[0] / ctx->n_submit, 1e3 * ctx->t_phase[1] / ctx->n_submit, 1e3 * ctx->t_phase[2] / ctx->n_submit,
                1e3 * ctx->t_phase[3] / ctx->n_submit, 1e3 * ctx->t_phase[4] / ctx->n_submit, 1e3 * ctx->t_phase[5] / ctx->n_submit);
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->nn_done) cudaEventDestroy(ctx->nn_done);
    for (int i = 0; i < N_SLOTS; ++i) {
        Slot& s = ctx->slots[i];
        Buf* bs[] = {&s.pos, &s.flag, &s.mapq, &s.hp, &s.cigar_off, &s.cigar, &s.seq_off, &s.seq, &s.ref, &s.admit,
                     &s.read_end, &s.op_x, &s.op_y, &s.op_info, &s.blockmax, &s.covA, &s.covE, &s.rowR, &s.cov_up, &s.ptile, &s.ctile, &s.csuper,
                     &s.word_base, &s.row_pos, &s.counts, &s.row_depth, &s.row_flag, &s.head_cnt, &s.tail_cnt,
                     &s.skipdiff, &s.max_skip, &s.row_ins, &s.row_del, &s.binc, &s.bin_cur, &s.events, &s.raw, &s.cov, &s.cov_tile, &s.refnib,
                     &s.cand_row, &s.cand_pos, &s.cand_depth, &s.tensor, &s.alt_off, &s.alt_n, &s.alt, &s.cur_ref,
                     &s.deleted, &s.probs, &s.scalars, &s.scan_scratch, &s.pbed, &s.cbed, &s.known, &s.covP, &s.xop, &s.d_calls,
                     &s.b_cdata, &s.b_blk, &s.b_win, &s.b_ubuf, &s.b_nrec, &s.b_soff, &s.b_scls, &s.b_skey, &s.b_snops, &s.b_snb,
                     &s.b_sdst, &s.b_sc, &s.d_vlen, &s.d_voff, &s.d_text, &s.d_contig};
        for (Buf* b : bs) release(*b);
        Pin* ps[] = {&s.h_scalars, &s.h_pos, &s.h_depth, &s.h_probs, &s.h_alt_off, &s.h_alt_n, &s.h_alt, &s.h_tensor,
                     &s.h_row_pos, &s.h_counts, &s.h_row_depth, &s.h_calls, &s.h_fsc, &s.h_rpos, &s.h_rflag, &s.h_rmapq,
                     &s.h_rhp, &s.h_rcoff, &s.h_rcig, &s.h_rsoff, &s.h_rseq, &s.h_text};
        for (Pin* b : ps) release(*b);
        for (int k = 0; k < N_EV; ++k) if (s.ev[k]) cudaEventDestroy(s.ev[k]);
        if (s.ev_alt) cudaEventDestroy(s.ev_alt);
        for (int k = 0; k < 2; ++k) if (s.ev_call[k]) cudaEventDestroy(s.ev_call[k]);
        for (int k = 0; k < 2; ++k) if (s.ev_vcf[k]) cudaEventDestroy(s.ev_vcf[k]);
        if (s.ev_cnt) cudaEventDestroy(s.ev_cnt);
        if (s.ev_parse) cudaEventDestroy(s.ev_parse);
        for (int k = 0; k < 6; ++k) if (s.ev_bam[k]) cudaEventDestroy(s.ev_bam[k]);
        if (s.st) cudaStreamDestroy(s.st);
        if (s.st_a) cudaStreamDestroy(s.st_a);
    }
    release(ctx->wbuf);
    release(ctx->nn_scratch);
    release(ctx->fwd_in);
    release(ctx->ref_res);
    release(ctx->refnib_res);
    release(ctx->thr);
    release(ctx->vcf_qtab);
    release(ctx->fwd_out);
    tc_release(ctx->tc);
    if (ctx->fwd_stream) cudaStreamDestroy(ctx->fwd_stream);
    delete ctx;
}

int c3r_host_alloc(void** out, int64_t n_bytes) {
    if (!out || n_bytes <= 0) return C3R_ERR_ARG;
    *out = nullptr;
    return cudaHostAlloc(out, (size_t)n_bytes, cudaHostAllocPortable) == cudaSuccess ? C3R_OK : C3R_ERR_CUDA;
}
void c3r_host_free(void* p) { if (p) cudaFreeHost(p); }

const char* c3r_last_error(c3r_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int c3r_set_weights(c3r_ctx* ctx, const c3r_weight_view* views, int n_views) {
    if (!ctx || !views) return C3R_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    std::map<std::string, std::pair<const float*, int64_t>> w;
    for (int i = 0; i < n_views; ++i) w[views[i].name] = std::make_pair(views[i].data, views[i].n_elem);
    return build_net(ctx, w);
}

int c3r_set_reference(c3r_ctx* ctx, const uint8_t* ref, int64_t ref_start1, int64_t ref_len) {
    if (!ctx || !ref || ref_len <= 0 || ref_start1 < 1) return C3R_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaDeviceSynchronize());
    if (ensure(ctx, ctx->ref_res, (size_t)ref_len + 16)) return C3R_ERR_CUDA;
    CK(cudaMemcpy(ctx->ref_res.p, ref, (size_t)ref_len, cudaMemcpyHostToDevice));
    ctx->ref_res_start0 = ref_start1 - 1;
    ctx->ref_res_len = ref_len;
    const int64_t nw = (ref_len + 7) / 8;
    if (ensure(ctx, ctx->refnib_res, (size_t)nw * 4)) return C3R_ERR_CUDA;
    k_refnib<<<(unsigned)((nw + 255) / 256), 256>>>((const uint8_t*)ctx->ref_res.p, ref_len, (uint32_t*)ctx->refnib_res.p, nw);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    return C3R_OK;
}

static void advance_all(c3r_ctx* ctx, bool block, uint64_t block_upto = ~0ull);
static int submit_once(c3r_ctx* ctx, const c3r_reads* rd, const uint8_t* ref, int64_t ref_start1, int64_t ref_len,
                       int64_t region_start1, int64_t region_end1, c3r_ticket* ticket);

// sorted, disjoint, non-touching intervals / strictly increasing sites: the device searches them by bisection
static int check_filter(c3r_ctx* ctx, const c3r_site_filter* f) {
    if (!f) return 0;
    const struct { const int32_t* iv; int64_t n; const char* what; } beds[2] = {
        {f->pileup_bed, f->n_pileup_bed, "pileup_bed"}, {f->confident_bed, f->n_confident_bed, "confident_bed"}};
    for (const auto& b : beds) {
        if (b.n > 0 && !b.iv) return fail(ctx, C3R_ERR_ARG, "site filter: interval count without intervals");
        if (b.n > 0x3fffffff) return fail(ctx, C3R_ERR_CAPACITY, "site filter: too many intervals");
        for (int64_t k = 0; k < b.n; ++k) {
            if (b.iv[2 * k] < 0 || b.iv[2 * k + 1] <= b.iv[2 * k] || (k && b.iv[2 * k] <= b.iv[2 * k - 1])) {
                char m[128];
                snprintf(m, sizeof m, "site filter: %s must be sorted, non-empty, disjoint and non-touching (interval %lld)", b.what, (long long)k);
                return fail(ctx, C3R_ERR_ARG, m);
            }
        }
    }
    if (f->n_known_sites > 0 && !f->known_sites) return fail(ctx, C3R_ERR_ARG, "site filter: site count without sites");
    if (f->n_known_sites > 0x7fffffff) return fail(ctx, C3R_ERR_CAPACITY, "site filter: too many sites");
    for (int64_t k = 1; k < f->n_known_sites; ++k)
        if (f->known_sites[k] <= f->known_sites[k - 1]) return fail(ctx, C3R_ERR_ARG, "site filter: known_sites must be strictly increasing");
    return 0;
}

int c3r_submit_chunk(c3r_ctx* ctx, const c3r_reads* rd, const uint8_t* ref, int64_t ref_start1, int64_t ref_len,
                     int64_t region_start1, int64_t region_end1, c3r_ticket* ticket) {
    return c3r_submit_chunk_filtered(ctx, rd, ref, ref_start1, ref_len, region_start1, region_end1, nullptr, ticket);
}

int c3r_submit_chunk_filtered(c3r_ctx* ctx, const c3r_reads* rd, const uint8_t* ref, int64_t ref_start1, int64_t ref_len,
                              int64_t region_start1, int64_t region_end1, const c3r_site_filter* filter,
                              c3r_ticket* ticket) {
    if (!ctx || !rd || !ticket) return C3R_ERR_ARG;
    if (int rc = check_filter(ctx, filter)) return rc;
    ctx->filter = filter;
    int rc = submit_once(ctx, rd, ref, ref_start1, ref_len, region_start1, region_end1, ticket);
    ctx->filter = nullptr;
    return rc;
}

// Row-space capacity of a slot and everything sized by it.  Rows = positions under an M/=/X/D op, dilated by 16 on
// each side of every N-separated block: a read contributes at most (its M/D length + 32 per block).  Without
// `cigar_host` the bounds are cheap ones that need no host pass over the CIGARs (M bases <= SEQ bases; deletions are
// assumed not to outnumber the sequenced bases; row events - indel tokens + read bases that differ from the
// reference - sized for one base in four); if a chunk breaks that, the device-side capacity checks fire and
// advance() comes back here with the CIGARs for exact bounds (events then sized for every base).
// The slot's scan state (scan.cuh), sized for scans of up to n elements.  Every scan of a slot uses the same layout
// (aggregates of SCAN_ELEM bytes): the status words of one layout must never lie over the aggregates of another.
constexpr size_t SCAN_ELEM = 32;
static_assert(sizeof(ScanElem) <= SCAN_ELEM && sizeof(c3rbgzf::Slot3) <= SCAN_ELEM && sizeof(c3rvcf::VcfTotals) <= SCAN_ELEM,
              "scan aggregates fit the layout");
static int ensure_scan(c3r_ctx* ctx, Slot& s, int64_t n) {
    const size_t elem = SCAN_ELEM;
    // scan state: 256 B of counters, then per tile a status word, an aggregate and an inclusive prefix
    const size_t tiles = (size_t)(n / SCAN_TILE + 2);
    const size_t need = 256 + tiles * 4 + 2 * tiles * elem + 64;
    if (s.scan_scratch.cap < need) {
        if (ensure(ctx, s.scan_scratch, need)) return C3R_ERR_CUDA;
        CK(cudaMemsetAsync(s.scan_scratch.p, 0, s.scan_scratch.cap, s.st_a));   // status words of epoch 0, ticket 0
    }
    uint8_t* sp = (uint8_t*)s.scan_scratch.p;
    const size_t cap_tiles = (s.scan_scratch.cap - 256 - 64) / (4 + 2 * elem);
    s.scan.ctrl = (unsigned int*)sp;
    s.scan.status = (uint32_t*)(sp + 256);
    s.scan.aggr = sp + 256 + ((cap_tiles * 4 + 15) / 16) * 16;
    s.scan.incl = (uint8_t*)s.scan.aggr + cap_tiles * elem;
    s.scan.err = P<int32_t>(s.scalars) + 6;
    return 0;
}

static int size_rows(c3r_ctx* ctx, Slot& s, const uint32_t* cigar_host) {
    Dev& d = s.d;
    int64_t md_len = 0, n_skip = 0, ev_ub = 0;
    if (cigar_host) {
        for (int64_t k = 0; k < d.n_ops; ++k) {
            const uint32_t c = cigar_host[k], op = c & 15u;
            const int64_t len = c >> 4;
            if (op == 0 || op == 2 || op == 7 || op == 8) md_len += len;
            if (op == 3) ++n_skip;
        }
        ev_ub = d.n_ops + 2 * s.n_seq_bytes;
    } else {
        md_len = 4 * s.n_seq_bytes;
        n_skip = d.n_ops;
        ev_ub = d.n_ops + s.n_seq_bytes / 2;
    }
    int64_t L_ub = md_len + 32 * (n_skip + d.n_reads) + 64;
    L_ub += 33 * s.n_known_sites;                    // rows around known sites
    if (L_ub > d.W) L_ub = d.W;
    if (L_ub < 64) L_ub = 64;
    d.L_ub = L_ub;
    d.events_ub = ev_ub + 8;
    d.cand_cap = L_ub;
#define EN(b, bytes) if (ensure(ctx, s.b, (size_t)(bytes))) return C3R_ERR_CUDA
    EN(row_pos, (L_ub + 2) * 4); EN(counts, ((L_ub + 32) * d.C) * 4); EN(row_depth, (L_ub + 2) * 4); EN(row_flag, L_ub + 2);
    EN(head_cnt, (L_ub + 2) * 4); EN(tail_cnt, (L_ub + 2) * 4); EN(skipdiff, (L_ub + 2) * 8); EN(max_skip, (L_ub + 2) * 4);
    EN(row_ins, (L_ub + 2) * 4); EN(row_del, (L_ub + 2) * 4);
    EN(binc, (L_ub + 4) * 4); EN(bin_cur, (L_ub + 4) * 4);
    EN(events, d.events_ub * sizeof(RowEvent)); EN(raw, d.events_ub * sizeof(RowEvent));
    EN(cov, (L_ub + 4) * NCOV_MAX * 4); EN(cov_tile, (L_ub / COV_TILE + 4) * NCOV_MAX * 4);
    EN(ctile, (L_ub / COV_TILE + 4) * 4); EN(csuper, (L_ub / (64 * COV_TILE) + 4) * 4);
    EN(cand_row, (L_ub + 2) * 4); EN(cand_pos, (L_ub + 2) * 4); EN(cand_depth, (L_ub + 2) * 4);
    EN(cur_ref, (L_ub + 2) * 8); EN(deleted, L_ub + 2);
    {
        int64_t mx = d.n_ops > d.NW ? d.n_ops : d.NW;
        if (L_ub + 4 > mx) mx = L_ub + 4;
        if (int rc = ensure_scan(ctx, s, mx)) return rc;
    }
#undef EN
    d.row_pos = P<int32_t>(s.row_pos); d.counts = P<int32_t>(s.counts); d.row_depth = P<int32_t>(s.row_depth);
    d.row_flag = P<uint8_t>(s.row_flag); d.head_cnt = P<int32_t>(s.head_cnt); d.tail_cnt = P<int32_t>(s.tail_cnt);
    d.skipdiff = P<Int2>(s.skipdiff); d.max_skip = P<int32_t>(s.max_skip);
    d.row_inscnt = P<int32_t>(s.row_ins); d.row_delcnt = P<int32_t>(s.row_del);
    d.binc = P<int32_t>(s.binc); d.bin_cur = P<int32_t>(s.bin_cur);
    d.events = P<RowEvent>(s.events); d.raw = P<RowEvent>(s.raw); d.cov = P<int32_t>(s.cov); d.cov_tile = P<int32_t>(s.cov_tile);
    d.ctile = P<int32_t>(s.ctile); d.csuper = P<int32_t>(s.csuper);
    d.cand_row = P<int32_t>(s.cand_row); d.cand_pos = P<int32_t>(s.cand_pos); d.cand_depth = P<int32_t>(s.cand_depth);
    d.cur_ref = P<Int2>(s.cur_ref); d.deleted = P<uint8_t>(s.deleted);
    return 0;
}

// checks of a submit that need no reads; fills in the resident reference window when ref == NULL
static int check_submit(c3r_ctx* ctx, const uint8_t* ref, int64_t* ref_start1, int64_t* ref_len, int64_t region_start1,
                        int64_t region_end1) {
    if (!ref) {
        if (!ctx->ref_res_len) return fail(ctx, C3R_ERR_STATE, "ref == NULL but c3r_set_reference was never called");
        *ref_start1 = ctx->ref_res_start0 + 1;
        *ref_len = ctx->ref_res_len;
    }
    if (!ctx->have_weights) return fail(ctx, C3R_ERR_STATE, "c3r_set_weights must be called before c3r_submit_chunk");
    if (region_end1 < region_start1 || region_start1 < 1) return fail(ctx, C3R_ERR_ARG, "bad region");
    if (region_end1 > 0x7fff0000LL) return fail(ctx, C3R_ERR_CAPACITY, "positions must fit int32");
    return 0;
}

// the text options of the context, as the ticket in slot s is submitted
static void take_vcf(c3r_ctx* ctx, Slot& s) {
    s.vcf = ctx->vcf;
    s.vcf_show_ref = ctx->vcf_show_ref;
    s.vcf_q_min = ctx->vcf_q_min;
    s.vcf_contig = ctx->vcf_contig;
}

static int free_slot(c3r_ctx* ctx) {
    for (int i = 0; i < N_SLOTS; ++i) if (!ctx->slots[i].in_use) return i;
    return fail(ctx, C3R_ERR_STATE, "all tickets in flight; c3r_release one first");
}

static int queue_rec_write(c3r_ctx* ctx, Slot& s);

// Everything of a chunk from its reads onward: the slot's buffers sized from the read counts, the reads copied to
// the device (host reads) or written there by k_rec_write (a device fetch, reads_on_device), the filters and the
// reference, stage A and the copy of its counts.  The ticket is then pending_b.
static int queue_chunk(c3r_ctx* ctx, Slot& s, const c3r_reads* rd, bool reads_on_device, const uint8_t* ref,
                       int64_t ref_start1, int64_t ref_len, int64_t region_start1, int64_t region_end1,
                       const c3r_site_filter* flt) {
    if (rd->n_seq_bytes * 2 >= 0xffffffffLL) return fail(ctx, C3R_ERR_CAPACITY, "more than 4G bases in one chunk");
    if (rd->n_reads >= (1LL << 28)) return fail(ctx, C3R_ERR_CAPACITY, "more than 2^28 reads in one chunk");
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double tp = now();
    auto lap = [&](int k) { const double t = now(); ctx->t_phase[k] += t - tp; tp = t; };
    if (!reads_on_device) s.launches = 0;          // a device fetch counts its parse kernels too
    s.has_result = false;
    Dev& d = s.d;
    memset(&d, 0, sizeof d);
    const c3r_params& pr = ctx->prm;
    d.n_reads = rd->n_reads; d.n_ops = rd->n_ops;
    d.R0 = (int32_t)(region_start1 - 1); d.R1 = (int32_t)region_end1;
    d.W = (int64_t)d.R1 - d.R0; d.NW = (d.W + 31) / 32;
    d.C = pr.channels; d.min_cov = pr.min_coverage; d.min_mq = pr.min_mq; d.excl = pr.excl_flags;
    d.snp_af = pr.snp_min_af; d.indel_af = pr.indel_min_af; d.padding = pr.enable_padding;
    d.max_depth = pr.max_depth; d.skip_prop = pr.skip_proportion;
    d.dbg = getenv("C3R_DBG") ? atoi(getenv("C3R_DBG")) : 0;
    d.ref_start0 = ref_start1 - 1; d.ref_len = ref_len;
    d.thr_snp = (const uint16_t*)ctx->thr.p; d.thr_indel = (const uint16_t*)ctx->thr.p + THR_N;
    s.n_seq_bytes = rd->n_seq_bytes;
    s.n_known_sites = (flt && flt->n_known_sites > 0) ? flt->n_known_sites : 0;
    s.exact_bounds = false;
    s.deferred_rc = 0;
    const int64_t R = rd->n_reads > 0 ? rd->n_reads : 1, O = rd->n_ops > 0 ? rd->n_ops : 1;
#define EN(b, bytes) if (ensure(ctx, s.b, (size_t)(bytes))) return C3R_ERR_CUDA
    EN(pos, R * 4); EN(flag, R * 2); EN(mapq, R); EN(hp, R); EN(cigar_off, (R + 1) * 4); EN(cigar, O * 4);
    EN(seq_off, (R + 1) * 8); EN(seq, rd->n_seq_bytes + 64); if (ref) { EN(ref, ref_len + 16); }
    EN(admit, R); EN(read_end, R * 4); EN(op_x, O * 4); EN(op_y, O * 4); EN(op_info, O * 4);
    // position space: buffers padded to whole tiles of PT_WORDS words (k_row_bits / k_row_rank store 16 bytes per thread);
    // the summary levels of covA and covE (mark_range) share one buffer: level l has NW / 32^l + 2 words
    const int64_t NWp = ((d.NW + PT_WORDS - 1) / PT_WORDS) * PT_WORDS + 8;
    int64_t up_words[COV_UP], up_total = 0;
    { int64_t n = d.NW; for (int l = 0; l < COV_UP; ++l) { n = (n >> 5) + 2; up_words[l] = n; up_total += n; } }
    // everything a pass needs zeroed lives in ONE pool (one memset per pass instead of four): covA, covE, the summary
    // levels of both, blockmax
    const int64_t pool_words = 2 * NWp + 2 * up_total + (R / 256 + 2) + 16;
    EN(covA, pool_words * 4); EN(rowR, NWp * 4); EN(word_base, NWp * 4);
    s.zero_bytes = (size_t)pool_words * 4;
    EN(ptile, (NWp / PT_WORDS + 4) * 4);
    if (ref) { EN(refnib, ((ref_len + 7) / 8 + 1) * 4); }
    d.n_pbed = d.n_cbed = d.n_known = -1;
    if (flt) {
        if (flt->n_pileup_bed >= 0) { EN(pbed, (flt->n_pileup_bed + 1) * 8); EN(covP, (d.NW + 4) * 4); d.n_pbed = (int32_t)flt->n_pileup_bed; }
        if (flt->n_confident_bed >= 0) { EN(cbed, (flt->n_confident_bed + 1) * 8); d.n_cbed = (int32_t)flt->n_confident_bed; }
        if (flt->n_known_sites >= 0) { EN(known, (flt->n_known_sites + 1) * 4); d.n_known = (int32_t)flt->n_known_sites; }
    }
#undef EN
    d.pos = P<int32_t>(s.pos); d.flag = P<uint16_t>(s.flag); d.mapq = P<uint8_t>(s.mapq); d.hp = P<uint8_t>(s.hp);
    d.cigar_off = P<int32_t>(s.cigar_off); d.cigar = P<uint32_t>(s.cigar); d.seq_off = P<int64_t>(s.seq_off);
    d.seq = P<uint8_t>(s.seq); d.ref = ref ? P<uint8_t>(s.ref) : P<uint8_t>(ctx->ref_res);
    d.admit = P<uint8_t>(s.admit); d.read_end = P<int32_t>(s.read_end);
    d.op_x = P<int32_t>(s.op_x); d.op_y = P<uint32_t>(s.op_y); d.op_info = P<uint32_t>(s.op_info);
    d.covA = P<uint32_t>(s.covA); d.covE = d.covA + NWp; d.rowR = P<uint32_t>(s.rowR);
    d.word_base = P<int32_t>(s.word_base);
    {
        uint32_t* u = d.covE + NWp;
        for (int l = 0; l < COV_UP; ++l) { d.upA[l] = u; u += up_words[l]; }
        for (int l = 0; l < COV_UP; ++l) { d.upE[l] = u; u += up_words[l]; }
        d.blockmax = (int32_t*)u;
    }
    d.ptile = P<int32_t>(s.ptile); d.kctr = P<int32_t>(s.scalars) + 12;
    d.n_rows = P<int64_t>(s.scalars); d.n_cand = P<int64_t>(s.scalars) + 1; d.err = P<int32_t>(s.scalars) + 6;
    d.n_raw = P<int64_t>(s.scalars) + 5;
    if (int rc0 = size_rows(ctx, s, nullptr)) return rc0;     // row space: cheap capacity bounds first
    d.refnib = ref ? P<uint32_t>(s.refnib) : P<uint32_t>(ctx->refnib_res);
    d.n_ref_words = (ref_len + 7) / 8;
    d.pbed = P<int32_t>(s.pbed); d.cbed = P<int32_t>(s.cbed); d.known = P<int32_t>(s.known);
    d.covP = d.n_pbed >= 0 ? P<uint32_t>(s.covP) : d.covA;
    d.head_tail = pr.enable_head_tail;
    d.tail = P<int32_t>(s.scalars) + 8;

    cudaStream_t st = s.st_a;
    lap(0);
    if (reads_on_device) {
        if (int rc = queue_rec_write(ctx, s)) return rc;
    } else {
        CK(cudaEventRecord(s.ev[0], st));
        if (rd->n_reads > 0) {
            CK(cudaMemcpyAsync(s.pos.p, rd->pos, rd->n_reads * 4, cudaMemcpyHostToDevice, st));
            CK(cudaMemcpyAsync(s.flag.p, rd->flag, rd->n_reads * 2, cudaMemcpyHostToDevice, st));
            CK(cudaMemcpyAsync(s.mapq.p, rd->mapq, rd->n_reads, cudaMemcpyHostToDevice, st));
            CK(cudaMemcpyAsync(s.hp.p, rd->hp, rd->n_reads, cudaMemcpyHostToDevice, st));
            CK(cudaMemcpyAsync(s.cigar_off.p, rd->cigar_off, (rd->n_reads + 1) * 4, cudaMemcpyHostToDevice, st));
            CK(cudaMemcpyAsync(s.seq_off.p, rd->seq_off, (rd->n_reads + 1) * 8, cudaMemcpyHostToDevice, st));
        }
    }
    if (d.n_pbed > 0) CK(cudaMemcpyAsync(s.pbed.p, flt->pileup_bed, (size_t)d.n_pbed * 8, cudaMemcpyHostToDevice, st));
    if (d.n_cbed > 0) CK(cudaMemcpyAsync(s.cbed.p, flt->confident_bed, (size_t)d.n_cbed * 8, cudaMemcpyHostToDevice, st));
    if (d.n_known > 0) CK(cudaMemcpyAsync(s.known.p, flt->known_sites, (size_t)d.n_known * 4, cudaMemcpyHostToDevice, st));
    if (!reads_on_device) {
        if (rd->n_ops > 0) CK(cudaMemcpyAsync(s.cigar.p, rd->cigar, rd->n_ops * 4, cudaMemcpyHostToDevice, st));
        if (rd->n_seq_bytes > 0) CK(cudaMemcpyAsync(s.seq.p, rd->seq, rd->n_seq_bytes, cudaMemcpyHostToDevice, st));
    }
    if (ref && ref_len > 0) {
        CK(cudaMemcpyAsync(s.ref.p, ref, ref_len, cudaMemcpyHostToDevice, st));
        const int64_t nw = (ref_len + 7) / 8;
        k_refnib<<<(unsigned)((nw + 255) / 256), 256, 0, st>>>((const uint8_t*)s.ref.p, ref_len, (uint32_t*)s.refnib.p, nw);
        ++s.launches;
    }
    // The copies above overlap the network pass of the ticket before this one, and so do the position / row stages:
    // the network's partly filled rounds and its tail leave SMs idle that these ~20 short kernels take (9.66 M sites/s
    // end to end against 8.73 M when they wait for the pass to end).
    lap(1);
    int rc = run_stage_a(ctx, s);
    lap(2);
    // the counts of stage A travel to the host behind it; stage B is queued when they have arrived (advance)
    if (!rc) { cudaError_t e = cudaMemcpyAsync(s.h_scalars.p, s.scalars.p, 64, cudaMemcpyDeviceToHost, st); if (e != cudaSuccess) rc = fail(ctx, C3R_ERR_CUDA, cudaGetErrorString(e)); }
    if (!rc) { cudaError_t e = cudaEventRecord(s.ev_cnt, st); if (e != cudaSuccess) rc = fail(ctx, C3R_ERR_CUDA, cudaGetErrorString(e)); }
    if (rc) return rc;
    s.pending_b = true;
    return 0;
}

static int submit_once(c3r_ctx* ctx, const c3r_reads* rd, const uint8_t* ref, int64_t ref_start1, int64_t ref_len,
                       int64_t region_start1, int64_t region_end1, c3r_ticket* ticket) {
    if (int rc = check_submit(ctx, ref, &ref_start1, &ref_len, region_start1, region_end1)) return rc;
    CK(cudaSetDevice(ctx->device));
    ++ctx->n_submit;
    const int si = free_slot(ctx);
    if (si < 0) return si;
    Slot& s = ctx->slots[si];
    s.bam = false;
    s.pending_parse = false;
    s.calls = ctx->calls;
    take_vcf(ctx, s);
    int rc = queue_chunk(ctx, s, rd, false, ref, ref_start1, ref_len, region_start1, region_end1, ctx->filter);
    if (rc) { cudaStreamSynchronize(s.st_a); cudaStreamSynchronize(s.st); return rc; }
    s.in_use = true;
    s.order = ++ctx->submit_seq;
    *ticket = si;
    // tickets submitted earlier whose counts are in by now get their stage B queued here (never blocks)
    const auto t1 = std::chrono::steady_clock::now();
    advance_all(ctx, getenv("C3R_SYNC_SUBMIT") != nullptr);
    ctx->t_phase[3] += std::chrono::duration<double>(std::chrono::steady_clock::now() - t1).count();
    return C3R_OK;
}

// ------------------------------------------------------------ device BAM reading (csrc/bgzf.cuh)
static const char* fetch_err_text(int code) {
    switch (code) {
        case c3rbgzf::FE_INFLATE: return "BGZF inflate/CRC failure";
        case c3rbgzf::FE_HEADER: return "corrupt BGZF block header";
        case c3rbgzf::FE_BIG_BLOCK: return "BGZF block larger than 64 KiB";
        case c3rbgzf::FE_SHORT_READ: return "short read from the BAM";
        case c3rbgzf::FE_CROSS: return "record crosses the end of an index chunk";
        case c3rbgzf::FE_MALFORMED: return "malformed BAM record";
        default: return "malformed aux data in a BAM record";
    }
}

// the tables of a raw fetch come from outside the library: every offset is checked before the kernels use it
static int check_raw(c3r_ctx* ctx, const c3r_bam_raw* raw) {
    if (raw->n_windows < 0 || raw->n_blocks < 0 || raw->n_bytes < 0 || raw->n_ubytes < 0 ||
        (raw->n_bytes > 0 && !raw->data) || (raw->n_blocks > 0 && !raw->blocks) || (raw->n_windows > 0 && !raw->windows))
        return fail(ctx, C3R_ERR_ARG, "raw fetch: bad counts or null tables");
    if (raw->n_windows >= (1 << 20) || raw->n_ubytes >= (1LL << 40)) return fail(ctx, C3R_ERR_CAPACITY, "raw fetch too large");
    if (raw->beg < 0 || raw->end > (1LL << 31) || raw->tid < 0) return fail(ctx, C3R_ERR_ARG, "raw fetch: bad region");
    int64_t ub = 0, nb = 0;
    for (int32_t w = 0; w < raw->n_windows; ++w) {
        const c3r_bam_window& W = raw->windows[w];
        if (W.status) {
            if (W.status < c3rbgzf::FE_HEADER || W.status > c3rbgzf::FE_SHORT_READ || W.n_blocks != 0)
                return fail(ctx, C3R_ERR_ARG, "raw fetch: bad window status");
            continue;
        }
        if (W.ubase != ub || W.usize < 0 || W.ubeg < 0 || W.uend < 0 || W.first_block != nb || W.n_blocks < 0 ||
            W.n_blocks > raw->n_blocks - nb)
            return fail(ctx, C3R_ERR_ARG, "raw fetch: window table does not match its blocks");
        int64_t uo = W.ubase;
        for (int32_t k = 0; k < W.n_blocks; ++k) {
            const c3r_bgzf_block& B = raw->blocks[nb + k];
            if (B.window != w || B.uoff != uo || B.usize < 0 || B.usize > (int32_t)c3rbgzf::MAX_BLOCK || B.csize < 0 ||
                B.coff < 0 || B.coff > raw->n_bytes - B.csize)
                return fail(ctx, C3R_ERR_ARG, "raw fetch: block table out of bounds");
            uo += B.usize;
        }
        if (uo != W.ubase + W.usize) return fail(ctx, C3R_ERR_ARG, "raw fetch: window size does not match its blocks");
        ub += W.usize;
        nb += W.n_blocks;
    }
    if (nb != raw->n_blocks || ub != raw->n_ubytes) return fail(ctx, C3R_ERR_ARG, "raw fetch: tables do not add up");
    return 0;
}

int c3r_submit_bam_chunk(c3r_ctx* ctx, const c3r_bam_raw* raw, const uint8_t* ref, int64_t ref_start1, int64_t ref_len,
                         int64_t region_start1, int64_t region_end1, const c3r_site_filter* filter, c3r_ticket* ticket) {
    if (!ctx || !raw || !ticket) return C3R_ERR_ARG;
    if (int rc = check_filter(ctx, filter)) return rc;
    if (int rc = check_raw(ctx, raw)) return rc;
    if (int rc = check_submit(ctx, ref, &ref_start1, &ref_len, region_start1, region_end1)) return rc;
    CK(cudaSetDevice(ctx->device));
    const int si = free_slot(ctx);
    if (si < 0) return si;
    Slot& s = ctx->slots[si];
    s.bam = true;
    s.calls = ctx->calls;
    take_vcf(ctx, s);
    s.ref_host = ref; s.ref_start1 = ref_start1; s.ref_len = ref_len;
    s.region_start1 = region_start1; s.region_end1 = region_end1;
    // the filter is read during the call (as c3r_submit_chunk_filtered's): the slot keeps a copy for the deferred part
    s.has_filter = filter != nullptr;
    if (filter) {
        s.f_pbed.assign(filter->pileup_bed, filter->pileup_bed + (filter->n_pileup_bed > 0 ? 2 * filter->n_pileup_bed : 0));
        s.f_cbed.assign(filter->confident_bed, filter->confident_bed + (filter->n_confident_bed > 0 ? 2 * filter->n_confident_bed : 0));
        s.f_known.assign(filter->known_sites, filter->known_sites + (filter->n_known_sites > 0 ? filter->n_known_sites : 0));
        s.flt = *filter;
        s.flt.pileup_bed = s.f_pbed.data(); s.flt.confident_bed = s.f_cbed.data(); s.flt.known_sites = s.f_known.data();
    }
    // device windows and the record slot capacity: window w holds at most usize / 36 + 1 records (a record is at least
    // 36 bytes; the chain ends at a shorter one)
    const int32_t nw = raw->n_windows;
    std::vector<c3rbgzf::DevWindow> dw((size_t)(nw > 0 ? nw : 1));
    int64_t n_slots = 0;
    for (int32_t w = 0; w < nw; ++w) {
        const c3r_bam_window& W = raw->windows[w];
        c3rbgzf::DevWindow& x = dw[w];
        x.ubase = W.ubase; x.usize = W.usize; x.ubeg = W.ubeg; x.uend = W.uend;
        x.slot_base = n_slots; x.status = W.status; x.n_blocks = W.n_blocks;
        n_slots += W.usize / 36 + 1;
    }
    const int64_t NB = raw->n_blocks, S = n_slots > 0 ? n_slots : 1;
#define EN(b, bytes) if (ensure(ctx, s.b, (size_t)(bytes))) return C3R_ERR_CUDA
    EN(b_cdata, raw->n_bytes + 16); EN(b_blk, (NB + 1) * 32); EN(b_win, (size_t)(nw + 1) * sizeof(c3rbgzf::DevWindow));
    EN(b_ubuf, raw->n_ubytes + 64); EN(b_nrec, (nw + 1) * 4);
    EN(b_soff, S * 8); EN(b_scls, S); EN(b_skey, S * 8); EN(b_snops, S * 4); EN(b_snb, S * 8);
    EN(b_sdst, S * sizeof(c3rbgzf::Slot3)); EN(b_sc, sizeof(c3rbgzf::FetchSc));
#undef EN
    if (ensure_pin(ctx, s.h_fsc, sizeof(c3rbgzf::FetchSc))) return C3R_ERR_CUDA;
    if (int rc = ensure_scan(ctx, s, S)) return rc;
    // block table as columns
    std::vector<int64_t> bcol((size_t)(2 * NB + 1));
    std::vector<int32_t> icol((size_t)(3 * NB + 1));
    for (int64_t k = 0; k < NB; ++k) {
        const c3r_bgzf_block& B = raw->blocks[k];
        bcol[k] = B.coff; bcol[NB + k] = B.uoff;
        icol[k] = B.csize; icol[NB + k] = B.usize; icol[2 * NB + k] = B.window;
    }
    c3rbgzf::Fetch& f = s.fetch;
    f = c3rbgzf::Fetch{};
    f.tid = raw->tid; f.beg = raw->beg; f.end = raw->end; f.n_win = nw; f.n_slots = n_slots;
    f.cdata = P<uint8_t>(s.b_cdata);
    int64_t* b64 = P<int64_t>(s.b_blk);
    int32_t* b32 = (int32_t*)(b64 + 2 * NB);
    f.blk_coff = b64; f.blk_uoff = b64 + NB; f.blk_csize = b32; f.blk_usize = b32 + NB; f.blk_win = b32 + 2 * NB;
    f.win = P<c3rbgzf::DevWindow>(s.b_win);
    f.ubuf = P<uint8_t>(s.b_ubuf); f.n_rec = P<int32_t>(s.b_nrec);
    f.slot_off = P<int64_t>(s.b_soff); f.slot_cls = P<uint8_t>(s.b_scls); f.slot_key = P<uint64_t>(s.b_skey);
    f.slot_nops = P<int32_t>(s.b_snops); f.slot_nb = P<int64_t>(s.b_snb); f.slot_dst = P<c3rbgzf::Slot3>(s.b_sdst);
    f.sc = P<c3rbgzf::FetchSc>(s.b_sc);
    cudaStream_t st = s.st_a;
    int launches = 0;
    // the block tables are pageable host memory: the copies stage them before the call returns; the compressed bytes
    // are read by DMA after it (page-locked) or staged likewise
    if (raw->n_bytes > 0) CK(cudaMemcpyAsync(s.b_cdata.p, raw->data, raw->n_bytes, cudaMemcpyHostToDevice, st));
    if (NB > 0) {
        CK(cudaMemcpyAsync(b64, bcol.data(), (size_t)NB * 16, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(b32, icol.data(), (size_t)NB * 12, cudaMemcpyHostToDevice, st));
    }
    if (nw > 0) CK(cudaMemcpyAsync(s.b_win.p, dw.data(), (size_t)nw * sizeof(c3rbgzf::DevWindow), cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(s.b_sc.p, 0xff, 16, st));                 // no error, no stop
    CK(cudaMemsetAsync((uint8_t*)s.b_sc.p + 16, 0, sizeof(c3rbgzf::FetchSc) - 16, st));
    CK(cudaEventRecord(s.ev_bam[0], st));
    if (NB > 0) {
        static bool smem_set = false;
        if (!smem_set) {
            CK(cudaFuncSetAttribute(c3rbgzf::k_inflate, cudaFuncAttributeMaxDynamicSharedMemorySize, c3rbgzf::INFLATE_SMEM));
            smem_set = true;
        }
        c3rbgzf::k_inflate<<<(unsigned)NB, 32, c3rbgzf::INFLATE_SMEM, st>>>(f); ++launches;
    }
    CK(cudaEventRecord(s.ev_bam[1], st));
    if (nw > 0) { c3rbgzf::k_rec_bounds<<<(unsigned)nw, c3rbgzf::BOUNDS_THREADS, 0, st>>>(f); ++launches; }
    CK(cudaEventRecord(s.ev_bam[2], st));
    if (n_slots > 0) {
        const int64_t blocks = (n_slots + 255) / 256;
        c3rbgzf::k_rec_parse<<<(unsigned)(blocks < ctx->sm_count * 16 ? blocks : ctx->sm_count * 16), 256, 0, st>>>(f); ++launches;
        c3rbgzf::OpKeep op; op.f = f;
        launches += device_scan(op, n_slots, s.scan, s.scan_epoch, (c3rbgzf::Slot3*)&f.sc->n_reads, st);
    }
    CK(cudaEventRecord(s.ev_bam[3], st));
    CK(cudaMemcpyAsync(s.h_fsc.p, s.b_sc.p, sizeof(c3rbgzf::FetchSc), cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(s.ev_parse, st));
    CK(cudaGetLastError());
    s.launches = launches;
    s.in_use = true;
    s.has_result = false;
    s.deferred_rc = 0;
    s.pending_b = false;
    s.pending_parse = true;
    s.order = ++ctx->submit_seq;
    ++ctx->n_submit;
    *ticket = si;
    advance_all(ctx, getenv("C3R_SYNC_SUBMIT") != nullptr);
    return C3R_OK;
}

// k_rec_write into the read buffers queue_chunk sized, and the copy of the reads to the pinned host buffers
static int queue_rec_write(c3r_ctx* ctx, Slot& s) {
    cudaStream_t st = s.st_a;
    c3rbgzf::Fetch& f = s.fetch;
    c3r_reads& h = s.h_reads;
    f.pos = P<int32_t>(s.pos); f.flag = P<uint16_t>(s.flag); f.mapq = P<uint8_t>(s.mapq); f.hp = P<uint8_t>(s.hp);
    f.cigar_off = P<int32_t>(s.cigar_off); f.cigar = P<uint32_t>(s.cigar); f.seq_off = P<int64_t>(s.seq_off);
    f.seq = P<uint8_t>(s.seq);
    CK(cudaEventRecord(s.ev[0], st));
    CK(cudaEventRecord(s.ev_bam[4], st));
    CK(cudaMemsetAsync(s.cigar_off.p, 0, 4, st));
    CK(cudaMemsetAsync(s.seq_off.p, 0, 8, st));
    if (h.n_reads > 0) {
        const int64_t blocks = (f.n_slots * 32 + 255) / 256;
        c3rbgzf::k_rec_write<<<(unsigned)(blocks < ctx->sm_count * 16 ? blocks : ctx->sm_count * 16), 256, 0, st>>>(f);
        ++s.launches;
    }
    CK(cudaEventRecord(s.ev_bam[5], st));
    const int64_t R = h.n_reads;
    if (ensure_pin(ctx, s.h_rpos, R * 4) || ensure_pin(ctx, s.h_rflag, R * 2) || ensure_pin(ctx, s.h_rmapq, R) ||
        ensure_pin(ctx, s.h_rhp, R) || ensure_pin(ctx, s.h_rcoff, (R + 1) * 4) || ensure_pin(ctx, s.h_rcig, h.n_ops * 4) ||
        ensure_pin(ctx, s.h_rsoff, (R + 1) * 8) || ensure_pin(ctx, s.h_rseq, h.n_seq_bytes)) return C3R_ERR_CUDA;
    CK(cudaMemcpyAsync(s.h_rcoff.p, s.cigar_off.p, (R + 1) * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(s.h_rsoff.p, s.seq_off.p, (R + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (R > 0) {
        CK(cudaMemcpyAsync(s.h_rpos.p, s.pos.p, R * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(s.h_rflag.p, s.flag.p, R * 2, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(s.h_rmapq.p, s.mapq.p, R, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(s.h_rhp.p, s.hp.p, R, cudaMemcpyDeviceToHost, st));
    }
    if (h.n_ops > 0) CK(cudaMemcpyAsync(s.h_rcig.p, s.cigar.p, h.n_ops * 4, cudaMemcpyDeviceToHost, st));
    if (h.n_seq_bytes > 0) CK(cudaMemcpyAsync(s.h_rseq.p, s.seq.p, h.n_seq_bytes, cudaMemcpyDeviceToHost, st));
    h.pos = (const int32_t*)s.h_rpos.p; h.flag = (const uint16_t*)s.h_rflag.p; h.mapq = (const uint8_t*)s.h_rmapq.p;
    h.hp = (const uint8_t*)s.h_rhp.p; h.cigar_off = (const int32_t*)s.h_rcoff.p; h.cigar = (const uint32_t*)s.h_rcig.p;
    h.seq_off = (const int64_t*)s.h_rsoff.p; h.seq = (const uint8_t*)s.h_rseq.p;
    return 0;
}

// The parse counts of a device fetch are on the host: the first error before the first stop fails the ticket,
// otherwise the read buffers are sized from the counts and the rest of the chunk is queued
static int advance_parse(c3r_ctx* ctx, Slot& s) {
    const c3rbgzf::FetchSc& sc = *(const c3rbgzf::FetchSc*)s.h_fsc.p;
    if (sc.err_key < sc.stop_key) return fail(ctx, C3R_ERR_ARG, fetch_err_text((int)(sc.err_key & 7)));
    memset(&s.h_reads, 0, sizeof s.h_reads);
    s.h_reads.n_reads = sc.n_reads;
    s.h_reads.n_ops = sc.n_ops;
    s.h_reads.n_seq_bytes = sc.n_bases / 2;
    if (sc.n_ops >= (1LL << 31)) return fail(ctx, C3R_ERR_CAPACITY, "more than 2^31 CIGAR operations in one chunk");
    return queue_chunk(ctx, s, &s.h_reads, true, s.ref_host, s.ref_start1, s.ref_len, s.region_start1, s.region_end1,
                       s.has_filter ? &s.flt : nullptr);
}

// Queue stage B of a ticket whose stage A counts have arrived (block: wait for them).  Errors of this deferred part
// are kept in the slot and reported by c3r_wait(ticket).
static int advance(c3r_ctx* ctx, Slot& s, bool block) {
    if (s.in_use && s.pending_parse) {               // a device fetch: its parse counts first
        if (!block && cudaEventQuery(s.ev_parse) == cudaErrorNotReady) return 0;
        const auto t0 = std::chrono::steady_clock::now();
        int rc = 0;
        { cudaError_t e = cudaEventSynchronize(s.ev_parse); if (e != cudaSuccess) rc = fail(ctx, C3R_ERR_CUDA, cudaGetErrorString(e)); }
        s.pending_parse = false;
        if (!rc) rc = advance_parse(ctx, s);
        if (rc) { cudaStreamSynchronize(s.st_a); cudaStreamSynchronize(s.st); s.pending_b = false; s.deferred_rc = rc; s.deferred_err = ctx->err; }
        ctx->t_phase[4] += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        return 0;                                    // stage A is queued: its counts come later
    }
    if (!s.in_use || !s.pending_b) return 0;
    if (!block) {
        const cudaError_t q = cudaEventQuery(s.ev_cnt);
        if (q == cudaErrorNotReady) return 0;
    }
    const auto t0 = std::chrono::steady_clock::now();
    int rc = 0;
    { cudaError_t e = cudaEventSynchronize(s.ev_cnt); if (e != cudaSuccess) rc = fail(ctx, C3R_ERR_CUDA, cudaGetErrorString(e)); }
    s.pending_b = false;
    if (!rc) rc = parse_scalars(ctx, s);
    if (rc == C3R_ERR_CAPACITY && !s.exact_bounds && ctx->err.find("device capacity") != std::string::npos) {
        // unusual CIGARs (more deleted than sequenced bases, ...): exact bounds from the CIGARs, which are still on
        // the device, and stage A again
        s.exact_bounds = true;
        std::vector<uint32_t> cig((size_t)(s.d.n_ops > 0 ? s.d.n_ops : 1));
        rc = 0;
        if (s.d.n_ops > 0 && cudaMemcpy(cig.data(), s.cigar.p, (size_t)s.d.n_ops * 4, cudaMemcpyDeviceToHost) != cudaSuccess)
            rc = fail(ctx, C3R_ERR_CUDA, "could not read the CIGARs back for exact capacity bounds");
        if (!rc) rc = size_rows(ctx, s, cig.data());
        if (!rc) rc = run_stage_a(ctx, s);
        if (!rc) rc = read_scalars(ctx, s);
    }
    if (!rc) rc = ensure_stage_b(ctx, s);             // (stage A has ended: the host has seen its counts)
    if (!rc) rc = run_stage_b(ctx, s);
    if (!rc) rc = queue_d2h(ctx, s);
    if (!rc) { cudaError_t e = cudaEventRecord(s.ev[8], s.st); if (e != cudaSuccess) rc = fail(ctx, C3R_ERR_CUDA, cudaGetErrorString(e)); }
    if (rc) { cudaStreamSynchronize(s.st_a); cudaStreamSynchronize(s.st); s.deferred_rc = rc; s.deferred_err = ctx->err; }
    ctx->t_phase[4] += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return 0;
}

// every pending ticket, in submit order; tickets up to submit number `block_upto` are waited for, later ones only
// taken when their counts are already in
static void advance_all(c3r_ctx* ctx, bool block, uint64_t block_upto) {
    for (;;) {
        Slot* next = nullptr;
        for (int i = 0; i < N_SLOTS; ++i) {
            Slot& s = ctx->slots[i];
            if (s.in_use && (s.pending_b || s.pending_parse) && (!next || s.order < next->order)) next = &s;
        }
        if (!next) return;
        const bool parse = next->pending_parse;
        advance(ctx, *next, block && next->order <= block_upto);
        if (parse && !next->pending_parse) continue;  // its stage A is queued now: take its counts in the next round
        if (next->pending_b || next->pending_parse) return;   // not ready yet (non-blocking): the later ones wait their turn
    }
}

int c3r_wait(c3r_ctx* ctx, c3r_ticket ticket, c3r_result* res) {
    if (!ctx || !res || ticket < 0 || ticket >= N_SLOTS) return C3R_ERR_ARG;
    Slot& s = ctx->slots[ticket];
    if (!s.in_use) return fail(ctx, C3R_ERR_STATE, "ticket not in flight");
    CK(cudaSetDevice(ctx->device));
    // Stage B of this ticket and of the one submitted after it is queued first (the latter's counts arrive while the
    // pass of the ticket waited for still runs), so that the device goes from one pass to the next without waiting
    // for the host; tickets further ahead are taken along when their counts happen to be in.
    advance_all(ctx, true, s.order + 1);
    if (s.deferred_rc) {                             // the deferred part failed: report it and give the ticket back
        const int rc = s.deferred_rc;
        ctx->err = s.deferred_err;
        s.deferred_rc = 0;
        s.in_use = false;
        return rc;
    }
    CK(cudaStreamSynchronize(s.st));
    Dev& d = s.d;
    const int32_t err = ((const int32_t*)s.h_scalars.p)[6];
    if (err) return fail(ctx, C3R_ERR_CAPACITY, "device capacity check failed in the candidate stages");
    if (int rc = check_tc(ctx, s.st)) return rc;
    s.alt_total = ((const int64_t*)s.h_scalars.p)[2];
    if (!s.has_result) {
        // alt entries: sized by the device-side total, copied after the first sync
        const int64_t n = s.n_cand;
        if (n > 0 && s.alt_total > 0) {
            if (ensure_pin(ctx, s.h_alt, (size_t)s.alt_total * sizeof(AltEntry))) return C3R_ERR_CUDA;
            CK(cudaMemcpyAsync(s.h_alt.p, s.alt.p, (size_t)s.alt_total * sizeof(AltEntry), cudaMemcpyDeviceToHost, s.st));
            CK(cudaStreamSynchronize(s.st));
        }
        if (ctx->prm.keep_rows) {                    // header: row_pos is 1-based
            int32_t* rp = (int32_t*)s.h_row_pos.p;
            for (int64_t i = 0; i < s.n_rows; ++i) rp[i] += 1;
        }
        s.has_result = true;
    }
    c3r_result& r = s.res;
    memset(&r, 0, sizeof r);
    r.n_rows = s.n_rows;
    r.n_cand = s.n_cand;
    r.pos = (const int32_t*)s.h_pos.p; r.depth = (const int32_t*)s.h_depth.p; r.probs = (const float*)s.h_probs.p;
    r.alt_off = (const int64_t*)s.h_alt_off.p; r.alt_n = (const int32_t*)s.h_alt_n.p; r.alt = (const c3r_alt_entry*)s.h_alt.p;
    r.tensor = ctx->prm.keep_tensor ? (const int32_t*)s.h_tensor.p : nullptr;
    if (ctx->prm.keep_rows) {
        r.row_pos = (const int32_t*)s.h_row_pos.p; r.row_counts = (const int32_t*)s.h_counts.p;
        r.row_depth = (const int32_t*)s.h_row_depth.p;
    }
    for (int k = 0; k < 8; ++k) {
        float ms = 0.f;
        // D2H: after k_call and the text kernels
        cudaEventElapsedTime(&ms, k != 7 ? s.ev[k] : s.vcf ? s.ev_vcf[1] : s.calls ? s.ev_call[1] : s.ev[7], s.ev[k + 1]);
        r.stage_ms[k] = ms;
    }
    r.kernel_launches = s.launches;
    *res = r;
    (void)d;
    return C3R_OK;
}

int c3r_enable_calls(c3r_ctx* ctx, int on) {
    if (!ctx) return C3R_ERR_ARG;
    ctx->calls = on != 0;
    return C3R_OK;
}

int c3r_wait_calls(c3r_ctx* ctx, c3r_ticket ticket, const c3r_call** calls, int64_t* n, float* device_ms) {
    if (!ctx || !calls || !n || ticket < 0 || ticket >= N_SLOTS) return C3R_ERR_ARG;
    Slot& s = ctx->slots[ticket];
    if (!s.in_use || !s.has_result) return fail(ctx, C3R_ERR_STATE, "c3r_wait_calls needs a ticket c3r_wait has returned");
    if (!s.calls) return fail(ctx, C3R_ERR_STATE, "call records were off when this ticket was submitted (c3r_enable_calls)");
    *calls = s.n_cand > 0 ? (const c3r_call*)s.h_calls.p : nullptr;
    *n = s.n_cand;
    if (device_ms) {
        CK(cudaSetDevice(ctx->device));
        CK(cudaEventElapsedTime(device_ms, s.ev_call[0], s.ev_call[1]));
    }
    return C3R_OK;
}

int c3r_set_vcf(c3r_ctx* ctx, const c3r_vcf_options* opts) {
    if (!ctx || !opts) return C3R_ERR_ARG;
    if (!opts->on) { ctx->vcf = false; return C3R_OK; }
    if (!opts->contig) return fail(ctx, C3R_ERR_ARG, "c3r_set_vcf: no contig name");
    const size_t len = strlen(opts->contig);
    if (len > (size_t)c3rvcf::CONTIG_MAX) return fail(ctx, C3R_ERR_ARG, "c3r_set_vcf: contig name longer than 1024 bytes");
    if (!ctx->vcf_q_n) {                             // once per context: the QUAL table, the texts, k_vcf_write's shared memory
        CK(cudaSetDevice(ctx->device));
        int32_t q_n = 0;
        const float* t = c3rvcf::qual_table(&q_n);
        if (ensure(ctx, ctx->vcf_qtab, (size_t)q_n * sizeof(float))) return C3R_ERR_CUDA;
        CK(cudaMemcpy(ctx->vcf_qtab.p, t, (size_t)q_n * sizeof(float), cudaMemcpyHostToDevice));
        c3rvcf::special_texts(ctx->nan_text, ctx->ninf_text);
        CK(cudaFuncSetAttribute(c3rvcf::k_vcf_write, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)c3rvcf::vcf_write_smem(c3rvcf::row_max(c3rvcf::CONTIG_MAX))));
        ctx->vcf_q_n = q_n;
    }
    ctx->vcf = true;
    ctx->vcf_show_ref = opts->show_ref != 0;
    ctx->vcf_q_min = c3rvcf::qual_q_min(opts->qual_cut);
    ctx->vcf_contig.assign(opts->contig, len);
    return C3R_OK;
}

int c3r_wait_vcf(c3r_ctx* ctx, c3r_ticket ticket, const char** text, int64_t* n_bytes, int64_t* n_rows, float* device_ms) {
    if (!ctx || !text || !n_bytes || !n_rows || ticket < 0 || ticket >= N_SLOTS) return C3R_ERR_ARG;
    Slot& s = ctx->slots[ticket];
    if (!s.in_use || !s.has_result) return fail(ctx, C3R_ERR_STATE, "c3r_wait_vcf needs a ticket c3r_wait has returned");
    if (!s.vcf) return fail(ctx, C3R_ERR_STATE, "VCF text was off when this ticket was submitted (c3r_set_vcf)");
    const int64_t* hs = (const int64_t*)s.h_scalars.p;
    const int64_t nb = s.n_cand > 0 ? hs[8] : 0, nr = s.n_cand > 0 ? hs[9] : 0;
    if (nb < 0 || nb > s.n_cand * s.vcf_row_max || nr < 0 || nr > s.n_cand)
        return fail(ctx, C3R_ERR_CUDA, "VCF text totals out of range");
    *text = nb > 0 ? (const char*)s.h_text.p : "";
    *n_bytes = nb;
    *n_rows = nr;
    if (device_ms) {
        CK(cudaSetDevice(ctx->device));
        CK(cudaEventElapsedTime(device_ms, s.ev_vcf[0], s.ev_vcf[1]));
    }
    return C3R_OK;
}

int c3r_wait_reads(c3r_ctx* ctx, c3r_ticket ticket, c3r_reads* out, float* device_ms) {
    if (!ctx || !out || ticket < 0 || ticket >= N_SLOTS) return C3R_ERR_ARG;
    Slot& s = ctx->slots[ticket];
    if (!s.in_use || !s.has_result) return fail(ctx, C3R_ERR_STATE, "c3r_wait_reads needs a ticket c3r_wait has returned");
    if (!s.bam) return fail(ctx, C3R_ERR_STATE, "the ticket was submitted from host reads (c3r_submit_chunk)");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(s.st_a));
    *out = s.h_reads;
    if (device_ms) {
        float ms[3];
        if (int rc = c3r_wait_reads_stages(ctx, ticket, ms)) return rc;
        *device_ms = ms[0] + ms[1] + ms[2];
    }
    return C3R_OK;
}

int c3r_wait_reads_stages(c3r_ctx* ctx, c3r_ticket ticket, float stage_ms[3]) {
    if (!ctx || !stage_ms || ticket < 0 || ticket >= N_SLOTS) return C3R_ERR_ARG;
    Slot& s = ctx->slots[ticket];
    if (!s.in_use || !s.has_result) return fail(ctx, C3R_ERR_STATE, "c3r_wait_reads_stages needs a ticket c3r_wait has returned");
    if (!s.bam) return fail(ctx, C3R_ERR_STATE, "the ticket was submitted from host reads (c3r_submit_chunk)");
    CK(cudaSetDevice(ctx->device));
    float w = 0.f;
    CK(cudaEventElapsedTime(&stage_ms[0], s.ev_bam[0], s.ev_bam[1]));
    CK(cudaEventElapsedTime(&stage_ms[1], s.ev_bam[1], s.ev_bam[2]));
    CK(cudaEventElapsedTime(&stage_ms[2], s.ev_bam[2], s.ev_bam[3]));
    CK(cudaEventElapsedTime(&w, s.ev_bam[4], s.ev_bam[5]));
    stage_ms[2] += w;
    return C3R_OK;
}

int c3r_release(c3r_ctx* ctx, c3r_ticket ticket) {
    if (!ctx || ticket < 0 || ticket >= N_SLOTS) return C3R_ERR_ARG;
    Slot& s = ctx->slots[ticket];
    if (s.in_use) { cudaSetDevice(ctx->device); cudaStreamSynchronize(s.st_a); cudaStreamSynchronize(s.st); }
    s.in_use = false;
    s.pending_b = false;                             // released before its stage B was queued: nothing more to run
    s.pending_parse = false;
    s.deferred_rc = 0;
    s.has_result = false;
    return C3R_OK;
}

int c3r_rerun_resident(c3r_ctx* ctx, c3r_ticket ticket, float* total_ms, float* stage_ms8) {
    if (!ctx || ticket < 0 || ticket >= N_SLOTS) return C3R_ERR_ARG;
    Slot& s = ctx->slots[ticket];
    if (!s.in_use) return fail(ctx, C3R_ERR_STATE, "ticket not in flight");
    CK(cudaSetDevice(ctx->device));
    advance_all(ctx, true);
    if (s.deferred_rc) { ctx->err = s.deferred_err; return s.deferred_rc; }
    CK(cudaStreamSynchronize(s.st));
    s.launches = 0;
    CK(cudaEventRecord(s.ev[0], s.st_a));
    int rc = run_stage_a(ctx, s);
    if (!rc) rc = read_scalars(ctx, s);
    if (!rc) rc = ensure_stage_b(ctx, s);
    if (!rc) rc = run_stage_b(ctx, s);
    if (rc) return rc;
    CK(cudaEventRecord(s.ev[8], s.st));
    CK(cudaStreamSynchronize(s.st));
    if (int rc3 = check_tc(ctx, s.st)) return rc3;
    if (total_ms) CK(cudaEventElapsedTime(total_ms, s.ev[0], s.ev[8]));
    if (stage_ms8) {
        for (int k = 0; k < 8; ++k) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, s.ev[k], s.ev[k + 1]);
            stage_ms8[k] = ms;
        }
    }
    return s.launches;
}

int c3r_forward(c3r_ctx* ctx, const int32_t* tensor, int64_t n, float* probs, float* device_ms) {
    if (!ctx || !tensor || !probs || n < 0) return C3R_ERR_ARG;
    if (!ctx->have_weights) return fail(ctx, C3R_ERR_STATE, "c3r_set_weights must be called first");
    if (n == 0) return C3R_OK;
    CK(cudaSetDevice(ctx->device));
    const size_t per = (size_t)WIN * ctx->prm.channels * 4;
    if (ensure(ctx, ctx->fwd_in, n * per) || ensure(ctx, ctx->fwd_out, n * 96)) return C3R_ERR_CUDA;
    cudaStream_t st = ctx->fwd_stream;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    CK(cudaMemcpyAsync(ctx->fwd_in.p, tensor, n * per, cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(e0, st));
    int nl = 0;
    int rc = nn_forward(ctx, (const int32_t*)ctx->fwd_in.p, n, (float*)ctx->fwd_out.p, st, &nl);
    if (rc) return rc;
    CK(cudaEventRecord(e1, st));
    CK(cudaMemcpyAsync(probs, ctx->fwd_out.p, n * 96, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (int rc2 = check_tc(ctx, st)) return rc2;
    if (device_ms) CK(cudaEventElapsedTime(device_ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return nl;
}

int c3r_debug_fetch(c3r_ctx* ctx, int which, void* dst, int64_t max_bytes, int64_t* n_bytes) {
    if (!ctx || !dst || !n_bytes) return C3R_ERR_ARG;
    TcNet& t = ctx->tc;
    if (!t.cap_tiles) return fail(ctx, C3R_ERR_STATE, "no tensor-core forward has run");
    CK(cudaSetDevice(ctx->device));
    CK(cudaDeviceSynchronize());
    const size_t tiles = (size_t)t.cap_tiles;
    const void* src = nullptr;
    size_t bytes = 0;
    switch (which) {
        case 0: src = t.h1_cur ? t.h1_cur : t.h1[0]; bytes = tiles * NT * 4 * TC_IMG * 2; break;
        case 2: src = t.h2; bytes = tiles * NT * 5 * TC_IMG * 2; break;
        case 3: src = t.l4; bytes = tiles * 128 * DENSE * 4; break;
        case 4: src = t.trace; bytes = t.trace ? 2 * 2 * NT * 8 * 8 * sizeof(long long) : 0; break;
        default: return fail(ctx, C3R_ERR_ARG, "unknown buffer");
    }
    if ((int64_t)bytes > max_bytes) bytes = (size_t)max_bytes;
    CK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    *n_bytes = (int64_t)bytes;
    return C3R_OK;
}

}  // extern "C"

// =============================================================== network glue
namespace {

constexpr int64_t NN_SUB = 4096;      // sites per fp32 sub-batch (bounds the fp32 scratch)

int build_net(c3r_ctx* ctx, const std::map<std::string, std::pair<const float*, int64_t>>& w) {
    const int C = ctx->prm.channels;
    struct Need { const char* name; int64_t n; };
    const Need needs[] = {
        {"LSTM1/forward/kernel", (int64_t)C * G1}, {"LSTM1/forward/recurrent_kernel", (int64_t)U1 * G1}, {"LSTM1/forward/bias", G1},
        {"LSTM1/backward/kernel", (int64_t)C * G1}, {"LSTM1/backward/recurrent_kernel", (int64_t)U1 * G1}, {"LSTM1/backward/bias", G1},
        {"LSTM2/forward/kernel", (int64_t)H1W * G2}, {"LSTM2/forward/recurrent_kernel", (int64_t)U2 * G2}, {"LSTM2/forward/bias", G2},
        {"LSTM2/backward/kernel", (int64_t)H1W * G2}, {"LSTM2/backward/recurrent_kernel", (int64_t)U2 * G2}, {"LSTM2/backward/bias", G2},
        {"L4/kernel", (int64_t)L4_IN * DENSE}, {"L4/bias", DENSE},
        {"L5_1/kernel", DENSE * DENSE}, {"L5_1/bias", DENSE}, {"L5_2/kernel", DENSE * DENSE}, {"L5_2/bias", DENSE},
        {"Y_gt21_logits/kernel", DENSE * 21}, {"Y_gt21_logits/bias", 21},
        {"Y_genotype_logits/kernel", DENSE * 3}, {"Y_genotype_logits/bias", 3}};
    for (const Need& nd : needs) {
        auto it = w.find(nd.name);
        if (it == w.end()) return fail(ctx, C3R_ERR_ARG, std::string("missing weight ") + nd.name);
        if (it->second.second != nd.n) return fail(ctx, C3R_ERR_ARG, std::string("wrong size for weight ") + nd.name);
    }
    auto W = [&](const char* n) { return w.find(n)->second.first; };
    // host staging in the fp32 kernels' layouts
    std::vector<float> h;
    auto push = [&](size_t n) { size_t o = h.size(); h.resize(o + ((n + 63) / 64) * 64, 0.f); return o; };
    const size_t o_w1 = push((size_t)C * 2 * G1), o_b1 = push(2 * G1), o_u1 = push((size_t)2 * U1 * G1);
    const size_t o_w2 = push((size_t)H1W * 2 * G2), o_b2 = push(2 * G2), o_u2 = push((size_t)2 * U2 * G2);
    const size_t o_k4 = push((size_t)L4_IN * DENSE), o_b4 = push(DENSE);
    const size_t o_k51 = push(DENSE * DENSE), o_b51 = push(DENSE), o_k52 = push(DENSE * DENSE), o_b52 = push(DENSE);
    const size_t o_ky1 = push(DENSE * 21), o_by1 = push(21), o_ky2 = push(DENSE * 3), o_by2 = push(3);
    for (int c = 0; c < C; ++c) {
        memcpy(&h[o_w1 + (size_t)c * 2 * G1], W("LSTM1/forward/kernel") + (size_t)c * G1, G1 * 4);
        memcpy(&h[o_w1 + (size_t)c * 2 * G1 + G1], W("LSTM1/backward/kernel") + (size_t)c * G1, G1 * 4);
    }
    memcpy(&h[o_b1], W("LSTM1/forward/bias"), G1 * 4);
    memcpy(&h[o_b1 + G1], W("LSTM1/backward/bias"), G1 * 4);
    memcpy(&h[o_u1], W("LSTM1/forward/recurrent_kernel"), (size_t)U1 * G1 * 4);
    memcpy(&h[o_u1 + (size_t)U1 * G1], W("LSTM1/backward/recurrent_kernel"), (size_t)U1 * G1 * 4);
    for (int c = 0; c < H1W; ++c) {
        memcpy(&h[o_w2 + (size_t)c * 2 * G2], W("LSTM2/forward/kernel") + (size_t)c * G2, G2 * 4);
        memcpy(&h[o_w2 + (size_t)c * 2 * G2 + G2], W("LSTM2/backward/kernel") + (size_t)c * G2, G2 * 4);
    }
    memcpy(&h[o_b2], W("LSTM2/forward/bias"), G2 * 4);
    memcpy(&h[o_b2 + G2], W("LSTM2/backward/bias"), G2 * 4);
    memcpy(&h[o_u2], W("LSTM2/forward/recurrent_kernel"), (size_t)U2 * G2 * 4);
    memcpy(&h[o_u2 + (size_t)U2 * G2], W("LSTM2/backward/recurrent_kernel"), (size_t)U2 * G2 * 4);
    memcpy(&h[o_k4], W("L4/kernel"), (size_t)L4_IN * DENSE * 4);
    memcpy(&h[o_b4], W("L4/bias"), DENSE * 4);
    memcpy(&h[o_k51], W("L5_1/kernel"), DENSE * DENSE * 4);
    memcpy(&h[o_b51], W("L5_1/bias"), DENSE * 4);
    memcpy(&h[o_k52], W("L5_2/kernel"), DENSE * DENSE * 4);
    memcpy(&h[o_b52], W("L5_2/bias"), DENSE * 4);
    memcpy(&h[o_ky1], W("Y_gt21_logits/kernel"), DENSE * 21 * 4);
    memcpy(&h[o_by1], W("Y_gt21_logits/bias"), 21 * 4);
    memcpy(&h[o_ky2], W("Y_genotype_logits/kernel"), DENSE * 3 * 4);
    memcpy(&h[o_by2], W("Y_genotype_logits/bias"), 3 * 4);
    if (ensure(ctx, ctx->wbuf, h.size() * 4)) return C3R_ERR_CUDA;
    CK(cudaMemcpy(ctx->wbuf.p, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
    const float* b = (const float*)ctx->wbuf.p;
    NetF32& n = ctx->net;
    n.C = C;
    n.w1 = b + o_w1; n.b1 = b + o_b1; n.u1 = b + o_u1; n.w2 = b + o_w2; n.b2 = b + o_b2; n.u2 = b + o_u2;
    n.k4 = b + o_k4; n.b4 = b + o_b4; n.k51 = b + o_k51; n.b51 = b + o_b51; n.k52 = b + o_k52; n.b52 = b + o_b52;
    n.ky1 = b + o_ky1; n.by1 = b + o_by1; n.ky2 = b + o_ky2; n.by2 = b + o_by2;
    // tensor-core path: repack into fp16 operand images
    std::string terr;
    if (tc_build(ctx->tc, n, h.data(), o_w1, o_b1, o_u1, o_w2, o_b2, o_u2, o_k4, o_b4, o_k51, o_b51, o_k52, o_b52, ctx->sm_count, &terr))
        return fail(ctx, C3R_ERR_CUDA, "tensor-core weight repack failed: " + terr);
    ctx->have_weights = true;
    return C3R_OK;
}

static int nn_forward_impl(c3r_ctx* ctx, const int32_t* tensor_dev, int64_t n, float* probs_dev, cudaStream_t st, int* launches,
                           const __half* xop_ready);

// Tickets run on their own streams but share the network's scratch buffers: passes are ordered by events.
int nn_forward(c3r_ctx* ctx, const int32_t* tensor_dev, int64_t n, float* probs_dev, cudaStream_t st, int* launches,
               const __half* xop_ready) {
    if (ctx->prm.nn_impl == 1)                       // the tensor-core pass orders itself buffer by buffer (TcPipe)
        return nn_forward_impl(ctx, tensor_dev, n, probs_dev, st, launches, xop_ready);
    if (!ctx->nn_done) CK(cudaEventCreateWithFlags(&ctx->nn_done, cudaEventDisableTiming));
    else CK(cudaStreamWaitEvent(st, ctx->nn_done, 0));
    const int rc = nn_forward_impl(ctx, tensor_dev, n, probs_dev, st, launches, nullptr);
    CK(cudaEventRecord(ctx->nn_done, st));
    return rc;
}

static int nn_forward_impl(c3r_ctx* ctx, const int32_t* tensor_dev, int64_t n, float* probs_dev, cudaStream_t st, int* launches,
                           const __half* xop_ready) {
    *launches = 0;
    if (ctx->prm.nn_impl == 1) {
        std::string terr;
        int nl = tc_forward(ctx->tc, ctx->net, tensor_dev, n, probs_dev, st, &terr, xop_ready);
        if (nl < 0) return fail(ctx, C3R_ERR_CUDA, "tensor-core forward failed: " + terr);
        *launches = nl;
        ctx->tc_dirty = true;
        return 0;
    }
    const int C = ctx->prm.channels;
    const int64_t cap = n < NN_SUB ? n : NN_SUB;
    if (ctx->nscr.cap < cap) {
        if (ensure(ctx, ctx->nn_scratch, netf32_scratch_bytes(cap, C))) return C3R_ERR_CUDA;
        float* p = (float*)ctx->nn_scratch.p;
        NetF32Scratch& s = ctx->nscr;
        s.cap = cap;
        s.x = p; p += (size_t)cap * NT * C;
        s.zx1 = p; p += (size_t)cap * NT * 2 * G1;
        s.h1 = p; p += (size_t)cap * NT * H1W;
        s.zx2 = p; p += (size_t)cap * NT * 2 * G2;
        s.h2 = p; p += (size_t)cap * NT * H2W;
        s.l4 = p; p += (size_t)cap * DENSE;
        s.hbuf = p; p += (size_t)cap * 2 * U2 * 2;
        s.cbuf = p;
    }
    for (int64_t o = 0; o < n; o += ctx->nscr.cap) {
        const int64_t m = n - o < ctx->nscr.cap ? n - o : ctx->nscr.cap;
        *launches += netf32_forward(ctx->net, ctx->nscr, tensor_dev + o * WIN * C, m, probs_dev + o * 24, st);
    }
    CK(cudaGetLastError());
    return 0;
}

}  // namespace
