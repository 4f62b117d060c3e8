// Call records -> VCF rows, natively and in parallel on the host (A7, SURVEY.md §8a / §8f-2).
//
// The genotype decision is csrc/call.cuh, the same code k_call runs on the GPU: c3r_decode_vcf makes each
// candidate's call record with it on the host, c3r_format_vcf takes records made elsewhere, and both print a record
// with csrc/vcf_row.cuh's put_call, the same code k_vcf_write runs on the GPU.  What is left here is QUAL on the host
// and the threaded row driver.  The row text is that of the reference's consumer
// (/root/reference/clair3_rna/call_variants.py):
//     output_with                          :1117-1392 (AD / AF / QUAL / FILTER / row text)
//     quality_score_from                   :383-389
// with the options call_var_bam always passes (--pileup --showRef --add_indel_length False, --qual 2;
// clair3_rna/call_var_bam.py:247-272).  clair3_rna_b200/decoder.py is the readable version, pinned by rows the
// reference's own output_with printed; this one exists because the Python decoder runs at ~7 k rows/s per core while
// the GPU emits millions of candidates/s.  QUAL is computed in double from the record's float32 probability (NumPy-1
// promotion, SURVEY.md §8c).
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/c3r_b200.h"
#include "call.cuh"
#include "vcf_row.cuh"

namespace c3rvcf {

const double PHRED_TRANS = -10.0 * (std::log(M_E) / std::log(10.0));      // call_variants.py:58

// round(max(PHRED_TRANS * log(((1 - p) + 1e-10) / (p + 1e-10)) + 10, 0), 2) in hundredths (Python's round() and
// "%.2f" are both the correct rounding of the binary value)
int32_t qual_q_host(float prob) {
    const double p = (double)prob;
    double x = PHRED_TRANS * std::log(((1.0 - p) + 1e-10) / (p + 1e-10)) + 10;
    if (!(x > 0)) x = 0;
    return (int32_t)round_scaled(x, 100.0);               // x <= 110: log's argument is >= 1e-10 / (1 + 1e-10)
}

// T[k - 1] = the smallest float32 p in [0, 1] with qual_q_host(p) >= k, k = 1 .. qual_q_host(1): bisection over the bit
// patterns of [0, 1], which order like the values
const float* qual_table(int32_t* n) {
    static std::vector<float> t;
    static std::once_flag once;
    std::call_once(once, [] {
        auto val = [](uint32_t b) { float f; memcpy(&f, &b, 4); return f; };
        const uint32_t one = 0x3f800000u;
        const int32_t q_max = qual_q_host(1.0f);
        if (q_max > QUAL_Q_MAX) abort();                  // the row bound assumes QUAL <= 110.00
        t.resize((size_t)q_max);
        uint32_t lo0 = 0;
        for (int32_t k = 1; k <= q_max; ++k) {
            uint32_t lo = lo0, hi = one;                  // q(hi) >= k; the answer is not below the previous one
            while (lo < hi) {
                const uint32_t mid = lo + (hi - lo) / 2;
                if (qual_q_host(val(mid)) >= k) hi = mid;
                else lo = mid + 1;
            }
            t[(size_t)k - 1] = val(lo);
            lo0 = lo;
        }
    });
    *n = (int32_t)t.size();
    return t.data();
}

int32_t qual_q_min(double qual_cut) {
    if (qual_cut < 0) return 0;
    if (!(qual_cut <= 1e7)) return INT32_MAX;             // NaN, or beyond any QUAL: every variant is LowQual
    int64_t q = (int64_t)std::floor(qual_cut * 100.0) - 2;
    if (q < 0) q = 0;
    while ((double)q / 100.0 < qual_cut) ++q;
    return (int32_t)q;
}

void special_texts(char nan_text[8], char ninf_text[8]) {
    volatile double zero = 0.0;                           // at run time, as the host's own divisions make them
    snprintf(nan_text, 8, "%.4f", zero / zero);
    snprintf(ninf_text, 8, "%.4f", -1.0 / zero);
}

}  // namespace c3rvcf

namespace {

// A growing text whose rows are printed in place: print(Sink&) is given the free room and called again with more
// when the row did not fit
struct Text {
    std::string s;
    size_t used = 0;
    template <class Print>
    bool row(const Print& print) {
        for (;;) {
            c3rvcf::Sink o = {&s[0] + used, (int64_t)(s.size() - used), 0};
            const bool any = print(o);
            if (o.n <= o.cap) { used += (size_t)o.n; return any; }
            s.resize(std::max(2 * s.size(), used + (size_t)o.n));
        }
    }
};

// rows(i, out) appends the line of candidate i to `out` and says whether it printed one; candidates are split into
// n_threads contiguous ranges whose texts are joined in order into one malloc'ed buffer
template <class Rows>
int rows_in_parallel(int64_t n, int n_threads, const Rows& rows, char** text, int64_t* n_bytes, int64_t* n_rows) {
    int nt = n_threads > 0 ? n_threads : (int)std::max(1u, std::thread::hardware_concurrency());
    if ((int64_t)nt > (n + 255) / 256) nt = (int)std::max<int64_t>(1, (n + 255) / 256);
    std::vector<Text> parts(nt);
    std::vector<int64_t> counted(nt, 0);
    auto work = [&](int t) {
        const int64_t a = n * t / nt, b = n * (t + 1) / nt;
        Text& out = parts[t];
        out.s.resize((size_t)(b - a) * 96 + 4096);
        for (int64_t i = a; i < b; ++i) if (rows(i, out)) ++counted[t];
    };
    if (nt <= 1) work(0);
    else {
        std::vector<std::thread> th;
        for (int t = 0; t < nt; ++t) th.emplace_back(work, t);
        for (auto& t : th) t.join();
    }
    size_t total = 0;
    for (const Text& s : parts) total += s.used;
    char* buf = (char*)malloc(total + 1);
    if (!buf) return C3R_ERR_ARG;
    size_t o = 0;
    for (const Text& s : parts) { memcpy(buf + o, s.s.data(), s.used); o += s.used; }
    buf[total] = 0;
    *text = buf;
    *n_bytes = (int64_t)total;
    for (int64_t r : counted) *n_rows += r;
    return C3R_OK;
}

c3rcall::CallIn call_input(const c3r_result* res, int64_t i, const c3r_reads* reads, const uint8_t* ref, int64_t ref_start1,
                           int64_t ref_len) {
    c3rcall::CallIn c;
    c.e = res->alt + res->alt_off[i];
    c.n = res->alt_n[i];
    c.probs = res->probs + 24 * i;
    c.ref = ref;
    c.ref_len = ref_len;
    c.p0 = (int64_t)res->pos[i] - ref_start1;
    c.seq = reads ? reads->seq : nullptr;
    return c;
}

c3rvcf::Fmt host_fmt(const char* contig, const uint8_t* ref, int64_t ref_start1, const c3r_reads* reads, double qual_cut,
                     int show_ref) {
    c3rvcf::Fmt f;
    f.contig = contig;
    f.contig_len = (int32_t)strlen(contig);
    f.q_min = c3rvcf::qual_q_min(qual_cut);
    f.ref = ref;
    f.ref_start1 = ref_start1;
    f.seq = reads ? reads->seq : nullptr;
    f.show_ref = show_ref != 0;
    c3rvcf::special_texts(f.nan_text, f.ninf_text);
    return f;
}

bool put_host_row(Text& out, const c3rvcf::Fmt& f, const c3r_call& c, int32_t pos, int32_t depth) {
    if (!c3rvcf::has_row(f, c)) return false;
    const int32_t q = c3rvcf::qual_q_host(c.prob);
    return out.row([&](c3rvcf::Sink& o) { return c3rvcf::put_call(o, f, c, pos, depth, q); });
}

// A record that cannot be printed - malformed, or made over another window or read pool than the one given - fails
// the call instead of losing its row.  REF letters 1.. are reference bases after the candidate; a candidate off the
// window (its context padded with 'A') has REF = ref_first alone and reads none.
bool records_printable(const c3r_result* res, const c3r_call* calls, const c3r_reads* reads, int64_t ref_start1,
                       int64_t ref_len) {
    const uint8_t* seq = reads ? reads->seq : nullptr;
    const int64_t n_bases = seq ? 2 * reads->n_seq_bytes : 0;
    for (int64_t i = 0; i < res->n_cand; ++i) {
        const c3r_call& c = calls[i];
        if (c.family == C3R_CALL_NO_ROW) continue;
        if (c.family > 9 || c.gt > 4 || c.n_alt > 2 || c.n_ad > 2 || c.ref_len < 1) return false;
        const int64_t p0 = (int64_t)res->pos[i] - ref_start1;
        const int64_t ds = p0 + 1 < 0 ? 0 : p0 + 1;
        if (c.ref_len > 1 && ds + c.ref_len - 1 > ref_len) return false;
        for (int a = 0; a < c.n_alt; ++a) {
            const c3r_call_allele& al = c.alt[a];
            if (al.suffix_from < 1 || al.suffix_from > c.ref_len) return false;
            if (seq && (int64_t)al.ins_seq_off + al.ins_len > n_bases) return false;
        }
    }
    return true;
}

}  // namespace

extern "C" {

// One VCF data line per candidate of `res`, in order, into a malloc'ed buffer (free with c3r_free_text).
// reads: the records the result was computed from (inserted bases are read from reads->seq);
// ref/ref_start1/ref_len: the reference window given to c3r_submit_chunk.  qual_cut < 0: no LowQual filter.
int c3r_decode_vcf(const c3r_result* res, const c3r_reads* reads, const uint8_t* ref, int64_t ref_start1, int64_t ref_len,
                   const char* contig, double qual_cut, int show_ref, int n_threads, char** text, int64_t* n_bytes, int64_t* n_rows) {
    if (!res || !ref || !contig || !text || !n_bytes || !n_rows) return C3R_ERR_ARG;
    const int64_t n = res->n_cand;
    *text = nullptr; *n_bytes = 0; *n_rows = 0;
    if (n > 0 && (!res->pos || !res->depth || !res->probs || !res->alt_off || !res->alt_n)) return C3R_ERR_ARG;
    const c3rvcf::Fmt f = host_fmt(contig, ref, ref_start1, reads, qual_cut, show_ref);
    auto rows = [&](int64_t i, Text& out) {
        c3r_call c;
        c3rcall::decide_call(call_input(res, i, reads, ref, ref_start1, ref_len), c);
        return put_host_row(out, f, c, res->pos[i], res->depth[i]);
    };
    return rows_in_parallel(n, n_threads, rows, text, n_bytes, n_rows);
}

// c3r_decode_vcf's lines from call records made elsewhere (k_call, c3r_debug_decide_calls)
int c3r_format_vcf(const c3r_result* res, const c3r_call* calls, const c3r_reads* reads, const uint8_t* ref,
                   int64_t ref_start1, int64_t ref_len, const char* contig, double qual_cut, int show_ref, int n_threads,
                   char** text, int64_t* n_bytes, int64_t* n_rows) {
    if (!res || !ref || !contig || !text || !n_bytes || !n_rows) return C3R_ERR_ARG;
    const int64_t n = res->n_cand;
    *text = nullptr; *n_bytes = 0; *n_rows = 0;
    if (n > 0 && (!res->pos || !res->depth || !calls)) return C3R_ERR_ARG;
    if (!records_printable(res, calls, reads, ref_start1, ref_len)) return C3R_ERR_ARG;
    const c3rvcf::Fmt f = host_fmt(contig, ref, ref_start1, reads, qual_cut, show_ref);
    auto rows = [&](int64_t i, Text& out) { return put_host_row(out, f, calls[i], res->pos[i], res->depth[i]); };
    return rows_in_parallel(n, n_threads, rows, text, n_bytes, n_rows);
}

int c3r_debug_decide_calls(const c3r_result* res, const c3r_reads* reads, const uint8_t* ref, int64_t ref_start1,
                           int64_t ref_len, c3r_call* out) {
    if (!res || !ref) return C3R_ERR_ARG;
    const int64_t n = res->n_cand;
    if (n > 0 && (!out || !res->pos || !res->probs || !res->alt_off || !res->alt_n)) return C3R_ERR_ARG;
    for (int64_t i = 0; i < n; ++i) c3rcall::decide_call(call_input(res, i, reads, ref, ref_start1, ref_len), out[i]);
    return C3R_OK;
}

void c3r_free_text(char* text) { free(text); }

// test hook: the decoder's "%.2f" / "%.4f" (exact round-half-even without libc) into out (>= 32 bytes, NUL terminated)
int c3r_debug_format_fixed(double x, int decimals, char* out) {
    if (!out || (decimals != 2 && decimals != 4) || !(x >= 0) || !(x < 1e12)) return C3R_ERR_ARG;
    c3rvcf::Sink o = {out, 31, 0};
    c3rvcf::put_fixed(o, x, decimals);
    out[o.n] = 0;
    return C3R_OK;
}

int64_t c3r_vcf_row_max(int64_t contig_len) { return contig_len < 0 ? -1 : c3rvcf::row_max(contig_len); }

// The device's way, on the host: QUAL from the table, every row's length counted first, the rows written at the
// exclusive prefix sums of the lengths, each of them checked to fill exactly its counted length (C3R_ERR_STATE if not)
int c3r_debug_vcf_rows(const c3r_result* res, const c3r_call* calls, const c3r_reads* reads, const uint8_t* ref,
                       int64_t ref_start1, int64_t ref_len, const char* contig, double qual_cut, int show_ref,
                       char** text, int64_t* n_bytes, int64_t* n_rows) {
    if (!res || !ref || !contig || !text || !n_bytes || !n_rows) return C3R_ERR_ARG;
    const int64_t n = res->n_cand;
    *text = nullptr; *n_bytes = 0; *n_rows = 0;
    if (n > 0 && (!res->pos || !res->depth || !calls)) return C3R_ERR_ARG;
    if (!records_printable(res, calls, reads, ref_start1, ref_len)) return C3R_ERR_ARG;
    const c3rvcf::Fmt f = host_fmt(contig, ref, ref_start1, reads, qual_cut, show_ref);
    int32_t q_n = 0;
    const float* qtab = c3rvcf::qual_table(&q_n);
    std::vector<int64_t> len((size_t)n), off((size_t)n + 1, 0);
    for (int64_t i = 0; i < n; ++i) {
        c3rvcf::Sink o = {nullptr, 0, 0};
        if (c3rvcf::has_row(f, calls[i]))
            c3rvcf::put_call(o, f, calls[i], res->pos[i], res->depth[i], c3rvcf::qual_q_table(qtab, q_n, calls[i].prob));
        len[i] = o.n;
        off[i + 1] = off[i] + o.n;
        *n_rows += o.n > 0;
    }
    char* buf = (char*)malloc((size_t)off[n] + 1);
    if (!buf) return C3R_ERR_ARG;
    for (int64_t i = 0; i < n; ++i) {
        if (!len[i]) continue;
        c3rvcf::Sink o = {buf + off[i], len[i], 0};
        c3rvcf::put_call(o, f, calls[i], res->pos[i], res->depth[i], c3rvcf::qual_q_table(qtab, q_n, calls[i].prob));
        if (o.n != len[i]) { free(buf); *n_rows = 0; return C3R_ERR_STATE; }
    }
    buf[off[n]] = 0;
    *text = buf;
    *n_bytes = off[n];
    return C3R_OK;
}

// QUAL by the table against QUAL by the formula for every float32 bit pattern: q and the text printed from it
int c3r_debug_vcf_qual_check(int n_threads, int64_t* n_checked, int64_t* n_mismatch) {
    if (!n_checked || !n_mismatch) return C3R_ERR_ARG;
    int32_t q_n = 0;
    const float* qtab = c3rvcf::qual_table(&q_n);
    const int nt = n_threads > 0 ? n_threads : (int)std::max(1u, std::thread::hardware_concurrency());
    std::atomic<int64_t> bad{0}, done{0};
    auto work = [&](int t) {
        int64_t my_bad = 0, my_done = 0;
        const uint64_t a = (1ull << 32) * (uint64_t)t / (uint64_t)nt, b = (1ull << 32) * (uint64_t)(t + 1) / (uint64_t)nt;
        for (uint64_t bits = a; bits < b; ++bits) {
            const uint32_t u = (uint32_t)bits;
            float p;
            memcpy(&p, &u, 4);
            const int32_t qt = c3rvcf::qual_q_table(qtab, q_n, p);
            const int32_t qh = c3rvcf::qual_q_host(p);
            ++my_done;
            if (qt != qh) { ++my_bad; continue; }
            if ((u & 0xfffu) == 0) {                     // the text, on one pattern in 4096: two ways of printing q
                double x = c3rvcf::PHRED_TRANS * std::log(((1.0 - (double)p) + 1e-10) / ((double)p + 1e-10)) + 10;
                if (!(x > 0)) x = 0;
                char s1[32], s2[32];
                c3rvcf::Sink o1 = {s1, 31, 0}, o2 = {s2, 31, 0};
                c3rvcf::put_fixed(o1, x, 2);
                c3rvcf::put_units(o2, (uint64_t)qt, 2);
                char ref_text[64];
                snprintf(ref_text, sizeof ref_text, "%.2f", x);
                if (o1.n != o2.n || memcmp(s1, s2, (size_t)o1.n) || strlen(ref_text) != (size_t)o2.n ||
                    memcmp(ref_text, s2, (size_t)o2.n)) ++my_bad;
            }
        }
        bad += my_bad;
        done += my_done;
    };
    std::vector<std::thread> th;
    for (int t = 0; t < nt; ++t) th.emplace_back(work, t);
    for (auto& t : th) t.join();
    *n_checked = done;
    *n_mismatch = bad;
    return C3R_OK;
}

int c3r_debug_vcf_q_min(double qual_cut, int32_t* q_min) {
    if (!q_min) return C3R_ERR_ARG;
    *q_min = c3rvcf::qual_q_min(qual_cut);
    return C3R_OK;
}

}  // extern "C"
