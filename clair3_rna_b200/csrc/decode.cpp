// Call records -> VCF rows, natively and in parallel on the host (A7, SURVEY.md §8a / §8f-2).
//
// The genotype decision is csrc/call.cuh, the same code k_call runs on the GPU: c3r_decode_vcf makes each
// candidate's call record with it on the host, c3r_format_vcf takes records made elsewhere, and both print a record
// with put_call.  What is left here is the row text of the reference's consumer
// (/root/reference/clair3_rna/call_variants.py):
//     output_with                          :1117-1392 (AD / AF / QUAL / FILTER / row text)
//     quality_score_from                   :383-389
// with the options call_var_bam always passes (--pileup --showRef --add_indel_length False, --qual 2;
// clair3_rna/call_var_bam.py:247-272).  clair3_rna_b200/decoder.py is the readable version, pinned by rows the
// reference's own output_with printed; this one exists because the Python decoder runs at ~7 k rows/s per core while
// the GPU emits millions of candidates/s.  QUAL is computed in double from the record's float32 probability (NumPy-1
// promotion, SURVEY.md §8c).
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/c3r_b200.h"
#include "call.cuh"

namespace {

const char NT16[17] = "=ACMGRSVTWYHKDBN";
const char* const GT_TEXT[5] = {"0/0", "1/1", "0/1", "1/2", "None"};       // c3rcall::Gt

const double PHRED_TRANS = -10.0 * (std::log(M_E) / std::log(10.0));      // call_variants.py:58

// x (0 <= x < 2^40) rounded to `scale` = 10^decimals units, to nearest with ties to even ON THE EXACT BINARY VALUE -
// what printf("%.*f") and Python's '%.*f' print.  x * scale = hi + lo exactly (fused multiply-add), so the comparison
// with one half is exact: a non-zero distance of the quotient's fraction from 0.5 is at least one ulp of hi and lo is
// below half an ulp.
inline uint64_t round_scaled(double x, double scale) {
    const double hi = x * scale;
    const double lo = std::fma(x, scale, -hi);
    const double fl = std::floor(hi);
    uint64_t q = (uint64_t)fl;
    const double d = (hi - fl) - 0.5;
    if (d > 0 || (d == 0 && (lo > 0 || (lo == 0 && (q & 1))))) ++q;
    return q;
}
inline char* put_uint(char* p, uint64_t v) {
    char tmp[24];
    int n = 0;
    do { tmp[n++] = (char)('0' + v % 10); v /= 10; } while (v);
    while (n) *p++ = tmp[--n];
    return p;
}
inline char* put_int(char* p, long v) {
    if (v < 0) { *p++ = '-'; return put_uint(p, (uint64_t)(-(v + 1)) + 1); }
    return put_uint(p, (uint64_t)v);
}
// "%.<decimals>f" of x >= 0 (decimals = 2 or 4); returns the end of the text (not NUL terminated)
inline char* put_fixed(char* p, double x, int decimals) {
    const uint64_t unit = decimals == 2 ? 100 : 10000;
    const uint64_t q = round_scaled(x, (double)unit);
    p = put_uint(p, q / unit);
    *p++ = '.';
    uint64_t f = q % unit;
    for (uint64_t u = unit / 10; u; u /= 10) { *p++ = (char)('0' + f / u); f %= u; }
    return p;
}

// round(max(x, 0), 2) as a double, through the correctly rounded 2-decimal text (Python's round() and "%.2f")
double round2(double x, char* text, size_t n) {
    (void)n;
    if (!(x > 0)) x = 0;
    if (!(x < 1e12)) { snprintf(text, n, "%.2f", x); return strtod(text, nullptr); }   // never reached by a QUAL
    const uint64_t q = round_scaled(x, 100.0);
    char* e = put_fixed(text, x, 2);
    *e = 0;
    return (double)q / 100.0;                        // == strtod(text): both are the correctly rounded q / 100
}

std::string iupac_to_n(const std::string& s) {
    if (s == ".") return s;
    std::string o = s;
    for (char& c : o) {
        const char u = (char)toupper((unsigned char)c);
        if (!(u == 'A' || u == 'C' || u == 'G' || u == 'T' || u == 'N' || u == ',' || u == '.')) c = 'N';
    }
    return o;
}

// output_with's row text from the decision: AF, QUAL, FILTER and the line (with '\n') appended to `out`
void put_row(const char* contig, int pos, std::string& ref_base, std::string& alt_base, bool is_ref, const char* gt,
             int depth, int ref_count, const long* counts, size_t n_counts, long support, float prob, double qual_cut,
             std::string& out) {
    double af = depth != 0 ? ((double)support + 0.0) / (double)depth : 0.0;
    if (af > 1) af = 1;
    const double p = (double)prob;
    char qtxt[64];
    const double qual = round2(PHRED_TRANS * std::log(((1.0 - p) + 1e-10) / (p + 1e-10)) + 10, qtxt, sizeof qtxt);
    const char* filt = is_ref ? "RefCall" : ((qual_cut < 0 || qual >= qual_cut) ? "PASS" : "LowQual");
    ref_base = iupac_to_n(ref_base);
    alt_base = iupac_to_n(alt_base);
    char buf[160];
    char* b = buf;
    out += contig;
    *b++ = '\t'; b = put_int(b, pos); *b++ = '\t'; *b++ = '.'; *b++ = '\t';
    out.append(buf, (size_t)(b - buf));
    out += ref_base; out += '\t'; out += alt_base; out += '\t'; out += qtxt; out += '\t'; out += filt;
    out += "\t.\tGT:GQ:DP:AD:AF\t";
    out += gt;
    b = buf;
    *b++ = ':'; b = put_int(b, (long)(int)qual); *b++ = ':'; b = put_int(b, depth); *b++ = ':'; b = put_int(b, ref_count);
    out.append(buf, (size_t)(b - buf));
    for (size_t i = 0; i < n_counts; ++i) { b = buf; *b++ = ','; b = put_int(b, counts[i]); out.append(buf, (size_t)(b - buf)); }
    out += ':';
    if (n_counts <= 1) {
        b = af >= 0 ? put_fixed(buf, af, 4) : buf + snprintf(buf, sizeof buf, "%.4f", af);
        out.append(buf, (size_t)(b - buf));
    } else {
        for (size_t i = 0; i < n_counts; ++i) {
            double a = 1.0 * (double)counts[i] / (double)depth;
            if (a > 1.0) a = 1.0;
            b = buf;
            if (i) *b++ = ',';
            b = (a >= 0) ? put_fixed(b, a, 4) : b + snprintf(b, 64, "%.4f", a);       // nan / negative: libc's text
            out.append(buf, (size_t)(b - buf));
        }
    }
    out += '\n';
}

// rows(i, out) appends the line of candidate i to `out` and says whether it printed one; candidates are split into
// n_threads contiguous ranges whose texts are joined in order into one malloc'ed buffer
template <class Rows>
int rows_in_parallel(int64_t n, int n_threads, const Rows& rows, char** text, int64_t* n_bytes, int64_t* n_rows) {
    int nt = n_threads > 0 ? n_threads : (int)std::max(1u, std::thread::hardware_concurrency());
    if ((int64_t)nt > (n + 255) / 256) nt = (int)std::max<int64_t>(1, (n + 255) / 256);
    std::vector<std::string> parts(nt);
    std::vector<int64_t> counted(nt, 0);
    auto work = [&](int t) {
        const int64_t a = n * t / nt, b = n * (t + 1) / nt;
        std::string& out = parts[t];
        out.reserve((size_t)(b - a) * 64);
        for (int64_t i = a; i < b; ++i) if (rows(i, out)) ++counted[t];
    };
    if (nt <= 1) work(0);
    else {
        std::vector<std::thread> th;
        for (int t = 0; t < nt; ++t) th.emplace_back(work, t);
        for (auto& t : th) t.join();
    }
    size_t total = 0;
    for (const std::string& s : parts) total += s.size();
    char* buf = (char*)malloc(total + 1);
    if (!buf) return C3R_ERR_ARG;
    size_t o = 0;
    for (const std::string& s : parts) { memcpy(buf + o, s.data(), s.size()); o += s.size(); }
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

// The text of one allele of a call record (see c3r_call_allele)
void put_allele(std::string& s, const c3r_call_allele& a, const uint8_t* seq, const uint8_t* ref, int64_t del_start,
                int ref_len) {
    s += (char)a.first;
    if (seq)
        for (uint32_t q = a.ins_seq_off; q < a.ins_seq_off + a.ins_len; ++q) s += NT16[c3rcall::nib(seq, q)];
    for (int k = a.suffix_from; k < ref_len; ++k) s += (char)ref[del_start + k - 1];
}

// The VCF line of one call record (with '\n') appended to `out`; false when the record has no row.  REF is ref_first
// and then the reference bases after the candidate, an ALT its allele, "." for a reference call.
bool put_call(const c3r_result* res, int64_t i, const c3r_call& c, const uint8_t* seq, const uint8_t* ref,
              int64_t ref_start1, const char* contig, double qual_cut, bool show_ref, std::string& out) {
    if (c.family == C3R_CALL_NO_ROW) return false;
    const bool is_ref = c.family == 0;
    if (!show_ref && is_ref) return false;
    static thread_local std::string ref_base, alt_base;
    const int64_t p0 = (int64_t)res->pos[i] - ref_start1;
    const int64_t ds = p0 + 1 < 0 ? 0 : p0 + 1;
    ref_base.assign(1, (char)c.ref_first);
    for (int k = 1; k < c.ref_len; ++k) ref_base += (char)ref[ds + k - 1];
    if (c.n_alt == 0) alt_base.assign(1, '.');
    else {
        alt_base.clear();
        for (int a = 0; a < c.n_alt; ++a) {
            if (a) alt_base += ',';
            put_allele(alt_base, c.alt[a], seq, ref, ds, c.ref_len);
        }
    }
    const long counts[2] = {c.ad[0], c.ad[1]};
    put_row(contig, res->pos[i], ref_base, alt_base, is_ref, GT_TEXT[c.gt], res->depth[i], c.ref_count, counts, c.n_ad,
            c.support, c.prob, qual_cut, out);
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
    const uint8_t* seq = reads ? reads->seq : nullptr;
    auto rows = [&](int64_t i, std::string& out) {
        c3r_call c;
        c3rcall::decide_call(call_input(res, i, reads, ref, ref_start1, ref_len), c);
        return put_call(res, i, c, seq, ref, ref_start1, contig, qual_cut, show_ref != 0, out);
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
    const uint8_t* seq = reads ? reads->seq : nullptr;
    const int64_t n_bases = seq ? 2 * reads->n_seq_bytes : 0;
    // A record that cannot be printed - malformed, or made over another window or read pool than the one given -
    // fails the call instead of losing its row.  REF letters 1.. are reference bases after the candidate; a
    // candidate off the window (its context padded with 'A') has REF = ref_first alone and reads none.
    for (int64_t i = 0; i < n; ++i) {
        const c3r_call& c = calls[i];
        if (c.family == C3R_CALL_NO_ROW) continue;
        if (c.family > 9 || c.gt > 4 || c.n_alt > 2 || c.n_ad > 2 || c.ref_len < 1) return C3R_ERR_ARG;
        const int64_t p0 = (int64_t)res->pos[i] - ref_start1;
        const int64_t ds = p0 + 1 < 0 ? 0 : p0 + 1;
        if (c.ref_len > 1 && ds + c.ref_len - 1 > ref_len) return C3R_ERR_ARG;
        for (int a = 0; a < c.n_alt; ++a) {
            const c3r_call_allele& al = c.alt[a];
            if (al.suffix_from < 1 || al.suffix_from > c.ref_len) return C3R_ERR_ARG;
            if (seq && (int64_t)al.ins_seq_off + al.ins_len > n_bases) return C3R_ERR_ARG;
        }
    }
    auto rows = [&](int64_t i, std::string& out) {
        return put_call(res, i, calls[i], seq, ref, ref_start1, contig, qual_cut, show_ref != 0, out);
    };
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
    *put_fixed(out, x, decimals) = 0;
    return C3R_OK;
}

}  // extern "C"
