// The VCF data line of one call record (c3r_call), in code that compiles for the host (c3r_decode_vcf,
// c3r_format_vcf, csrc/decode.cpp) and for sm_100a (k_vcf_len / k_vcf_write below, queued by csrc/c3r_abi.cu).
//
// It restates the row text of output_with (call_variants.py:1117-1392, decoder.py vcf_row()): AF, QUAL, FILTER, AD and
// the line.  Everything inexact is pinned down so that both sides print the same bytes:
//   * QUAL enters as q, an integer number of hundredths.  The host computes it from the record's float32 probability
//     with its own libm (qual_q_host, the formula decode.cpp always used); the device looks it up in a table the host
//     built with that same formula (qual_table: the smallest float32 at which each q is reached), which is exact
//     wherever the formula is monotone in the probability - checked for all 2^32 inputs by the CPU tests.
//     QUAL's text is q / 100 with two decimals, GQ is q / 100 (== (int)(q / 100.0): q / 100.0 is never within
//     rounding of an integer unless q is a multiple of 100), FILTER compares q with q_min, the smallest q with
//     q / 100.0 >= qual_cut (qual_q_min).
//   * AF is an IEEE double division and "%.4f" is exact rounding of its binary value (round_scaled); on the device the
//     operations are the _rn intrinsics, so nvcc cannot contract x * scale into an fma the host does not do.  The text
//     of a NaN AF (depth 0 with two AD counts: 0.0 / 0.0) and of -inf (a negative count over depth 0) is whatever the
//     host's printf makes of them; the device is handed those strings (special_texts).
// A row goes into a Sink that writes while it has room and always counts, so the length the device computes for the
// offsets and the bytes it then writes come from the same code.
#pragma once
#include <stdint.h>

#include "call.cuh"

namespace c3rvcf {

constexpr int QUAL_Q_MAX = 11000;          // q at probability 1: QUAL 110.00 (qual_table checks it)
constexpr int CONTIG_MAX = 1024;           // longest contig name c3r_set_vcf takes
// The longest row of a contig name of `contig_len` bytes.  A record k_call makes has REF <= 1 + MAX_INDEL letters (the
// centre and a deletion key) and at most two ALTs, each at most 1 + MAX_INDEL + MAX_INDEL letters (a letter, an
// insertion key's bases, REF's letters after the first); an int prints in at most 11 characters, an AF in at most
// 16 ("-2147483648.0000"), QUAL in 6 ("110.00"), GQ in 3.
constexpr int INT_CHARS = 11;
constexpr int AF_CHARS = 16;
constexpr int ALLELE_MAX = 1 + 2 * c3rcall::MAX_INDEL;
constexpr int64_t ROW_FIXED =
    1 + INT_CHARS + 3 +                    // \t POS \t . \t
    (1 + c3rcall::MAX_INDEL) + 1 +         // REF \t
    (2 * ALLELE_MAX + 1) + 1 +             // ALT \t
    6 + 1 + 7 +                            // QUAL \t FILTER
    18 +                                   // \t . \t GT:GQ:DP:AD:AF \t
    4 + 1 + 3 + 1 + INT_CHARS +            // GT : GQ : DP
    1 + INT_CHARS + 2 * (1 + INT_CHARS) +  // : ref_count , ad , ad
    1 + (2 * AF_CHARS + 1) + 1;            // : AF , AF \n
C3R_HD int64_t row_max(int64_t contig_len) { return contig_len + ROW_FIXED; }
static_assert(ROW_FIXED == 394, "the row bound is pinned: change it together with its tests");

struct Sink {
    char* p;                               // room for cap bytes; cap 0: count only
    int64_t cap;
    int64_t n;
    C3R_HD void c(char x) { if (n < cap) p[n] = x; ++n; }
    C3R_HD void s(const char* t) { while (*t) c(*t++); }
};

// What every row of a chunk shares
struct Fmt {
    const char* contig;
    int32_t contig_len;
    int32_t q_min;                         // FILTER PASS when q >= q_min (qual_q_min)
    const uint8_t* ref;                    // the reference window
    int64_t ref_start1;
    const uint8_t* seq;                    // nt16 pool of the reads; NULL: insertion keys print their base alone
    int32_t show_ref;
    char nan_text[8];                      // the host printf's "%.4f" of 0.0 / 0.0 and of -1.0 / 0.0
    char ninf_text[8];
};

C3R_HD double dmul(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
C3R_HD double dfma(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
    return __fma_rn(a, b, c);
#else
    return __builtin_fma(a, b, c);
#endif
}
C3R_HD double ddiv(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}
C3R_HD double dfloor(double x) {
#if defined(__CUDA_ARCH__)
    return floor(x);
#else
    return __builtin_floor(x);
#endif
}

// x (0 <= x < 2^40) rounded to `scale` = 10^decimals units, to nearest with ties to even ON THE EXACT BINARY VALUE -
// what printf("%.*f") and Python's '%.*f' print.  x * scale = hi + lo exactly (fused multiply-add), so the comparison
// with one half is exact: a non-zero distance of the quotient's fraction from 0.5 is at least one ulp of hi and lo is
// below half an ulp.
C3R_HD uint64_t round_scaled(double x, double scale) {
    const double hi = dmul(x, scale);
    const double lo = dfma(x, scale, -hi);
    const double fl = dfloor(hi);
    uint64_t q = (uint64_t)fl;
    const double d = (hi - fl) - 0.5;
    if (d > 0 || (d == 0 && (lo > 0 || (lo == 0 && (q & 1))))) ++q;
    return q;
}
C3R_HD void put_uint(Sink& o, uint64_t v) {
    char tmp[24];
    int n = 0;
    do { tmp[n++] = (char)('0' + v % 10); v /= 10; } while (v);
    while (n) o.c(tmp[--n]);
}
C3R_HD void put_int(Sink& o, int64_t v) {
    if (v < 0) { o.c('-'); put_uint(o, (uint64_t)(-(v + 1)) + 1); return; }
    put_uint(o, (uint64_t)v);
}
// q units of 10^-decimals as "%.<decimals>f"
C3R_HD void put_units(Sink& o, uint64_t q, int decimals) {
    const uint64_t unit = decimals == 2 ? 100 : 10000;
    put_uint(o, q / unit);
    o.c('.');
    uint64_t f = q % unit;
    for (uint64_t u = unit / 10; u; u /= 10) { o.c((char)('0' + f / u)); f %= u; }
}
// "%.<decimals>f" of 0 <= x < 2^40 (decimals = 2 or 4)
C3R_HD void put_fixed(Sink& o, double x, int decimals) { put_units(o, round_scaled(x, decimals == 2 ? 100.0 : 10000.0), decimals); }
// "%.4f" of an AF: a ratio of two int32, clamped to 1 - so finite below 2^31 unless it is NaN or -inf
C3R_HD void put_af(Sink& o, const Fmt& f, double a) {
    if (a >= 0) put_fixed(o, a, 4);
    else if (a != a) o.s(f.nan_text);
    else if (a < -4294967296.0) o.s(f.ninf_text);
    else { o.c('-'); put_fixed(o, -a, 4); }
}

// iupac_to_n of decoder.py, letter by letter: a letter outside ACGTN (either case) becomes 'N'; ',' and '.' stay
C3R_HD char iupac_n(char c) {
    const char u = (c >= 'a' && c <= 'z') ? (char)(c - 32) : c;
    return (u == 'A' || u == 'C' || u == 'G' || u == 'T' || u == 'N' || u == ',' || u == '.') ? c : 'N';
}

// REF letter k >= 1 of a record is ref[del_start + k - 1]
C3R_HD void put_allele(Sink& o, const Fmt& f, const c3r_call_allele& a, int64_t ds, int ref_len) {
    o.c(iupac_n((char)a.first));
    if (f.seq)
        for (uint32_t q = a.ins_seq_off; q < a.ins_seq_off + a.ins_len; ++q) o.c(iupac_n(c3rcall::seq_char(c3rcall::nib(f.seq, q))));
    for (int k = a.suffix_from; k < ref_len; ++k) o.c(iupac_n((char)f.ref[ds + k - 1]));
}

// Whether a record prints a row (the same test k_vcf_len and the host printers make)
C3R_HD bool has_row(const Fmt& f, const c3r_call& c) {
    return c.family != C3R_CALL_NO_ROW && (f.show_ref || c.family != 0);
}

// The VCF line of one call record (with '\n'); false, and nothing printed, when the record has no row.  REF is
// ref_first and then the reference bases after the candidate, an ALT its allele, "." for a reference call.
C3R_HD bool put_call(Sink& o, const Fmt& f, const c3r_call& c, int32_t pos, int32_t depth, int32_t q) {
    if (!has_row(f, c)) return false;
    const bool is_ref = c.family == 0;
    const int64_t p0 = (int64_t)pos - f.ref_start1;
    const int64_t ds = p0 + 1 < 0 ? 0 : p0 + 1;
    for (int i = 0; i < f.contig_len; ++i) o.c(f.contig[i]);
    o.c('\t'); put_int(o, pos); o.s("\t.\t");
    o.c(iupac_n((char)c.ref_first));
    for (int k = 1; k < c.ref_len; ++k) o.c(iupac_n((char)f.ref[ds + k - 1]));
    o.c('\t');
    if (c.n_alt == 0) o.c('.');
    for (int a = 0; a < c.n_alt; ++a) {
        if (a) o.c(',');
        put_allele(o, f, c.alt[a], ds, c.ref_len);
    }
    o.c('\t');
    put_units(o, (uint64_t)q, 2);
    o.c('\t');
    o.s(is_ref ? "RefCall" : q >= f.q_min ? "PASS" : "LowQual");
    o.s("\t.\tGT:GQ:DP:AD:AF\t");
    o.s(c.gt == 0 ? "0/0" : c.gt == 1 ? "1/1" : c.gt == 2 ? "0/1" : c.gt == 3 ? "1/2" : "None");   // c3rcall::Gt
    o.c(':'); put_int(o, q / 100); o.c(':'); put_int(o, depth); o.c(':'); put_int(o, c.ref_count);
    for (int i = 0; i < c.n_ad; ++i) { o.c(','); put_int(o, c.ad[i]); }
    o.c(':');
    if (c.n_ad <= 1) {
        double af = depth != 0 ? ddiv((double)c.support + 0.0, (double)depth) : 0.0;
        if (af > 1) af = 1;
        put_af(o, f, af);
    } else {
        for (int i = 0; i < c.n_ad; ++i) {
            double a = ddiv(1.0 * (double)c.ad[i], (double)depth);
            if (a > 1.0) a = 1.0;
            if (i) o.c(',');
            put_af(o, f, a);
        }
    }
    o.c('\n');
    return true;
}

// q of a probability by the table: the number of entries <= p.  The formula gives 0 below 0, above 1 and for NaN.
C3R_HD int32_t qual_q_table(const float* t, int32_t n, float p) {
    if (!(p >= 0.f && p <= 1.f)) return 0;
    int32_t lo = 0, hi = n;
    while (lo < hi) {
        const int32_t mid = (lo + hi) >> 1;
#if defined(__CUDA_ARCH__)
        const float v = __ldg(t + mid);
#else
        const float v = t[mid];
#endif
        if (v <= p) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// ---- host side (decode.cpp)
int32_t qual_q_host(float prob);                         // QUAL's formula in double, as hundredths
const float* qual_table(int32_t* n);                     // built once per process
int32_t qual_q_min(double qual_cut);                     // qual_cut < 0: 0 (no LowQual filter)
void special_texts(char nan_text[8], char ninf_text[8]);

#if defined(__CUDACC__)
// ---- device side: one row length per candidate, their offsets (scan.cuh), the rows
struct DevRows {
    Fmt f;                                 // contig, ref and seq in device memory
    const c3r_call* calls;
    const int32_t* pos;
    const int32_t* depth;
    int64_t n;
    const float* qtab;
    int32_t q_n;
    int32_t* len;                          // [n] row bytes, 0: no row
    long long* off;                        // [n] first byte of each row
    char* out;
};

__global__ void __launch_bounds__(128) k_vcf_len(const DevRows r) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < r.n; i += (int64_t)gridDim.x * blockDim.x) {
        const c3r_call c = r.calls[i];
        Sink o = {nullptr, 0, 0};
        if (has_row(r.f, c)) put_call(o, r.f, c, r.pos[i], r.depth[i], qual_q_table(r.qtab, r.q_n, c.prob));
        r.len[i] = (int32_t)o.n;
    }
}

struct VcfTotals { long long bytes, rows; };
struct OpVcfOff {
    typedef VcfTotals T;
    struct Ctx {};
    const int32_t* len;
    long long* off;
    int64_t n;
    __device__ void ctx_init(Ctx&) const {}
    __device__ T identity() const { return T{0, 0}; }
    __device__ T combine(const T& x, const T& y) const { return T{x.bytes + y.bytes, x.rows + y.rows}; }
    __device__ int64_t size() const { return n; }
    __device__ T load(int64_t i) const { const int32_t l = len[i]; return T{l, l > 0}; }
    __device__ void store(int64_t i, const T& incl, const T& own, Ctx&) const { off[i] = incl.bytes - own.bytes; }
};

// A block prints VCF_TILE consecutive candidates, one thread each, into shared memory; their rows are one contiguous
// range of the output, which the block then stores 16 bytes at a time (bytes of the range's partial first and last
// 16-byte words one by one: the neighbouring blocks own the rest of those words).
constexpr int VCF_TILE = 64;
inline size_t vcf_write_smem(int64_t row_max_bytes) { return (size_t)(VCF_TILE * row_max_bytes + 32); }

__global__ void __launch_bounds__(VCF_TILE) k_vcf_write(const DevRows r, int64_t row_max_bytes) {
    extern __shared__ __align__(16) char sm[];
    for (int64_t c0 = (int64_t)blockIdx.x * VCF_TILE; c0 < r.n; c0 += (int64_t)gridDim.x * VCF_TILE) {
        const int64_t c1 = c0 + VCF_TILE < r.n ? c0 + VCF_TILE : r.n;
        const int64_t g0 = r.off[c0], g1 = r.off[c1 - 1] + r.len[c1 - 1];
        const int64_t a0 = g0 & ~15LL;
        const int64_t i = c0 + threadIdx.x;
        if (i < c1 && r.len[i] > 0) {
            const c3r_call c = r.calls[i];
            Sink o = {sm + (r.off[i] - a0), row_max_bytes, 0};
            put_call(o, r.f, c, r.pos[i], r.depth[i], qual_q_table(r.qtab, r.q_n, c.prob));
        }
        __syncthreads();
        for (int64_t w = a0 + 16 * (int64_t)threadIdx.x; w < g1; w += 16 * VCF_TILE) {
            if (w >= g0 && w + 16 <= g1) *reinterpret_cast<uint4*>(r.out + w) = *reinterpret_cast<const uint4*>(sm + (w - a0));
            else
                for (int64_t b = w > g0 ? w : g0; b < w + 16 && b < g1; ++b) r.out[b] = sm[b - a0];
        }
        __syncthreads();                                 // the tile's text is stored before the next one is printed
    }
}
#endif

}  // namespace c3rvcf
