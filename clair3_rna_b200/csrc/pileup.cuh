// Integer half of the pileup calling path: flat alignment records -> per-position
// count rows -> candidates -> 33 x C windows + alt_info.  sm_100a, HBM-bound work:
// no tensor cores here.
//
// Reference semantics restated (all under /root/reference):
//   samtools mpileup column membership / tokens   src/create_tensor_pileup.py:436-451 (external htslib)
//   generate_tensor                                src/create_tensor_pileup.py:85-302
//   candidate predicate, ring buffer, padding      src/create_tensor_pileup.py:463-611
//   depth rescale                                  clair3_rna/utils.py:85-92,120
//
// Data layout in HBM (one chunk):
//   position space  region [R0, R1), W = R1-R0 positions, bitmaps of ceil(W/32)+2 words
//       covA   1 bit/position: covered by >=1 admitted read (incl. D and N)  -> run contiguity
//       covE   1 bit/position: covered by an M/=/X/D op (a base or a `*`/`#`)
//       rowR   = dilate16(covE) & covA : positions that get a count row
//       word_base[w] = rank of the first row of word w  (row(p) = word_base + popc(bits below p))
//   row space  L rows (device-side count), rows of consecutive positions are consecutive
//       counts[L][C] int32, row_pos[L], row_depth[L], row_flag[L], max_skip[L]
//       cov[L][4|6] coverage difference rows (per strand M and D coverage, M coverage per haplotype)
//   row events (CSR by row, 16 B each): read bases that differ from the reference, and indel tokens
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include "scan.cuh"

namespace c3r {

constexpr int MPILEUP_MAX_DEPTH = 8000;      // htslib bam_plp maxcnt as samtools mpileup sets it by default
constexpr int WIN = 33;
constexpr int FLANK = 16;
constexpr int TILE_ROWS = 32;
constexpr int COV_UP = 5;                    // summary levels above a coverage bitmap: 32^6 positions > int32
constexpr int PT_WORDS = 1024;               // bitmap words per position tile (k_row_bits / k_row_rank: 256 threads x 4 words)
constexpr uint32_t OP_SKIP = 0xffffffffu;
constexpr int COV_TILE = 256;                // rows per k_rows block / coverage aggregate

struct RowEvent {              // something other than "a base equal to the reference" at a row
    uint32_t info;             // rid << 4 | hp << 2 | is_del << 1 | reverse
    int32_t len;               // > 0: indel token of that length;  0: a read base that differs from the reference
    uint32_t yb;               // indel: base index of the inserted bases;  mismatch: 0..3 = A,C,G,T, 4 = N / ambiguity
                               // code (counts nothing, but is not the reference base)
    int32_t row;
};

struct AltEntry {              // mirrors c3r_alt_entry
    uint8_t kind, base;
    uint16_t len;
    int32_t count;
    uint32_t seq_off;
    uint32_t order;
};

struct ScanElem {              // segmented scan over CIGAR ops
    unsigned long long v;      // ref_len << 32 | qry_len (within the read so far)
    int32_t rid;
    int32_t flag;
};

struct Int2 { int32_t a, b; };

// Everything the kernels need, passed by value.
struct Dev {
    // ---- inputs
    int64_t n_reads, n_ops;
    const int32_t* pos; const uint16_t* flag; const uint8_t* mapq; const uint8_t* hp;
    const int32_t* cigar_off; const uint32_t* cigar; const int64_t* seq_off; const uint8_t* seq;
    const uint8_t* ref; int64_t ref_start0; int64_t ref_len;
    int32_t R0, R1; int64_t W; int64_t NW;            // region (0-based half open), words
    // ---- params
    int32_t C; int32_t min_cov; int32_t min_mq; uint32_t excl; double snp_af, indel_af;
    int32_t padding; int32_t max_depth; double skip_prop;
    int32_t dbg;                // experiments (C3R_DBG): 1 = no tie-break walk, 2 = no heavy-row path

    const uint16_t* thr_snp; const uint16_t* thr_indel;     // THR_N entries each (k_thr_table)
    // ---- optional site filters (create_tensor_pileup.py:446-451, 480-481, 551-556); n < 0: not given.
    // Intervals: sorted, disjoint, non-touching (start0, end0) pairs; known: sorted 1-based positions.
    const int32_t* pbed; int32_t n_pbed;                    // mpileup -l: rows exist only inside
    const int32_t* cbed; int32_t n_cbed;                    // confident BED: [pos-1, pos+max_del+1) must overlap
    const int32_t* known; int32_t n_known;                  // genotyping: candidates are exactly these sites
    // printed columns = covA inside the pileup BED (covA itself without one); head/tail mode: zero rows around runs
    const uint32_t* covP; int32_t head_tail;
    int32_t* tail;              // [0] offset of the last printed column + 1, [1] offset of the last gap below it + 1
    // ---- per read / per op
    uint8_t* admit; int32_t* read_end;
    int32_t* op_x; uint32_t* op_y;
    uint32_t* op_info;          // rid << 4 | hp << 2 | last op of its read << 1 | reverse;  OP_SKIP: read not admitted
    // ---- position space
    uint32_t* covA; uint32_t* covE; uint32_t* rowR; int32_t* word_base;
    uint32_t* upA[COV_UP]; uint32_t* upE[COV_UP];   // "whole word set" summaries of covA / covE, level l+1 over level l (mark_range)
    int32_t* ptile;             // [NW / PT_WORDS + 2]: rows per tile of PT_WORDS bitmap words, then their exclusive prefix
    int32_t* kctr;              // [4] block tickets of the kernels whose last block finishes a job (zeroed with the scalars)
    // ---- row space
    int64_t L_ub;
    int64_t* n_rows;            // device scalar L
    int32_t* row_pos; int32_t* counts; int32_t* row_depth; uint8_t* row_flag;
    int32_t* head_cnt; int32_t* tail_cnt; Int2* skipdiff; int32_t* max_skip;
    int32_t* row_inscnt; int32_t* row_delcnt;
    // ---- row events (CSR by row): binc = event counts, then offsets (L_ub+2); cov = coverage difference rows
    int32_t* binc; int32_t* bin_cur; RowEvent* events;
    RowEvent* raw; int64_t* n_raw; // events in discovery order (k_cmp) before the counting sort (k_scatter_aggr)
    int64_t events_ub;
    int32_t* cov;                  // [L_ub+2][4 or 6]: Mf Mr Df Dr [M_hp1 M_hp2]
    int32_t* cov_tile;             // [L_ub/256+2][4 or 6]: sums of cov over tiles of 256 rows, then their exclusive prefix
    const uint32_t* refnib; int64_t n_ref_words;     // one-hot reference nibbles of the loaded window (k_refnib)
    int32_t* blockmax;             // [n_reads/256+1]: largest end of the admitted reads of each block of 256 reads
    int32_t* ctile;                // [L_ub/256+2]: candidates per tile of 256 rows (k_rows)
    int32_t* csuper;               // [L_ub/16384+2]: candidates per group of 64 tiles
    // ---- candidates
    int64_t* n_cand; int32_t* cand_row; int64_t cand_cap;
    int32_t* cand_pos; int32_t* cand_depth;
    int32_t* tensor;            // [n_cand][33][C]
    int64_t* alt_off; int32_t* alt_n; AltEntry* alt; int64_t alt_cap;
    // padding pass scratch
    Int2* cur_ref; uint8_t* deleted;
    int32_t* err;               // device error flag
};

// ------------------------------------------------------------------ helpers
__device__ __forceinline__ bool op_consumes_ref(uint32_t op) { return op == 0 || op == 2 || op == 3 || op == 7 || op == 8; }
__device__ __forceinline__ bool op_consumes_qry(uint32_t op) { return op == 0 || op == 1 || op == 4 || op == 7 || op == 8; }
__device__ __forceinline__ bool op_is_match(uint32_t op) { return op == 0 || op == 7 || op == 8; }

// rank of position p (0-based genome coordinate, inside the region) among rows: number of row bits below p
__device__ __forceinline__ int32_t row_lower_bound(const Dev& d, int32_t p) {
    if (p <= d.R0) return 0;
    int64_t o = (int64_t)p - d.R0;
    if (o >= d.W) o = d.W;
    const int64_t w = o >> 5;
    const uint32_t m = (1u << (o & 31)) - 1u;
    return d.word_base[w] + __popc(d.rowR[w] & m);
}
__device__ __forceinline__ bool bit_at(const uint32_t* bm, int64_t o) { return (bm[o >> 5] >> (o & 31)) & 1u; }

__device__ __forceinline__ uint32_t nib_at(const uint8_t* seq, uint32_t q) {
    const uint32_t b = seq[q >> 1];
    return (q & 1u) ? (b & 15u) : (b >> 4);
}
// reference base at genome position p -> channel index 0..3 (non-ACGT -> 0 like evc_base_from), acgt flag
__device__ __forceinline__ int ref_index(const Dev& d, int32_t p, bool* is_acgt) {
    const int64_t o = (int64_t)p - d.ref_start0;
    uint8_t c = (o >= 0 && o < d.ref_len) ? d.ref[o] : (uint8_t)'N';
    if (c >= 'a') c -= 32;
    int idx = c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1;
    *is_acgt = idx >= 0;
    return idx < 0 ? 0 : idx;
}

// set bits [a, b) (region offsets, already clipped) of bitmap bm.  The two end words take an atomicOr each; the whole
// words between them are not written: they become a bit range of the next level ("this whole word is set"), marked
// the same way - at most two atomics per level, whatever the length (a read spanning introns of 100 kb is 3 000
// words).  k_row_bits folds the levels back into level 0.
// (testing the word first and skipping the atomic when the bits are already there was measured slower: 44 against
// 33 us for k_cigar at config 2 - the dependent load costs more than the atomics it saves)
__device__ __forceinline__ void or_bits(uint32_t* w, uint32_t m) { atomicOr(w, m); }
__device__ __forceinline__ void mark_range(uint32_t* bm, uint32_t* const* up, int64_t a, int64_t b) {
    if (b <= a) return;
    int64_t lo = a, hi = b;
#pragma unroll 1
    for (int l = 0;; ++l) {
        const int64_t wa = lo >> 5, wb = (hi - 1) >> 5;
        const uint32_t ma = 0xffffffffu << (lo & 31);
        const uint32_t mb = 0xffffffffu >> (31 - ((hi - 1) & 31));
        if (wa == wb) { or_bits(&bm[wa], ma & mb); return; }
        or_bits(&bm[wa], ma);
        or_bits(&bm[wb], mb);
        if (wb <= wa + 1) return;
        if (l == COV_UP) {                               // beyond the top level (not reachable with int32 positions)
            for (int64_t w = wa + 1; w < wb; ++w) or_bits(&bm[w], 0xffffffffu);
            return;
        }
        lo = wa + 1; hi = wb; bm = up[l];
    }
}
// is level-0 word w inside a range marked at a higher level?  (4 consecutive words, w4 % 4 == 0: bit j = word w4 + j)
__device__ __forceinline__ uint32_t up_full4(uint32_t* const* up, int64_t w4) {
    uint32_t m = (up[0][w4 >> 5] >> (w4 & 31)) & 0xfu;
    int64_t idx = w4 >> 5;
#pragma unroll
    for (int l = 1; l < COV_UP; ++l) {
        if ((up[l][idx >> 5] >> (idx & 31)) & 1u) m = 0xfu;
        idx >>= 5;
    }
    return m;
}
__device__ __forceinline__ bool up_full(uint32_t* const* up, int64_t w) { return (up_full4(up, w & ~3ll) >> (w & 3)) & 1u; }

// ------------------------------------------------- K1: CIGAR geometry per read
// G lanes per read (G = 32, or 8 when reads carry few ops): the group walks the read's ops G at a time, an
// inclusive scan inside the group (shuffles) gives every op the reference / query lengths consumed before it, and
// the running totals carry over to the next G ops.  Per op: reference start op_x, base index op_y, op_info
// (read ordinal, haplotype, strand, last-op flag; OP_SKIP when the read is not admitted); the runs of M/=/X/D ops
// between ref-skips mark covE (one interval per run), the read's whole span marks covA.  Also the admit flag per read (samtools mpileup filters, SURVEY.md 8a A0).
// No device-wide scan, no segment heads: reads are independent (this replaced a segmented look-back scan over all
// ops that took 50 us for a million ops, most of it waiting on its own cross-block protocol).
template <int G>
__global__ void __launch_bounds__(256) k_cigar(Dev d) {
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
    const int gl = threadIdx.x & (G - 1);
    if (r >= d.n_reads) return;                          // whole groups leave together (256 % G == 0)
    const uint32_t gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (threadIdx.x & 31 & ~(G - 1)));
    const uint32_t f = d.flag[r];
    const int32_t a = d.cigar_off[r], b = d.cigar_off[r + 1];
    const int32_t pos = d.pos[r];
    bool ok = !(f & (0x4u | 0x100u | 0x200u | 0x400u)) && !(f & d.excl) && (int)d.mapq[r] >= d.min_mq;
    if ((f & 0x1u) && !(f & 0x2u)) ok = false;
    if (b <= a) ok = false;
    uint32_t hp = d.hp[r];
    hp = hp == 1 ? 1u : hp == 2 ? 2u : 0u;
    const uint32_t info = ((uint32_t)r << 4) | (hp << 2) | ((f >> 4) & 1u);
    uint32_t x = 0, y = (uint32_t)d.seq_off[r];          // reference bases consumed so far, base index in the sequence pool
    for (int32_t k0 = a; k0 < b; k0 += G) {
        const int32_t k = k0 + gl;
        const uint32_t c = k < b ? d.cigar[k] : 0u;
        const uint32_t op = c & 15u, len = c >> 4;
        const uint32_t rl = op_consumes_ref(op) ? len : 0u, ql = op_consumes_qry(op) ? len : 0u;
        uint32_t ir = rl, iq = ql;
#pragma unroll
        for (int o = 1; o < G; o <<= 1) {
            const uint32_t ur = __shfl_up_sync(gmask, ir, o, G), uq = __shfl_up_sync(gmask, iq, o, G);
            if (gl >= o) { ir += ur; iq += uq; }
        }
        const int32_t ox = pos + (int32_t)(x + ir - rl);
        if (k < b) {
            d.op_x[k] = ox;
            d.op_y[k] = y + iq - ql;
            d.op_info[k] = ok ? (info | (k + 1 == b ? 2u : 0u)) : OP_SKIP;
        }
        // covE: consecutive M/=/X/D ops of a read are adjacent on the reference (insertions and clips take no
        // reference), so the run of them between two ref-skips is ONE interval: its first lane marks it (a third to
        // a tenth of the atomics of marking every op on its own)
        {
            const int sh = threadIdx.x & 31 & ~(G - 1);                          // the group's first lane in the warp
            const bool md = ok && k < b && rl && (op_is_match(op) || op == 2);
            const bool sk = k < b && op == 3 && len;
            const uint32_t gm = G == 32 ? 0xffffffffu : (1u << G) - 1u;
            const uint32_t md_mask = (__ballot_sync(gmask, md) >> sh) & gm, sk_mask = (__ballot_sync(gmask, sk) >> sh) & gm;
            const uint32_t below = (1u << gl) - 1u;
            const int prev_sk = 31 - __clz((sk_mask & below) | 0u) ;            // -1 when none ( __clz(0) == 32 )
            const uint32_t seg_lo = prev_sk < 0 ? 0u : (prev_sk >= 31 ? 0xffffffffu : (2u << prev_sk) - 1u);   // lanes up to prev_sk
            const bool first = md && (md_mask & below & ~seg_lo) == 0u;
            const uint32_t above = gl >= 31 ? 0u : ~((2u << gl) - 1u);
            const uint32_t nsk = sk_mask & above;
            const uint32_t seg_hi = nsk ? ~((nsk & (0u - nsk)) - 1u) : 0u;       // lanes from the next skip on
            const uint32_t mine = md_mask & ~below & ~seg_hi & gm;                // md lanes of my segment from me on
            const int last = mine ? 31 - __clz(mine) : gl;
            const int32_t end = __shfl_sync(gmask, ox + (int32_t)rl, sh + last, 32);
            if (first) {
                int64_t lo = (int64_t)ox - d.R0, hi = (int64_t)end - d.R0;
                if (lo < 0) lo = 0;
                if (hi > d.W) hi = d.W;
                mark_range(d.covE, d.upE, lo, hi);
            }
        }
        x += __shfl_sync(gmask, ir, G - 1, G);
        y += __shfl_sync(gmask, iq, G - 1, G);
    }
    if (gl == 0) {
        d.admit[r] = ok ? 1 : 0;
        const int32_t end = pos + (int32_t)x;
        d.read_end[r] = b > a ? end : pos;
        if (ok) {                                        // the read's whole span
            atomicMax(&d.blockmax[r >> 8], end);
            int64_t lo = (int64_t)pos - d.R0, hi = (int64_t)end - d.R0;
            if (lo < 0) lo = 0;
            if (hi > d.W) hi = d.W;
            mark_range(d.covA, d.upA, lo, hi);
        }
    }
}

// Genotyping mode: a known site is a candidate even in the middle of an intron, where the columns only carry
// `>` / `<`; marking the site like an aligned base gives it and its 16 neighbours on each side count rows.
__global__ void k_mark_known(Dev d) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d.n_known) return;
    const int64_t o = (int64_t)d.known[i] - 1 - d.R0;
    if (o >= 0 && o < d.W) atomicOr(&d.covE[o >> 5], 1u << (o & 31));
}

// -------------------------------------------- S3: rows = dilate16(E) & A, rank
// rowR word from covA word `a` and the covE words below / at / above it
__device__ __forceinline__ uint32_t row_word(const Dev& d, int64_t w, uint32_t a, uint32_t e0, uint32_t e1, uint32_t e2) {
    if (a == 0u) return 0u;                          // most of a contig: no read, no row
    // 96-bit smear by 16 to the left and to the right; only the middle word is needed
    unsigned long long lo = ((unsigned long long)e1 << 32) | e0;      // positions of (w-1, w)
    unsigned long long hi = ((unsigned long long)e2 << 32) | e1;      // positions of (w, w+1)
    unsigned long long up = lo;                                       // smear towards higher bits
    up |= up << 1; up |= up << 2; up |= up << 4; up |= up << 8; up |= up << 1;   // 1+2+4+8+1 = 16
    unsigned long long dn = hi;                                       // smear towards lower bits
    dn |= dn >> 1; dn |= dn >> 2; dn |= dn >> 4; dn |= dn >> 8; dn |= dn >> 1;
    const uint32_t dil = (uint32_t)(up >> 32) | (uint32_t)dn;
    const int64_t last = d.W - (w << 5);             // clear bits beyond the region end
    if (last < 32) a &= last <= 0 ? 0u : (0xffffffffu >> (32 - last));
    return dil & a;
}

// exclusive prefix of a[0 .. n) in place by ONE block of 256 threads (8 values per thread and round); the values were
// written by other blocks of the same kernel (read through L2).  Returns the total to thread 255 only.
__device__ int32_t block_scan_inplace_256(int32_t* a, int n, int32_t* wsum8, int32_t* carry_s) {
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) *carry_s = 0;
    int32_t total = 0;
    for (int b0 = 0; b0 < n; b0 += 2048) {
        const int i0 = b0 + 8 * t;
        int32_t v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = i0 + k < n ? __ldcg(a + i0 + k) : 0;
        int32_t own = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) own += v[k];
        int32_t x = own;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
        __syncthreads();                             // wsum8 / carry_s of the previous round are consumed
        if (lane == 31) wsum8[warp] = x;
        __syncthreads();
        int32_t run = *carry_s + x - own;
#pragma unroll
        for (int w = 0; w < 8; ++w) if (w < warp) run += wsum8[w];
#pragma unroll
        for (int k = 0; k < 8; ++k) { if (i0 + k < n) a[i0 + k] = run; run += v[k]; }
        total = run;
        __syncthreads();
        if (t == 255) *carry_s = run;
    }
    __syncthreads();
    return total;
}

// Position space in two elementwise kernels over tiles of PT_WORDS bitmap words (thread = 4 consecutive words, 16-byte
// accesses) instead of two device-wide scans over all words - 98 % of the words of a contig carry no row:
//   k_row_bits  folds the summary levels into covA / covE (covA is written back: the printed-column tests read it),
//               builds rowR and counts the rows of the tile; the last block to finish turns the tile counts into
//               their exclusive prefix (a few thousand values) and publishes the row count
//   k_row_rank  word_base, row_pos, and zeroes the row-space accumulators of the tile's rows (what k_clear_rows did)
__global__ void __launch_bounds__(256) k_row_bits(Dev d) {
    __shared__ uint32_t sE[PT_WORDS + 2];            // folded covE of the tile, one halo word on each side
    __shared__ int32_t wsum[8];
    __shared__ int32_t carry_s;
    __shared__ bool is_last;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int64_t w0 = (int64_t)blockIdx.x * PT_WORDS;
    const int64_t w4 = w0 + 4 * t;
    uint32_t a[4] = {0u, 0u, 0u, 0u}, e[4] = {0u, 0u, 0u, 0u};
    if (w4 < d.NW) {                                 // the bitmaps hold NW + 4 zeroed words
        const uint4 A = *(const uint4*)(d.covA + w4);
        const uint32_t mA = up_full4(d.upA, w4);
        a[0] = A.x; a[1] = A.y; a[2] = A.z; a[3] = A.w;
        // covE is a subset of covA (every M/D op lies inside its read's span): where no read covers anything - 98 % of
        // a chromosome - the covE words and their summary levels need not even be read
        // (genotyping mode marks known sites in covE whether a read covers them or not: no short cut there)
        if ((A.x | A.y | A.z | A.w | mA) != 0u || d.n_known > 0) {
            const uint4 E = *(const uint4*)(d.covE + w4);
            const uint32_t mE = up_full4(d.upE, w4);
            e[0] = E.x; e[1] = E.y; e[2] = E.z; e[3] = E.w;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (w4 + j >= d.NW) { a[j] = 0u; e[j] = 0u; continue; }
                if ((mA >> j) & 1u) a[j] = 0xffffffffu;
                if ((mE >> j) & 1u) e[j] = 0xffffffffu;
            }
            if (mA) *(uint4*)(d.covA + w4) = make_uint4(a[0], a[1], a[2], a[3]);
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) sE[1 + 4 * t + j] = e[j];
    if (t == 0) sE[0] = w0 > 0 ? (up_full(d.upE, w0 - 1) ? 0xffffffffu : d.covE[w0 - 1]) : 0u;
    if (t == 32) {
        const int64_t w = w0 + PT_WORDS;
        sE[PT_WORDS + 1] = w < d.NW ? (up_full(d.upE, w) ? 0xffffffffu : d.covE[w]) : 0u;
    }
    __syncthreads();
    uint32_t rr[4];
    int32_t cnt = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        rr[j] = row_word(d, w4 + j, a[j], sE[4 * t + j], sE[4 * t + j + 1], sE[4 * t + j + 2]);
        cnt += __popc(rr[j]);
    }
    *(uint4*)(d.rowR + w4) = make_uint4(rr[0], rr[1], rr[2], rr[3]);      // buffers are padded to whole tiles
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) wsum[warp] = cnt;
    __syncthreads();
    if (t == 0) {
        int32_t tot = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) tot += wsum[i];
        d.ptile[blockIdx.x] = tot;
        __threadfence();
        is_last = atomicAdd(&d.kctr[0], 1) == (int)gridDim.x - 1;
        carry_s = 0;
    }
    __syncthreads();
    if (!is_last) return;
    // ---- the last block: exclusive prefix of the tile counts in place
    __threadfence();
    const int n = (int)gridDim.x;
    const int32_t total = block_scan_inplace_256(d.ptile, n, wsum, &carry_s);
    if (t == 255) {
        d.ptile[n] = total;
        *d.n_rows = total;
        if (total > d.L_ub) atomicExch(d.err, 1);
    }
}

__global__ void __launch_bounds__(256) k_row_rank(Dev d) {
    __shared__ int32_t wsum[8];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int NC = d.C == 30 ? 6 : 4;
    const int64_t w4 = (int64_t)blockIdx.x * PT_WORDS + 4 * t;
    const int32_t tile_base = d.ptile[blockIdx.x], tile_end = d.ptile[blockIdx.x + 1];
    if (tile_end == tile_base && blockIdx.x != gridDim.x - 1 && blockIdx.x != 0) {
        // a tile without rows (98 % of them): every word has the same rank, nothing to zero (block-uniform exit)
        *(int4*)(d.word_base + w4) = make_int4(tile_base, tile_base, tile_base, tile_base);
        return;
    }
    const uint4 R = *(const uint4*)(d.rowR + w4);
    const uint32_t r[4] = {R.x, R.y, R.z, R.w};
    const int32_t c0 = __popc(r[0]), c1 = __popc(r[1]), c2 = __popc(r[2]), c3 = __popc(r[3]);
    int32_t x = c0 + c1 + c2 + c3;
    const int32_t own = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    int32_t b = tile_base + x - own;
#pragma unroll
    for (int i = 0; i < 8; ++i) if (i < warp) b += wsum[i];
    *(int4*)(d.word_base + w4) = make_int4(b, b + c0, b + c0 + c1, b + c0 + c1 + c2);
    if (own) {
        int32_t idx = b;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int32_t p0 = d.R0 + (int32_t)((w4 + j) << 5);
            if (r[j] == 0xffffffffu) {                   // the usual case inside an exon
                for (int q = 0; q < 32; ++q) if (idx + q < d.L_ub) d.row_pos[idx + q] = p0 + q;
                idx += 32;
            } else {
                for (uint32_t m = r[j]; m; m &= m - 1) { if (idx < d.L_ub) d.row_pos[idx] = p0 + __ffs(m) - 1; ++idx; }
            }
        }
    }
    // ---- zero the row-space accumulators of the tile's rows; the last tile also takes the two slack rows
    int64_t z0 = tile_base, z1 = tile_end;
    if (blockIdx.x == gridDim.x - 1) z1 += 2;
    if (z1 > d.L_ub + 2) z1 = d.L_ub + 2;
    for (int64_t i = z0 + t; i < z1; i += 256) {
        d.binc[i] = 0;
        d.bin_cur[i] = 0;
        for (int c = 0; c < NC; ++c) d.cov[i * NC + c] = 0;
        if (d.padding) {
            d.head_cnt[i] = 0; d.tail_cnt[i] = 0;
            Int2 z; z.a = 0; z.b = 0;
            d.skipdiff[i] = z;
            d.deleted[i] = 0;
        }
    }
    if (blockIdx.x == 0)
        for (int64_t i = t; i < d.L_ub / (64 * COV_TILE) + 2; i += 256) d.csuper[i] = 0;
    for (int64_t i = z0 / COV_TILE + t; i <= (z1 > z0 ? (z1 - 1) / COV_TILE : z0 / COV_TILE); i += 256) d.ctile[i] = 0;
    if (z1 > z0) {                                       // coverage tiles these rows fall into (neighbours overlap: all zero)
        const int64_t ct0 = z0 / COV_TILE, ct1 = (z1 - 1) / COV_TILE + 1;
        for (int64_t i = ct0 * NC + t; i < (ct1 + 1) * NC; i += 256) d.cov_tile[i] = 0;
    }
}

__device__ __forceinline__ uint32_t nibmask(int n) {         // low n nibbles set, n clamped to 0..8
    uint32_t m;                                              // shl.b32 clamps the shift amount: 1 << 32 == 0
    asm("shl.b32 %0, 1, %1;" : "=r"(m) : "r"((uint32_t)(n < 0 ? 0 : 4 * n)));
    return m - 1u;
}

// ------------------------------------------------ reference as one-hot nibbles
// refnib: one 4-bit code per reference position of the loaded window (A=1, C=2, G=4, T=8 like BAM's
// nt16, anything else 0), position i of the window at bits 4*(i&7) of word i>>3.  Built once per
// reference window; read bases are compared against it eight at a time.
__global__ void k_refnib(const uint8_t* __restrict__ ref, int64_t ref_len, uint32_t* __restrict__ out, int64_t n_words) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_words) return;
    uint32_t v = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int64_t o = w * 8 + j;
        uint8_t c = o < ref_len ? ref[o] : (uint8_t)'N';
        if (c >= 'a') c -= 32;
        const uint32_t nib = c == 'A' ? 1u : c == 'C' ? 2u : c == 'G' ? 4u : c == 'T' ? 8u : 0u;
        v |= nib << (4 * j);
    }
    out[w] = v;
}

// --------------------------------------------------- row events: compare pass
// K2 counts relative to the reference: a read base that equals the reference base leaves no trace of
// its own; it is accounted for by the per-strand coverage of its op (a +1/-1 pair in the row-space
// difference array `cov`, prefix-summed in k_rows).  Only bases that differ from the reference (1-3 % of
// them), N / ambiguity codes, and the indel tokens become *row events*.
//   ref-base count of a row = coverage - mismatch events;  other bases = their mismatch events.
// k_cmp: one thread per CIGAR op for the bookkeeping; the sequence words of a warp's 32 ops are then dealt
// out to its lanes one word each.  Read bases are compared 8 at a time (one 32-bit word of nt16 nibbles against the one-hot reference
// nibbles, funnel-shifted into register).  Events are staged in shared memory and appended to the raw
// list with one global atomic per flush; k_scatter_aggr then counting-sorts them by row (CSR).
constexpr int NCOV_MAX = 6;                  // Mf Mr Df Dr [M_hp1 M_hp2]
constexpr int CMP_THREADS = 256;
constexpr int CMP_STAGE = 1536;              // events staged per block (24 KB)

struct __align__(16) CmpOp {                 // an M/=/X op clipped to the region (32 bytes: two 16-byte shared loads)
    int32_t w0, w1;                          // sequence words [w0, w1] holding its bases
    int32_t kw;                              // reference-nibble word of sequence word w: w + kw
    uint32_t sh;                             // funnel shift (bits) between the two
    int32_t rbase;                           // row of base 8*w + j: rbase + 8*w + j
    uint32_t info;                           // rid << 4 | hp << 2 | rev   (is_del bit clear)
    uint32_t m0, m1;                         // nibbles of word w0 / of word w1 that belong to the op
};

struct EventStage {
    RowEvent buf[CMP_STAGE];
    int n;
    int base;
};

__device__ __forceinline__ void emit_event(const Dev& d, EventStage& st, int32_t row, uint32_t info, int32_t len, uint32_t yb) {
    RowEvent e;
    e.info = info; e.len = len; e.yb = yb; e.row = row;
    const int i = atomicAdd(&st.n, 1);
    if (i < CMP_STAGE) { st.buf[i] = e; return; }
    const long long slot = (long long)atomicAdd((unsigned long long*)d.n_raw, 1ull);     // stage full: straight to the list
    if (slot < d.events_ub) { d.raw[slot] = e; atomicAdd(&d.binc[row], 1); } else atomicExch(d.err, 3);
}

__device__ __forceinline__ void cmp_emit(const Dev& d, EventStage& st, const CmpOp& c, int32_t w, uint32_t rw, uint32_t x) {
    while (x) {
        const int j = (__ffs(x) - 1) >> 2;
        x &= ~(0xfu << (4 * j));
        const uint32_t nib = (rw >> (4 * j)) & 15u;
        const uint32_t code = nib == 1 ? 0u : nib == 2 ? 1u : nib == 4 ? 2u : nib == 8 ? 3u : 4u;
        emit_event(d, st, c.rbase + 8 * w + j, c.info, 0, code);
    }
}

// sequence word w (8 bases) of one op against the reference
__device__ __forceinline__ void cmp_one(const Dev& d, EventStage& st, const CmpOp& c, int32_t w) {
    uint32_t rw = ((const uint32_t*)d.seq)[w];
    rw = ((rw & 0x0f0f0f0fu) << 4) | ((rw >> 4) & 0x0f0f0f0fu);              // base j of the word at bits 4j..4j+3
    const int32_t wi = w + c.kw;
    uint32_t f0, f1;
    if ((uint32_t)wi < (uint32_t)(d.n_ref_words - 1)) { f0 = d.refnib[wi]; f1 = d.refnib[wi + 1]; }
    else {                                                                   // op reaches over an end of the loaded reference
        f0 = (wi >= 0 && wi < d.n_ref_words) ? d.refnib[wi] : 0u;
        f1 = (wi + 1 >= 0 && wi + 1 < d.n_ref_words) ? d.refnib[wi + 1] : 0u;
    }
    uint32_t x = rw ^ __funnelshift_r(f0, f1, c.sh);
    x &= (w == c.w0 ? c.m0 : 0xffffffffu) & (w == c.w1 ? c.m1 : 0xffffffffu);
    if (x) cmp_emit(d, st, c, w, rw, x);
}

// staged events -> raw list (one global atomic per flush), per-row counters
__device__ __forceinline__ void cmp_flush(const Dev& d, EventStage& st) {
    __syncthreads();
    const int n = st.n < CMP_STAGE ? st.n : CMP_STAGE;
    if (threadIdx.x == 0 && n > 0) st.base = (int)atomicAdd((unsigned long long*)d.n_raw, (unsigned long long)n);
    __syncthreads();
    if (n > 0) {
        const long long base = st.base;
        if (base + n > d.events_ub) { if (threadIdx.x == 0) atomicExch(d.err, 3); }
        else {
            for (int i = threadIdx.x; i < n; i += CMP_THREADS) {
                const RowEvent e = st.buf[i];
                d.raw[base + i] = e;
                atomicAdd(&d.binc[e.row], 1);
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) st.n = 0;
    __syncthreads();
}

// Persistent blocks: a block walks chunks of CMP_THREADS ops and appends its staged events to the raw list when
// the stage is half full - a few hundred atomics on the list's end counter per pass instead of one per 256 ops
// (same-address atomics are served one per ~27 cycles: 4 135 of them were most of this kernel's 63 us).
__global__ void __launch_bounds__(CMP_THREADS) k_cmp(Dev d) {
    __shared__ EventStage st;
    __shared__ CmpOp wops[CMP_THREADS / 32][32];         // the warp's ops, so that any lane can take any word
    __shared__ int32_t wpre[CMP_THREADS / 32][32];       // exclusive prefix of their word counts
    const int lane = threadIdx.x & 31;
    const int NC = d.C == 30 ? 6 : 4;
    if (*d.err == 1) return;                             // more rows than the buffers hold: the host retries with exact bounds
    __shared__ int chunk_s;
    if (threadIdx.x == 0) st.n = 0;
    // chunks of CMP_THREADS ops are handed out by a counter: a chunk's cost goes with the bases under its ops (a HiFi
    // match of kilobases next to 3-base exon ends), a static split leaves the blocks finishing far apart
    for (;;) {
    if (threadIdx.x == 0) chunk_s = atomicAdd(&d.kctr[3], 1);
    __syncthreads();
    const int64_t k0 = (int64_t)chunk_s * CMP_THREADS;
    if (k0 >= d.n_ops) break;
    const int64_t k = k0 + threadIdx.x;
    CmpOp cmp;
    cmp.w0 = 0; cmp.w1 = -1; cmp.kw = 0; cmp.sh = 0; cmp.rbase = 0; cmp.info = 0; cmp.m0 = 0; cmp.m1 = 0;
    do {
        if (k >= d.n_ops) break;
        const uint32_t oi = d.op_info[k];                // from k_cigar: read ordinal, haplotype, strand, last-op flag
        if (oi == OP_SKIP) break;                        // read not admitted
        const int32_t r = (int32_t)(oi >> 4);
        const uint32_t c = d.cigar[k];
        const uint32_t op = c & 15u;
        const int32_t len = (int32_t)(c >> 4);
        if (!op_consumes_ref(op) || len == 0) break;
        const int32_t x = d.op_x[k];
        const uint32_t rev = oi & 1u;
        const uint32_t hp = (oi >> 2) & 3u;
        const int32_t a = x < d.R0 ? d.R0 : x;
        const int32_t b = x + len > d.R1 ? d.R1 : x + len;

        if (op == 3) {                                   // N: `>` / `<` over [a, b)
            if (d.padding && b > a) {
                const int32_t ra = row_lower_bound(d, a), rb = row_lower_bound(d, b);
                if (rb > ra) {
                    int32_t* f = rev ? &d.skipdiff[0].b : &d.skipdiff[0].a;
                    atomicAdd(&f[2 * (int64_t)ra], 1);
                    atomicAdd(&f[2 * (int64_t)rb], -1);
                }
            }
            break;
        }
        if (b > a) {                                     // M/=/X or D segment: rows ra .. ra + (b - a) - 1 are consecutive
            const int32_t ra = row_lower_bound(d, a), rb = ra + (b - a);
            const int ch = (op == 2 ? 2 : 0) + (int)rev;
            atomicAdd(d.cov + (int64_t)ra * NC + ch, 1);
            atomicAdd(d.cov + (int64_t)rb * NC + ch, -1);
            const bool hpc = NC == 6 && op != 2 && hp;
            if (hpc) { atomicAdd(d.cov + (int64_t)ra * NC + 3 + hp, 1); atomicAdd(d.cov + (int64_t)rb * NC + 3 + hp, -1); }
            if (ra / COV_TILE != rb / COV_TILE) {        // the pair straddles coverage tiles: keep the tile sums right
                atomicAdd(d.cov_tile + (int64_t)(ra / COV_TILE) * NC + ch, 1);
                atomicAdd(d.cov_tile + (int64_t)(rb / COV_TILE) * NC + ch, -1);
                if (hpc) {
                    atomicAdd(d.cov_tile + (int64_t)(ra / COV_TILE) * NC + 3 + hp, 1);
                    atomicAdd(d.cov_tile + (int64_t)(rb / COV_TILE) * NC + 3 + hp, -1);
                }
            }
            if (op != 2) {
                const int64_t qa = (int64_t)d.op_y[k] + (a - x);             // base index of position a
                const int64_t qb = qa + (b - a);
                cmp.w0 = (int32_t)(qa >> 3); cmp.w1 = (int32_t)((qb - 1) >> 3);
                cmp.m0 = ~nibmask((int)(qa & 7)); cmp.m1 = nibmask((int)(qb - 8 * (int64_t)cmp.w1));
                const int64_t K = ((int64_t)a - d.ref_start0) - qa;          // reference offset of base q: q + K
                cmp.kw = (int32_t)(K >> 3);
                cmp.sh = ((uint32_t)K & 7u) * 4u;
                cmp.rbase = (int32_t)((int64_t)ra - qa);
                cmp.info = oi & ~2u;
            }
        }
        // head / tail marks (only consumed by the padding rule)
        if (d.padding) {
            if (x == d.pos[r] && x >= d.R0 && x < d.R1) {
                bool first = true;                       // first reference-consuming op of the read
                for (int32_t j = d.cigar_off[r]; j < k; ++j)
                    if (op_consumes_ref(d.cigar[j] & 15u) && (d.cigar[j] >> 4)) first = false;
                if (first) atomicAdd(&d.head_cnt[row_lower_bound(d, x)], 1);
            }
            const int32_t end = d.read_end[r];
            if (x + len == end && end - 1 >= d.R0 && end - 1 < d.R1)
                atomicAdd(&d.tail_cnt[row_lower_bound(d, end - 1)], 1);
        }
        // indel tokens attach to the last column of an M/=/X/D op (htslib resolve_cigar2)
        const int32_t last = x + len - 1;
        if (last < d.R0 || last >= d.R1) break;
        if (oi & 2u) break;                              // last op of its read: nothing follows
        int64_t j = k + 1;
        bool more = true;                                // op j belongs to this read
        int32_t ins_len = 0, del_len = 0;
        const uint32_t op2 = d.cigar[j] & 15u;
        if (op2 != 1 && !(op2 == 2 && op != 2)) break;
        if (op2 == 1) {
            while (more) {
                const uint32_t cj = d.cigar[j], o = cj & 15u;
                if (o == 1) ins_len += (int32_t)(cj >> 4);
                else if (o != 6) break;
                more = !(d.op_info[j] & 2u);
                ++j;
            }
        }
        if (more && (d.cigar[j] & 15u) == 2 && op != 2) {
            while (more) {
                const uint32_t cj = d.cigar[j];
                if ((cj & 15u) != 2) break;
                del_len += (int32_t)(cj >> 4);
                more = !(d.op_info[j] & 2u);
                ++j;
            }
        }
        if (!ins_len && !del_len) break;
        const int32_t row = row_lower_bound(d, last);
        for (int which = 0; which < 2; ++which) {
            const int32_t l = which ? del_len : ins_len;
            if (!l) continue;
            // inserted bases start right after this op's query bases (M) or at its query position (D)
            emit_event(d, st, row, ((uint32_t)r << 4) | (hp << 2) | ((uint32_t)which << 1) | rev, l,
                       d.op_y[k] + (op_is_match(op) ? (uint32_t)len : 0u));
        }
    } while (0);

    // ---- read bases against the reference: the words of the warp's 32 ops are dealt out lane by lane, so lanes
    // stay busy whatever the op lengths (M ops of 3 bases next to HiFi matches of kilobases)
    {
        const int warp = threadIdx.x >> 5;
        const int32_t cnt = cmp.w1 - cmp.w0 + 1;         // 0 for everything that is not an M/=/X op
        int32_t incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int32_t y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
        const int32_t total = __shfl_sync(0xffffffffu, incl, 31);
        wops[warp][lane] = cmp;
        wpre[warp][lane] = incl - cnt;
        __syncwarp();
        for (int32_t g = lane; g < total; g += 32) {
            int i = 0;                                   // last op whose prefix is <= g (ops without words share a prefix
#pragma unroll                                           // with their successor, so the last one is the owner)
            for (int stp = 16; stp > 0; stp >>= 1) if (wpre[warp][i + stp] <= g) i += stp;
            const CmpOp c = wops[warp][i];
            cmp_one(d, st, c, c.w0 + (g - wpre[warp][i]));
        }
    }
    __syncthreads();
    const bool fl = st.n >= CMP_STAGE / 2;               // block-uniform: read between two barriers
    __syncthreads();
    if (fl) cmp_flush(d, st);
    }
    cmp_flush(d, st);
}

// exclusive scan of the per-row event counters in place
struct OpEvents {
    typedef int32_t T;
    struct Ctx {};
    Dev d;
    __device__ void ctx_init(Ctx&) const {}
    __device__ T identity() const { return 0; }
    __device__ T combine(const T& x, const T& y) const { return x + y; }
    __device__ int64_t size() const { return *d.n_rows + 1; }
    __device__ T load(int64_t i) const { return d.binc[i]; }
    __device__ void store(int64_t i, const T& incl, const T& own, Ctx&) const { d.binc[i] = incl - own; }
};
struct OpSkip {
    typedef Int2 T;
    struct Ctx {};
    Dev d;
    __device__ void ctx_init(Ctx&) const {}
    __device__ T identity() const { T t; t.a = 0; t.b = 0; return t; }
    __device__ T combine(const T& x, const T& y) const { T t; t.a = x.a + y.a; t.b = x.b + y.b; return t; }
    __device__ int64_t size() const { return *d.n_rows; }
    __device__ T load(int64_t i) const { return d.skipdiff[i]; }
    __device__ void store(int64_t i, const T& incl, const T&, Ctx&) const {
        // '>' forward skips, '<' reverse skips, '^' heads, '$' tails (create_tensor_pileup.py:178)
        int32_t m = incl.a > incl.b ? incl.a : incl.b;
        const int32_t h = d.head_cnt[i], t = d.tail_cnt[i];
        m = m > h ? m : h;
        m = m > t ? m : t;
        d.max_skip[i] = m;
    }
};

// ------------------------------------------------------------- site filters
// index of the last interval whose start is <= q, or -1
__device__ __forceinline__ int iv_last_start_le(const int32_t* iv, int n, int32_t q) {
    int lo = 0, hi = n;                                  // first interval with start > q
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (iv[2 * mid] <= q) lo = mid + 1; else hi = mid; }
    return lo - 1;
}
// [a, b) lies inside one interval (the intervals do not touch, so a gap-free run cannot span two)
__device__ __forceinline__ bool iv_contains(const int32_t* iv, int n, int32_t a, int32_t b) {
    const int k = iv_last_start_le(iv, n, a);
    return k >= 0 && iv[2 * k + 1] >= b;
}
// some interval has start < b and end > a (IntervalTree.overlap, shared/interval_tree.py:80-89)
__device__ __forceinline__ bool iv_overlaps(const int32_t* iv, int n, int32_t a, int32_t b) {
    const int k = iv_last_start_le(iv, n, b - 1);
    return k >= 0 && iv[2 * k + 1] > a;
}
__device__ __forceinline__ bool known_site(const int32_t* ks, int n, int32_t pos1) {
    int lo = 0, hi = n;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (ks[mid] < pos1) lo = mid + 1; else hi = mid; }
    return lo < n && ks[lo] == pos1;
}

// printed columns of word w: covA restricted to the pileup BED (mpileup -l)
__global__ void k_bed_mask(Dev d, uint32_t* out) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= d.NW + 4) return;
    uint32_t bits = 0u;
    const uint32_t a = w < d.NW ? d.covA[w] : 0u;
    if (a) {
        const int64_t lo = (int64_t)d.R0 + (w << 5), hi = lo + 32;           // genome positions of the word
        for (int k = iv_last_start_le(d.pbed, d.n_pbed, (int32_t)(hi - 1)); k >= 0 && d.pbed[2 * k + 1] > lo; --k) {
            const int64_t x = d.pbed[2 * k] > lo ? d.pbed[2 * k] - lo : 0, y = d.pbed[2 * k + 1] < hi ? d.pbed[2 * k + 1] - lo : 32;
            bits |= (y >= 32 ? 0xffffffffu : (1u << y) - 1u) & (0xffffffffu << x);
        }
    }
    out[w] = a & bits;
}
// head/tail mode: the last printed column of the stream and the last gap below it (the final run starts after it)
__global__ void k_last_col(Dev d) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= d.NW) return;
    const uint32_t b = d.covP[w];
    if (b) atomicMax(&d.tail[0], (int32_t)(w << 5) + 32 - __clz(b));
}
__global__ void k_last_gap(Dev d) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int32_t last = d.tail[0] - 1;
    if (last < 0 || w > (last >> 5)) return;
    uint32_t m = ~d.covP[w];
    if (w == (last >> 5)) m &= (1u << (last & 31)) - 1u;
    if (m) atomicMax(&d.tail[1], (int32_t)(w << 5) + 32 - __clz(m));
}
// printed columns right below / above region offset o, up to 16 each (the part of the 33-column window that lies in
// the candidate's own run)
__device__ __forceinline__ void printed_run(const Dev& d, int64_t o, int* n_before, int* n_after) {
    const int64_t w = o >> 5;
    const unsigned long long up = (d.covP[w] | ((unsigned long long)d.covP[w + 1] << 32)) >> (o & 31);   // bit 0 = o
    const int na = __ffsll((long long)~(up >> 1)) - 1;
    *n_after = na > FLANK ? FLANK : na;
    const int64_t s = o - FLANK < 0 ? 0 : o - FLANK;
    const int wb = (int)(o - s);                                                                         // columns s .. o-1
    int nb = 0;
    if (wb > 0) {
        const int64_t ws = s >> 5;
        const unsigned long long dn = (d.covP[ws] | ((unsigned long long)d.covP[ws + 1] << 32)) >> (s & 31);   // bit 0 = s
        const unsigned long long x = ~dn << (64 - wb);                    // bit 63 = column o-1
        nb = x ? __clzll((long long)x) : wb;
        if (nb > wb) nb = wb;
    }
    *n_before = nb;
}

// ------------------------------------------------------------- K2: rows
__device__ __forceinline__ bool ins_equal(const Dev& d, const RowEvent& a, const RowEvent& b, bool fold_strand) {
    if (a.len != b.len) return false;
    if (!fold_strand && ((a.info ^ b.info) & 1u)) return false;
    for (int32_t i = 0; i < a.len; ++i)
        if (nib_at(d.seq, a.yb + i) != nib_at(d.seq, b.yb + i)) return false;
    return true;
}

// first read (BAM order) that shows the reference base at position p, as key rid * 2.  Reference-relative
// counting keeps no per-read record of matching bases, so this walks reads: it starts at the first block of 256 reads
// whose running maximum of read ends passes p (no earlier read can reach p) and stops at the first read starting
// after p.  Only count ties ask for it.
__device__ uint32_t first_ref_read(const Dev& d, int32_t p, uint32_t ref_nib) {
    const int64_t n_blocks = (d.n_reads + 255) >> 8;
    int64_t b = 0;
    while (b < n_blocks && d.blockmax[b] <= p) ++b;
    for (int64_t r = b << 8; r < d.n_reads && d.pos[r] <= p; ++r) {
        if (!d.admit[r] || d.read_end[r] <= p) continue;
        int32_t x = d.pos[r];
        uint32_t y = (uint32_t)d.seq_off[r];
        for (int32_t k = d.cigar_off[r]; k < d.cigar_off[r + 1]; ++k) {
            const uint32_t c = d.cigar[k], op = c & 15u;
            const int32_t len = (int32_t)(c >> 4);
            if (op_consumes_ref(op)) {
                if (p < x + len) {
                    if (op_is_match(op) && nib_at(d.seq, y + (uint32_t)(p - x)) == ref_nib) return (uint32_t)r * 2u;
                    break;
                }
                x += len;
            }
            if (op_consumes_qry(op)) y += (uint32_t)len;
        }
    }
    return 0xffffffffu;
}

// first-occurrence key (read ordinal * 2 + is_indel_token) of each allele class at a row;
// only needed to break count ties the way Counter/dict insertion order does.
__device__ void first_keys(const Dev& d, int32_t row, int32_t p, int ri, bool acgt, uint32_t key[6]) {
    for (int i = 0; i < 6; ++i) key[i] = 0xffffffffu;
    const int32_t e0 = d.binc[row] - d.binc[0], e1 = d.binc[row + 1] - d.binc[0];
    for (int32_t s = e0; s < e1; ++s) {
        const RowEvent e = d.events[s];
        int c;
        uint32_t kk = (e.info >> 4) * 2u;
        if (e.len == 0) { if (e.yb > 3u) continue; c = (int)e.yb; }
        else { c = (e.info & 2u) ? 5 : 4; kk += 1u; }
        if (kk < key[c]) key[c] = kk;
    }
    if (acgt) key[ri] = first_ref_read(d, p, 1u << ri);
}

// allele-frequency thresholds as integer tables: thr[depth] = smallest count c >= 1 with
// (double)c / (double)max(depth, 1) >= af, the reference's float64 test (create_tensor_pileup.py:270-277)
// evaluated once per depth instead of once per row and class.  Depths >= THR_N use the division.
constexpr int THR_N = 4096;
__global__ void k_thr_table(uint16_t* thr_snp, uint16_t* thr_indel, double snp_af, double indel_af) {
    const int dpt = blockIdx.x * blockDim.x + threadIdx.x;
    if (dpt >= THR_N) return;
    const double den = dpt > 0 ? (double)dpt : 1.0;
    for (int which = 0; which < 2; ++which) {
        const double af = which ? indel_af : snp_af;
        int c = 1;
        const int lim = dpt > 1 ? dpt : 1;
        while (c <= lim && !((double)c / den >= af)) ++c;
        (which ? thr_indel : thr_snp)[dpt] = (uint16_t)(c <= lim ? c : 0xffff);
    }
}

// raw events -> CSR by row (counting sort: the scan above made binc the bin offsets); block 0 meanwhile turns the
// coverage tile sums into their exclusive prefix, in place (one tile per 256 rows: a few thousand values, a job for
// one block that used to be a 12 us kernel of its own between the scatter and k_rows)
template <int NC>
__global__ void __launch_bounds__(1024) k_scatter_aggr(Dev d) {
    if (*d.err == 1) return;
    if (blockIdx.x != 0) {
        const int64_t n = *d.n_raw < d.events_ub ? *d.n_raw : d.events_ub;
        const int64_t stride = (int64_t)(gridDim.x - 1) * blockDim.x;
        const int32_t b0 = d.binc[0];
        for (int64_t i = (int64_t)(blockIdx.x - 1) * blockDim.x + threadIdx.x; i < n; i += stride) {
            const RowEvent e = d.raw[i];
            const int64_t slot = (int64_t)d.binc[e.row] - b0 + atomicAdd(&d.bin_cur[e.row], 1);
            d.events[slot] = e;
        }
        return;
    }
    __shared__ int32_t wtot[32][NC];
    __shared__ int32_t carry[NC];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t nt = *d.n_rows / COV_TILE + 1;
    if (threadIdx.x < NC) carry[threadIdx.x] = 0;
    __syncthreads();
    for (int64_t b0 = 0; b0 < nt; b0 += 1024) {
        const int64_t i = b0 + threadIdx.x;
        int32_t own[NC], x[NC];
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            own[c] = i < nt ? d.cov_tile[i * NC + c] : 0;
            x[c] = own[c];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int32_t y = __shfl_up_sync(0xffffffffu, x[c], o); if (lane >= o) x[c] += y; }
        }
        if (lane == 31)
#pragma unroll
            for (int c = 0; c < NC; ++c) wtot[warp][c] = x[c];
        __syncthreads();
        if (warp == 0) {                                 // scan of the 32 warp totals
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                int32_t t = wtot[lane][c];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const int32_t y = __shfl_up_sync(0xffffffffu, t, o); if (lane >= o) t += y; }
                wtot[lane][c] = t;                       // inclusive
            }
        }
        __syncthreads();
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const int32_t before = carry[c] + (warp ? wtot[warp - 1][c] : 0);
            if (i < nt) d.cov_tile[i * NC + c] = before + x[c] - own[c];
        }
        __syncthreads();
        if (threadIdx.x < NC) carry[threadIdx.x] += wtot[31][threadIdx.x];
        __syncthreads();
    }
}

// Distinct indel alleles among the n events of one row (mismatch events, len == 0, are skipped), enumerated by the
// whole warp: the first unassigned token becomes the leader and every lane compares its own tokens with it at once.
// An insertion compare is a chain of dependent sequence loads; done serially per pair it costs about a microsecond,
// which a het insertion under 500x coverage used to pay tens of thousands of times.  `done` is the warp's bitmap
// in shared memory (IND_WORDS words: rows of up to IND_MAX events; the callers walk longer rows serially).
// FOLD merges the two strands of an allele (alt_info keys are case-folded) and tracks the earliest read; without
// FOLD the strands stay apart (I1/D1 are per strand).
// visit(leader event, count, first-occurrence key, base index of the first occurrence's inserted bases).
constexpr int IND_WORDS = 128;
constexpr int IND_MAX = IND_WORDS * 32;
template <bool FOLD, class Visit>
__device__ __forceinline__ void for_each_indel_allele(const Dev& d, const RowEvent* evs, int n, int lane, uint32_t* done,
                                                      Visit visit) {
    const int nw = (n + 31) >> 5;
    for (int w = 0; w < nw; ++w) {
        const int q = w * 32 + lane;
        const uint32_t m = __ballot_sync(0xffffffffu, q >= n || evs[q < n ? q : n - 1].len == 0);
        if (lane == 0) done[w] = m;
    }
    __syncwarp();
    int w0 = 0;
    for (;;) {
        while (w0 < nw && done[w0] == 0xffffffffu) ++w0;
        if (w0 >= nw) break;
        const RowEvent ev = evs[w0 * 32 + __ffs(~done[w0]) - 1];
        const bool is_del = ev.info & 2u;
        int32_t cnt = 0;
        uint32_t first = 0xffffffffu, first_y = ev.yb;
        for (int w = w0; w < nw; ++w) {
            const uint32_t dw = done[w];
            if (dw == 0xffffffffu) continue;
            bool match = false;
            if (!((dw >> lane) & 1u)) {
                const RowEvent o = evs[w * 32 + lane];
                const bool same_kind = FOLD ? ((o.info ^ ev.info) & 2u) == 0 : ((o.info ^ ev.info) & 3u) == 0;
                match = same_kind && (is_del ? o.len == ev.len : ins_equal(d, o, ev, FOLD));
                if (match) {
                    const uint32_t kk = (o.info >> 4) * 2u + 1u;
                    if (kk < first) { first = kk; first_y = o.yb; }
                }
            }
            const uint32_t mm = __ballot_sync(0xffffffffu, match);
            cnt += __popc(mm);
            __syncwarp();                                    // every lane has read done[w] (keeps racecheck quiet: the ballot already orders them)
            if (lane == 0) done[w] = dw | mm;
        }
        __syncwarp();
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const uint32_t of = __shfl_xor_sync(0xffffffffu, first, o), oy = __shfl_xor_sync(0xffffffffu, first_y, o);
            if (of < first) { first = of; first_y = oy; }
        }
        visit(ev, cnt, first, first_y);
    }
}

// indel tokens of one row: per strand totals and the largest distinct allele per strand (I, I1, D, D1 and, phased,
// IP/DP/IM/DM) into the row vector v.  evs[0..n) may also hold mismatch events (len == 0), which are skipped.
template <int C>
__device__ void row_indels(const Dev& d, const RowEvent* evs, int32_t n, int32_t* v, int32_t& ins_cnt, int32_t& del_cnt) {
    for (int32_t s = 0; s < n; ++s) {
        const RowEvent e = evs[s];
        if (e.len == 0) continue;
        const uint32_t rev = e.info & 1u;
        const uint32_t hp = (e.info >> 2) & 3u;
        const bool is_del = e.info & 2u;
        if (is_del) { ++del_cnt; ++v[rev ? 15 : 6]; } else { ++ins_cnt; ++v[rev ? 13 : 4]; }
        if (C == 30) {
            if (hp == 1) ++v[is_del ? 23 : 22]; else if (hp == 2) ++v[is_del ? 29 : 28];
        }
        bool seen = false;
        for (int32_t q = 0; q < s && !seen; ++q) {
            const RowEvent o = evs[q];
            if (o.len != 0 && ((o.info ^ e.info) & 3u) == 0 && (is_del ? o.len == e.len : ins_equal(d, o, e, false))) seen = true;
        }
        if (seen) continue;
        int32_t same = 1;
        for (int32_t q = s + 1; q < n; ++q) {
            const RowEvent o = evs[q];
            if (o.len != 0 && ((o.info ^ e.info) & 3u) == 0 && (is_del ? o.len == e.len : ins_equal(d, o, e, false))) ++same;
        }
        const int ch = is_del ? (rev ? 16 : 7) : (rev ? 14 : 5);
        if (same > v[ch]) v[ch] = same;
    }
}

// K2 proper.  Block = one coverage tile of 256 rows (grid-stride); thread = row, warp = 32 consecutive
// rows.  Coverage = tile prefix + in-block prefix of the difference rows; the row's events give everything else:
// mismatching bases, I/I1/D/D1, phased channels; then the candidate predicate (integer AF threshold
// tables, first-occurrence tie-break) and the row leaves through shared memory as 16-byte coalesced stores.
// K3's test: the 33 columns c-16 .. c+16 are all printed (one gap-free run of covP): restates "pop when pos - c == 16
// and the ring has no empty slot" (create_tensor_pileup.py:565-568).  Head/tail mode: zero rows stand in for the
// columns before the run; the columns after it are only supplied when the stream ends, i.e. for the final run
// (create_tensor_pileup.py:508-511, 613-637).
// (out of line and with its operands by value: it runs for the few eligible rows only and must not cost k_rows registers)
__device__ __noinline__ bool window_printed(const uint32_t* covP, int64_t o, int64_t W, int head_tail, int32_t tail1) {
    if (head_tail) {
        if (!((covP[o >> 5] >> (o & 31)) & 1u)) return false;
        const unsigned long long up = (covP[o >> 5] | ((unsigned long long)covP[(o >> 5) + 1] << 32)) >> (o & 31);   // bit 0 = o
        const int na = __ffsll((long long)~(up >> 1)) - 1;                    // printed columns right above o (printed_run)
        return na >= FLANK || o >= tail1;
    }
    if (o - FLANK < 0 || o + FLANK >= W) return false;
    // 33 consecutive printed columns starting at o-16 (covP = covA inside the pileup BED: mpileup -l never prints
    // the others, so the ring buffer restarts there)
    const int64_t s = o - FLANK;
    const int64_t w = s >> 5;
    const int sh = (int)(s & 31);
    const unsigned long long lo = covP[w] | ((unsigned long long)covP[w + 1] << 32);
    const unsigned long long bits = lo >> sh;              // 64 - sh >= 33 bits are valid
    const unsigned long long need = (1ull << 33) - 1ull;
    return (bits & need) == need;
}

constexpr int ROWS_WARPS = 8;
constexpr int ROWS_HEAVY = 32;               // rows with more events than this are walked by the whole warp
#ifndef C3R_ROWS_BLOCKS
#define C3R_ROWS_BLOCKS 5
#endif
template <int C>
__global__ void __launch_bounds__(ROWS_WARPS * 32, C == 30 ? 4 : C3R_ROWS_BLOCKS) k_rows(Dev d) {
    constexpr int NC = C == 30 ? 6 : 4;
    static_assert(ROWS_WARPS * 32 == COV_TILE, "one block per coverage tile");
    __shared__ __align__(16) int32_t stage[ROWS_WARPS][TILE_ROWS * C];
    __shared__ uint32_t done_s[ROWS_WARPS][IND_WORDS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (*d.err == 1) return;                             // more rows than the buffers hold: the host retries with exact bounds
    const int64_t L = *d.n_rows;
    const int32_t ev_base = d.binc[0];
    for (int64_t tile = blockIdx.x; tile * COV_TILE < L; tile += gridDim.x) {
        const int64_t base = tile * COV_TILE;
        const int64_t row = base + threadIdx.x;
        const bool live = row < L;
        int32_t carry[NC];
#pragma unroll
        for (int c = 0; c < NC; ++c) carry[c] = d.cov_tile[tile * NC + c];
        // ---- operands of the row, requested together
        int32_t cv[NC];
#pragma unroll
        for (int c = 0; c < NC; ++c) cv[c] = 0;
        int32_t p = 0, e0 = 0, e1 = 0;
        uint8_t rc = (uint8_t)'N';
        if (live) {
            if (NC == 4) { const int4 t = *(const int4*)(d.cov + row * 4); cv[0] = t.x; cv[1] = t.y; cv[2] = t.z; cv[3] = t.w; }
            else {
                const int2* q = (const int2*)(d.cov + row * 6);
                const int2 t0 = q[0], t1 = q[1], t2 = q[2];
                cv[0] = t0.x; cv[1] = t0.y; cv[2] = t1.x; cv[3] = t1.y; cv[NC - 2] = t2.x; cv[NC - 1] = t2.y;
            }
            p = d.row_pos[row];
            e0 = d.binc[row] - ev_base; e1 = d.binc[row + 1] - ev_base;
            const int64_t ro = (int64_t)p - d.ref_start0;
            if (ro >= 0 && ro < d.ref_len) rc = d.ref[ro];
        }
        // ---- inclusive prefix of the coverage differences.  A warp works out its own starting coverage - the tile's
        // carry plus the difference rows of the warps before it in the tile, which it simply reads as well (the same
        // lines its neighbours load: cache hits) - so the tile loop has NO block barrier: a warp held up by a row with
        // hundreds of indel tokens used to hold the other seven at the barriers (30 % of this kernel's stall samples).
        int32_t pre[NC];
#pragma unroll
        for (int c = 0; c < NC; ++c) pre[c] = 0;
        for (int w = 0; w < warp; ++w) {
            const int64_t rw = base + w * 32 + lane;             // rows before this warp's rows
            if (rw >= L) continue;                               // (only in a warp that has no live row itself)
            if (NC == 4) { const int4 t = *(const int4*)(d.cov + rw * 4); pre[0] += t.x; pre[1] += t.y; pre[2] += t.z; pre[3] += t.w; }
            else {
                const int2* q = (const int2*)(d.cov + rw * 6);
                const int2 t0 = q[0], t1 = q[1], t2 = q[2];
                pre[0] += t0.x; pre[1] += t0.y; pre[2] += t1.x; pre[3] += t1.y; pre[NC - 2] += t2.x; pre[NC - 1] += t2.y;
            }
        }
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            int32_t x = cv[c];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
            int32_t b = pre[c];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) b += __shfl_xor_sync(0xffffffffu, b, o);
            cv[c] = x + b + carry[c];
        }
        // ---- events of the warp's 32 rows.  They are contiguous in the CSR list, so the warp reads them together
        // (32 events = 512 contiguous bytes per step) and counts the mismatching bases into per-row counters in
        // shared memory (the row's slice of the staging tile) - a thread walking its own row's events one dependent
        // load after the other was what this kernel spent its time on.  Indel tokens only set the row's bit here.
        int32_t* v = &stage[warp][lane * C];
        constexpr int KA = C == 30 ? 20 : 10;                        // [fwd A C G T N][rev A C G T N] ([hp1 ..][hp2 ..])
        static_assert(KA <= C, "the counters of a row fit its slice of the staging tile");
#pragma unroll
        for (int i = 0; i < KA; ++i) v[i] = 0;
        const int32_t E1w = __reduce_max_sync(0xffffffffu, live ? e1 : 0);
        const int32_t E0w = min(__reduce_min_sync(0xffffffffu, live ? e0 : 0x7fffffff), E1w);    // a warp without live rows: empty range
        const int32_t ev_row0 = (int32_t)(base + warp * 32);
        uint32_t indel_rows = 0;
        __syncwarp();
        for (int32_t s = E0w + lane; s < E1w; s += 32) {
            const RowEvent e = d.events[s];
            const int rl = e.row - ev_row0;
            if (e.len != 0) indel_rows |= 1u << rl;
            else if (e.yb <= 4u) {
                int32_t* a = &stage[warp][rl * C];
                atomicAdd(&a[(e.info & 1u) * 5 + e.yb], 1);
                if (C == 30) {
                    const uint32_t hp = (e.info >> 2) & 3u;
                    if (hp == 1 || hp == 2) atomicAdd(&a[10 + (hp - 1) * 5 + e.yb], 1);
                }
            }
        }
        indel_rows = __reduce_or_sync(0xffffffffu, indel_rows);
        __syncwarp();
        unsigned long long wf = 0, wr = 0, wp = 0, wm = 0;           // mismatching A,C,G,T as four 16-bit fields
        int32_t mm_f = 0, mm_r = 0, mm_p = 0, mm_m = 0;              // all mismatch events incl. N / ambiguity codes
#pragma unroll
        for (int b = 0; b < 5; ++b) {
            const int32_t cf = v[b], cr = v[5 + b];
            mm_f += cf; mm_r += cr;
            if (b < 4) { wf |= (unsigned long long)cf << (16 * b); wr |= (unsigned long long)cr << (16 * b); }
            if (C == 30) {
                const int32_t cp = v[10 + b], cm = v[15 + b];
                mm_p += cp; mm_m += cm;
                if (b < 4) { wp |= (unsigned long long)cp << (16 * b); wm |= (unsigned long long)cm << (16 * b); }
            }
        }
        __syncwarp();                                                // every lane holds its counters: the tile is free
#pragma unroll
        for (int i = 0; i < C; ++i) v[i] = 0;
        int32_t ins_cnt = 0, del_cnt = 0;
        const bool has_indel = live && ((indel_rows >> lane) & 1u);
        const bool heavy_me = has_indel && (e1 - e0) > ROWS_HEAVY;
        bool is_cand = false;
        // rows with indel tokens among many events (a het indel under deep coverage is hundreds of them): the whole warp
        // walks one such row at a time - token totals by ballots, distinct alleles by leader enumeration
        for (uint32_t heavy = __ballot_sync(0xffffffffu, heavy_me); heavy; heavy &= heavy - 1) {
            const int src = __ffs(heavy) - 1;
            const int32_t E0 = __shfl_sync(0xffffffffu, e0, src), E1 = __shfl_sync(0xffffffffu, e1, src);
            int32_t t[8] = {0, 0, 0, 0, 0, 0, 0, 0};         // indel tokens: ins f, ins r, del f, del r, IP, DP, IM, DM (warp-uniform)
            for (int32_t s0 = E0; s0 < E1; s0 += 32) {
                const int32_t s = s0 + lane;
                RowEvent e;
                e.info = 0; e.len = 0; e.yb = 5u; e.row = 0;
                if (s < E1) e = d.events[s];
                const uint32_t hp = (e.info >> 2) & 3u;
                if (__any_sync(0xffffffffu, e.len != 0)) {
                    const int x = e.len != 0 ? (int)(e.info & 3u) : -1;       // is_del << 1 | rev
#pragma unroll
                    for (int y = 0; y < 4; ++y) t[y] += __popc(__ballot_sync(0xffffffffu, x == y));
                    if (C == 30) {
#pragma unroll
                        for (int y = 0; y < 4; ++y)          // (hp 1, ins) (hp 1, del) (hp 2, ins) (hp 2, del)
                            t[4 + y] += __popc(__ballot_sync(0xffffffffu, x >= 0 && (int)hp == 1 + (y >> 1) && (x >> 1) == (y & 1)));
                    }
                }
            }
            const int32_t n_ind = t[0] + t[1] + t[2] + t[3];
            if (n_ind > 0 && E1 - E0 > IND_MAX) {            // longer than the bitmap: serial walk of the list
                if (lane == src) row_indels<C>(d, d.events + E0, E1 - E0, v, ins_cnt, del_cnt);
            } else if (n_ind > 0) {
                int32_t best[4] = {0, 0, 0, 0};              // largest distinct allele: I1, i1, D1, d1
                for_each_indel_allele<false>(d, d.events + E0, E1 - E0, lane, done_s[warp],
                                             [&](const RowEvent& ev, int32_t cnt, uint32_t, uint32_t) {
                    const int x = (int)(ev.info & 3u);
#pragma unroll
                    for (int y = 0; y < 4; ++y) if (y == x && cnt > best[y]) best[y] = cnt;
                });
                if (lane == src) {
                    ins_cnt = t[0] + t[1]; del_cnt = t[2] + t[3];
                    v[4] = t[0]; v[13] = t[1]; v[6] = t[2]; v[15] = t[3];
                    v[5] = best[0]; v[14] = best[1]; v[7] = best[2]; v[16] = best[3];
                    if (C == 30) { v[22] = t[4]; v[23] = t[5]; v[28] = t[6]; v[29] = t[7]; }
                }
            }
            __syncwarp();
        }
        if (live) {
            if (has_indel && !heavy_me) row_indels<C>(d, d.events + e0, e1 - e0, v, ins_cnt, del_cnt);
            if (rc >= 'a') rc -= 32;
            const int ri_raw = rc == 'A' ? 0 : rc == 'C' ? 1 : rc == 'G' ? 2 : rc == 'T' ? 3 : -1;
            const bool acgt = ri_raw >= 0;
            const int ri = acgt ? ri_raw : 0;
            int32_t bf[4], br[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                bf[i] = (int32_t)((wf >> (16 * i)) & 0xffff);
                br[i] = (int32_t)((wr >> (16 * i)) & 0xffff);
                if (acgt && i == ri) { bf[i] += cv[0] - mm_f; br[i] += cv[1] - mm_r; }   // matching bases = coverage - mismatches
                v[i] = bf[i];
                v[9 + i] = br[i];
            }
            const int32_t star_f = cv[2], star_r = cv[3];
            v[8] = star_f; v[17] = star_r;
            if (C == 30) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    int32_t a1 = (int32_t)((wp >> (16 * i)) & 0xffff), a2 = (int32_t)((wm >> (16 * i)) & 0xffff);
                    if (acgt && i == ri) { a1 += cv[NC - 2] - mm_p; a2 += cv[NC - 1] - mm_m; }
                    v[18 + i] = a1;
                    v[24 + i] = a2;
                }
            }
            const int32_t fsum = bf[0] + bf[1] + bf[2] + bf[3], rsum = br[0] + br[1] + br[2] + br[3];
            const int32_t depth = fsum + rsum + star_f + star_r;
            // candidate predicate (create_tensor_pileup.py:268-299, 536, 555)
            int32_t cls[6];
#pragma unroll
            for (int i = 0; i < 4; ++i) cls[i] = bf[i] + br[i];
            cls[4] = ins_cnt; cls[5] = del_cnt;
            const int32_t cls_ref = ri == 0 ? cls[0] : ri == 1 ? cls[1] : ri == 2 ? cls[2] : cls[3];
            bool pass_snp = false, pass_indel = false;
            if (depth < THR_N) {
                const int32_t ts = d.thr_snp[depth], ti = d.thr_indel[depth];
#pragma unroll
                for (int i = 0; i < 4; ++i) if (i != ri && cls[i] >= ts) pass_snp = true;
                pass_indel = cls[4] >= ti || cls[5] >= ti;
            } else {
                const double den = (double)depth;
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (i != ri && cls[i] > 0 && (double)cls[i] / den >= d.snp_af) pass_snp = true;
                if (cls[4] > 0 && (double)cls[4] / den >= d.indel_af) pass_indel = true;
                if (cls[5] > 0 && (double)cls[5] / den >= d.indel_af) pass_indel = true;
            }
            bool pass = pass_snp || pass_indel;
            if (!pass) {
                int32_t top = 0;
#pragma unroll
                for (int i = 0; i < 6; ++i) top = cls[i] > top ? cls[i] : top;
                if (top > 0) {
                    if (cls_ref < top) pass = true;
                    else {
                        bool tie = false;
#pragma unroll
                        for (int i = 0; i < 6; ++i) if (i != ri && cls[i] == top) tie = true;
                        if (tie && !(d.dbg & 1)) {
                            uint32_t key[6];
                            first_keys(d, (int32_t)row, p, ri, acgt, key);
                            for (int i = 0; i < 6; ++i) if (i != ri && cls[i] == top && key[i] < key[ri]) pass = true;
                        }
                    }
                }
            }
            if (depth > 0 && (d.snp_af == 0.0 || d.indel_af == 0.0)) pass = true;
            bool cand = acgt && pass && depth >= d.min_cov;
            if (d.n_known >= 0) cand = known_site(d.known, d.n_known, p + 1);        // :555-556 - AF, depth and base ignored
            else if (cand && d.n_cbed >= 0) {
                // longest deleted reference string of the row, clipped where the loaded reference ends (:234-237)
                int32_t max_del = 0;
                const int32_t room = (int32_t)min((int64_t)0x7fffffff, d.ref_len - ((int64_t)p - d.ref_start0) - 1);
                for (int32_t s = e0; s < e1; ++s) {
                    const RowEvent e = d.events[s];
                    if (e.len != 0 && (e.info & 2u)) max_del = max(max_del, min(e.len, max(room, 0)));
                }
                cand = iv_overlaps(d.cbed, d.n_cbed, p, p + max_del + 2);
            }
            is_cand = cand && window_printed(d.covP, (int64_t)p - d.R0, d.W, d.head_tail, d.head_tail ? d.tail[1] : 0);   // K3
            const uint8_t flag = is_cand ? 1 : 0;
            v[ri] = -fsum;
            v[9 + ri] = -rsum;
            d.row_depth[row] = depth;
            // samtools mpileup keeps at most 8000 reads per position (-d default; the reference never passes
            // --max-depth, create_tensor_pileup.py:442) and drops the reads beyond - in a read-order dependent way
            // that is not reproduced here: such a chunk is refused instead of being called differently
            if (depth > MPILEUP_MAX_DEPTH) atomicExch(d.err, 7);
            d.row_flag[row] = flag;
            d.row_inscnt[row] = ins_cnt;
            d.row_delcnt[row] = del_cnt + star_f + star_r;
            if (d.padding) { Int2 cr; cr.a = -fsum; cr.b = -rsum; d.cur_ref[row] = cr; }
        }
        // rows of a warp are contiguous in HBM: write 16 B per lane per step from the staging tile
        __syncwarp();
        const int64_t wrow0 = base + warp * 32;
        if (wrow0 < L) {
            const int64_t rows_here = min((int64_t)TILE_ROWS, L - wrow0);
            const int n_int = (int)rows_here * C;
            int32_t* out = d.counts + wrow0 * C;                 // 32*C*4 bytes per warp tile: 16 B aligned
            for (int i = lane * 4; i < n_int; i += 128) {
                if (i + 4 <= n_int) *(int4*)(out + i) = *(const int4*)(&stage[warp][i]);
                else for (int q = i; q < n_int; ++q) out[q] = stage[warp][q];
            }
        }
        __syncwarp();
        // candidates of the tile and of its group of 64 tiles (K3's list is built from these counts: k_cand_emit)
        const int nc = __popc(__ballot_sync(0xffffffffu, is_cand));
        if (lane == 0 && nc) {
            atomicAdd(&d.ctile[tile], nc);
            atomicAdd(&d.csuper[tile >> 6], nc);
        }
    }
}

// ------------------------------------------------------- K3: candidate list
// k_rows flagged the candidates (eligible and 33 printed columns) and counted them per tile of 256 rows and per group
// of 64 tiles.  Block = tile; its first slot = the groups before its group + the tiles before it in its group (a few
// dozen cached loads, no scan and no serial tail); a candidate's slot = that + its rank in the tile (position order).
__global__ void __launch_bounds__(256) k_cand_emit(Dev d) {
    __shared__ int32_t wsum[8];
    const int64_t L = *d.n_rows;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t n_ct = (L + COV_TILE - 1) / COV_TILE;
    auto block_sum = [&](int32_t v) {                    // sum over the block, returned to every thread
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        __syncthreads();
        if (lane == 0) wsum[warp] = v;
        __syncthreads();
        int32_t t = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += wsum[w];
        return t;
    };
    if (blockIdx.x == 0) {                               // the candidate count
        int32_t v = 0;
        for (int64_t i = threadIdx.x; i < (n_ct + 63) / 64; i += 256) v += d.csuper[i];
        const int32_t total = block_sum(v);
        if (threadIdx.x == 0) *d.n_cand = total;
    }
    for (int64_t tile = blockIdx.x; tile < n_ct; tile += gridDim.x) {
        if (d.ctile[tile] == 0) continue;                // block-uniform
        int32_t v = 0;
        for (int64_t i = threadIdx.x; i < (tile >> 6); i += 256) v += d.csuper[i];
        for (int64_t i = (tile & ~63ll) + threadIdx.x; i < tile; i += 256) v += d.ctile[i];
        const int32_t base = block_sum(v);
        const int64_t row = tile * COV_TILE + threadIdx.x;
        const bool c = row < L && d.row_flag[row];
        const uint32_t m = __ballot_sync(0xffffffffu, c);
        __syncthreads();
        if (lane == 0) wsum[warp] = __popc(m);
        __syncthreads();
        if (c) {
            int64_t i = base + __popc(m & ((1u << lane) - 1u));
#pragma unroll
            for (int w = 0; w < 8; ++w) if (w < warp) i += wsum[w];
            if (i < d.cand_cap) {
                d.cand_row[i] = (int32_t)row;
                d.cand_pos[i] = d.row_pos[row] + 1;
                d.cand_depth[i] = d.row_depth[row];
            }
        }
    }
}

// ------------------------------------------------------- K4: window assembly
// tensor[i][k][c] = counts[row_i - 16 + k][c]  (rows of consecutive positions are consecutive);
// with depth > 1.5*max_depth the window is divided by depth/max_depth in fp64 and truncated
// (clair3_rna/utils.py:85-92,120).  `scale` is skipped when the padding pass still has to patch.
__device__ __forceinline__ int32_t rescale(int32_t v, int32_t depth, int32_t max_depth) {
    const double sf = __ddiv_rn((double)depth, (double)max_depth);
    return (int32_t)__ddiv_rn((double)v, sf);
}
__global__ void k_window(Dev d, int apply_scale) {
    const int64_t n = *d.n_cand < d.cand_cap ? *d.n_cand : d.cand_cap;
    const int per = WIN * d.C;
    for (int64_t i = blockIdx.x; i < n; i += gridDim.x) {
        const int32_t row = d.cand_row[i];
        const int32_t depth = d.cand_depth[i];
        const bool sc = apply_scale && depth > 0 && (double)depth > (double)d.max_depth * 1.5;
        const int32_t* src = d.counts + ((int64_t)row - FLANK) * d.C;
        int32_t* dst = d.tensor + i * per;
        if (!d.head_tail) {
            for (int j = threadIdx.x; j < per; j += blockDim.x) {
                int32_t v = src[j];
                if (sc) v = rescale(v, depth, d.max_depth);
                dst[j] = v;
            }
            continue;
        }
        int nb, na;                                        // window rows that are columns of the candidate's run
        printed_run(d, (int64_t)d.cand_pos[i] - 1 - d.R0, &nb, &na);
        const int j0 = (FLANK - nb) * d.C, j1 = (FLANK + na + 1) * d.C;
        for (int j = threadIdx.x; j < per; j += blockDim.x) {
            int32_t v = (j >= j0 && j < j1) ? src[j] : 0;
            if (sc) v = rescale(v, depth, d.max_depth);
            dst[j] = v;
        }
    }
}
// K4 fused with the network's input stage: the window goes straight into LSTM1's fp16 operand images
//   xop[tile][33][KX/8][128 rows][8 halfs]   (k < C: x_hi = fp16(x), C <= k < 2C: x_hi again - it meets W_lo -,
//   2C <= k < 3C: x_lo = x - x_hi, k = 3C, 3C+1: 1 - they meet the bias rows -, rest 0; nn_tc.cuh, k_xop)
// instead of int32 tensor[n][33][C] that k_xop would read back: no 2.4 KB per site round trip through HBM.  Used
// when nobody asks for the tensor itself (keep_tensor) and no padding pass has to patch it.
// Block = (tile of 128 sites, window row t), thread = site: a thread reads the C counts of ITS row (72 / 120 contiguous
// bytes, 8-byte loads) and writes the KX/8 16-byte cells of the image; the lanes of a warp are consecutive sites, so
// every store instruction of a warp is 512 contiguous bytes.  Sites beyond n (the tile pair's padding) are zero rows.
template <int C, int KX>
__global__ void __launch_bounds__(128) k_window_xop(Dev d, __half* __restrict__ xop) {
    static_assert(KX >= 3 * C + 2 && KX % 16 == 0, "x_hi | x_hi | x_lo | 1 | 1 must fit the input part");
    const int64_t n = *d.n_cand < d.cand_cap ? *d.n_cand : d.cand_cap;
    const int64_t n_tiles = ((n + 255) / 256) * 2;             // tiles come in pairs
    const int r = threadIdx.x;
    for (int64_t b = blockIdx.x; b < n_tiles * WIN; b += gridDim.x) {
        const int64_t tile = b / WIN;
        const int t = (int)(b - tile * WIN);
        const int64_t i = tile * 128 + r;
        float x[C];
#pragma unroll
        for (int c = 0; c < C; ++c) x[c] = 0.0f;
        bool live = i < n;
        if (live) {
            const int32_t depth = d.cand_depth[i];
            const int32_t row = d.cand_row[i];
            if (d.head_tail) {                                 // window rows that are columns of the candidate's own run
                int nb, na;
                printed_run(d, (int64_t)d.cand_pos[i] - 1 - d.R0, &nb, &na);
                live = t >= FLANK - nb && t < FLANK + na + 1;
            }
            if (live) {
                const int2* src = (const int2*)(d.counts + ((int64_t)row - FLANK + t) * C);     // C is even: 8-byte aligned
                int32_t v[C];
#pragma unroll
                for (int c = 0; c < C / 2; ++c) { const int2 q = src[c]; v[2 * c] = q.x; v[2 * c + 1] = q.y; }
                if (depth > 0 && (double)depth > (double)d.max_depth * 1.5) {
#pragma unroll
                    for (int c = 0; c < C; ++c) v[c] = rescale(v[c], depth, d.max_depth);
                }
#pragma unroll
                for (int c = 0; c < C; ++c) x[c] = (float)v[c];
            }
        }
        __half xh[C], xl[C];                                   // x = xh + xl exactly (|x| <= 8000)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            xh[c] = __float2half(x[c]);
            xl[c] = __float2half(x[c] - __half2float(xh[c]));
        }
        __half* base = xop + ((size_t)tile * WIN + t) * (size_t)(KX * 128) + r * 8;
#pragma unroll
        for (int k8 = 0; k8 < KX / 8; ++k8) {
            __align__(16) __half hv[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int k = k8 * 8 + j;                      // compile-time after unrolling
                hv[j] = k < C ? xh[k < C ? k : 0] : k < 2 * C ? xh[k < 2 * C && k >= C ? k - C : 0]
                      : k < 3 * C ? xl[k < 3 * C && k >= 2 * C ? k - 2 * C : 0]
                      : __float2half(k < 3 * C + 2 ? 1.0f : 0.0f);
            }
            *(uint4*)(base + (size_t)k8 * (128 * 8)) = *(const uint4*)hv;
        }
    }
}
__global__ void k_rescale(Dev d) {
    const int64_t n = *d.n_cand < d.cand_cap ? *d.n_cand : d.cand_cap;
    const int per = WIN * d.C;
    for (int64_t i = blockIdx.x; i < n; i += gridDim.x) {
        const int32_t depth = d.cand_depth[i];
        if (!(depth > 0 && (double)depth > (double)d.max_depth * 1.5)) continue;
        int32_t* dst = d.tensor + i * per;
        for (int j = threadIdx.x; j < per; j += blockDim.x) dst[j] = rescale(dst[j], depth, d.max_depth);
    }
}

// splice-junction padding (create_tensor_pileup.py:573-593, 611): sequential along chains of
// emitted candidates <= 32 bp apart because padded rows persist (shared row objects) and an
// emitted centre disappears from depth_dict.  One thread per chain head.
__global__ void k_padding(Dev d) {
    const int64_t n = *d.n_cand < d.cand_cap ? *d.n_cand : d.cand_cap;
    const int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= n) return;
    // chains: consecutive candidates of one run <= 32 bp apart.  In head/tail mode a window also looks at the depth
    // of columns of neighbouring runs (and at whether their centres were emitted), so there the chain is by distance only.
    auto linked = [&](int64_t i) {
        const int32_t dp = d.cand_pos[i] - d.cand_pos[i - 1];
        return dp <= 2 * FLANK && (d.head_tail || d.cand_row[i] - d.cand_row[i - 1] == dp);
    };
    if (h > 0 && linked(h)) return;                  // not a chain head
    const int per = WIN * d.C;
    // head/tail mode: the slots of the ring that no column of the run has overwritten yet all reference ONE zero row
    // (`[[0] * C] * 33`), so a padding write into such a slot shows in all of them until the run has 33 columns
    int32_t zf[4] = {0, 0, 0, 0}, zr[4] = {0, 0, 0, 0};
    int32_t z_run = -1;
    for (int64_t i = h; i < n; ++i) {
        if (i > h && !linked(i)) break;
        const int32_t row = d.cand_row[i];
        const int32_t depth = d.cand_depth[i];
        const int32_t p = d.cand_pos[i] - 1;
        int nb = FLANK, na = FLANK;
        if (d.head_tail) {
            printed_run(d, (int64_t)p - d.R0, &nb, &na);
            if (nb < FLANK && z_run != p - nb) {         // a new run: a new shared zero row
                z_run = p - nb;
                for (int b = 0; b < 4; ++b) zf[b] = zr[b] = 0;
            }
        }
        // row of window slot k: the run's own column, else (head/tail mode) a column of another run if one is
        // printed there - such a column has its depth in depth_dict but is a zero row in this window
        auto slot_row = [&](int k, bool* own) -> int32_t {
            *own = k >= FLANK - nb && k <= FLANK + na;
            if (*own) return row - FLANK + k;
            const int64_t o = (int64_t)p - FLANK + k - d.R0;
            if (o < 0 || o >= d.W || !bit_at(d.covP, o)) return -1;
            return row_lower_bound(d, p - FLANK + k);
        };
        const bool flushed = d.head_tail && na < FLANK;   // emitted when the stream ends: no padding step (:613-637)
        if (!flushed) {
            int32_t mx_depth = 0, mx_skip = 0;
            bool any = false;
            for (int k = 0; k < WIN; ++k) {
                bool own;
                const int32_t r = slot_row(k, &own);
                if (r < 0) continue;
                if (!d.deleted[r]) { const int32_t dd = d.row_depth[r]; if (!any || dd > mx_depth) mx_depth = dd; any = true; }
                const int32_t ms = d.max_skip[r];
                mx_skip = ms > mx_skip ? ms : mx_skip;
            }
            if (any && mx_depth > 0 && __ddiv_rn((double)mx_skip, (double)mx_depth) > d.skip_prop) {
                const Int2 c = d.cur_ref[row];
                const int32_t sf = c.a < 0 ? -c.a : c.a, sr = c.b < 0 ? -c.b : c.b;
                const double pf = sf + sr > 0 ? __ddiv_rn((double)sf, (double)(sf + sr)) : 0.0;
                const double pr = 1.0 - pf;
                const int32_t vf = -(int32_t)__dmul_rn((double)depth, pf);
                const int32_t vr = -(int32_t)__dmul_rn((double)depth, pr);
                const double thr = __dmul_rn((double)depth, d.skip_prop);
                for (int k = 0; k < WIN; ++k) {
                    if (k == FLANK) continue;
                    bool own;
                    const int32_t r = slot_row(k, &own);
                    const int32_t cd = (r < 0 || d.deleted[r]) ? 0 : d.row_depth[r];
                    if ((double)cd < thr) {
                        bool acgt;
                        const int ri = ref_index(d, p - FLANK + k, &acgt);
                        if (!acgt) continue;
                        if (own) { Int2 nv; nv.a = vf; nv.b = vr; d.cur_ref[r] = nv; }
                        else { zf[ri] = vf; zr[ri] = vr; }
                    }
                }
            }
        }
        int32_t* dst = d.tensor + i * per;
        for (int k = 0; k < WIN; ++k) {
            if (k >= FLANK - nb && k <= FLANK + na) {
                const int32_t r = row - FLANK + k;
                bool acgt;
                const int ri = ref_index(d, d.row_pos[r], &acgt);
                const Int2 c = d.cur_ref[r];
                dst[k * d.C + ri] = c.a;
                dst[k * d.C + 9 + ri] = c.b;
            } else if (k < FLANK) {                      // not yet overwritten slots: the shared zero row
                for (int b = 0; b < 4; ++b) { dst[k * d.C + b] = zf[b]; dst[k * d.C + 9 + b] = zr[b]; }
            }                                            // slots after the end of the stream: fresh zero rows
        }
        if (!flushed) d.deleted[row] = 1;
    }
}

// ------------------------------------------------------------- alt_info
// upper bound of alleles per candidate: 3 alt bases + its indel events + reference
struct OpAltOff {
    typedef long long T;
    struct Ctx {};
    Dev d;
    __device__ void ctx_init(Ctx&) const {}
    __device__ T identity() const { return 0; }
    __device__ T combine(const T& x, const T& y) const { return x + y; }
    __device__ int64_t size() const { return *d.n_cand < d.cand_cap ? *d.n_cand : d.cand_cap; }
    __device__ T load(int64_t i) const {
        const int32_t row = d.cand_row[i];
        return 4 + (d.binc[row + 1] - d.binc[row]);
    }
    __device__ void store(int64_t i, const T& incl, const T& own, Ctx&) const { d.alt_off[i] = incl - own; }
};

// alleles in alt_dict insertion order (create_tensor_pileup.py:223,235,251,259-261): keys are
// case-folded, so the two strands of one allele merge and keep the earlier first occurrence.
// One warp per candidate: the lanes split the row's events to find the first read showing each
// non-reference base and to collect the indel tokens; lane 0 then builds the (short) allele list.
__global__ void __launch_bounds__(256) k_altinfo(Dev d) {
    const int64_t n = *d.n_cand < d.cand_cap ? *d.n_cand : d.cand_cap;
    const int lane = threadIdx.x & 31;
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= n) return;
    const int32_t row = d.cand_row[i];
    const int32_t p = d.row_pos[row];
    const int64_t off = d.alt_off[i];
    const int32_t e0 = d.binc[row] - d.binc[0], e1 = d.binc[row + 1] - d.binc[0];
    // One pass over the row's events by all lanes: first-occurrence key of each non-reference base (the earliest read
    // among the mismatch events), and the indel tokens compacted into shared memory so that the allele loop below does
    // not walk the whole event list with one dependent global load per event.
    __shared__ uint32_t done_s[8][IND_WORDS];
    const int wip = threadIdx.x >> 5;
    uint32_t key[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
    bool any_ind = false;
    for (int32_t s0 = e0; s0 < e1; s0 += 32) {
        const int32_t s = s0 + lane;
        RowEvent e;
        e.info = 0; e.len = 0; e.yb = 4u; e.row = 0;
        if (s < e1) e = d.events[s];
        if (e.len == 0 && e.yb <= 3u) {
            const uint32_t kk = (e.info >> 4) * 2u;
#pragma unroll
            for (int b = 0; b < 4; ++b) if (b == (int)e.yb && kk < key[b]) key[b] = kk;
        }
        any_ind |= e.len != 0;
    }
    any_ind = __any_sync(0xffffffffu, any_ind);
#pragma unroll
    for (int b = 0; b < 4; ++b)
#pragma unroll
        for (int sft = 16; sft > 0; sft >>= 1) key[b] = min(key[b], __shfl_xor_sync(0xffffffffu, key[b], sft));
    __syncwarp();
    if (off + 4 + (e1 - e0) > d.alt_cap) { if (lane == 0) { atomicExch(d.err, 4); d.alt_n[i] = 0; } return; }
    AltEntry* out = d.alt + off;
    int m = 0;                                       // lane 0's count of entries
    bool acgt;
    const int ri = ref_index(d, p, &acgt);
    const char L4[4] = {'A', 'C', 'G', 'T'};
    const int32_t* v = d.counts + (int64_t)row * d.C;
    int32_t alt_cnt = 0;
    if (lane == 0) {
        for (int b = 0; b < 4; ++b) {
            if (b == ri) continue;
            const int32_t c = v[b] + v[9 + b];
            if (c <= 0) continue;
            alt_cnt += c;
            AltEntry e; e.kind = 'X'; e.base = L4[b]; e.len = 0; e.count = c; e.seq_off = 0; e.order = key[b];
            out[m++] = e;
        }
    }
    // distinct indel alleles (strands folded), their counts and first occurrences
    if (!any_ind) {
    } else if (e1 - e0 <= IND_MAX) {
        for_each_indel_allele<true>(d, d.events + e0, e1 - e0, lane, done_s[wip],
                                    [&](const RowEvent& ev, int32_t cnt, uint32_t first, uint32_t first_y) {
            if (lane != 0) return;
            AltEntry e;
            e.kind = (ev.info & 2u) ? 'D' : 'I'; e.base = L4[ri];
            e.len = (uint16_t)(ev.len > 65535 ? 65535 : ev.len);
            e.count = cnt; e.seq_off = first_y; e.order = first;
            out[m++] = e;
        });
    } else if (lane == 0) {                          // longer than the bitmap: serial walk of the row's list
        const RowEvent* evs = d.events + e0;
        const int32_t n_ev = e1 - e0;
        for (int32_t s = 0; s < n_ev; ++s) {
            const RowEvent ev = evs[s];
            if (ev.len == 0) continue;
            const bool is_del = ev.info & 2u;
            bool seen = false;
            for (int32_t q = 0; q < s && !seen; ++q) {
                const RowEvent o = evs[q];
                if (o.len != 0 && ((o.info ^ ev.info) & 2u) == 0 && (is_del ? o.len == ev.len : ins_equal(d, o, ev, true))) seen = true;
            }
            if (seen) continue;
            int32_t cnt = 0;
            uint32_t first = 0xffffffffu, first_y = ev.yb;
            for (int32_t q = s; q < n_ev; ++q) {
                const RowEvent o = evs[q];
                if (o.len != 0 && ((o.info ^ ev.info) & 2u) == 0 && (is_del ? o.len == ev.len : ins_equal(d, o, ev, true))) {
                    ++cnt;
                    const uint32_t kk = (o.info >> 4) * 2u + 1u;
                    if (kk < first) { first = kk; first_y = o.yb; }
                }
            }
            AltEntry e;
            e.kind = is_del ? 'D' : 'I'; e.base = L4[ri];
            e.len = (uint16_t)(ev.len > 65535 ? 65535 : ev.len);
            e.count = cnt; e.seq_off = first_y; e.order = first;
            out[m++] = e;
        }
    }
    if (lane != 0) return;
    // insertion sort by first occurrence
    for (int a = 1; a < m; ++a) {
        AltEntry e = out[a];
        int b = a - 1;
        while (b >= 0 && out[b].order > e.order) { out[b + 1] = out[b]; --b; }
        out[b + 1] = e;
    }
    const int32_t depth = d.row_depth[row];
    const int32_t ref_cnt = depth - d.row_delcnt[row] - d.row_inscnt[row] - alt_cnt;
    if (ref_cnt > 0) {
        AltEntry e; e.kind = 'R'; e.base = L4[ri]; e.len = 0; e.count = ref_cnt; e.seq_off = 0; e.order = 0xffffffffu;
        out[m++] = e;
    }
    d.alt_n[i] = m;
}

}  // namespace c3r
