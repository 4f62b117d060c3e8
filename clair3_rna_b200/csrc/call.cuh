// The genotype decision of one candidate as a fixed-size call record (c3r_call, include/c3r_b200.h), in code that
// compiles for the host (c3r_debug_decide_calls, csrc/decode.cpp) and for sm_100a (k_call, csrc/c3r_abi.cu).
//
// It restates decide() and the allele-count part of vcf_row() in csrc/decode.cpp statement by statement, quirks
// included: a failed family zeroes its probability and retries without clearing REF / ALT, find_alt_base ranks the
// X alleles by descending count (ties stable) and falls back when the wanted base trails by >= 9 reads, indel dicts
// keep a repeated key at its first position with its last value, keys longer than MAX_INDEL are cut, SNP counts are
// cumulative, deletion counts are matched by length (first_len_match), and a candidate whose centre base is outside
// the IUPAC table gives no row.
//
// Strings become positions: an allele is {first letter, an insertion key's inserted bases, a suffix of REF}, and
// keys are compared by content - insertion keys by their sequence nibbles, deletion keys by their length, because
// every deletion key of a candidate is a prefix of the same reference bases (a key cut at the window end is shorter).
// The only arithmetic is IEEE float32 products and comparisons, so the device's record equals the host's bit for bit.
// Everything inexact (QUAL's log, AF's division) and all text stay in the host formatter (c3r_format_vcf).
//
// Two facts the record relies on, both true of the library's inputs: reference bytes and allele letters are never
// ',' (a ',' in the text is always the separator of two alleles), and allele counts are at most the 8000-read depth
// cap, so sums of two of them fit int32.
#pragma once
#include <stdint.h>

#include "../../include/c3r_b200.h"

#if defined(__CUDACC__)
#define C3R_HD __host__ __device__ __forceinline__
#define C3R_UNROLL _Pragma("unroll")
#else
#define C3R_HD inline
#define C3R_UNROLL
#endif

namespace c3rcall {

constexpr int FLANK = 16;
constexpr int MAX_INDEL = 50;                       // param_p.py maximum_variant_length_that_need_infer
enum Fam { REF = 0, HOMO_SNP, HET_SNP, HOMO_INS, HET_ACGT_INS, HET_INSINS, HOMO_DEL, HET_ACGT_DEL, HET_DELDEL, INSDEL, N_FAM };
enum Gt { GT_00 = 0, GT_11, GT_01, GT_12, GT_NONE };
// the 23 outcome probabilities, family by family: members of family f are [FAM_OFF[f], FAM_OFF[f + 1])
constexpr int N_OUTCOME = 23;
C3R_HD int fam_off(int f) {
    return f <= HOMO_SNP ? 0 : f == HET_SNP ? 4 : f == HOMO_INS ? 10 : f == HET_ACGT_INS ? 11 : f == HET_INSINS ? 15
         : f == HOMO_DEL ? 16 : f == HET_ACGT_DEL ? 17 : f == HET_DELDEL ? 21 : f == INSDEL ? 22 : 23;
}

// One candidate's inputs.  The same pointers are device memory in k_call and host memory in the CPU hook.
struct CallIn {
    const c3r_alt_entry* e;     // its alleles (c3r_result.alt + alt_off[i]), alt_n[i] of them
    int32_t n;
    const float* probs;         // its 24 probabilities
    const uint8_t* ref;         // the reference window
    int64_t ref_len;
    int64_t p0;                 // candidate offset in the window (pos - ref_start1)
    const uint8_t* seq;         // nt16 pool of the reads; NULL: an insertion key is its base alone (like decode.cpp)
};

C3R_HD char base2acgt(char c) {                     // shared/utils.py:41-44; 0 when the base is not in the table
    const char* K = "ACGTURYSWKMBDHVN";
    const char* V = "ACGTTACCAGACAAAA";
    for (int i = 0; i < 16; ++i) if (K[i] == c) return V[i];
    return 0;
}
C3R_HD uint8_t nib(const uint8_t* seq, uint32_t q) {
    const uint8_t b = seq[q >> 1];
    return (q & 1u) ? (b & 15) : (b >> 4);
}
C3R_HD int64_t del_start(const CallIn& c) { return c.p0 + 1 < 0 ? 0 : c.p0 + 1; }
C3R_HD int ins_len(const CallIn& c, const c3r_alt_entry& e) { return c.seq ? e.len : 0; }
// letters of a deletion key: the reference bases after the candidate, cut at the window end
C3R_HD int del_len(const CallIn& c, const c3r_alt_entry& e) {
    const int64_t lo = del_start(c);
    int64_t hi = c.p0 + 1 + (int64_t)e.len;
    if (hi > c.ref_len) hi = c.ref_len;
    return hi > lo ? (int)(hi - lo) : 0;
}
C3R_HD int key_len(const CallIn& c, const c3r_alt_entry& e) {
    return e.kind == 'I' ? 1 + ins_len(c, e) : e.kind == 'D' ? del_len(c, e) : 1;
}
// same kind assumed
C3R_HD bool key_eq(const CallIn& c, const c3r_alt_entry& a, const c3r_alt_entry& b) {
    if (a.kind == 'D') return del_len(c, a) == del_len(c, b);
    if (a.base != b.base) return false;
    if (a.kind != 'I') return true;
    const int n = ins_len(c, a);
    if (n != ins_len(c, b)) return false;
    for (int k = 0; k < n; ++k) if (nib(c.seq, a.seq_off + k) != nib(c.seq, b.seq_off + k)) return false;
    return true;
}

// ---- the allele dicts of decide(): keys of one kind, 1 <= length <= MAX_INDEL, first position, last value
C3R_HD bool dict_key(const CallIn& c, int k, char kind) {
    if (c.e[k].kind != kind) return false;
    const int l = key_len(c, c.e[k]);
    if (l < 1 || l > MAX_INDEL) return false;
    for (int j = 0; j < k; ++j) if (c.e[j].kind == kind && key_eq(c, c.e[j], c.e[k])) return false;
    return true;
}
C3R_HD int32_t last_value(const CallIn& c, int k) {
    int32_t v = c.e[k].count;
    for (int j = k + 1; j < c.n; ++j) if (c.e[j].kind == c.e[k].kind && key_eq(c, c.e[j], c.e[k])) v = c.e[j].count;
    return v;
}
// best_indel: first maximum of the dict; -1 when it is empty
C3R_HD int best_indel(const CallIn& c, char kind) {
    int b = -1;
    int32_t bv = 0;
    for (int k = 0; k < c.n; ++k) {
        if (!dict_key(c, k, kind)) continue;
        const int32_t v = last_value(c, k);
        if (b < 0 || v > bv) { b = k; bv = v; }
    }
    return b;
}
// two_indels: the dict sorted by value (stable), then reversed - descending values, ties in reverse dict order -
// and its first two; for deletions the longer key first, and nothing unless there are two.  Returns how many.
C3R_HD int two_indels(const CallIn& c, char kind, int* out) {
    int t1 = -1, t2 = -1;
    int32_t v1 = 0, v2 = 0;
    for (int k = 0; k < c.n; ++k) {
        if (!dict_key(c, k, kind)) continue;
        const int32_t v = last_value(c, k);
        if (t1 < 0 || v >= v1) { t2 = t1; v2 = v1; t1 = k; v1 = v; }
        else if (t2 < 0 || v >= v2) { t2 = k; v2 = v; }
    }
    if (kind == 'I') {
        out[0] = t1; out[1] = t2;
        return t1 < 0 ? 0 : t2 < 0 ? 1 : 2;
    }
    if (t2 < 0) return 0;
    if (key_len(c, c.e[t1]) > key_len(c, c.e[t2])) { out[0] = t1; out[1] = t2; }
    else { out[0] = t2; out[1] = t1; }
    return 2;
}
// find_alt_base: the X alleles by descending count (stable); *chosen = want, or the top base when want is absent or
// trails it by >= 9 reads; 0 without X alleles.  Returns how many there are, the top two in r[0], r[1].
C3R_HD int snp_alts(const CallIn& c, char want, char* chosen, char* r) {
    int n = 0, t1 = -1, t2 = -1;
    bool have = false;
    int32_t mine = 0;
    for (int k = 0; k < c.n; ++k) {
        const c3r_alt_entry& e = c.e[k];
        if (e.kind != 'X') continue;
        ++n;
        if (t1 < 0 || e.count > c.e[t1].count) { t2 = t1; t1 = k; }
        else if (t2 < 0 || e.count > c.e[t2].count) t2 = k;
        // the first of the ranked list with this base: the largest count among them
        if (want && (char)e.base == want && (!have || e.count > mine)) { have = true; mine = e.count; }
    }
    *chosen = 0;
    if (!n) return 0;
    if (!have || c.e[t1].count - mine >= 9) want = (char)c.e[t1].base;
    *chosen = want;
    r[0] = (char)c.e[t1].base;
    r[1] = t2 >= 0 ? (char)c.e[t2].base : 0;
    return n;
}

// ---- REF / ALT as positions.  REF letter 0 is ref_first, letter k >= 1 is ref[del_start + k - 1].
struct Al {
    char first;
    int16_t ins;                // entry of an insertion key whose inserted bases follow `first`, -1: none
    uint16_t sf;                // then REF letters [sf, ref_len)
};
struct Dec {
    bool flags[N_FAM];
    bool has_ref, has_alt;
    char ref_first;
    int ref_len;
    int n_alt;                  // 0: empty
    Al alt[2];
    float prob;
    int fam;                    // branch of the last retry-loop pass (REF for a reference call)
    uint16_t retries;
};
C3R_HD Al al_key(const CallIn& c, int k, int ref_len) {        // an insertion key as an allele
    Al a; a.first = (char)c.e[k].base; a.ins = (int16_t)k; a.sf = (uint16_t)ref_len; return a;
}
C3R_HD Al al_ref(char first, int sf) { Al a; a.first = first; a.ins = -1; a.sf = (uint16_t)sf; return a; }
C3R_HD int al_ins(const CallIn& c, const Al& a) { return a.ins >= 0 ? ins_len(c, c.e[a.ins]) : 0; }
C3R_HD int al_len(const CallIn& c, const Dec& D, const Al& a) { return 1 + al_ins(c, a) + (D.ref_len - a.sf); }
C3R_HD char ref_char(const CallIn& c, const Dec& D, int k) {
    return k == 0 ? D.ref_first : (char)c.ref[del_start(c) + k - 1];
}
C3R_HD char seq_char(uint8_t code) { return "=ACMGRSVTWYHKDBN"[code]; }
C3R_HD char al_char(const CallIn& c, const Dec& D, const Al& a, int k) {
    if (k == 0) return a.first;
    const int ni = al_ins(c, a);
    if (k <= ni) return seq_char(nib(c.seq, c.e[a.ins].seq_off + (k - 1)));
    return ref_char(c, D, a.sf + (k - 1 - ni));
}
C3R_HD bool al_eq(const CallIn& c, const Dec& D, const Al& a, const Al& b) {
    const int n = al_len(c, D, a);
    if (n != al_len(c, D, b)) return false;
    for (int k = 0; k < n; ++k) if (al_char(c, D, a, k) != al_char(c, D, b, k)) return false;
    return true;
}
C3R_HD bool al_eq_ref(const CallIn& c, const Dec& D, const Al& a) {
    if (al_len(c, D, a) != D.ref_len) return false;
    for (int k = 0; k < D.ref_len; ++k) if (al_char(c, D, a, k) != ref_char(c, D, k)) return false;
    return true;
}
// the first `len` letters of allele a against an insertion key
C3R_HD bool al_eq_ins_key(const CallIn& c, const Dec& D, const Al& a, int len, const c3r_alt_entry& e) {
    if (len != 1 + ins_len(c, e)) return false;
    if (al_char(c, D, a, 0) != (char)e.base) return false;
    for (int k = 1; k < len; ++k) if (al_char(c, D, a, k) != seq_char(nib(c.seq, e.seq_off + (k - 1)))) return false;
    return true;
}

// ---- output_from (decode.cpp decide())
C3R_HD int fam_index_of(const float* v, int f, float x) {
    for (int j = fam_off(f); j < fam_off(f + 1); ++j) if (v[j] == x) return j - fam_off(f);
    return -1;
}
C3R_HD int fam_argmax(const float* v, int f) {
    const int o = fam_off(f);
    int b = 0;
    for (int j = 1; j < fam_off(f + 1) - o; ++j) if (v[o + j] > v[o + b]) b = j;
    return b;
}

C3R_HD void decide(const CallIn& c, char center, Dec& D) {
    for (int f = 0; f < N_FAM; ++f) D.flags[f] = false;
    D.has_ref = D.has_alt = false;
    D.ref_first = 0; D.ref_len = 0; D.n_alt = 0; D.prob = 0.f; D.fam = REF; D.retries = 0;
    const char ref_acgt = base2acgt(center);
    const float* gt21 = c.probs;
    const float p00 = c.probs[21], p11 = c.probs[22], p01 = c.probs[23];
    const int HOMO_IX[4] = {0, 4, 7, 9};
    const int HET_IX[6] = {1, 2, 3, 5, 6, 8};
    const char ACGT[4] = {'A', 'C', 'G', 'T'};
    const char HET_L[6][2] = {{'A', 'C'}, {'A', 'G'}, {'A', 'T'}, {'C', 'G'}, {'C', 'T'}, {'G', 'T'}};
    const float rr = gt21[HOMO_IX[ref_acgt == 'A' ? 0 : ref_acgt == 'C' ? 1 : ref_acgt == 'G' ? 2 : 3]];
    const float p_ref = p00 * rr;
    auto as_ref = [&](float p) {
        for (int f = 0; f < N_FAM; ++f) D.flags[f] = false;
        D.flags[REF] = true;
        D.has_ref = D.has_alt = true;
        D.ref_first = ref_acgt; D.ref_len = 1;
        D.n_alt = 1; D.alt[0] = al_ref(ref_acgt, 1);
        D.prob = p;
        D.fam = REF;
    };
    if (p00 >= 0.5f && rr >= 0.5f) { as_ref(p_ref); return; }
    float v[N_OUTCOME];
    C3R_UNROLL
    for (int i = 0; i < 4; ++i) v[fam_off(HOMO_SNP) + i] = p11 * gt21[HOMO_IX[i]];
    C3R_UNROLL
    for (int i = 0; i < 6; ++i) v[fam_off(HET_SNP) + i] = p01 * gt21[HET_IX[i]];
    v[fam_off(HOMO_INS)] = p11 * gt21[15];
    v[fam_off(HET_INSINS)] = p01 * gt21[15];
    C3R_UNROLL
    for (int i = 0; i < 4; ++i) v[fam_off(HET_ACGT_INS) + i] = gt21[16 + i] * p01;
    v[fam_off(HOMO_DEL)] = p11 * gt21[10];
    v[fam_off(HET_DELDEL)] = p01 * gt21[10];
    C3R_UNROLL
    for (int i = 0; i < 4; ++i) v[fam_off(HET_ACGT_DEL) + i] = gt21[11 + i] * p01;
    v[fam_off(INSDEL)] = p01 * gt21[20];
    float best = 0.f;
    for (int guard = 0; (!D.has_ref || !D.has_alt) && guard < 64; ++guard) {
        best = p_ref;
        for (int j = 0; j < N_OUTCOME; ++j) if (v[j] > best) best = v[j];
        if (best == p_ref) { as_ref(best); return; }
        for (int f = HOMO_SNP; f < N_FAM; ++f) D.flags[f] = fam_index_of(v, f, best) >= 0;
        D.flags[REF] = false;
        auto retry = [&](int f, int i, int bit) { v[fam_off(f) + i] = 0.f; D.retries |= (uint16_t)(1u << bit); };
        auto set_ref = [&](int del) {                       // REF = centre (+ the bases of a deletion key)
            D.ref_first = center; D.ref_len = 1 + (del >= 0 ? del_len(c, c.e[del]) : 0); D.has_ref = true;
        };
        auto one_snp = [&](int f, int i, char want, int bit_none, int bit_same) {   // ALT = find_alt_base(want)
            char chosen, r[2];
            snp_alts(c, want, &chosen, r);
            if (chosen) { D.n_alt = 1; D.alt[0] = al_ref(chosen, D.ref_len); D.has_alt = true; }
            else { D.has_alt = false; D.n_alt = 0; }
            if (!chosen) { retry(f, i, bit_none); return false; }
            if (chosen == center) { retry(f, i, bit_same); return false; }
            return true;
        };
        if (D.flags[HOMO_SNP]) {
            D.fam = HOMO_SNP;
            set_ref(-1);
            const int i = fam_index_of(v, HOMO_SNP, best);
            const char lab = ACGT[fam_argmax(v, HOMO_SNP)];
            if (!one_snp(HOMO_SNP, i, lab, C3R_RETRY_HOMO_SNP_NO_X, C3R_RETRY_HOMO_SNP_IS_REF)) continue;
        } else if (D.flags[HET_SNP]) {
            D.fam = HET_SNP;
            const int a = fam_argmax(v, HET_SNP);
            const char l0 = HET_L[a][0], l1 = HET_L[a][1];
            const int i = fam_index_of(v, HET_SNP, best);
            set_ref(-1);
            if (l0 != center && l1 != center) {
                char chosen, r[2];
                if (snp_alts(c, 0, &chosen, r) < 2) { retry(HET_SNP, i, C3R_RETRY_HET_SNP_LT2_X); continue; }
                D.n_alt = 2; D.alt[0] = al_ref(r[0], 1); D.alt[1] = al_ref(r[1], 1); D.has_alt = true;
            } else if (!one_snp(HET_SNP, i, l0 != center ? l0 : l1, C3R_RETRY_HET_SNP_NO_X, C3R_RETRY_HET_SNP_IS_REF)) continue;
        } else if (D.flags[HOMO_INS]) {
            D.fam = HOMO_INS;
            const int i = fam_index_of(v, HOMO_INS, best);
            const int ins = best_indel(c, 'I');
            if (ins < 0) { retry(HOMO_INS, i, C3R_RETRY_HOMO_INS_NO_I); continue; }
            set_ref(-1);
            D.n_alt = 1; D.alt[0] = al_key(c, ins, 1); D.has_alt = true;
        } else if (D.flags[HET_ACGT_INS]) {
            D.fam = HET_ACGT_INS;
            const int i = fam_index_of(v, HET_ACGT_INS, best);
            const int ins = best_indel(c, 'I');
            if (ins < 0) { retry(HET_ACGT_INS, i, C3R_RETRY_HET_ACGT_INS_NO_I); continue; }
            set_ref(-1);
            D.n_alt = 1; D.alt[0] = al_key(c, ins, 1); D.has_alt = true;
            if (ACGT[i] != center) {
                char chosen, r[2];
                if (!snp_alts(c, 0, &chosen, r)) { retry(HET_ACGT_INS, i, C3R_RETRY_HET_ACGT_INS_NO_X); continue; }
                D.n_alt = 2; D.alt[1] = D.alt[0]; D.alt[0] = al_ref(r[0], 1);
            }
        } else if (D.flags[HET_INSINS]) {
            D.fam = HET_INSINS;
            const int i = fam_index_of(v, HET_INSINS, best);
            int two[2];
            if (two_indels(c, 'I', two) < 2) { retry(HET_INSINS, i, C3R_RETRY_HET_INSINS_LT2_I); continue; }
            set_ref(-1);
            D.n_alt = 1; D.alt[0] = al_key(c, two[0], 1); D.has_alt = true;
            if (!key_eq(c, c.e[two[1]], c.e[two[0]])) { D.n_alt = 2; D.alt[0] = al_key(c, two[1], 1); D.alt[1] = al_key(c, two[0], 1); }
            else { retry(HET_INSINS, i, C3R_RETRY_HET_INSINS_SAME); continue; }
        } else if (D.flags[HOMO_DEL]) {
            D.fam = HOMO_DEL;
            const int i = fam_index_of(v, HOMO_DEL, best);
            const int del = best_indel(c, 'D');
            if (del < 0) { retry(HOMO_DEL, i, C3R_RETRY_HOMO_DEL_NO_D); continue; }
            set_ref(del);
            D.n_alt = 1; D.alt[0] = al_ref(center, D.ref_len); D.has_alt = true;
        } else if (D.flags[HET_ACGT_DEL]) {
            D.fam = HET_ACGT_DEL;
            const int i = fam_index_of(v, HET_ACGT_DEL, best);
            const int del = best_indel(c, 'D');
            if (del < 0) { retry(HET_ACGT_DEL, i, C3R_RETRY_HET_ACGT_DEL_NO_D); continue; }
            set_ref(del);
            D.n_alt = 1; D.alt[0] = al_ref(center, D.ref_len); D.has_alt = true;
            if (ACGT[i] != D.ref_first) { D.n_alt = 2; D.alt[1] = al_ref(ACGT[i], 1); }
        } else if (D.flags[HET_DELDEL]) {
            D.fam = HET_DELDEL;
            const int i = fam_index_of(v, HET_DELDEL, best);
            int two[2];
            if (two_indels(c, 'D', two) < 2) { retry(HET_DELDEL, i, C3R_RETRY_HET_DELDEL_LT2_D); continue; }
            set_ref(two[0]);
            D.n_alt = 1; D.alt[0] = al_ref(center, D.ref_len); D.has_alt = true;
            const int other = del_len(c, c.e[two[1]]);
            const Al a1 = D.alt[0];
            const Al a2 = al_ref(center, other + 1 <= D.ref_len ? other + 1 : D.ref_len);
            if (!al_eq(c, D, a1, a2) && !al_eq_ref(c, D, a1) && !al_eq_ref(c, D, a2)) { D.n_alt = 2; D.alt[1] = a2; }
            else { retry(HET_DELDEL, i, C3R_RETRY_HET_DELDEL_SAME); continue; }
        } else if (D.flags[INSDEL]) {
            D.fam = INSDEL;
            const int i = fam_index_of(v, INSDEL, best);
            const int ins = best_indel(c, 'I'), del = best_indel(c, 'D');
            if (ins < 0 || del < 0) { retry(INSDEL, i, C3R_RETRY_INSDEL_NO_I_OR_D); continue; }
            set_ref(del);
            D.n_alt = 2; D.alt[0] = al_ref(center, D.ref_len); D.alt[1] = al_key(c, ins, 1);
            D.has_alt = true;
        }
    }
    D.prob = best;
}

// ---- vcf_row(): which row, its GT and its allele counts
C3R_HD int32_t snp_count(const CallIn& c, char b) {      // dict_get(snp, b): last X allele of that base
    int32_t v = 0;
    for (int k = 0; k < c.n; ++k) if (c.e[k].kind == 'X' && (char)c.e[k].base == b) v = c.e[k].count;
    return v;
}
C3R_HD int32_t del_count(const CallIn& c, int len) {     // dict_get(dele, key of that length) == first_len_match
    int32_t v = 0;
    for (int k = 0; k < c.n; ++k) if (c.e[k].kind == 'D' && del_len(c, c.e[k]) == len) v = c.e[k].count;
    return v;
}
C3R_HD int32_t ins_count(const CallIn& c, const Dec& D, const Al& a, int len) {   // dict_get(ins, a[:len])
    int32_t v = 0;
    for (int k = 0; k < c.n; ++k) if (c.e[k].kind == 'I' && al_eq_ins_key(c, D, a, len, c.e[k])) v = c.e[k].count;
    return v;
}

C3R_HD void record_allele(const CallIn& c, const Al& a, c3r_call_allele& o) {
    o.first = (uint8_t)a.first;
    o.reserved = 0;
    o.ins_len = (uint16_t)(a.ins >= 0 ? ins_len(c, c.e[a.ins]) : 0);
    o.ins_seq_off = a.ins >= 0 ? c.e[a.ins].seq_off : 0;
    o.suffix_from = a.sf;
    o.reserved2 = 0;
}

// The call record of one candidate.
C3R_HD void decide_call(const CallIn& c, c3r_call& out) {
    out.prob = 0.f; out.ref_count = 0; out.support = 0; out.ad[0] = out.ad[1] = 0;
    out.family = C3R_CALL_NO_ROW; out.gt = GT_NONE; out.n_ad = 0; out.n_alt = 0;
    out.ref_first = 0; out.reserved = 0; out.ref_len = 0; out.retries = 0; out.flags = 0;
    for (int a = 0; a < 2; ++a) record_allele(c, al_ref(0, 0), out.alt[a]);
    // 33-base context padded with 'A' off the loaded reference: only its centre matters
    const char center = (c.p0 >= 0 && c.p0 < c.ref_len) ? (char)c.ref[c.p0] : 'A';
    if (!base2acgt(center)) return;                                  // clair3_rna/utils.py:113
    Dec D;
    decide(c, center, D);
    out.retries = D.retries;
    for (int f = 0; f < N_FAM; ++f) if (D.flags[f]) out.flags |= (uint16_t)(1u << f);
    out.prob = D.prob;
    const bool* f = D.flags;
    const bool is_ref = f[REF];
    if (!is_ref && D.has_ref && D.has_alt) {
        // ref_base == alt_base: an ALT with a ',' never equals REF
        if (D.n_alt == 1 && al_eq_ref(c, D, D.alt[0])) return;
    }
    if (!D.has_ref || !D.has_alt) return;
    const bool multi = D.n_alt == 2;
    int gt = GT_NONE;
    if (is_ref) gt = GT_00;
    else if (f[HOMO_SNP] || f[HOMO_INS] || f[HOMO_DEL]) gt = GT_11;
    else if (f[HET_SNP] || f[HET_ACGT_INS] || f[HET_INSINS] || f[HET_ACGT_DEL] || f[HET_DELDEL]) gt = GT_01;
    if (multi) gt = GT_12;
    int32_t ref_count = 0;
    for (int k = 0; k < c.n; ++k) if (c.e[k].kind == 'R') ref_count = c.e[k].count;
    if (ref_count < 0) ref_count = 0;
    int32_t support = 0, counts[2] = {0, 0};
    int n_counts = 0;
    auto push = [&](int32_t v) { if (n_counts < 2) counts[n_counts] = v; ++n_counts; };
    int n_alt = D.n_alt;
    if (is_ref) {
        support = ref_count;
        n_alt = 0;                                                  // ALT "."
    } else if (f[HOMO_SNP] || f[HET_SNP]) {
        for (int a = 0; a < D.n_alt; ++a)
            for (int k = 0; k < al_len(c, D, D.alt[a]); ++k) {
                support += snp_count(c, al_char(c, D, D.alt[a], k));
                push(support);                                      // cumulative, as the reference does
            }
    } else if (f[HOMO_INS] || f[HET_INSINS]) {
        for (int a = 0; a < D.n_alt; ++a) {
            const int32_t n = ins_count(c, D, D.alt[a], al_len(c, D, D.alt[a]));
            support += n;
            push(n);
        }
    } else if (f[HET_ACGT_INS]) {
        const Al& ins_b = multi ? D.alt[1] : D.alt[0];
        const int32_t c_snp = multi ? snp_count(c, D.alt[0].first) : 0;
        const int32_t c_ins = ins_count(c, D, ins_b, al_len(c, D, ins_b));
        support = c_ins + c_snp;
        if (multi) push(c_snp);
        push(c_ins);
    } else if (f[HOMO_DEL] || f[HET_DELDEL]) {
        // the dele dict of vcf_row: every deletion key, its size the number of distinct key lengths
        int n_keys = 0, len0 = -1;
        for (int k = 0; k < c.n; ++k) {
            if (c.e[k].kind != 'D') continue;
            const int l = del_len(c, c.e[k]);
            if (n_keys == 0) { n_keys = 1; len0 = l; }
            else if (l != len0) n_keys = 2;
        }
        if (n_keys) {
            if (f[HOMO_DEL]) {
                support = D.ref_len > 1 ? del_count(c, D.ref_len - 1) : 0;
                push(support);
            } else if (f[HET_DELDEL] && n_keys > 1) {
                for (int a = 0; a < D.n_alt; ++a) {
                    const int ln = D.ref_len - al_len(c, D, D.alt[a]);
                    const int32_t n = ln >= 0 ? del_count(c, ln) : 0;
                    push(n);
                    support += n;
                }
            }
        }
    } else if (f[HET_ACGT_DEL]) {
        const int32_t c_snp = multi ? snp_count(c, D.alt[1].first) : 0;
        const int32_t c_del = D.ref_len > 1 ? del_count(c, D.ref_len - 1) : 0;
        support = c_del + c_snp;
        if (multi) push(c_snp);
        push(c_del);
    } else if (f[INSDEL]) {
        for (int a = 0; a < D.n_alt; ++a) {
            const int len = al_len(c, D, D.alt[a]);
            const int ln = D.ref_len - len;
            int32_t n;
            if (ln < 0) n = ins_count(c, D, D.alt[a], D.ref_len > 1 ? len - (D.ref_len - 1) : len);
            else n = del_count(c, ln);
            push(n);
            support += n;
        }
    }
    out.family = (uint8_t)D.fam;
    out.gt = (uint8_t)gt;
    out.ref_count = ref_count;
    out.support = support;
    out.ad[0] = counts[0];
    out.ad[1] = counts[1];
    out.n_ad = (uint8_t)n_counts;
    out.n_alt = (uint8_t)n_alt;
    out.ref_first = (uint8_t)D.ref_first;
    out.ref_len = (uint16_t)D.ref_len;
    for (int a = 0; a < n_alt; ++a) record_allele(c, D.alt[a], out.alt[a]);
}

}  // namespace c3rcall
