// Probabilities + allele table -> VCF rows, natively and in parallel on the host (A7, SURVEY.md §8a / §8f-2).
//
// Restates the pileup-mode behaviour of the reference's consumer (/root/reference/clair3_rna/call_variants.py):
//     possible_outcome_probabilites_from   :518-667   (add_indel_length=False branch)
//     find_alt_base                        :670-681
//     insertion_/deletion_bases_using_alt_info_from   :112-196
//     output_from                          :684-1020  (retry loop over outcome families)
//     output_with                          :1117-1392 (AD / AF / QUAL / FILTER / row text)
//     quality_score_from                   :383-389
// with the options call_var_bam always passes (--pileup --showRef --add_indel_length False, --qual 2;
// clair3_rna/call_var_bam.py:247-272).  It follows clair3_rna_b200/decoder.py statement by statement (that
// file is the readable version, pinned by rows the reference's own output_with printed); this one exists
// because the Python decoder runs at ~7 k rows/s per core while the GPU emits millions of candidates/s.
// Products of probabilities are float32 like the reference's numpy scalars; QUAL is computed in double
// from the float32 product (NumPy-1 promotion, SURVEY.md §8c).
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

constexpr int FLANK = 16;
constexpr int MAX_INDEL = 50;                       // param_p.py maximum_variant_length_that_need_infer
const char* const GT21_LABELS[21] = {"AA", "AC", "AG", "AT", "CC", "CG", "CT", "GG", "GT", "TT", "DelDel", "ADel", "CDel",
                                     "GDel", "TDel", "InsIns", "AIns", "CIns", "GIns", "TIns", "InsDel"};   // task/gt21.py:3-25
const char ACGT[5] = "ACGT";
const char NT16[17] = "=ACMGRSVTWYHKDBN";

char base2acgt(char c) {                            // shared/utils.py:41-44; 0 when the base is not in the table
    static const char* K = "ACGTURYSWKMBDHVN";
    static const char* V = "ACGTTACCAGACAAAA";
    const char* p = strchr(K, c);
    return (p && c) ? V[p - K] : 0;
}

struct Allele {
    char kind;                                      // X I D R
    std::string key;                                // alt_info key without its first letter
    int count;
};

enum Fam { REF = 0, HOMO_SNP, HET_SNP, HOMO_INS, HET_ACGT_INS, HET_INSINS, HOMO_DEL, HET_ACGT_DEL, HET_DELDEL, INSDEL, N_FAM };

// find_alt_base: X alleles by descending count (stable); falls back to the best supported base when `want`
// is absent or trails it by >= 9 reads.  Returns the ranked bases; *chosen = 0 when there is no X allele.
// (scratch vectors are per thread and reused: this runs once or twice per candidate, millions of times per genome)
const std::vector<char>& snp_alts(const std::vector<Allele>& alt, char want, char* chosen) {
    static thread_local std::vector<std::pair<char, int>> ranked;
    static thread_local std::vector<char> out;
    ranked.clear();
    out.clear();
    for (const Allele& a : alt) if (a.kind == 'X') {
        // stable insertion by descending count (at most a handful of entries)
        size_t i = ranked.size();
        ranked.emplace_back(a.key[0], a.count);
        while (i > 0 && ranked[i - 1].second < a.count) { std::swap(ranked[i - 1], ranked[i]); --i; }
    }
    *chosen = 0;
    if (ranked.empty()) return out;
    bool have = false;
    int mine = 0;
    for (const auto& r : ranked) if (r.first == want && want) { have = true; mine = r.second; break; }
    if (!have || ranked[0].second - mine >= 9) want = ranked[0].first;
    *chosen = want;
    for (const auto& r : ranked) out.push_back(r.first);
    return out;
}

std::vector<std::pair<std::string, int>> indel_keys(const std::vector<Allele>& alt, char kind) {
    std::vector<std::pair<std::string, int>> d;     // dict semantics: a repeated key keeps its first position, last value
    for (const Allele& a : alt) {
        if (a.kind != kind || a.key.size() < 1 || (int)a.key.size() > MAX_INDEL) continue;
        bool found = false;
        for (auto& kv : d) if (kv.first == a.key) { kv.second = a.count; found = true; break; }
        if (!found) d.emplace_back(a.key, a.count);
    }
    return d;
}
std::string best_indel(const std::vector<Allele>& alt, char kind) {
    const auto d = indel_keys(alt, kind);
    if (d.empty()) return "";
    size_t b = 0;
    for (size_t i = 1; i < d.size(); ++i) if (d[i].second > d[b].second) b = i;     // max(): first maximum
    return d[b].first;
}
std::vector<std::string> two_indels(const std::vector<Allele>& alt, char kind) {
    auto d = indel_keys(alt, kind);
    std::stable_sort(d.begin(), d.end(), [](const auto& x, const auto& y) { return x.second < y.second; });
    std::reverse(d.begin(), d.end());               // sorted ascending (stable), then [::-1]
    std::vector<std::string> r;
    if (kind == 'I') {
        for (size_t i = 0; i < d.size() && i < 2; ++i) r.push_back(d[i].first);
        return r;
    }
    if (d.size() <= 1) return r;
    const std::string &a = d[0].first, &b = d[1].first;
    if (a.size() > b.size()) { r.push_back(a); r.push_back(b); } else { r.push_back(b); r.push_back(a); }
    return r;
}

struct FamV {                                       // probabilities of one outcome family (at most 6 members)
    float v[6];
    int n = 0;
    void push_back(float x) { v[n++] = x; }
};

struct Decision {
    bool flags[N_FAM];
    bool has_ref = false, has_alt = false;
    std::string ref_base, alt_base;
    float prob = 0.f;
};

// output_from
Decision decide(char center, const float* probs, const std::vector<Allele>& alt) {
    Decision D;
    for (bool& f : D.flags) f = false;
    const char ref_acgt = base2acgt(center);
    const float* gt21 = probs;
    const float p00 = probs[21], p11 = probs[22], p01 = probs[23];
    // GT21_LABELS indices: AA 0, CC 4, GG 7, TT 9; AC 1, AG 2, AT 3, CG 5, CT 6, GT 8
    static const int HOMO_IX[4] = {0, 4, 7, 9};
    static const int HET_IX[6] = {1, 2, 3, 5, 6, 8};
    const float rr = gt21[HOMO_IX[ref_acgt == 'A' ? 0 : ref_acgt == 'C' ? 1 : ref_acgt == 'G' ? 2 : 3]];
    const float p_ref = p00 * rr;
    auto as_ref = [&](float p) {
        for (bool& f : D.flags) f = false;
        D.flags[REF] = true;
        D.has_ref = D.has_alt = true;
        D.ref_base = D.alt_base = std::string(1, ref_acgt);
        D.prob = p;
    };
    if (p00 >= 0.5f && rr >= 0.5f) { as_ref(p_ref); return D; }
    static const char* HOMO[4] = {"AA", "CC", "GG", "TT"};
    static const char* HET[6] = {"AC", "AG", "AT", "CG", "CT", "GT"};
    FamV fam[N_FAM];
    for (int i = 0; i < 4; ++i) fam[HOMO_SNP].push_back(p11 * gt21[HOMO_IX[i]]);
    for (int i = 0; i < 6; ++i) fam[HET_SNP].push_back(p01 * gt21[HET_IX[i]]);
    fam[HOMO_INS].push_back(p11 * gt21[15]);
    fam[HET_INSINS].push_back(p01 * gt21[15]);
    for (int i = 0; i < 4; ++i) fam[HET_ACGT_INS].push_back(gt21[16 + i] * p01);
    fam[HOMO_DEL].push_back(p11 * gt21[10]);
    fam[HET_DELDEL].push_back(p01 * gt21[10]);
    for (int i = 0; i < 4; ++i) fam[HET_ACGT_DEL].push_back(gt21[11 + i] * p01);
    fam[INSDEL].push_back(p01 * gt21[20]);
    const std::string ctr(1, center);
    auto index_of = [](const FamV& v, float x) { for (int i = 0; i < v.n; ++i) if (v.v[i] == x) return i; return -1; };
    auto argmax = [](const FamV& v) { int b = 0; for (int i = 1; i < v.n; ++i) if (v.v[i] > v.v[b]) b = i; return b; };
    float best = 0.f;
    // A failed family zeroes its probability and `continue`s WITHOUT clearing ref_base/alt_base, exactly like the
    // reference: the loop ends as soon as both happen to be set.
    for (int guard = 0; (!D.has_ref || !D.has_alt) && guard < 64; ++guard) {
        best = p_ref;
        for (int f = HOMO_SNP; f < N_FAM; ++f) for (int i = 0; i < fam[f].n; ++i) if (fam[f].v[i] > best) best = fam[f].v[i];
        if (best == p_ref) { as_ref(best); return D; }
        for (int f = HOMO_SNP; f < N_FAM; ++f) D.flags[f] = index_of(fam[f], best) >= 0;
        D.flags[REF] = false;
        if (D.flags[HOMO_SNP]) {
            FamV& v = fam[HOMO_SNP];
            D.ref_base = ctr; D.has_ref = true;
            const int i = index_of(v, best);
            const char* lab = HOMO[argmax(v)];
            char chosen;
            snp_alts(alt, lab[0] != center ? lab[0] : lab[1], &chosen);
            if (chosen) { D.alt_base = std::string(1, chosen); D.has_alt = true; } else { D.has_alt = false; D.alt_base.clear(); }
            if (!chosen || D.alt_base == D.ref_base) { v.v[i] = 0; continue; }
        } else if (D.flags[HET_SNP]) {
            FamV& v = fam[HET_SNP];
            const char* lab = HET[argmax(v)];
            const int i = index_of(v, best);
            D.ref_base = ctr; D.has_ref = true;
            if (lab[0] != center && lab[1] != center) {
                char chosen;
                const std::vector<char>& ranked = snp_alts(alt, 0, &chosen);
                if (ranked.size() < 2) { v.v[i] = 0; continue; }
                D.alt_base = std::string(1, ranked[0]) + "," + std::string(1, ranked[1]); D.has_alt = true;
            } else {
                char chosen;
                snp_alts(alt, lab[0] != center ? lab[0] : lab[1], &chosen);
                if (chosen) { D.alt_base = std::string(1, chosen); D.has_alt = true; } else { D.has_alt = false; D.alt_base.clear(); }
                if (!chosen || D.alt_base == D.ref_base) { v.v[i] = 0; continue; }
            }
        } else if (D.flags[HOMO_INS]) {
            FamV& v = fam[HOMO_INS];
            const int i = index_of(v, best);
            const std::string ins = best_indel(alt, 'I');
            if (ins.empty()) { v.v[i] = 0; continue; }
            D.ref_base = ctr; D.alt_base = ins; D.has_ref = D.has_alt = true;
        } else if (D.flags[HET_ACGT_INS]) {
            FamV& v = fam[HET_ACGT_INS];
            const int i = index_of(v, best);
            const std::string ins = best_indel(alt, 'I');
            if (ins.empty()) { v.v[i] = 0; continue; }
            D.ref_base = ctr; D.alt_base = ins; D.has_ref = D.has_alt = true;
            if (ACGT[i] != center) {
                char chosen;
                const std::vector<char>& ranked = snp_alts(alt, 0, &chosen);
                if (ranked.empty()) { v.v[i] = 0; continue; }
                D.alt_base = std::string(1, ranked[0]) + "," + D.alt_base;
            }
        } else if (D.flags[HET_INSINS]) {
            FamV& v = fam[HET_INSINS];
            const int i = index_of(v, best);
            const std::vector<std::string> two = two_indels(alt, 'I');
            if (two.size() < 2) { v.v[i] = 0; continue; }
            D.ref_base = ctr; D.alt_base = two[0]; D.has_ref = D.has_alt = true;
            if (two[1] != two[0]) D.alt_base = two[1] + "," + two[0];
            else { v.v[i] = 0; continue; }
        } else if (D.flags[HOMO_DEL]) {
            FamV& v = fam[HOMO_DEL];
            const int i = index_of(v, best);
            const std::string dele = best_indel(alt, 'D');
            if (dele.empty()) { v.v[i] = 0; continue; }
            D.ref_base = ctr + dele; D.alt_base = D.ref_base.substr(0, 1); D.has_ref = D.has_alt = true;
        } else if (D.flags[HET_ACGT_DEL]) {
            FamV& v = fam[HET_ACGT_DEL];
            const int i = index_of(v, best);
            const std::string dele = best_indel(alt, 'D');
            if (dele.empty()) { v.v[i] = 0; continue; }
            D.ref_base = ctr + dele; D.alt_base = D.ref_base.substr(0, 1); D.has_ref = D.has_alt = true;
            if (ACGT[i] != D.ref_base[0]) D.alt_base = D.alt_base + "," + std::string(1, ACGT[i]) + D.ref_base.substr(1);
        } else if (D.flags[HET_DELDEL]) {
            FamV& v = fam[HET_DELDEL];
            const int i = index_of(v, best);
            const std::vector<std::string> two = two_indels(alt, 'D');
            if (two.size() < 2) { v.v[i] = 0; continue; }
            const std::string &longer = two[0], &other = two[1];
            D.ref_base = ctr + longer; D.alt_base = D.ref_base.substr(0, 1); D.has_ref = D.has_alt = true;
            const std::string a1 = D.alt_base;
            const std::string a2 = D.ref_base.substr(0, 1) + (other.size() + 1 <= D.ref_base.size() ? D.ref_base.substr(other.size() + 1) : "");
            if (a1 != a2 && D.ref_base != a1 && D.ref_base != a2) D.alt_base = a1 + "," + a2;
            else { v.v[i] = 0; continue; }
        } else if (D.flags[INSDEL]) {
            FamV& v = fam[INSDEL];
            const int i = index_of(v, best);
            const std::string ins = best_indel(alt, 'I'), dele = best_indel(alt, 'D');
            if (ins.empty() || dele.empty()) { v.v[i] = 0; continue; }
            D.ref_base = ctr + dele;
            D.alt_base = D.ref_base.substr(0, 1) + "," + ins + D.ref_base.substr(1);
            D.has_ref = D.has_alt = true;
        }
    }
    D.prob = best;
    return D;
}

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

std::vector<std::string> split(const std::string& s, char sep) {
    std::vector<std::string> out;
    size_t a = 0;
    for (;;) {
        const size_t b = s.find(sep, a);
        if (b == std::string::npos) { out.push_back(s.substr(a)); return out; }
        out.push_back(s.substr(a, b - a));
        a = b + 1;
    }
}

int dict_get(const std::vector<std::pair<std::string, int>>& d, const std::string& k, bool have_key = true) {
    if (!have_key) return 0;
    for (const auto& kv : d) if (kv.first == k) return kv.second;
    return 0;
}
void dict_set(std::vector<std::pair<std::string, int>>& d, const std::string& k, int v) {
    for (auto& kv : d) if (kv.first == k) { kv.second = v; return; }
    d.emplace_back(k, v);
}

// output_with's row text from the decision: AF, QUAL, FILTER and the line (with '\n') appended to `out`.  Shared by
// c3r_decode_vcf and c3r_format_vcf, so that both print the same bytes.
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

// output_with: appends one VCF line (with '\n') to `out`; returns false when the reference prints nothing
bool vcf_row(const char* contig, int pos, const std::string& ref33, int depth, const std::vector<Allele>& alt,
             const float* probs, double qual_cut, bool show_ref, std::string& out) {
    const char center = ref33.size() > 1 ? ref33[FLANK] : ref33[0];
    Decision D = decide(center, probs, alt);
    const bool* f = D.flags;
    const bool is_ref = f[REF];
    if ((!show_ref && is_ref) || (!is_ref && D.has_ref && D.has_alt && D.ref_base == D.alt_base)) return false;
    if (!D.has_ref || !D.has_alt) return false;
    std::string ref_base = D.ref_base, alt_base = D.alt_base;
    const bool multi = alt_base.find(',') != std::string::npos;
    const char* gt = "None";
    if (is_ref) gt = "0/0";
    else if (f[HOMO_SNP] || f[HOMO_INS] || f[HOMO_DEL]) gt = "1/1";
    else if (f[HET_SNP] || f[HET_ACGT_INS] || f[HET_INSINS] || f[HET_ACGT_DEL] || f[HET_DELDEL]) gt = "0/1";
    if (multi) gt = "1/2";
    static thread_local std::vector<std::pair<std::string, int>> snp, ins, dele;
    static thread_local std::vector<long> counts;
    snp.clear(); ins.clear(); dele.clear(); counts.clear();
    int ref_count = 0;
    for (const Allele& a : alt) {
        if (a.kind == 'X') dict_set(snp, a.key.substr(0, 1), a.count);
        else if (a.kind == 'I') dict_set(ins, a.key, a.count);
        else if (a.kind == 'D') dict_set(dele, a.key, a.count);
        else if (a.kind == 'R') ref_count = a.count;
    }
    if (ref_count < 0) ref_count = 0;
    long support = 0;
    auto first_len_match = [&](size_t ln) { for (const auto& kv : dele) if (kv.first.size() == ln) return kv.second; return 0; };
    if (is_ref) {
        support = ref_count;
        alt_base = ".";
    } else if (f[HOMO_SNP] || f[HET_SNP]) {
        for (char b : alt_base) {
            if (b == ',') continue;
            support += dict_get(snp, std::string(1, b));
            counts.push_back(support);                  // cumulative, as the reference does
        }
    } else if (f[HOMO_INS] || f[HET_INSINS]) {
        for (const std::string& s : split(alt_base, ',')) {
            const int c = dict_get(ins, s);
            support += c;
            counts.push_back(c);
        }
    } else if (f[HET_ACGT_INS]) {
        const std::vector<std::string> parts = split(alt_base, ',');
        const bool has_snp = multi;
        const std::string snp_b = multi ? parts[0].substr(0, 1) : "";
        const std::string ins_b = multi ? parts[1] : alt_base;
        const int c_snp = multi ? dict_get(snp, snp_b) : 0;
        const int c_ins = dict_get(ins, ins_b);
        support = c_ins + c_snp;
        if (has_snp && !snp_b.empty()) counts.push_back(c_snp);
        counts.push_back(c_ins);
    } else if (f[HOMO_DEL] || f[HET_DELDEL]) {
        if (!dele.empty()) {
            if (f[HOMO_DEL]) {
                support = ref_base.size() > 1 ? dict_get(dele, ref_base.substr(1)) : 0;
                counts.push_back(support);
            } else if (f[HET_DELDEL] && dele.size() > 1) {
                for (const std::string& s : split(alt_base, ',')) {
                    const long ln = (long)ref_base.size() - (long)s.size();
                    const int c = ln >= 0 ? first_len_match((size_t)ln) : 0;
                    counts.push_back(c);
                    support += c;
                }
            }
        }
    } else if (f[HET_ACGT_DEL]) {
        const std::vector<std::string> parts = split(alt_base, ',');
        std::string snp_b;
        if (multi && parts.size() > 1) snp_b = parts[1].substr(0, 1);
        const int c_snp = multi ? (snp_b.empty() ? 0 : dict_get(snp, snp_b)) : 0;
        const int c_del = ref_base.size() > 1 ? dict_get(dele, ref_base.substr(1)) : 0;
        support = c_del + c_snp;
        if (!snp_b.empty()) counts.push_back(c_snp);
        counts.push_back(c_del);
    } else if (f[INSDEL]) {
        for (const std::string& s : split(alt_base, ',')) {
            const long ln = (long)ref_base.size() - (long)s.size();
            int c;
            if (ln < 0) {
                const std::string ib = ref_base.size() > 1 ? s.substr(0, s.size() - (ref_base.size() - 1)) : s;
                c = dict_get(ins, ib);
            } else c = first_len_match((size_t)ln);
            counts.push_back(c);
            support += c;
        }
    }
    put_row(contig, pos, ref_base, alt_base, is_ref, gt, depth, ref_count, counts.data(), counts.size(), support, D.prob,
            qual_cut, out);
    return true;
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
    auto rows = [&](int64_t i, std::string& out) {
        static thread_local std::vector<Allele> alt;
        static thread_local std::string ref33;
        const int64_t p0 = (int64_t)res->pos[i] - ref_start1;            // offset of the candidate in ref
        // 33-base context, padded with 'A' off the loaded reference (create_tensor_pileup.py:313-331)
        ref33.assign(2 * FLANK + 1, 'A');
        for (int k = -FLANK; k <= FLANK; ++k) {
            const int64_t o = p0 + k;
            if (o >= 0 && o < ref_len) ref33[k + FLANK] = (char)ref[o];
        }
        if (!base2acgt(ref33[FLANK])) return false;                      // clair3_rna/utils.py:113
        alt.clear();
        const c3r_alt_entry* e = res->alt + res->alt_off[i];
        for (int32_t k = 0; k < res->alt_n[i]; ++k) {
            Allele al;
            al.kind = (char)e[k].kind;
            al.count = e[k].count;
            if (al.kind == 'X' || al.kind == 'R') al.key.assign(1, (char)e[k].base);
            else if (al.kind == 'I') {
                al.key.assign(1, (char)e[k].base);
                if (reads && reads->seq)
                    for (uint32_t q = e[k].seq_off; q < e[k].seq_off + e[k].len; ++q) {
                        const uint8_t by = reads->seq[q >> 1];
                        al.key.push_back(NT16[(q & 1) ? (by & 15) : (by >> 4)]);
                    }
            } else {
                for (int64_t o = p0 + 1; o < p0 + 1 + (int64_t)e[k].len && o < ref_len; ++o) if (o >= 0) al.key.push_back((char)ref[o]);
            }
            alt.push_back(std::move(al));
        }
        return vcf_row(contig, res->pos[i], ref33, res->depth[i], alt, res->probs + 24 * i, qual_cut, show_ref != 0, out);
    };
    return rows_in_parallel(n, n_threads, rows, text, n_bytes, n_rows);
}

// c3r_decode_vcf's lines from call records: what is left of output_with once the decision is made
int c3r_format_vcf(const c3r_result* res, const c3r_call* calls, const c3r_reads* reads, const uint8_t* ref,
                   int64_t ref_start1, int64_t ref_len, const char* contig, double qual_cut, int show_ref, int n_threads,
                   char** text, int64_t* n_bytes, int64_t* n_rows) {
    if (!res || !ref || !contig || !text || !n_bytes || !n_rows) return C3R_ERR_ARG;
    const int64_t n = res->n_cand;
    *text = nullptr; *n_bytes = 0; *n_rows = 0;
    if (n > 0 && (!res->pos || !res->depth || !calls)) return C3R_ERR_ARG;
    static const char* const GT_TEXT[5] = {"0/0", "1/1", "0/1", "1/2", "None"};
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
        const c3r_call& c = calls[i];
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
        put_row(contig, res->pos[i], ref_base, alt_base, is_ref, GT_TEXT[c.gt], res->depth[i], c.ref_count, counts,
                c.n_ad, c.support, c.prob, qual_cut, out);
        return true;
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
