// The BAM record format (SAMv1 §4.2) in code that compiles for the host (c3r_bam_fetch, csrc/bam_io.cpp) and for
// sm_100a (k_rec_parse / k_rec_write, csrc/bgzf.cuh): the one copy of the record checks, the aux walk, the CIGAR
// lengths and the fetch's per-record decision in the tree.  Every read of a record is bounded by its block_size.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#ifndef C3R_HD
#define C3R_HD __host__ __device__ __forceinline__
#endif
#else
#ifndef C3R_HD
#define C3R_HD inline
#endif
#endif

namespace c3rbam {

C3R_HD uint16_t rd16(const uint8_t* p) { return (uint16_t)(p[0] | (p[1] << 8)); }
C3R_HD uint32_t rd32(const uint8_t* p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

struct RecView {
    int32_t tid, pos;
    uint16_t flag, n_cigar;
    uint8_t mapq, l_name;
    int32_t l_seq;
    const uint8_t* cigar;      // n_cigar u32
    const uint8_t* seq;
    const uint8_t* aux;
    const uint8_t* aux_end;
};

// p: the record after its block_size field
C3R_HD bool view_record(const uint8_t* p, uint32_t block_size, RecView& r) {
    if (block_size < 32) return false;
    r.tid = (int32_t)rd32(p);
    r.pos = (int32_t)rd32(p + 4);
    r.l_name = p[8];
    r.mapq = p[9];
    r.n_cigar = rd16(p + 12);
    r.flag = rd16(p + 14);
    r.l_seq = (int32_t)rd32(p + 16);
    if (r.l_seq < 0) return false;
    const uint64_t need = 32ull + r.l_name + 4ull * r.n_cigar + (uint64_t)(r.l_seq + 1) / 2 + (uint64_t)r.l_seq;
    if (need > block_size) return false;
    r.cigar = p + 32 + r.l_name;
    r.seq = r.cigar + 4 * r.n_cigar;
    r.aux = r.seq + (r.l_seq + 1) / 2 + r.l_seq;
    r.aux_end = p + block_size;
    return true;
}

// walks the aux fields; returns false on malformed data.  Finds HP (any integer type) and CG (B,I long CIGAR).
C3R_HD bool scan_aux(const RecView& r, int64_t* hp, const uint8_t** cg, uint32_t* cg_n) {
    const uint8_t* a = r.aux;
    const uint8_t* e = r.aux_end;
    *hp = -1; *cg = nullptr; *cg_n = 0;
    while (a + 3 <= e) {
        const uint8_t t0 = a[0], t1 = a[1], ty = a[2];
        a += 3;
        int64_t iv = 0;
        bool is_int = false;
        switch (ty) {
            case 'A': case 'c': case 'C':
                if (a + 1 > e) return false;
                iv = ty == 'c' ? (int8_t)a[0] : a[0]; is_int = ty != 'A'; a += 1; break;
            case 's': case 'S':
                if (a + 2 > e) return false;
                iv = ty == 's' ? (int16_t)rd16(a) : rd16(a); is_int = true; a += 2; break;
            case 'i': case 'I':
                if (a + 4 > e) return false;
                iv = ty == 'i' ? (int64_t)(int32_t)rd32(a) : (int64_t)rd32(a); is_int = true; a += 4; break;
            case 'f':
                if (a + 4 > e) return false;
                a += 4; break;
            case 'Z': case 'H':
                while (a < e && *a) ++a;
                if (a >= e) return false;
                ++a; break;
            case 'B': {
                if (a + 5 > e) return false;
                const uint8_t sub = a[0];
                const uint32_t cnt = rd32(a + 1);
                const uint32_t sz = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : (sub == 'i' || sub == 'I' || sub == 'f') ? 4 : 0;
                if (!sz) return false;
                a += 5;
                if ((uint64_t)(e - a) < (uint64_t)cnt * sz) return false;
                if (t0 == 'C' && t1 == 'G' && sub == 'I') { *cg = a; *cg_n = cnt; }
                a += (size_t)cnt * sz;
                break;
            }
            default:
                return false;
        }
        if (is_int && t0 == 'H' && t1 == 'P') *hp = iv;
    }
    return a == e;
}

C3R_HD int64_t cigar_ref_len(const uint8_t* c, uint32_t n) {
    int64_t l = 0;
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t v = rd32(c + 4 * i), op = v & 15;
        if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) l += v >> 4;
    }
    return l;
}
C3R_HD int64_t cigar_qry_len(const uint8_t* c, uint32_t n) {
    int64_t l = 0;
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t v = rd32(c + 4 * i), op = v & 15;
        if (op == 0 || op == 1 || op == 4 || op == 7 || op == 8) l += v >> 4;
    }
    return l;
}

// What a region fetch does with one record, in the order c3r_bam_fetch checks it.
enum RecClass { REC_KEEP = 1, REC_SKIP, REC_STOP, REC_ERR_MALFORMED, REC_ERR_AUX };

struct RecInfo {
    RecView r;
    const uint8_t* cig;        // the CIGAR the fetch keeps (CG:B,I when the record carries its long CIGAR there)
    uint32_t n_cig;
    int64_t hp;                // -1: absent
    int64_t n_bases;           // l_seq, or the CIGAR's query length for SEQ '*'
};

// p / block_size as for view_record; records of contig `tid` overlapping the 0-based half-open [beg, end)
C3R_HD int classify_record(const uint8_t* p, uint32_t block_size, int32_t tid, int64_t beg, int64_t end, RecInfo& x) {
    RecView& r = x.r;
    if (!view_record(p, block_size, r)) return REC_ERR_MALFORMED;
    if (r.tid != tid) return (r.tid > tid || r.tid < 0) ? REC_STOP : REC_SKIP;
    if (r.pos >= end) return REC_STOP;
    const uint8_t* cg;
    uint32_t cg_n;
    if (!scan_aux(r, &x.hp, &cg, &cg_n)) return REC_ERR_AUX;
    x.cig = r.cigar;
    x.n_cig = r.n_cigar;
    if (cg && x.n_cig == 2 && (rd32(x.cig) & 15) == 4 && (int64_t)(rd32(x.cig) >> 4) == r.l_seq && (rd32(x.cig + 4) & 15) == 3) {
        x.cig = cg; x.n_cig = cg_n;                 // long CIGAR kept in the CG:B,I tag (SAMv1 §4.2.2)
    }
    const int64_t rlen = cigar_ref_len(x.cig, x.n_cig);
    const int64_t rend = r.pos + (rlen > 0 ? rlen : 1);
    if (rend <= beg) return REC_SKIP;
    // SEQ '*': samtools prints 'N' for every query position (bam_plcmd.c pileup_seq)
    x.n_bases = r.l_seq > 0 ? (int64_t)r.l_seq : cigar_qry_len(x.cig, x.n_cig);
    return REC_KEEP;
}

C3R_HD uint8_t clamp_hp(int64_t hp) { return hp <= 0 ? 0 : (uint8_t)(hp > 255 ? 255 : hp); }

}  // namespace c3rbam
