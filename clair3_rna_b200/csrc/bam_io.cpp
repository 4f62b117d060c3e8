// BAM / BGZF / BAI reader and writer feeding the flat alignment records (c3r_reads) the
// kernels consume.  Host C++ with zlib only (no htslib in this image).
//
// What it replaces in the reference: the BAM is only ever touched through external samtools,
//   `samtools mpileup <bam> -r ctg:s-e ...`   /root/reference/src/create_tensor_pileup.py:436-451
//   `samtools idxstats <bam>`                 /root/reference/run_clair3_rna:187
// i.e. an index fetch of the records overlapping a region, in file (coordinate) order, plus the
// per-contig mapped-read counts.  Record filtering (flags, MAPQ) stays on the GPU (k_read_prepare).
//
// Formats follow the SAM/BAM specification (SAMv1 §4 BAM, §4.1 BGZF, §5.2 BAI).  Reader design:
// the compressed byte range of a fetch is cut into BGZF blocks by their headers, the blocks are
// inflated in parallel by a small thread pool into one contiguous buffer (ISIZE trailers give the
// output offsets up front), records are then walked once and copied into struct-of-arrays.
#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>
#include <zlib.h>

#include "../../include/c3r_b200.h"
#include "bam_rec.cuh"
#include "bgzf.cuh"

namespace {

using c3rbam::rd16;
using c3rbam::rd32;
inline uint64_t rd64(const uint8_t* p) { return (uint64_t)rd32(p) | ((uint64_t)rd32(p + 4) << 32); }
inline void wr16(std::vector<uint8_t>& v, uint16_t x) { v.push_back(x & 0xff); v.push_back(x >> 8); }
inline void wr32(std::vector<uint8_t>& v, uint32_t x) { for (int i = 0; i < 4; ++i) v.push_back((x >> (8 * i)) & 0xff); }
inline void wr64(std::vector<uint8_t>& v, uint64_t x) { wr32(v, (uint32_t)x); wr32(v, (uint32_t)(x >> 32)); }

// UCSC binning scheme (SAMv1 §5.3)
inline int reg2bin(int64_t beg, int64_t end) {
    --end;
    if (beg >> 14 == end >> 14) return (int)(((1 << 15) - 1) / 7 + (beg >> 14));
    if (beg >> 17 == end >> 17) return (int)(((1 << 12) - 1) / 7 + (beg >> 17));
    if (beg >> 20 == end >> 20) return (int)(((1 << 9) - 1) / 7 + (beg >> 20));
    if (beg >> 23 == end >> 23) return (int)(((1 << 6) - 1) / 7 + (beg >> 23));
    if (beg >> 26 == end >> 26) return (int)(((1 << 3) - 1) / 7 + (beg >> 26));
    return 0;
}
inline void reg2bins(int64_t beg, int64_t end, std::vector<int>& out) {
    out.clear();
    --end;
    out.push_back(0);
    for (int64_t k = 1 + (beg >> 26); k <= 1 + (end >> 26); ++k) out.push_back((int)k);
    for (int64_t k = 9 + (beg >> 23); k <= 9 + (end >> 23); ++k) out.push_back((int)k);
    for (int64_t k = 73 + (beg >> 20); k <= 73 + (end >> 20); ++k) out.push_back((int)k);
    for (int64_t k = 585 + (beg >> 17); k <= 585 + (end >> 17); ++k) out.push_back((int)k);
    for (int64_t k = 4681 + (beg >> 14); k <= 4681 + (end >> 14); ++k) out.push_back((int)k);
}
constexpr int META_BIN = 37450;
constexpr int BGZF_MAX_PAYLOAD = 0xff00;          // uncompressed bytes per block (as htslib)

struct Chunk { uint64_t beg, end; };
struct RefIndex {
    std::vector<std::pair<uint32_t, std::vector<Chunk>>> bins;
    std::vector<uint64_t> linear;
    uint64_t n_mapped = 0, n_unmapped = 0;
    bool has_meta = false;
};

struct Block { uint64_t coff; uint32_t csize; uint32_t usize; uint64_t uoff; };

}  // namespace

struct c3r_bam {
    std::string path, err;
    FILE* fp = nullptr;
    int n_threads = 4;
    std::vector<std::string> ref_names;
    std::vector<int64_t> ref_lens;
    std::string header_text;
    std::vector<RefIndex> index;
    uint64_t file_size = 0;
    // fetch output (owned here, exposed through c3r_reads)
    std::vector<int32_t> pos, cigar_off;
    std::vector<uint16_t> flag;
    std::vector<uint8_t> mapq, hp, seq;
    std::vector<uint32_t> cigar;
    std::vector<int64_t> seq_off;
    // scratch
    std::vector<uint8_t> cbuf, ubuf;
    // tables of the last raw fetch (c3r_bam_fetch_raw)
    std::vector<c3r_bgzf_block> raw_blocks;
    std::vector<c3r_bam_window> raw_windows;
};

namespace {

int bfail(c3r_bam* h, int code, const std::string& m) { h->err = m; return code; }

// inflate one BGZF block (raw deflate payload after the 18-byte header)
bool inflate_block(const uint8_t* src, uint32_t csize, uint8_t* dst, uint32_t usize) {
    if (csize < 26) return false;
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (inflateInit2(&zs, -15) != Z_OK) return false;
    const uint32_t xlen = rd16(src + 10);
    zs.next_in = const_cast<Bytef*>(src + 12 + xlen);
    zs.avail_in = csize - 12 - xlen - 8;
    zs.next_out = dst;
    zs.avail_out = usize;
    const int rc = inflate(&zs, Z_FINISH);
    const bool ok = (rc == Z_STREAM_END) && zs.total_out == usize;
    inflateEnd(&zs);
    if (!ok) return false;
    return (uint32_t)crc32(crc32(0L, Z_NULL, 0), dst, usize) == rd32(src + csize - 8);
}

// BSIZE from a BGZF header (total block size - 1), 0 if the header is not BGZF
uint32_t bgzf_block_size(const uint8_t* p, size_t avail) {
    if (avail < 18) return 0;
    if (p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) return 0;
    const uint32_t xlen = rd16(p + 10);
    if (avail < 12 + xlen) return 0;
    const uint8_t* x = p + 12;
    const uint8_t* xe = x + xlen;
    while (x + 4 <= xe) {
        const uint32_t slen = rd16(x + 2);
        if (x[0] == 'B' && x[1] == 'C' && slen == 2) return (uint32_t)rd16(x + 4) + 1;
        x += 4 + slen;
    }
    return 0;
}

// the messages of c3rbgzf::FetchErr
std::string fetch_err_text(const c3r_bam* h, int code) {
    switch (code) {
        case c3rbgzf::FE_INFLATE: return "BGZF inflate/CRC failure in " + h->path;
        case c3rbgzf::FE_HEADER: return "corrupt BGZF block header in " + h->path;
        case c3rbgzf::FE_BIG_BLOCK: return "BGZF block larger than 64 KiB";
        case c3rbgzf::FE_SHORT_READ: return "short read from " + h->path;
        case c3rbgzf::FE_CROSS: return "record crosses the end of an index chunk";
        case c3rbgzf::FE_MALFORMED: return "malformed BAM record";
        default: return "malformed aux data in a BAM record";
    }
}

// Bytes read for the blocks starting at compressed offset `cbeg` up to (and including) the block that contains
// compressed offset `cend_block` (or to EOF when cend_block == UINT64_MAX): one block more than the range, so that
// the last block is whole.  0 when cbeg is at or past the end of the file.
uint64_t range_bytes(const c3r_bam* h, uint64_t cbeg, uint64_t cend_block) {
    if (cbeg >= h->file_size) return 0;
    const uint64_t last = cend_block == UINT64_MAX ? h->file_size : std::min<uint64_t>(h->file_size, cend_block + 0x10000);
    return last - cbeg;
}

// Reads range_bytes(cbeg, cend_block) bytes of the file into `dst` and cuts them into the block table (`blocks`,
// uoff relative to the range, `*ubytes` their inflated size).  Returns a c3rbgzf::FetchErr.  The one reading of a
// fetch's blocks: the host fetch inflates what it returns, the raw fetch hands it to the device.
int read_blocks(c3r_bam* h, uint64_t cbeg, uint64_t cend_block, uint8_t* dst, std::vector<Block>& blocks, uint64_t* ubytes) {
    blocks.clear();
    *ubytes = 0;
    const uint64_t n = range_bytes(h, cbeg, cend_block);
    if (n == 0) return 0;
    if (fseeko(h->fp, (off_t)cbeg, SEEK_SET) != 0 || fread(dst, 1, n, h->fp) != n) return c3rbgzf::FE_SHORT_READ;
    size_t o = 0;
    uint64_t uoff = 0;
    while (o < n) {
        const uint32_t bs = bgzf_block_size(dst + o, n - o);
        if (bs == 0 || o + bs > n) {
            if (cend_block != UINT64_MAX && cbeg + o > cend_block) break;      // partial block past the range: ignore
            if (o + 18 > n && cend_block != UINT64_MAX) break;
            return c3rbgzf::FE_HEADER;
        }
        Block b;
        b.coff = cbeg + o; b.csize = bs; b.usize = rd32(dst + o + bs - 4); b.uoff = uoff;
        if (b.usize > 0x10000) return c3rbgzf::FE_BIG_BLOCK;
        blocks.push_back(b);
        uoff += b.usize;
        o += bs;
        if (cend_block != UINT64_MAX && b.coff > cend_block) break;
    }
    *ubytes = uoff;
    return 0;
}

// Inflate the blocks of read_blocks(cbeg, cend_block) into h->ubuf; `blocks` gets the block table.
int inflate_range(c3r_bam* h, uint64_t cbeg, uint64_t cend_block, std::vector<Block>& blocks) {
    h->cbuf.resize(range_bytes(h, cbeg, cend_block));
    uint64_t uoff = 0;
    if (int e = read_blocks(h, cbeg, cend_block, h->cbuf.data(), blocks, &uoff)) return bfail(h, C3R_ERR_ARG, fetch_err_text(h, e));
    const uint8_t* base = h->cbuf.data();
    h->ubuf.resize(uoff);
    std::atomic<size_t> next(0);
    std::atomic<int> bad(0);
    auto work = [&]() {
        for (;;) {
            const size_t i = next.fetch_add(1);
            if (i >= blocks.size()) return;
            const Block& b = blocks[i];
            if (b.usize == 0) continue;
            if (!inflate_block(base + (b.coff - cbeg), b.csize, h->ubuf.data() + b.uoff, b.usize)) bad.store(1);
        }
    };
    const int nt = (int)std::min<size_t>((size_t)std::max(1, h->n_threads), std::max<size_t>(1, blocks.size() / 4));
    if (nt <= 1) work();
    else {
        std::vector<std::thread> th;
        for (int i = 0; i < nt; ++i) th.emplace_back(work);
        for (auto& t : th) t.join();
    }
    if (bad.load()) return bfail(h, C3R_ERR_ARG, fetch_err_text(h, c3rbgzf::FE_INFLATE));
    return 0;
}

int load_header(c3r_bam* h) {
    // the header may span several blocks: inflate from the start until it is complete
    std::vector<Block> blocks;
    uint64_t want = 1 << 20;
    for (;;) {
        const uint64_t upto = std::min<uint64_t>(h->file_size, want);
        if (int rc = inflate_range(h, 0, upto >= h->file_size ? UINT64_MAX : upto, blocks)) return rc;
        const std::vector<uint8_t>& u = h->ubuf;
        bool complete = false;
        do {
            if (u.size() < 12) break;
            if (memcmp(u.data(), "BAM\1", 4) != 0) return bfail(h, C3R_ERR_ARG, h->path + " is not a BAM file");
            const uint64_t l_text = rd32(u.data() + 4);
            uint64_t o = 8 + l_text;
            if (u.size() < o + 4) break;
            const uint32_t n_ref = rd32(u.data() + o);
            o += 4;
            std::vector<std::string> names;
            std::vector<int64_t> lens;
            bool ok = true;
            for (uint32_t i = 0; i < n_ref; ++i) {
                if (u.size() < o + 4) { ok = false; break; }
                const uint32_t l_name = rd32(u.data() + o);
                if (u.size() < o + 4 + l_name + 4) { ok = false; break; }
                names.emplace_back((const char*)u.data() + o + 4, l_name ? l_name - 1 : 0);
                lens.push_back((int64_t)rd32(u.data() + o + 4 + l_name));
                o += 8 + l_name;
            }
            if (!ok) break;
            h->header_text.assign((const char*)u.data() + 8, l_text);
            h->ref_names = names;
            h->ref_lens = lens;
            complete = true;
        } while (0);
        if (complete) return 0;
        if (upto >= h->file_size) return bfail(h, C3R_ERR_ARG, "truncated BAM header in " + h->path);
        want *= 4;
    }
}

int load_index(c3r_bam* h, const std::string& ipath) {
    FILE* f = fopen(ipath.c_str(), "rb");
    if (!f) return bfail(h, C3R_ERR_ARG, "cannot open BAM index " + ipath);
    fseeko(f, 0, SEEK_END);
    const size_t n = (size_t)ftello(f);
    fseeko(f, 0, SEEK_SET);
    std::vector<uint8_t> b(n);
    const bool ok = fread(b.data(), 1, n, f) == n;
    fclose(f);
    if (!ok || n < 8 || memcmp(b.data(), "BAI\1", 4) != 0) return bfail(h, C3R_ERR_ARG, ipath + " is not a BAI index");
    size_t o = 4;
    const uint32_t n_ref = rd32(b.data() + o);
    o += 4;
    h->index.assign(n_ref, RefIndex());
    for (uint32_t r = 0; r < n_ref; ++r) {
        RefIndex& ri = h->index[r];
        if (o + 4 > n) return bfail(h, C3R_ERR_ARG, "truncated BAI");
        const uint32_t n_bin = rd32(b.data() + o);
        o += 4;
        for (uint32_t k = 0; k < n_bin; ++k) {
            if (o + 8 > n) return bfail(h, C3R_ERR_ARG, "truncated BAI");
            const uint32_t bin = rd32(b.data() + o);
            const uint32_t n_chunk = rd32(b.data() + o + 4);
            o += 8;
            if (o + 16ull * n_chunk > n) return bfail(h, C3R_ERR_ARG, "truncated BAI");
            std::vector<Chunk> cs(n_chunk);
            for (uint32_t c = 0; c < n_chunk; ++c) { cs[c].beg = rd64(b.data() + o); cs[c].end = rd64(b.data() + o + 8); o += 16; }
            if (bin == (uint32_t)META_BIN && n_chunk == 2) {
                ri.has_meta = true;
                ri.n_mapped = cs[1].beg;
                ri.n_unmapped = cs[1].end;
            } else ri.bins.emplace_back(bin, std::move(cs));
        }
        if (o + 4 > n) return bfail(h, C3R_ERR_ARG, "truncated BAI");
        const uint32_t n_intv = rd32(b.data() + o);
        o += 4;
        if (o + 8ull * n_intv > n) return bfail(h, C3R_ERR_ARG, "truncated BAI");
        ri.linear.resize(n_intv);
        for (uint32_t i = 0; i < n_intv; ++i) { ri.linear[i] = rd64(b.data() + o); o += 8; }
        std::sort(ri.bins.begin(), ri.bins.end(), [](const auto& a, const auto& c) { return a.first < c.first; });
    }
    return 0;
}

// ------------------------------------------------------------------ record decoding (bam_rec.cuh)
void append_record(c3r_bam* h, const c3rbam::RecInfo& x) {
    const c3rbam::RecView& r = x.r;
    h->pos.push_back(r.pos);
    h->flag.push_back(r.flag);
    h->mapq.push_back(r.mapq);
    h->hp.push_back(c3rbam::clamp_hp(x.hp));
    const size_t c0 = h->cigar.size();
    h->cigar.resize(c0 + x.n_cig);
    for (uint32_t i = 0; i < x.n_cig; ++i) h->cigar[c0 + i] = rd32(x.cig + 4 * i);
    h->cigar_off.push_back((int32_t)h->cigar.size());
    const int64_t n_bases = x.n_bases;
    const size_t s0 = h->seq.size();
    if (r.l_seq > 0) {
        h->seq.insert(h->seq.end(), r.seq, r.seq + (r.l_seq + 1) / 2);
        if (r.l_seq & 1) h->seq.back() &= 0xf0;
    } else {
        h->seq.resize(s0 + (size_t)(n_bases + 1) / 2, 0xff);
        if ((n_bases & 1) && n_bases > 0) h->seq.back() = 0xf0;
    }
    h->seq_off.push_back(h->seq_off.back() + ((n_bases + 1) & ~1LL));
}

void reset_out(c3r_bam* h) {
    h->pos.clear(); h->flag.clear(); h->mapq.clear(); h->hp.clear(); h->cigar.clear(); h->seq.clear();
    h->cigar_off.assign(1, 0);
    h->seq_off.assign(1, 0);
}

void export_out(c3r_bam* h, c3r_reads* out) {
    memset(out, 0, sizeof *out);
    out->n_reads = (int64_t)h->pos.size();
    out->n_ops = (int64_t)h->cigar.size();
    out->n_seq_bytes = (int64_t)h->seq.size();
    out->pos = h->pos.data(); out->flag = h->flag.data(); out->mapq = h->mapq.data(); out->hp = h->hp.data();
    out->cigar_off = h->cigar_off.data(); out->cigar = h->cigar.data(); out->seq_off = h->seq_off.data(); out->seq = h->seq.data();
}

}  // namespace

// =============================================================== C ABI
extern "C" {

int c3r_bam_open(const char* path, const char* index_path, int n_threads, c3r_bam** out) {
    if (!path || !out) return C3R_ERR_ARG;
    c3r_bam* h = new c3r_bam();
    *out = h;                                   // returned even on failure so the caller can read the error
    h->path = path;
    h->n_threads = n_threads > 0 ? n_threads : (int)std::max(1u, std::thread::hardware_concurrency());
    h->fp = fopen(path, "rb");
    if (!h->fp) return bfail(h, C3R_ERR_ARG, std::string("cannot open ") + path);
    fseeko(h->fp, 0, SEEK_END);
    h->file_size = (uint64_t)ftello(h->fp);
    if (int rc = load_header(h)) return rc;
    std::string ip = index_path ? index_path : "";
    if (ip.empty()) {
        ip = h->path + ".bai";
        FILE* t = fopen(ip.c_str(), "rb");
        if (t) fclose(t);
        else if (h->path.size() > 4) ip = h->path.substr(0, h->path.size() - 4) + ".bai";
    }
    if (int rc = load_index(h, ip)) return rc;
    reset_out(h);
    return C3R_OK;
}

void c3r_bam_close(c3r_bam* h) {
    if (!h) return;
    if (h->fp) fclose(h->fp);
    delete h;
}

const char* c3r_bam_error(c3r_bam* h) { return h ? h->err.c_str() : "null handle"; }
int c3r_bam_n_ref(c3r_bam* h) { return h ? (int)h->ref_names.size() : 0; }
const char* c3r_bam_ref_name(c3r_bam* h, int tid) {
    return (h && tid >= 0 && tid < (int)h->ref_names.size()) ? h->ref_names[tid].c_str() : nullptr;
}
int64_t c3r_bam_ref_len(c3r_bam* h, int tid) {
    return (h && tid >= 0 && tid < (int)h->ref_lens.size()) ? h->ref_lens[tid] : -1;
}
const char* c3r_bam_header_text(c3r_bam* h) { return h ? h->header_text.c_str() : nullptr; }

int c3r_bam_idxstats(c3r_bam* h, int tid, int64_t* n_mapped, int64_t* n_unmapped) {
    if (!h || tid < 0 || tid >= (int)h->index.size()) return C3R_ERR_ARG;
    const RefIndex& ri = h->index[tid];
    if (n_mapped) *n_mapped = ri.has_meta ? (int64_t)ri.n_mapped : 0;
    if (n_unmapped) *n_unmapped = ri.has_meta ? (int64_t)ri.n_unmapped : 0;
    return ri.has_meta ? C3R_OK : C3R_ERR_STATE;
}

}  // extern "C"

namespace {

// The index query of a fetch: the chunks of the bins overlapping [beg, end), cut by the linear index, sorted and
// merged (beg <= previous end).  Each merged chunk is one window of the fetch.
void query_chunks(const c3r_bam* h, int tid, int64_t beg, int64_t end, std::vector<Chunk>& merged) {
    merged.clear();
    if (tid >= (int)h->index.size() || beg >= end) return;
    const RefIndex& ri = h->index[tid];
    uint64_t min_off = 0;
    if (!ri.linear.empty()) {
        const size_t w = (size_t)(beg >> 14);
        min_off = w < ri.linear.size() ? ri.linear[w] : ri.linear.back();
        if (w >= ri.linear.size()) min_off = ri.linear.back();
    }
    std::vector<int> bins;
    reg2bins(beg, end, bins);
    std::vector<Chunk> chunks;
    for (int b : bins) {
        auto it = std::lower_bound(ri.bins.begin(), ri.bins.end(), (uint32_t)b, [](const auto& a, uint32_t v) { return a.first < v; });
        if (it == ri.bins.end() || it->first != (uint32_t)b) continue;
        for (const Chunk& c : it->second) if (c.end > min_off) chunks.push_back(c);
    }
    std::sort(chunks.begin(), chunks.end(), [](const Chunk& a, const Chunk& c) { return a.beg < c.beg; });
    for (const Chunk& c : chunks) {
        if (!merged.empty() && c.beg <= merged.back().end) merged.back().end = std::max(merged.back().end, c.end);
        else merged.push_back(c);
    }
}

// compressed range of a window and the record walk bounds in its inflated bytes (usize of them)
inline uint64_t window_cbeg(const Chunk& c) { return c.beg >> 16; }
inline uint64_t window_cend(const Chunk& c) { return c.end >> 16; }
void window_bounds(const Chunk& c, const std::vector<Block>& blocks, uint64_t usize, uint64_t* ubeg, uint64_t* uend) {
    *ubeg = c.beg & 0xffff;
    *uend = usize;
    for (const Block& b : blocks) if (b.coff == window_cend(c)) { *uend = b.uoff + (c.end & 0xffff); break; }
}

int check_fetch_args(c3r_bam* h, int tid, int64_t start1, int64_t end1) {
    if (tid < 0 || tid >= (int)h->ref_names.size()) return bfail(h, C3R_ERR_ARG, "reference id out of range");
    if (start1 < 1 || end1 < start1) return bfail(h, C3R_ERR_ARG, "bad region");
    return 0;
}

}  // namespace

extern "C" {

int c3r_bam_fetch(c3r_bam* h, int tid, int64_t start1, int64_t end1, c3r_reads* out) {
    if (!h || !out) return C3R_ERR_ARG;
    if (int rc = check_fetch_args(h, tid, start1, end1)) return rc;
    reset_out(h);
    const int64_t beg = start1 - 1, end = std::min<int64_t>(end1, 1LL << 29);      // 0-based half open
    std::vector<Chunk> merged;
    query_chunks(h, tid, beg, end, merged);
    std::vector<Block> blocks;
    bool past_end = false;
    for (const Chunk& c : merged) {
        if (past_end) break;
        if (int rc = inflate_range(h, window_cbeg(c), window_cend(c), blocks)) return rc;
        if (blocks.empty()) continue;
        uint64_t ubeg, uend;
        window_bounds(c, blocks, h->ubuf.size(), &ubeg, &uend);
        const uint8_t* u = h->ubuf.data();
        uint64_t o = ubeg;
        while (o + 4 <= uend) {
            const uint32_t bs = rd32(u + o);
            if (o + 4 + bs > h->ubuf.size()) return bfail(h, C3R_ERR_ARG, fetch_err_text(h, c3rbgzf::FE_CROSS));
            c3rbam::RecInfo x;
            const int cls = c3rbam::classify_record(u + o + 4, bs, tid, beg, end, x);
            o += 4 + bs;
            if (cls == c3rbam::REC_ERR_MALFORMED) return bfail(h, C3R_ERR_ARG, fetch_err_text(h, c3rbgzf::FE_MALFORMED));
            if (cls == c3rbam::REC_ERR_AUX) return bfail(h, C3R_ERR_ARG, fetch_err_text(h, c3rbgzf::FE_AUX));
            if (cls == c3rbam::REC_STOP) { past_end = true; break; }
            if (cls == c3rbam::REC_KEEP) append_record(h, x);
        }
    }
    export_out(h, out);
    return C3R_OK;
}

int c3r_bam_fetch_raw(c3r_bam* h, int tid, int64_t start1, int64_t end1, uint8_t* buf, int64_t cap, c3r_bam_raw* out) {
    if (!h || !out || cap < 0 || (cap > 0 && !buf)) return C3R_ERR_ARG;
    if (int rc = check_fetch_args(h, tid, start1, end1)) return rc;
    memset(out, 0, sizeof *out);
    h->raw_blocks.clear();
    h->raw_windows.clear();
    const int64_t beg = start1 - 1, end = std::min<int64_t>(end1, 1LL << 29);
    out->tid = tid;
    out->beg = beg;
    out->end = end;
    std::vector<Chunk> merged;
    query_chunks(h, tid, beg, end, merged);
    int64_t need = 0;
    for (const Chunk& c : merged) need += (int64_t)range_bytes(h, window_cbeg(c), window_cend(c));
    out->n_bytes = need;
    if (need > cap) return bfail(h, C3R_ERR_CAPACITY, "buffer too small for the compressed blocks of the region");
    std::vector<Block> blocks;
    int64_t coff = 0, ubase = 0;
    for (const Chunk& c : merged) {
        c3r_bam_window w;
        memset(&w, 0, sizeof w);
        uint64_t usize = 0;
        w.status = read_blocks(h, window_cbeg(c), window_cend(c), buf + coff, blocks, &usize);
        w.first_block = (int32_t)h->raw_blocks.size();
        if (!w.status) {
            uint64_t ubeg, uend;
            window_bounds(c, blocks, usize, &ubeg, &uend);
            w.ubase = ubase; w.usize = (int64_t)usize; w.ubeg = (int64_t)ubeg; w.uend = (int64_t)uend;
            w.n_blocks = (int32_t)blocks.size();
            for (const Block& b : blocks) {
                c3r_bgzf_block o;
                o.coff = coff + (int64_t)(b.coff - window_cbeg(c));
                o.uoff = ubase + (int64_t)b.uoff;
                o.csize = (int32_t)b.csize; o.usize = (int32_t)b.usize;
                o.window = (int32_t)h->raw_windows.size();
                o.reserved = 0;
                h->raw_blocks.push_back(o);
            }
            ubase += (int64_t)usize;
        }
        coff += (int64_t)range_bytes(h, window_cbeg(c), window_cend(c));
        h->raw_windows.push_back(w);
        if (w.status) break;                         // the host fetch returns here: nothing after it is read
    }
    out->n_windows = (int32_t)h->raw_windows.size();
    out->n_blocks = (int64_t)h->raw_blocks.size();
    out->n_ubytes = ubase;
    out->data = buf;
    out->blocks = h->raw_blocks.data();
    out->windows = h->raw_windows.data();
    return C3R_OK;
}

int c3r_debug_inflate(const uint8_t* block, int64_t n, uint8_t* out, int64_t cap, int64_t* n_out) {
    if (!block || !n_out || n < 26 || n > 0x10000 || cap < 0 || (cap > 0 && !out)) return C3R_ERR_ARG;
    const uint32_t bs = bgzf_block_size(block, (size_t)n);
    if (bs != (uint32_t)n) return C3R_ERR_ARG;
    const uint32_t usize = rd32(block + n - 4);
    *n_out = usize;
    if (usize > c3rbgzf::MAX_BLOCK || (int64_t)usize > cap) return C3R_ERR_ARG;
    uint32_t off, len;
    if (!c3rbgzf::bgzf_payload(block, (uint32_t)n, &off, &len)) return C3R_ERR_ARG;
    c3rbgzf::HostSink sink;
    sink.out = out; sink.cap = usize; sink.pos = 0;
    c3rbgzf::Tables t;
    if (c3rbgzf::inflate_core(block + off, len, sink, t) != c3rbgzf::IE_OK || sink.pos != usize) return C3R_ERR_ARG;
    // the device's CRC: 32 segments combined
    uint32_t tab[256];
    for (uint32_t k = 0; k < 256; ++k) tab[k] = c3rbgzf::crc_table_entry(k);
    const uint32_t seg = (usize + 31) / 32;
    uint32_t acc = 0;
    for (uint32_t a = 0; a < usize; a += seg) {
        const uint32_t l = std::min(seg, usize - a);
        acc = c3rbgzf::crc32_combine(acc, c3rbgzf::crc32_bytes(tab, out + a, l), l);
    }
    return acc == rd32(block + n - 8) ? C3R_OK : C3R_ERR_ARG;
}

// ---------------------------------------------------------------- writer (synthetic fixtures)
namespace {
struct BgzfWriter {
    FILE* fp = nullptr;
    std::vector<uint8_t> buf;
    uint64_t coff = 0;
    int level = 6;
    bool ok = true;
    uint64_t tell() const { return (coff << 16) | (uint64_t)buf.size(); }
    void flush_block() {
        uint8_t out[0x10000 + 64];
        z_stream zs;
        memset(&zs, 0, sizeof zs);
        if (deflateInit2(&zs, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) { ok = false; return; }
        zs.next_in = buf.data();
        zs.avail_in = (uInt)buf.size();
        zs.next_out = out + 18;
        zs.avail_out = sizeof(out) - 18 - 8;
        if (deflate(&zs, Z_FINISH) != Z_STREAM_END) { ok = false; deflateEnd(&zs); return; }
        const uint32_t clen = (uint32_t)zs.total_out;
        deflateEnd(&zs);
        const uint32_t total = clen + 26;
        const uint8_t hdr[18] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0,
                                 (uint8_t)((total - 1) & 0xff), (uint8_t)((total - 1) >> 8)};
        memcpy(out, hdr, 18);
        const uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), buf.data(), (uInt)buf.size());
        uint8_t* t = out + 18 + clen;
        for (int i = 0; i < 4; ++i) t[i] = (crc >> (8 * i)) & 0xff;
        for (int i = 0; i < 4; ++i) t[4 + i] = ((uint32_t)buf.size() >> (8 * i)) & 0xff;
        if (fwrite(out, 1, total, fp) != total) ok = false;
        coff += total;
        buf.clear();
    }
    void write(const uint8_t* p, size_t n) {
        while (n) {
            const size_t room = BGZF_MAX_PAYLOAD - buf.size();
            const size_t k = n < room ? n : room;
            buf.insert(buf.end(), p, p + k);
            p += k; n -= k;
            if (buf.size() == (size_t)BGZF_MAX_PAYLOAD) flush_block();
        }
    }
    void finish() {
        if (!buf.empty()) flush_block();
        flush_block();                              // empty EOF block
    }
};
}  // namespace

// Writes a coordinate-sorted BAM (+ .bai next to it) from flat records: batches[r] holds the records of
// reference r (may be NULL / empty).  Read names are synthetic, qualities are absent (0xff), HP:i is
// written (type C) for hp != 0.  Used to build fixtures for the reader and the drop-in entry point.
int c3r_bam_write(const char* path, int n_ref, const char* const* names, const int64_t* lens,
                  const c3r_reads* const* batches, int level, const char* header_text) {
    if (!path || n_ref < 0 || (n_ref && (!names || !lens || !batches))) return C3R_ERR_ARG;
    BgzfWriter w;
    w.fp = fopen(path, "wb");
    if (!w.fp) return C3R_ERR_ARG;
    w.level = level < 0 ? 6 : level;
    std::vector<uint8_t> hd;
    std::string text = header_text ? header_text : "";
    if (text.empty()) {
        text = "@HD\tVN:1.6\tSO:coordinate\n";
        for (int r = 0; r < n_ref; ++r) text += std::string("@SQ\tSN:") + names[r] + "\tLN:" + std::to_string(lens[r]) + "\n";
    }
    hd.insert(hd.end(), {'B', 'A', 'M', 1});
    wr32(hd, (uint32_t)text.size());
    hd.insert(hd.end(), text.begin(), text.end());
    wr32(hd, (uint32_t)n_ref);
    for (int r = 0; r < n_ref; ++r) {
        const size_t l = strlen(names[r]) + 1;
        wr32(hd, (uint32_t)l);
        hd.insert(hd.end(), names[r], names[r] + l);
        wr32(hd, (uint32_t)lens[r]);
    }
    w.write(hd.data(), hd.size());
    w.flush_block();                                // records start on a block boundary
    std::vector<RefIndex> index(n_ref);
    std::vector<std::vector<std::pair<uint32_t, std::vector<Chunk>>>> dummy;
    std::vector<uint8_t> rec;
    uint64_t serial = 0;
    for (int r = 0; r < n_ref; ++r) {
        const c3r_reads* b = batches[r];
        RefIndex& ri = index[r];
        if (!b || b->n_reads == 0) continue;
        std::vector<std::pair<uint32_t, Chunk>> bin_chunks;
        uint64_t ref_beg = w.tell(), ref_end = ref_beg;
        for (int64_t i = 0; i < b->n_reads; ++i, ++serial) {
            const int32_t c0 = b->cigar_off[i], c1 = b->cigar_off[i + 1];
            const uint32_t n_cig = (uint32_t)(c1 - c0);
            const int64_t l_seq = b->seq_off[i + 1] - b->seq_off[i];           // even-padded base count
            // the flat layout pads odd reads with one zero nibble: recover l_seq from the CIGAR
            int64_t ql = 0, rl = 0;
            for (int32_t k = c0; k < c1; ++k) {
                const uint32_t v = b->cigar[k], op = v & 15;
                if (op == 0 || op == 1 || op == 4 || op == 7 || op == 8) ql += v >> 4;
                if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) rl += v >> 4;
            }
            const int64_t ls = (ql <= l_seq && ql + 1 >= l_seq) ? ql : l_seq;
            char name[32];
            const int l_name = snprintf(name, sizeof name, "r%llu", (unsigned long long)serial) + 1;
            const int64_t end = b->pos[i] + (rl > 0 ? rl : 1);
            const bool long_cig = n_cig > 65535;
            rec.clear();
            wr32(rec, 0);                                           // block_size, patched below
            wr32(rec, (uint32_t)r);
            wr32(rec, (uint32_t)b->pos[i]);
            rec.push_back((uint8_t)l_name);
            rec.push_back(b->mapq[i]);
            wr16(rec, (uint16_t)reg2bin(b->pos[i], end));
            wr16(rec, (uint16_t)(long_cig ? 2 : n_cig));
            wr16(rec, b->flag[i]);
            wr32(rec, (uint32_t)ls);
            wr32(rec, 0xffffffffu); wr32(rec, 0xffffffffu); wr32(rec, 0);    // next refID, next pos, tlen
            rec.insert(rec.end(), name, name + l_name);
            if (long_cig) {
                wr32(rec, ((uint32_t)ls << 4) | 4u);
                wr32(rec, ((uint32_t)rl << 4) | 3u);
            } else for (int32_t k = c0; k < c1; ++k) wr32(rec, b->cigar[k]);
            const uint8_t* sq = b->seq + b->seq_off[i] / 2;
            rec.insert(rec.end(), sq, sq + (ls + 1) / 2);
            rec.insert(rec.end(), (size_t)ls, (uint8_t)0xff);
            if (b->hp[i]) { rec.push_back('H'); rec.push_back('P'); rec.push_back('C'); rec.push_back(b->hp[i]); }
            if (long_cig) {
                rec.push_back('C'); rec.push_back('G'); rec.push_back('B'); rec.push_back('I');
                wr32(rec, n_cig);
                for (int32_t k = c0; k < c1; ++k) wr32(rec, b->cigar[k]);
            }
            const uint32_t bs = (uint32_t)rec.size() - 4;
            for (int k = 0; k < 4; ++k) rec[k] = (bs >> (8 * k)) & 0xff;
            const uint64_t v0 = w.tell();
            w.write(rec.data(), rec.size());
            const uint64_t v1 = w.tell();
            ref_end = v1;
            const uint32_t bin = (uint32_t)reg2bin(b->pos[i], end);
            if (!bin_chunks.empty() && bin_chunks.back().first == bin && bin_chunks.back().second.end == v0) bin_chunks.back().second.end = v1;
            else bin_chunks.push_back({bin, {v0, v1}});
            const size_t w0 = (size_t)(b->pos[i] >> 14), w1 = (size_t)((end - 1) >> 14);
            if (ri.linear.size() <= w1) ri.linear.resize(w1 + 1, 0);
            for (size_t k = w0; k <= w1; ++k) if (ri.linear[k] == 0) ri.linear[k] = v0;
            if (b->flag[i] & 4) ++ri.n_unmapped; else ++ri.n_mapped;
        }
        // htslib fills empty linear-index windows with the following non-empty value's predecessor; the reader only
        // needs a lower bound, so carry the previous offset forward
        uint64_t last = ref_beg;
        for (uint64_t& v : ri.linear) { if (v == 0) v = last; else last = v; }
        std::sort(bin_chunks.begin(), bin_chunks.end(), [](const auto& a, const auto& c) {
            return a.first != c.first ? a.first < c.first : a.second.beg < c.second.beg; });
        for (const auto& bc : bin_chunks) {
            if (ri.bins.empty() || ri.bins.back().first != bc.first) ri.bins.emplace_back(bc.first, std::vector<Chunk>());
            ri.bins.back().second.push_back(bc.second);
        }
        ri.has_meta = true;
        std::vector<Chunk> meta = {{ref_beg, ref_end}, {ri.n_mapped, ri.n_unmapped}};
        ri.bins.emplace_back((uint32_t)META_BIN, meta);
    }
    w.finish();
    const bool ok = w.ok;
    fclose(w.fp);
    if (!ok) return C3R_ERR_ARG;
    std::vector<uint8_t> ix;
    ix.insert(ix.end(), {'B', 'A', 'I', 1});
    wr32(ix, (uint32_t)n_ref);
    for (int r = 0; r < n_ref; ++r) {
        const RefIndex& ri = index[r];
        wr32(ix, (uint32_t)ri.bins.size());
        for (const auto& bn : ri.bins) {
            wr32(ix, bn.first);
            wr32(ix, (uint32_t)bn.second.size());
            for (const Chunk& c : bn.second) { wr64(ix, c.beg); wr64(ix, c.end); }
        }
        wr32(ix, (uint32_t)ri.linear.size());
        for (uint64_t v : ri.linear) wr64(ix, v);
    }
    wr64(ix, 0);                                    // n_no_coor
    const std::string ip = std::string(path) + ".bai";
    FILE* f = fopen(ip.c_str(), "wb");
    if (!f) return C3R_ERR_ARG;
    const bool iok = fwrite(ix.data(), 1, ix.size(), f) == ix.size();
    fclose(f);
    return iok ? C3R_OK : C3R_ERR_ARG;
}

// bgzip + tabix of a VCF text (what `sort_vcf --compress_vcf True` does through the external tools,
// src/sort_vcf.py:70-76): writes `path` as BGZF and `path`.tbi (tabix index, VCF preset: sequence column 1, begin
// column 2, meta '#'; 16 kb linear index and the UCSC binning scheme like BAI; interval of a record =
// [POS-1, POS-1+len(REF))).  The text must be header lines ('#') followed by position-sorted data lines.
int c3r_vcf_write_bgzf(const char* path, const char* text, int64_t n_bytes, int level) {
    if (!path || (!text && n_bytes) || n_bytes < 0) return C3R_ERR_ARG;
    BgzfWriter w;
    w.level = level <= 0 ? 6 : level;
    w.fp = fopen(path, "wb");
    if (!w.fp) return C3R_ERR_ARG;
    std::vector<std::string> names;
    std::vector<RefIndex> index;
    std::vector<std::vector<std::pair<uint32_t, Chunk>>> chunks;
    int cur = -1;
    int64_t last_beg = -1;
    bool sorted = true;
    const char* p = text;
    const char* const e = text + n_bytes;
    while (p < e) {
        const char* nl = (const char*)memchr(p, '\n', (size_t)(e - p));
        const char* le = nl ? nl + 1 : e;                       // line incl. its newline
        const uint64_t v0 = w.tell();
        w.write((const uint8_t*)p, (size_t)(le - p));
        const uint64_t v1 = w.tell();
        if (*p != '#' && le - p > 1) {
            // CHROM \t POS \t ID \t REF
            const char* t1 = (const char*)memchr(p, '\t', (size_t)(le - p));
            const char* t2 = t1 ? (const char*)memchr(t1 + 1, '\t', (size_t)(le - t1 - 1)) : nullptr;
            const char* t3 = t2 ? (const char*)memchr(t2 + 1, '\t', (size_t)(le - t2 - 1)) : nullptr;
            const char* t4 = t3 ? (const char*)memchr(t3 + 1, '\t', (size_t)(le - t3 - 1)) : nullptr;
            if (!t4) { fclose(w.fp); return C3R_ERR_ARG; }
            const std::string chrom(p, t1);
            const int64_t beg = strtoll(t1 + 1, nullptr, 10) - 1;
            const int64_t end = beg + (t4 - t3 - 1 > 0 ? (int64_t)(t4 - t3 - 1) : 1);
            if (beg < 0) { fclose(w.fp); return C3R_ERR_ARG; }
            if (cur < 0 || names[cur] != chrom) {
                for (const std::string& nm : names) if (nm == chrom) sorted = false;   // a contig must be one block
                names.push_back(chrom);
                index.emplace_back();
                chunks.emplace_back();
                cur = (int)names.size() - 1;
                last_beg = -1;
            }
            if (beg < last_beg) sorted = false;
            last_beg = beg;
            RefIndex& ri = index[cur];
            auto& bc = chunks[cur];
            const uint32_t bin = (uint32_t)reg2bin(beg, end);
            if (!bc.empty() && bc.back().first == bin && bc.back().second.end == v0) bc.back().second.end = v1;
            else bc.push_back({bin, {v0, v1}});
            const size_t w0 = (size_t)(beg >> 14), w1 = (size_t)((end - 1) >> 14);
            if (ri.linear.size() <= w1) ri.linear.resize(w1 + 1, 0);
            for (size_t k = w0; k <= w1; ++k) if (ri.linear[k] == 0) ri.linear[k] = v0;
            ++ri.n_mapped;
        }
        p = le;
    }
    w.finish();
    const bool ok = w.ok;
    fclose(w.fp);
    if (!ok || !sorted) return C3R_ERR_ARG;
    std::vector<uint8_t> ix;
    ix.insert(ix.end(), {'T', 'B', 'I', 1});
    wr32(ix, (uint32_t)names.size());
    wr32(ix, 2); wr32(ix, 1); wr32(ix, 2); wr32(ix, 0); wr32(ix, (uint32_t)'#'); wr32(ix, 0);
    uint32_t l_nm = 0;
    for (const std::string& nm : names) l_nm += (uint32_t)nm.size() + 1;
    wr32(ix, l_nm);
    for (const std::string& nm : names) { ix.insert(ix.end(), nm.begin(), nm.end()); ix.push_back(0); }
    for (size_t r = 0; r < names.size(); ++r) {
        RefIndex& ri = index[r];
        uint64_t last = 0;
        for (uint64_t& v : ri.linear) { if (v == 0) v = last; else last = v; }
        auto& bc = chunks[r];
        std::stable_sort(bc.begin(), bc.end(), [](const auto& a, const auto& c) {
            return a.first != c.first ? a.first < c.first : a.second.beg < c.second.beg; });
        std::vector<std::pair<uint32_t, std::vector<Chunk>>> bins;
        for (const auto& x : bc) {
            if (bins.empty() || bins.back().first != x.first) bins.emplace_back(x.first, std::vector<Chunk>());
            bins.back().second.push_back(x.second);
        }
        wr32(ix, (uint32_t)bins.size());
        for (const auto& bn : bins) {
            wr32(ix, bn.first);
            wr32(ix, (uint32_t)bn.second.size());
            for (const Chunk& c : bn.second) { wr64(ix, c.beg); wr64(ix, c.end); }
        }
        wr32(ix, (uint32_t)ri.linear.size());
        for (uint64_t v : ri.linear) wr64(ix, v);
    }
    BgzfWriter wi;
    const std::string ip = std::string(path) + ".tbi";
    wi.fp = fopen(ip.c_str(), "wb");
    if (!wi.fp) return C3R_ERR_ARG;
    wi.write(ix.data(), ix.size());
    wi.finish();
    const bool iok = wi.ok;
    fclose(wi.fp);
    return iok ? C3R_OK : C3R_ERR_ARG;
}

}  // extern "C"
