// BGZF blocks inflated and BAM records parsed on the device: the device half of c3r_submit_bam_chunk.
//
// The host (c3r_bam_fetch_raw, csrc/bam_io.cpp) does the index query and reads the compressed bytes of each merged
// index chunk ("window"); the kernels here turn them into the flat c3r_reads arrays c3r_bam_fetch makes:
//   k_inflate      one BGZF block per CTA (one warp): RFC 1951 in full into shared memory, ISIZE and CRC32 checked
//                  (the CRC per lane over 1/32 of the block, combined), then written to the window's bytes;
//   k_rec_bounds   one CTA per window: the record length chain followed through shared-memory tiles of the window;
//   k_rec_parse    one thread per record: the fetch's checks, filters and stop rule (bam_rec.cuh), its CIGAR op and
//                  sequence byte counts;
//   (scan.cuh)     the output offsets of the records kept;
//   k_rec_write    one warp per record: pos, flag, mapq, hp, CIGAR and sequence into the slot's read buffers.
// The host fetch works a window at a time and returns at the first error or stops at the first record past the
// region, so the device orders both by one key, (window, stage, offset in the window): an inflate error of a window
// comes before its records, records in file order.  The first error is reported when it comes before the first stop.
//
// The DEFLATE decoder and the CRC arithmetic are C3R_HD code: c3r_debug_inflate runs them on the host.  Only the
// output sink (a warp copying matches lane-parallel in shared memory) is device-only.  Corrupt input is a status:
// every read is bounded by the block, the window or the record, every write by the output capacity.
#pragma once
#include <stdint.h>

#include "bam_rec.cuh"

namespace c3rbgzf {

constexpr uint32_t MAX_BLOCK = 0x10000;         // BGZF ISIZE limit

// error codes of a device fetch, in c3r_abi.cu's messages (the host fetch's texts)
enum FetchErr { FE_NONE = 0, FE_INFLATE = 1, FE_HEADER = 2, FE_BIG_BLOCK = 3, FE_SHORT_READ = 4, FE_CROSS = 5,
                FE_MALFORMED = 6, FE_AUX = 7 };

// (window, stage, offset) -> one ordered key; stage 0 = the window's blocks, 1 = its records.  The low 3 bits carry
// the error code.
C3R_HD uint64_t order_key(uint32_t w, uint32_t stage, uint64_t off, uint32_t code) {
    return ((uint64_t)w << 44) | ((uint64_t)stage << 43) | ((off & ((1ull << 40) - 1)) << 3) | code;
}

// ------------------------------------------------------------------ CRC32 (zlib's polynomial)
constexpr uint32_t CRC_POLY = 0xedb88320u;

C3R_HD uint32_t crc_table_entry(uint32_t n) {
    uint32_t c = n;
    for (int k = 0; k < 8; ++k) c = c & 1 ? (c >> 1) ^ CRC_POLY : c >> 1;
    return c;
}
// CRC of bytes [p, p + n) (finalised: ~ in and out), table of 256 entries
C3R_HD uint32_t crc32_bytes(const uint32_t* tab, const uint8_t* p, uint32_t n) {
    uint32_t c = 0xffffffffu;
    for (uint32_t i = 0; i < n; ++i) c = tab[(c ^ p[i]) & 0xff] ^ (c >> 8);
    return c ^ 0xffffffffu;
}
// a * b modulo the CRC polynomial (bit-reflected), as zlib's multmodp
C3R_HD uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ CRC_POLY : b >> 1;
    }
    return p;
}
// CRC of A followed by B from crc(A), crc(B) and len(B) (zlib's crc32_combine): crc(A) times x^(8 len(B))
C3R_HD uint32_t crc32_combine(uint32_t crc_a, uint32_t crc_b, uint32_t len_b) {
    uint32_t sq = 1u << 30;                      // x^1
    for (int k = 0; k < 3; ++k) sq = multmodp(sq, sq);   // x^8: one byte
    uint32_t p = 1u << 31;                       // x^0
    for (uint32_t n = len_b; n; n >>= 1) {
        if (n & 1) p = multmodp(sq, p);
        sq = multmodp(sq, sq);
    }
    return multmodp(p, crc_a) ^ crc_b;
}

// ------------------------------------------------------------------ DEFLATE (RFC 1951)
// Canonical Huffman code by counts per length and symbols in code order (the form of zlib's puff.c).
constexpr int MAXBITS = 15;
struct Huff {
    int16_t count[MAXBITS + 1];
    int16_t symbol[288];
};
// Shared state of one block's decode: the tables and the code-length scratch.  On the device it lives in shared
// memory; only the sink's leader lane writes it.
struct Tables {
    Huff lencode, distcode;
    int16_t lengths[320];
    int32_t left;                 // construct()'s result, for the lanes that did not build the table
};

// codes left over (> 0: incomplete, < 0: over-subscribed, 0: complete)
C3R_HD int construct(Huff& h, const int16_t* length, int n) {
    for (int len = 0; len <= MAXBITS; ++len) h.count[len] = 0;
    for (int s = 0; s < n; ++s) h.count[length[s]]++;
    if (h.count[0] == n) return 0;
    int left = 1;
    for (int len = 1; len <= MAXBITS; ++len) {
        left <<= 1;
        left -= h.count[len];
        if (left < 0) return left;
    }
    int16_t offs[MAXBITS + 1];
    offs[1] = 0;
    for (int len = 1; len < MAXBITS; ++len) offs[len + 1] = offs[len] + h.count[len];
    for (int s = 0; s < n; ++s)
        if (length[s] != 0) h.symbol[offs[length[s]]++] = (int16_t)s;
    return left;
}

// LSB-first bit reader over [p, p + n)
struct BitIn {
    const uint8_t* p;
    uint32_t n, pos;
    uint64_t buf;
    int cnt;
    C3R_HD void refill() {
        while (cnt <= 56 && pos < n) { buf |= (uint64_t)p[pos++] << cnt; cnt += 8; }
    }
    // false when the stream has fewer than k bits left
    C3R_HD bool bits(int k, uint32_t* v) {
        if (cnt < k) refill();
        if (cnt < k) return false;
        *v = (uint32_t)(buf & ((1ull << k) - 1));
        buf >>= k;
        cnt -= k;
        return true;
    }
};

// one symbol; < 0 on a code not in the table or a truncated stream
C3R_HD int decode(BitIn& in, const Huff& h) {
    if (in.cnt < MAXBITS) in.refill();
    uint32_t b = (uint32_t)in.buf;
    int code = 0, first = 0, index = 0;
    for (int len = 1; len <= MAXBITS; ++len) {
        code |= b & 1;
        b >>= 1;
        const int count = h.count[len];
        if (code - count < first) {
            if (len > in.cnt) return -2;
            in.buf >>= len;
            in.cnt -= len;
            return h.symbol[index + (code - first)];
        }
        index += count;
        first += count;
        first <<= 1;
        code <<= 1;
    }
    return -1;
}

enum InflateErr { IE_OK = 0, IE_TRUNCATED = -1, IE_BLOCK_TYPE = -2, IE_STORED_LEN = -3, IE_OVERFLOW = -4,
                  IE_CODES = -5, IE_SYMBOL = -6, IE_DISTANCE = -7, IE_ISIZE = -8, IE_CRC = -9, IE_HEADER = -10 };

// Inflates the raw DEFLATE stream [in, in + n) through `out` (a sink: pos, lit, match, stored, leader, sync).
// The output ends at the end of the final block; bytes after it are ignored, as zlib's inflate does.
template <class Sink>
C3R_HD int inflate_core(const uint8_t* in, uint32_t n, Sink& out, Tables& t) {
    BitIn bi;
    bi.p = in; bi.n = n; bi.pos = 0; bi.buf = 0; bi.cnt = 0;
    const uint16_t LBASE[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
    const uint8_t LEXT[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
    const uint16_t DBASE[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
    const uint8_t DEXT[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
    const uint8_t ORDER[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    uint32_t last = 0;
    do {
        uint32_t type;
        if (!bi.bits(1, &last) || !bi.bits(2, &type)) return IE_TRUNCATED;
        if (type == 0) {                                             // stored
            bi.buf >>= bi.cnt & 7;
            bi.cnt &= ~7;
            uint32_t len, nlen;
            if (!bi.bits(16, &len) || !bi.bits(16, &nlen)) return IE_TRUNCATED;
            if (len != (~nlen & 0xffffu)) return IE_STORED_LEN;
            bi.pos -= (uint32_t)(bi.cnt >> 3);                       // give the buffered whole bytes back
            bi.buf = 0;
            bi.cnt = 0;
            if (len > bi.n - bi.pos) return IE_TRUNCATED;
            if (!out.stored(bi.p + bi.pos, len)) return IE_OVERFLOW;
            bi.pos += len;
            continue;
        }
        if (type == 3) return IE_BLOCK_TYPE;
        if (type == 1) {                                             // fixed Huffman codes (RFC 1951 §3.2.6)
            if (out.leader()) {
                int s = 0;
                for (; s < 144; ++s) t.lengths[s] = 8;
                for (; s < 256; ++s) t.lengths[s] = 9;
                for (; s < 280; ++s) t.lengths[s] = 7;
                for (; s < 288; ++s) t.lengths[s] = 8;
                construct(t.lencode, t.lengths, 288);
                for (s = 0; s < 30; ++s) t.lengths[s] = 5;
                construct(t.distcode, t.lengths, 30);
            }
            out.sync();
        } else {                                                     // dynamic codes (RFC 1951 §3.2.7)
            uint32_t nlen, ndist, ncode;
            if (!bi.bits(5, &nlen) || !bi.bits(5, &ndist) || !bi.bits(4, &ncode)) return IE_TRUNCATED;
            nlen += 257; ndist += 1; ncode += 4;
            if (nlen > 286 || ndist > 30) return IE_CODES;
            if (out.leader()) for (int k = 0; k < 19; ++k) t.lengths[k] = 0;
            out.sync();
            for (uint32_t k = 0; k < ncode; ++k) {
                uint32_t v;
                if (!bi.bits(3, &v)) return IE_TRUNCATED;
                if (out.leader()) t.lengths[ORDER[k]] = (int16_t)v;
            }
            out.sync();
            if (out.leader()) t.left = construct(t.lencode, t.lengths, 19);
            out.sync();
            if (t.left != 0) return IE_CODES;                        // the code-length code must be complete
            uint32_t idx = 0;
            int prev = -1;
            while (idx < nlen + ndist) {
                int sym = decode(bi, t.lencode);
                if (sym < 0) return sym == -2 ? IE_TRUNCATED : IE_CODES;
                if (sym < 16) {
                    if (out.leader()) t.lengths[idx] = (int16_t)sym;
                    ++idx;
                    prev = sym;
                    continue;
                }
                int len = 0;
                uint32_t rep;
                if (sym == 16) {
                    if (prev < 0) return IE_CODES;                   // repeat with no length before it
                    len = prev;
                    if (!bi.bits(2, &rep)) return IE_TRUNCATED;
                    rep += 3;
                } else if (sym == 17) {
                    if (!bi.bits(3, &rep)) return IE_TRUNCATED;
                    rep += 3;
                } else {
                    if (!bi.bits(7, &rep)) return IE_TRUNCATED;
                    rep += 11;
                }
                if (idx + rep > nlen + ndist) return IE_CODES;
                for (uint32_t k = 0; k < rep; ++k) {
                    if (out.leader()) t.lengths[idx] = (int16_t)len;
                    ++idx;
                }
                prev = len;
            }
            out.sync();
            if (t.lengths[256] == 0) return IE_CODES;                // no end-of-block code
            if (out.leader()) {
                int err = construct(t.lencode, t.lengths, (int)nlen);
                // an incomplete code is allowed only as a single code of length 1 (zlib, puff)
                if (err < 0 || (err > 0 && (int)nlen != t.lencode.count[0] + t.lencode.count[1])) t.left = 1;
                else {
                    err = construct(t.distcode, t.lengths + nlen, (int)ndist);
                    t.left = (err < 0 || (err > 0 && (int)ndist != t.distcode.count[0] + t.distcode.count[1])) ? 1 : 0;
                }
            }
            out.sync();
            if (t.left != 0) return IE_CODES;
        }
        // the compressed data of the block
        for (;;) {
            int sym = decode(bi, t.lencode);
            if (sym < 0) return sym == -2 ? IE_TRUNCATED : IE_SYMBOL;
            if (sym < 256) {
                if (!out.lit((uint8_t)sym)) return IE_OVERFLOW;
                continue;
            }
            if (sym == 256) break;
            sym -= 257;
            if (sym >= 29) return IE_SYMBOL;
            uint32_t e = 0;
            if (LEXT[sym] && !bi.bits(LEXT[sym], &e)) return IE_TRUNCATED;
            const uint32_t len = LBASE[sym] + e;
            const int ds = decode(bi, t.distcode);
            if (ds < 0) return ds == -2 ? IE_TRUNCATED : IE_SYMBOL;
            if (ds >= 30) return IE_SYMBOL;
            e = 0;
            if (DEXT[ds] && !bi.bits(DEXT[ds], &e)) return IE_TRUNCATED;
            const uint32_t dist = DBASE[ds] + e;
            if (dist > out.pos) return IE_DISTANCE;
            if (!out.match(len, dist)) return IE_OVERFLOW;
        }
    } while (!last);
    return IE_OK;
}

// The deflate payload of a BGZF block of csize bytes (header, payload, CRC32, ISIZE); false if it does not fit
C3R_HD bool bgzf_payload(const uint8_t* blk, uint32_t csize, uint32_t* off, uint32_t* len) {
    if (csize < 26) return false;
    const uint32_t xlen = c3rbam::rd16(blk + 10);
    if (12u + xlen + 8u > csize) return false;
    *off = 12 + xlen;
    *len = csize - 12 - xlen - 8;
    return true;
}

// serial sink: the host test hook
struct HostSink {
    uint8_t* out;
    uint32_t cap, pos;
    bool leader() const { return true; }
    void sync() const {}
    bool lit(uint8_t b) { if (pos >= cap) return false; out[pos++] = b; return true; }
    bool match(uint32_t len, uint32_t dist) {
        if (len > cap - pos) return false;
        for (uint32_t k = 0; k < len; ++k, ++pos) out[pos] = out[pos - dist];
        return true;
    }
    bool stored(const uint8_t* src, uint32_t len) {
        if (len > cap - pos) return false;
        for (uint32_t k = 0; k < len; ++k) out[pos++] = src[k];
        return true;
    }
};

#if defined(__CUDACC__)
// ================================================================== device half
// A block of a device fetch (copied from c3r_bgzf_block) and the window geometry the kernels use.
struct DevWindow {
    int64_t ubase, usize, ubeg, uend;
    int64_t slot_base;                 // first record slot of the window; capacity usize / 36 + 1
    int32_t status;                    // FetchErr found by the host while reading the window, 0 = none
    int32_t n_blocks;
};

// Per-ticket scalars of a device fetch (zeroed / set to all ones before the kernels)
struct FetchSc {
    unsigned long long err_key;        // first error (order_key), ~0 = none
    unsigned long long stop_key;       // first record that ends the fetch, ~0 = none
    long long n_reads, n_ops, n_bases; // totals of the records kept (n_bases even-padded per read)
};

struct Slot3 { long long r, o, b; };

struct Fetch {
    int32_t tid;
    int64_t beg, end;
    int32_t n_win;
    int64_t n_slots;                   // slot capacity of all windows
    const uint8_t* cdata;              // compressed bytes
    const int64_t* blk_coff; const int64_t* blk_uoff;
    const int32_t* blk_csize; const int32_t* blk_usize; const int32_t* blk_win;
    const DevWindow* win;
    uint8_t* ubuf;                     // inflated windows, back to back
    int32_t* n_rec;                    // [n_win] records found in each window
    int64_t* slot_off;                 // [n_slots] record offset in its window
    uint8_t* slot_cls;                 // [n_slots] RecClass, 0 = empty slot
    uint64_t* slot_key;                // [n_slots] order_key of the record
    int32_t* slot_nops;                // [n_slots]
    int64_t* slot_nb;                  // [n_slots] even-padded bases
    Slot3* slot_dst;                   // [n_slots] output read / op / base offsets of a kept record
    FetchSc* sc;
    // outputs (the slot's read buffers)
    int32_t* pos; uint16_t* flag; uint8_t* mapq; uint8_t* hp; int32_t* cigar_off; uint32_t* cigar;
    int64_t* seq_off; uint8_t* seq;
};

// warp sink over the block's shared-memory staging buffer: every lane runs the decoder (same bits, same branches);
// lane 0 writes literals and the tables, the warp copies matches and stored runs
struct WarpSink {
    uint8_t* out;
    uint32_t cap, pos;
    __device__ bool leader() const { return (threadIdx.x & 31) == 0; }
    __device__ void sync() const { __syncwarp(); }
    __device__ bool lit(uint8_t b) {
        if (pos >= cap) return false;
        if (leader()) out[pos] = b;
        ++pos;
        return true;
    }
    __device__ bool match(uint32_t len, uint32_t dist) {
        if (len > cap - pos) return false;
        __syncwarp();                                  // literals of lane 0 are visible
        // byte k of the copy is byte (k mod dist) of the dist bytes before it: every source byte precedes `pos`
        for (uint32_t k = threadIdx.x & 31; k < len; k += 32) out[pos + k] = out[pos - dist + (k < dist ? k : k % dist)];
        __syncwarp();
        pos += len;
        return true;
    }
    __device__ bool stored(const uint8_t* src, uint32_t len) {
        if (len > cap - pos) return false;
        for (uint32_t k = threadIdx.x & 31; k < len; k += 32) out[pos + k] = src[k];
        __syncwarp();
        pos += len;
        return true;
    }
};

constexpr int INFLATE_SMEM = (int)MAX_BLOCK + 256 * 4 + (int)sizeof(Tables) + 16;

__device__ __forceinline__ void fetch_error(FetchSc* sc, uint64_t key) { atomicMin(&sc->err_key, (unsigned long long)key); }

// one BGZF block per CTA of 32 threads
__global__ void __launch_bounds__(32) k_inflate(const Fetch f) {
    extern __shared__ __align__(16) uint8_t sm[];
    uint32_t* crc_tab = (uint32_t*)sm;
    Tables& t = *(Tables*)(sm + 1024);
    uint8_t* out = sm + 1024 + ((sizeof(Tables) + 15) / 16) * 16;
    const int lane = threadIdx.x;
    const int64_t b = blockIdx.x;
    const uint32_t usize = (uint32_t)f.blk_usize[b], csize = (uint32_t)f.blk_csize[b];
    const int w = f.blk_win[b];
    if (usize == 0) return;                             // empty blocks are not inflated (as the host fetch)
    const uint8_t* src = f.cdata + f.blk_coff[b];
    for (int k = lane; k < 256; k += 32) crc_tab[k] = crc_table_entry((uint32_t)k);
    uint32_t off, len;
    int rc = IE_HEADER;
    WarpSink sink;
    sink.out = out; sink.cap = usize; sink.pos = 0;
    if (usize <= MAX_BLOCK && bgzf_payload(src, csize, &off, &len)) rc = inflate_core(src + off, len, sink, t);
    if (rc == IE_OK && sink.pos != usize) rc = IE_ISIZE;
    __syncwarp();
    if (rc == IE_OK) {
        const uint32_t seg = (usize + 31) / 32;
        const uint32_t a = lane * seg < usize ? lane * seg : usize;
        const uint32_t e = a + seg < usize ? a + seg : usize;
        uint32_t c = crc32_bytes(crc_tab, out + a, e - a);
        uint32_t acc = 0;
        for (int k = 0; k < 32; ++k) {
            const uint32_t ck = __shfl_sync(0xffffffffu, c, k), lk = __shfl_sync(0xffffffffu, e - a, k);
            if (lane == 0 && lk) acc = crc32_combine(acc, ck, lk);
        }
        acc = __shfl_sync(0xffffffffu, acc, 0);
        if (acc != c3rbam::rd32(src + csize - 8)) rc = IE_CRC;
    }
    if (rc != IE_OK) {
        if (lane == 0) fetch_error(f.sc, order_key((uint32_t)w, 0, 0, FE_INFLATE));
        return;
    }
    uint8_t* dst = f.ubuf + f.blk_uoff[b];
    for (uint32_t k = lane; k < usize; k += 32) dst[k] = out[k];
}

constexpr int BOUNDS_THREADS = 256;
constexpr int BOUNDS_TILE = 32768;

// one CTA per window: the length chain of its records, through tiles of the window staged in shared memory
__global__ void __launch_bounds__(BOUNDS_THREADS) k_rec_bounds(const Fetch f) {
    __shared__ __align__(16) uint8_t tile[BOUNDS_TILE];
    __shared__ long long s_o;
    __shared__ int s_n, s_done;
    const int w = blockIdx.x;
    const DevWindow W = f.win[w];
    if (W.status) {
        if (threadIdx.x == 0) { fetch_error(f.sc, order_key((uint32_t)w, 0, 0, (uint32_t)W.status)); f.n_rec[w] = 0; }
        return;
    }
    const uint8_t* u = f.ubuf + W.ubase;
    const int64_t cap = W.usize / 36 + 1;
    if (threadIdx.x == 0) { s_o = W.ubeg; s_n = 0; s_done = W.n_blocks == 0; }
    __syncthreads();
    while (!s_done) {
        const int64_t base = s_o;
        const int64_t lim = W.usize - base < BOUNDS_TILE ? W.usize - base : BOUNDS_TILE;
        for (int64_t k = threadIdx.x; k < lim; k += BOUNDS_THREADS) tile[k] = u[base + k];
        __syncthreads();
        if (threadIdx.x == 0) {
            int64_t o = base;
            int n = s_n;
            bool done = false;
            for (;;) {
                if (o + 4 > W.uend) { done = true; break; }
                if (o + 4 > base + lim) break;                 // the length field is in the next tile
                const uint32_t bs = c3rbam::rd32(tile + (o - base));
                if ((uint64_t)o + 4 + bs > (uint64_t)W.usize) {
                    fetch_error(f.sc, order_key((uint32_t)w, 1, (uint64_t)o, FE_CROSS));
                    done = true;
                    break;
                }
                if (n >= cap) { done = true; break; }          // cannot happen: records of >= 36 bytes but the last
                f.slot_off[W.slot_base + n] = o;
                ++n;
                o += 4 + (int64_t)bs;
                if (bs < 32) { done = true; break; }           // malformed (k_rec_parse reports it): the chain ends
            }
            s_o = o;
            s_n = n;
            s_done = done || o == base;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) f.n_rec[w] = s_n;
}

__device__ __forceinline__ int window_of(const Fetch& f, int64_t slot) {
    int lo = 0, hi = f.n_win - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (f.win[mid].slot_base <= slot) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// one thread per record slot
__global__ void __launch_bounds__(256) k_rec_parse(const Fetch f) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < f.n_slots; i += (int64_t)gridDim.x * blockDim.x) {
        const int w = window_of(f, i);
        const DevWindow& W = f.win[w];
        uint8_t cls = 0;
        int32_t nops = 0;
        int64_t nb = 0;
        uint64_t key = ~0ull;
        if (i - W.slot_base < f.n_rec[w]) {
            const int64_t o = f.slot_off[i];
            const uint8_t* p = f.ubuf + W.ubase + o;
            c3rbam::RecInfo x;
            cls = (uint8_t)c3rbam::classify_record(p + 4, c3rbam::rd32(p), f.tid, f.beg, f.end, x);
            key = order_key((uint32_t)w, 1, (uint64_t)o, 0);
            if (cls == c3rbam::REC_STOP) atomicMin(&f.sc->stop_key, (unsigned long long)key);
            else if (cls == c3rbam::REC_ERR_MALFORMED) fetch_error(f.sc, key | FE_MALFORMED);
            else if (cls == c3rbam::REC_ERR_AUX) fetch_error(f.sc, key | FE_AUX);
            else if (cls == c3rbam::REC_KEEP) { nops = (int32_t)x.n_cig; nb = (x.n_bases + 1) & ~1LL; }
        }
        f.slot_cls[i] = cls;
        f.slot_key[i] = key;
        f.slot_nops[i] = nops;
        f.slot_nb[i] = nb;
    }
}

// scan.cuh operator: output offsets of the records kept (before the first stop)
struct OpKeep {
    typedef Slot3 T;
    Fetch f;
    struct Ctx {};
    __device__ void ctx_init(Ctx&) const {}
    __device__ T identity() const { T t; t.r = 0; t.o = 0; t.b = 0; return t; }
    __device__ T combine(const T& a, const T& b) const { T t; t.r = a.r + b.r; t.o = a.o + b.o; t.b = a.b + b.b; return t; }
    __device__ T load(int64_t i) const {
        T t = identity();
        if (f.slot_cls[i] == c3rbam::REC_KEEP && f.slot_key[i] < f.sc->stop_key) { t.r = 1; t.o = f.slot_nops[i]; t.b = f.slot_nb[i]; }
        return t;
    }
    __device__ void store(int64_t i, const T& inc, const T& own, Ctx&) const {
        if (own.r) { T d; d.r = inc.r - own.r; d.o = inc.o - own.o; d.b = inc.b - own.b; f.slot_dst[i] = d; }
    }
    __device__ int64_t size() const { return f.n_slots; }
};

// one warp per record slot: the kept records into the read buffers (cigar_off[0] / seq_off[0] are zeroed before)
__global__ void __launch_bounds__(256) k_rec_write(const Fetch f) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t i = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); i < f.n_slots; i += warps) {
        if (f.slot_cls[i] != c3rbam::REC_KEEP || f.slot_key[i] >= f.sc->stop_key) continue;
        const int w = window_of(f, i);
        const uint8_t* p = f.ubuf + f.win[w].ubase + f.slot_off[i];
        c3rbam::RecInfo x;
        c3rbam::classify_record(p + 4, c3rbam::rd32(p), f.tid, f.beg, f.end, x);
        const Slot3 d = f.slot_dst[i];
        const int64_t nb = (x.n_bases + 1) & ~1LL;
        if (lane == 0) {
            f.pos[d.r] = x.r.pos;
            f.flag[d.r] = x.r.flag;
            f.mapq[d.r] = x.r.mapq;
            f.hp[d.r] = c3rbam::clamp_hp(x.hp);
            f.cigar_off[d.r + 1] = (int32_t)(d.o + x.n_cig);
            f.seq_off[d.r + 1] = d.b + nb;
        }
        for (uint32_t k = lane; k < x.n_cig; k += 32) f.cigar[d.o + k] = c3rbam::rd32(x.cig + 4 * k);
        uint8_t* s = f.seq + d.b / 2;
        const int64_t nbytes = (x.n_bases + 1) / 2;
        const bool odd = x.n_bases & 1;
        if (x.r.l_seq > 0) {
            for (int64_t k = lane; k < nbytes; k += 32) s[k] = (odd && k == nbytes - 1) ? (x.r.seq[k] & 0xf0) : x.r.seq[k];
        } else {
            for (int64_t k = lane; k < nbytes; k += 32) s[k] = (odd && k == nbytes - 1) ? 0xf0 : 0xff;
        }
    }
}
#endif  // __CUDACC__

}  // namespace c3rbgzf
