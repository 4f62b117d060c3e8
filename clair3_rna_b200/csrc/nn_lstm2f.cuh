// LSTM2 with its input projection fused into the recurrent step ("fused LSTM2").
//
// The projection never leaves the SM: every step's accumulator is
//   z_t = h1_t . W2_hi + h1_t . W2_lo + h2_{t-1} . U2 + [1 1 0..] . [b_hi ; b_lo ; 0..]  (K = 688) in TMEM,
// issued as tcgen05 cta_group::2 MMAs (M = 256 sites, N = 128 gate columns per chunk) by the pair's leader.
// W2 (hi + lo fp16 terms) and U2 do not fit next to the operands in 227 KB, so the weights are not resident: they
// stream from L2 through a ring of 16 KB stages in exactly the order the MMAs consume them - the same 430 KB
// sequence every step - and NP CTA pairs of one cluster (2*NP CTAs, all working on the same direction) share one
// copy of the stream by bulk-copy multicast: stage `it` is fetched by pair it % NP and lands in all NP pairs.
// A ring slot is handed back by tcgen05.commit multicast to every CTA of the cluster (one arrival per pair).
// The h1_t tile (x operand, 64 KB per CTA) sits in four 64-wide k blocks, each re-loaded for step t+1 as soon as
// the last chunk of step t has consumed it.
//
//   K order of a chunk: [x kb0 . W2_hi] [x kb0 . W2_lo] [kb1 ..] [kb2 ..] [kb3 ..] [h . U2 (160)] [ones . bias (16)]
//   = 6 stages (5 x 16 KB + 6 KB), 43 MMAs of K = 16; 5 chunks (32 units x 4 gates) per step.
// One thread issues every MMA of a pair, so its instruction path sets the pace: stages are large (8 MMAs per
// barrier round), the barrier tests of the next stage are issued before the current stage's MMAs, and the thread is
// chosen by elect.sync (straight-line UTCHMMA, ~40 cycles each).
//
// The projection part of a chunk has no dependency on h_{t-1}, so it is issued while the gate warps still work on
// the previous chunk, in the tensor pipe's idle time of the recurrence.
// This kernel replaced a hoisted form (k_gemm_zx + k_lstm_tc<5,0>) that wrote the projection zx2 = h1 . W2 + b to HBM
// (127 KB per site) and read it back - 4.5 of the 5.4 GB a pass moved - while its recurrence left the tensor pipe
// idle 83 % of the time.
// Math restated from /root/reference/clair3_rna/model.py:132-136,181 (Bidirectional LSTM, 160 units, Keras gate
// order i,f,c,o); gate stage identical to k_lstm_tc.
#pragma once
// (included from the middle of nn_tc.cuh: uses its tile constants, PTX wrappers and gate math)

namespace c3r {

namespace ptx {
// global -> shared bulk copy delivered to the same CTA-relative offset (data and mbarrier) of every CTA in `mask`
__device__ __forceinline__ void bulk_g2s_mcast(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint16_t mask) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;"
        ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "h"(mask) : "memory");
}
}  // namespace ptx

constexpr int L2F_CH = 5;                         // chunks per step
constexpr int L2F_IMG = 8192;                     // one [64 columns x 64 k] weight image
constexpr int L2F_STAGES = 6;                     // weight stages per chunk: 4 x (W2_hi | W2_lo of a k block), U2 rows 0..127, the rest
constexpr int L2F_SLOT = 2 * L2F_IMG;             // ring slot = one stage = two images
constexpr int L2F_LAST = 64 * 48 * 2;             // the last stage of a chunk: U2 rows 128..159 + the bias block
constexpr int L2F_CHUNK_BYTES = 10 * L2F_IMG + L2F_LAST;
constexpr int L2F_STREAM_BYTES = L2F_CH * L2F_CHUNK_BYTES;     // per (direction, pair half): 440 320 B
constexpr int L2F_NS = 4;                         // ring slots
constexpr int L2F_GATE_WARPS = 16;
constexpr int L2F_THREADS = 128 + 32 * L2F_GATE_WARPS;   // warp 0 MMA / acc relay, 1 x loader, 2 weight ring, 3 landed relay
constexpr int L2F_AH = TC_TILE * U2 * 2;          // one h buffer: 40 KB
constexpr int L2F_XB = TC_IMG * 2;                // one x k block: 16 KB
constexpr int L2F_OFF_X = 2 * L2F_AH;
constexpr int L2F_OFF_ONE = L2F_OFF_X + 4 * L2F_XB;
constexpr int L2F_OFF_W = L2F_OFF_ONE + TC_TILE * 16 * 2;
constexpr int L2F_OFF_BAR = L2F_OFF_W + L2F_NS * L2F_SLOT;
constexpr int L2F_SMEM = L2F_OFF_BAR + 1024;
static_assert(L2F_SMEM <= 232448, "fused LSTM2 shared memory");

struct Lstm2fArgs {
    const uint8_t* wstream;   // [2 dirs][2 halves][L2F_STREAM_BYTES]
    const __half* h1;         // [tile][33][4][TC_IMG] (LSTM1 output, high-order fp16 term)
    __half* hout;             // [tile][33][5][TC_IMG]
    __half* hout_lo;          // low-order term or nullptr
    int n_tiles;              // 128-site tiles (even)
    int* err;
    long long* prof;          // optional [32]: SM-clock totals of cluster 0's waits (C3R_L2F_PROF), see tools/lstm2f_probe.py
};

// wait + account the cycles spent to prof slot k (PROF instantiation only)
#define L2F_WAIT(bar, par, code, k) do { if (PROF && pf) { const long long t0__ = clock64(); ptx::mbar_wait(bar, par, a.err, code); pw[k] += clock64() - t0__; } else ptx::mbar_wait(bar, par, a.err, code); } while (0)

template <int NP, bool PROF>
__global__ void __launch_bounds__(L2F_THREADS, 1) k_lstm2_fused(Lstm2fArgs a) {
    constexpr int CH = L2F_CH;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t s_base = ptx::smem_u32(smem);
    const uint32_t s_AH = s_base, s_X = s_base + L2F_OFF_X, s_ONE = s_base + L2F_OFF_ONE, s_W = s_base + L2F_OFF_W;
    uint64_t* bars = (uint64_t*)(smem + L2F_OFF_BAR);
    const uint32_t b0 = ptx::smem_u32(bars);
    // Barriers (8 bytes each).  Where the leader needs "done in both CTAs of the pair" its barrier simply counts one
    // more arrival: the peer's relay thread, which waits for the peer's own barrier and arrives remotely (relaxed: the
    // data moved through the async proxy / TMEM and was ordered by its producers), so the issuing thread tests ONE
    // barrier per event.
    const uint32_t b_wf = b0;                         // [NS] weight stage landed (bulk copy tx) [+ relay on the leader]
    const uint32_t b_we = b_wf + 8 * L2F_NS;          // [NS] stage consumed by every pair of the cluster (NP commits)
    const uint32_t b_xf = b_we + 8 * L2F_NS;          // [4] x block landed [+ relay on the leader]
    const uint32_t b_xfree = b_xf + 32;               // [4] x block consumed by the step's last chunk (commit)
    const uint32_t b_accf = b_xfree + 32;             // [2] accumulator slot complete (commit)
    const uint32_t b_acce = b_accf + 16;              // [2] slot drained by this CTA's gate warps [+ relay on the leader]
    const uint32_t b_hrdy = b_acce + 16;              // h_t complete in this CTA [+ relay on the leader]
    uint32_t* tmem_ptr_s = (uint32_t*)(bars + 2 * L2F_NS + 8 + 4 + 1 + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = ptx::cluster_ctarank();
    const uint32_t pr = rank >> 1, hr = rank & 1, leader = rank & ~1u;
    constexpr int CSIZE = 2 * NP;
    const int cluster_id = blockIdx.x / CSIZE;
    const int dir = cluster_id & 1;
    const int J = (int)(gridDim.x / CSIZE / 2) * NP;  // pairs working on this direction
    const int j = (cluster_id >> 1) * NP + (int)pr;
    const int n_tile_pairs = a.n_tiles / 2;
    const int n_rounds = (n_tile_pairs + J - 1) / J;
    const uint16_t mask_all = (uint16_t)((1u << CSIZE) - 1);
    const uint16_t mask_pair = (uint16_t)(3u << (2 * pr));
    uint16_t mask_half = 0;                           // the CTAs that hold the same half of the gate columns
#pragma unroll
    for (int q = 0; q < NP; ++q) mask_half |= (uint16_t)(1u << (2 * q + hr));

    if (threadIdx.x == 0) {
        const uint32_t relay = hr == 0 ? 1u : 0u;     // the leader's barriers also count the peer's relay
        for (int i = 0; i < L2F_NS; ++i) { ptx::mbar_init(b_wf + 8 * i, 1 + relay); ptx::mbar_init(b_we + 8 * i, NP); }
        for (int i = 0; i < 4; ++i) { ptx::mbar_init(b_xf + 8 * i, 1 + relay); ptx::mbar_init(b_xfree + 8 * i, 1); }
        for (int i = 0; i < 2; ++i) { ptx::mbar_init(b_accf + 8 * i, 1); ptx::mbar_init(b_acce + 8 * i, L2F_GATE_WARPS + relay); }
        ptx::mbar_init(b_hrdy, L2F_GATE_WARPS + relay);
        ptx::fence_barrier_init();
    }
    // the constant A tile that meets the bias rows: k = 0, 1 are one, the other 14 k zero
    for (int i = threadIdx.x; i < TC_TILE * 16 / 2; i += blockDim.x) {
        const int cell = i / (TC_TILE * 4), w = i % 4;             // 32-bit words: [2 k8 cells][128 rows][4 words]
        ((uint32_t*)(smem + L2F_OFF_ONE))[i] = (cell == 0 && w == 0) ? 0x3c003c00u : 0u;
    }
    ptx::fence_proxy_async();
    if (warp == 0) {
        ptx::tmem_alloc<2>(ptx::smem_u32(tmem_ptr_s), 512);
        ptx::tmem_relinquish<2>();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync();
    ptx::tc_fence_after();
    const uint32_t tmem = *tmem_ptr_s;
    constexpr uint32_t IDESC = ptx::make_idesc_f16(256, 128);
    constexpr uint32_t C_COL = 256;
    const uint32_t n_steps = (uint32_t)n_rounds * NT;
    const bool pf = PROF && a.prof != nullptr && blockIdx.x == 0;

    if (warp == 0) {
        if (hr == 0) {
            // ---------------------------------------------------- MMA issue (pair leader): one thread chosen by elect.sync -
            // under that predicate ptxas emits straight-line UTCHMMA with uniform-register descriptors (a `lane == 0`
            // test or a converged warp with a per-lane predicate gets an ELECT / R2UR loop around every MMA: ~100 cycles each)
            if (ptx::elect_one()) {
                uint32_t wslot = 0, wph = 0, use = 0;
                long long pw[6] = {0, 0, 0, 0, 0, 0};
                const long long t_begin = PROF ? clock64() : 0;
                constexpr uint64_t KA = (2 * TC_TILE * 16) >> 4, KB = (2 * 64 * 16) >> 4;   // one k16 step in descriptor units
                const uint64_t dW = ptx::make_smem_desc(s_W, 64 * 16, 128);
                const uint64_t dX = ptx::make_smem_desc(s_X, TC_TILE * 16, 128);
                const uint64_t dH = ptx::make_smem_desc(s_AH, TC_TILE * 16, 128);
                const uint64_t d1 = ptx::make_smem_desc(s_ONE, TC_TILE * 16, 128);
                bool w_ok = false;                                  // result of the barrier test issued one stage ahead
                bool a_ok = false;                                  // the same for the next chunk's accumulator slot
                for (uint32_t g = 0; g < n_steps; ++g) {
                    const int step = (int)(g % NT);
                    const uint64_t dHb = dH + (uint64_t)((g & 1) * (L2F_AH >> 4));
#pragma unroll 1
                    for (int c = 0; c < CH; ++c, ++use) {
                        const uint32_t slot = use & 1, aph = (use >> 1) & 1;
                        if (!a_ok) L2F_WAIT(b_acce + 8 * slot, aph ^ 1, 303, 0);
                        ptx::tc_fence_after();
                        const uint32_t dacc = tmem + slot * 128;
#pragma unroll
                        for (int s = 0; s < L2F_STAGES; ++s) {
                            const bool tr = PROF && pf && g == 3;
                            long long* trp = a.prof + 16 + (c * L2F_STAGES + s) * 4;
                            if (tr) trp[0] = clock64();
                            if (c == 0 && s < 4) L2F_WAIT(b_xf + 8 * s, g & 1, 302, 2);                  // first use of this step's x block
                            if (s == 4 && c == 0 && step > 0) L2F_WAIT(b_hrdy, (g - 1) & 1, 304, 3);     // h_{t-1} complete in both CTAs
                            if (!w_ok) L2F_WAIT(b_wf + 8 * wslot, wph, 305, 4);
                            ptx::tc_fence_after();
                            // the next stage's barrier is tested now: the answer comes back under this stage's MMAs
                            const uint32_t nslot = wslot + 1 == L2F_NS ? 0 : wslot + 1, nph = wslot + 1 == L2F_NS ? wph ^ 1 : wph;
                            w_ok = ptx::mbar_try_wait(b_wf + 8 * nslot, nph);
                            if (s == L2F_STAGES - 1) a_ok = ptx::mbar_try_wait(b_acce + 8 * (slot ^ 1), (((use + 1) >> 1) & 1) ^ 1);
                            if (tr) trp[1] = clock64();
                            const uint64_t dB0 = dW + (uint64_t)(wslot * (L2F_SLOT >> 4));
                            if (s < 4) {
                                const uint64_t dA0 = dX + (uint64_t)(s * (L2F_XB >> 4));
#pragma unroll
                                for (int k = 0; k < 8; ++k)          // k16 steps 0..3 meet W2_hi, the same x again meets W2_lo
                                    ptx::mma_f16<2>(dacc, dA0 + (uint64_t)(k & 3) * KA, dB0 + (uint64_t)k * KB, IDESC, (s | k) ? 1u : 0u);
                            } else if (s == 4) {
                                if (step > 0) {
#pragma unroll
                                    for (int k = 0; k < 8; ++k) ptx::mma_f16<2>(dacc, dHb + (uint64_t)k * KA, dB0 + (uint64_t)k * KB, IDESC, 1u);
                                }
                            } else {
                                if (step > 0) {
#pragma unroll
                                    for (int k = 0; k < 2; ++k) ptx::mma_f16<2>(dacc, dHb + (uint64_t)(8 + k) * KA, dB0 + (uint64_t)k * KB, IDESC, 1u);
                                }
                                ptx::mma_f16<2>(dacc, d1, dB0 + 2 * KB, IDESC, 1u);
                            }
                            if (tr) trp[2] = clock64();
                            ptx::mma_commit_2_mcast(b_we + 8 * wslot, mask_all);
                            if (c == CH - 1 && s < 4) ptx::mma_commit_2_mcast(b_xfree + 8 * s, mask_pair);
                            if (tr) trp[3] = clock64();
                            wslot = nslot; wph = nph;
                        }
                        ptx::mma_commit_2_mcast(b_accf + 8 * slot, mask_pair);
                    }
                }
                if (PROF && pf) {
                    for (int k = 0; k < 6; ++k) a.prof[k] = pw[k];
                    a.prof[6] = clock64() - t_begin;
                    a.prof[7] = n_steps;
                }
            }
            __syncwarp();
        } else if (lane == 0) {
            // ---------------------------------------------------- peer: relay "slot drained" / "h complete" to the leader
            uint32_t use = 0;
            for (uint32_t g = 0; g < n_steps; ++g) {
                for (int c = 0; c < CH; ++c, ++use) {
                    const uint32_t slot = use & 1;
                    ptx::mbar_wait(b_acce + 8 * slot, (use >> 1) & 1, a.err, 320);
                    ptx::mbar_arrive_cluster_relaxed(b_acce + 8 * slot, leader);
                }
                ptx::mbar_wait(b_hrdy, g & 1, a.err, 321);
                ptx::mbar_arrive_cluster_relaxed(b_hrdy, leader);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // ---------------------------------------------------- x loader: this CTA's 128 rows of h1_t, four k blocks
            for (uint32_t g = 0; g < n_steps; ++g) {
                const int r = (int)(g / NT), step = (int)(g % NT);
                int tp = j + r * J;
                if (tp >= n_tile_pairs) tp = n_tile_pairs - 1;      // idle pair: keeps the protocol, stores nothing
                const int tile = tp * 2 + (int)hr;
                const int t = dir == 0 ? step : NT - 1 - step;
                const __half* src = a.h1 + ((size_t)tile * NT + t) * 4 * TC_IMG;
                for (int kb = 0; kb < 4; ++kb) {
                    ptx::mbar_wait(b_xfree + 8 * kb, (g & 1) ^ 1, a.err, 330);
                    ptx::mbar_arrive_expect_tx(b_xf + 8 * kb, L2F_XB);
                    ptx::bulk_g2s(s_X + kb * L2F_XB, src + (size_t)kb * TC_IMG, L2F_XB, b_xf + 8 * kb);
                }
            }
            if (n_steps > 0)
                for (int kb = 0; kb < 4; ++kb) ptx::mbar_wait(b_xfree + 8 * kb, (n_steps - 1) & 1, a.err, 331);
        }
    } else if (warp == 2) {
        if (lane == 0) {
            // ---------------------------------------------------- weight ring: every CTA arms its slot, pair it % NP fetches
            const uint8_t* wsrc = a.wstream + ((size_t)dir * 2 + hr) * L2F_STREAM_BYTES;
            uint32_t wslot = 0, wph = 0, it = 0;
            long long pw[1] = {0};
            for (uint32_t g = 0; g < n_steps; ++g) {
                uint32_t off = 0;
                for (int cs = 0; cs < CH * L2F_STAGES; ++cs, ++it) {
                    const uint32_t bytes = (cs % L2F_STAGES) == L2F_STAGES - 1 ? L2F_LAST : L2F_SLOT;
                    L2F_WAIT(b_we + 8 * wslot, wph ^ 1, 340, 0);
                    ptx::mbar_arrive_expect_tx(b_wf + 8 * wslot, bytes);
                    if (NP == 1) ptx::bulk_g2s(s_W + wslot * L2F_SLOT, wsrc + off, bytes, b_wf + 8 * wslot);
                    else if (it % NP == pr) ptx::bulk_g2s_mcast(s_W + wslot * L2F_SLOT, wsrc + off, bytes, b_wf + 8 * wslot, mask_half);
                    off += bytes;
                    if (++wslot == L2F_NS) { wslot = 0; wph ^= 1; }
                }
            }
            if (PROF && pf) a.prof[8] = pw[0];
            // commits still on their way to this CTA must land before it exits
            const uint32_t total = n_steps * CH * L2F_STAGES;
            for (uint32_t k = total > (uint32_t)L2F_NS ? total - L2F_NS : 0; k < total; ++k)
                ptx::mbar_wait(b_we + 8 * (k % L2F_NS), (k / L2F_NS) & 1, a.err, 341);
        }
    } else if (warp == 3) {
        if (lane == 0 && hr == 1) {
            // ---------------------------------------------------- peer: relay "landed" (x blocks, weight stages) in consumption order
            uint32_t wslot = 0, wph = 0;
            for (uint32_t g = 0; g < n_steps; ++g)
                for (int c = 0; c < CH; ++c)
                    for (int s = 0; s < L2F_STAGES; ++s) {
                        if (c == 0 && s < 4) {
                            ptx::mbar_wait(b_xf + 8 * s, g & 1, a.err, 350);
                            ptx::mbar_arrive_cluster_relaxed(b_xf + 8 * s, leader);
                        }
                        ptx::mbar_wait(b_wf + 8 * wslot, wph, a.err, 351);
                        ptx::mbar_arrive_cluster_relaxed(b_wf + 8 * wslot, leader);
                        if (++wslot == L2F_NS) { wslot = 0; wph ^= 1; }
                    }
        }
    } else {
        // -------------------------------------------------------- gates: TMEM -> c, h (as k_lstm_tc)
        const int gw = warp - 4;
        const int q = warp & 3;                          // TMEM lane quarter this warp may access
        const int sub = gw >> 2;                         // which 8 units of the chunk's 32
        const int row = q * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        uint32_t use = 0;
        const bool pfg = pf && gw == 0;
        long long pw[1] = {0};
        for (uint32_t g = 0; g < n_steps; ++g) {
            const int r = (int)(g / NT), step = (int)(g % NT);
            const int tp = j + r * J;
            const bool valid = tp < n_tile_pairs;
            const int tile = (valid ? tp : n_tile_pairs - 1) * 2 + (int)hr;
            const uint32_t nbuf = (g + 1) & 1;           // h_t goes to the buffer step+1 reads
            const int t = dir == 0 ? step : NT - 1 - step;
            uint8_t* ah = smem + nbuf * L2F_AH;
            __half* hout_t = a.hout + ((size_t)tile * NT + t) * 5 * TC_IMG;
            __half* hout_lo_t = a.hout_lo + ((size_t)tile * NT + t) * 5 * TC_IMG;
#pragma unroll
            for (int c = 0; c < CH; ++c, ++use) {
                const uint32_t slot = use & 1;
                if (PROF && pfg) { const long long t0 = clock64(); ptx::mbar_wait(b_accf + 8 * slot, (use >> 1) & 1, a.err, 308); pw[0] += clock64() - t0; }
                else ptx::mbar_wait(b_accf + 8 * slot, (use >> 1) & 1, a.err, 308);
                ptx::tc_fence_after();
                uint32_t cprev[8];
                uint32_t v[4][8];
#pragma unroll
                for (int gte = 0; gte < 4; ++gte) ptx::tmem_ld8(tmem + lane_addr + slot * 128 + gte * 32 + sub * 8, v[gte]);
                if (step > 0) ptx::tmem_ld8(tmem + lane_addr + C_COL + c * 32 + sub * 8, cprev);
                ptx::tmem_wait_ld();
                ptx::tc_fence_before();                  // the accumulator slot is in registers: hand it back
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(b_acce + 8 * slot);
                uint32_t cnew[8];
                __align__(16) __half hh[8];
                __align__(16) __half hl[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const float zi = __uint_as_float(v[0][u]), zf = __uint_as_float(v[1][u]);
                    const float zg = __uint_as_float(v[2][u]), zo = __uint_as_float(v[3][u]);
                    const float cp = step > 0 ? __uint_as_float(cprev[u]) : 0.0f;
                    float cn, hv;
                    lstm_cell(zi, zf, zg, zo, cp, cn, hv);
                    cnew[u] = __float_as_uint(cn);
                    hh[u] = __float2half(hv);
                    hl[u] = __float2half(hv - __half2float(hh[u]));
                }
                ptx::tmem_st8(tmem + lane_addr + C_COL + c * 32 + sub * 8, cnew);
                const uint4 pk = *(const uint4*)hh;
                const int k8 = c * 4 + sub;
                *(uint4*)(ah + (size_t)k8 * (TC_TILE * 16) + row * 16) = pk;
                ptx::tmem_wait_st();
                if (c == CH - 1) {                       // this warp's part of h_t is in shared memory
                    ptx::tc_fence_before();
                    ptx::fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive(b_hrdy);
                }
                if (valid) {
                    const int col8 = (dir * U2) / 8 + k8;            // 8-column group in the concat [fwd | bwd]
                    const size_t oo = (size_t)(col8 / 8) * TC_IMG + (size_t)(col8 % 8) * (TC_TILE * 8) + row * 8;
                    *(uint4*)(hout_t + oo) = pk;
                    if (a.hout_lo) *(uint4*)(hout_lo_t + oo) = *(const uint4*)hl;
                }
            }
        }
        if (PROF && pfg && lane == 0) a.prof[9] = pw[0];
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync();
    if (warp == 0) ptx::tmem_dealloc<2>(tmem, 512);
}

// weight stream of one (direction, pair half): for each chunk the 11 stages in K order, every stage a
// [64 columns x K_s] K-major core-matrix image.  Column j of half hr in chunk c is gate (hr*64+j)/32, unit
// c*32 + (hr*64+j)%32; i, f, o columns carry 0.5 * z like every other packed LSTM weight.
inline void lstm2f_pack(std::vector<uint8_t>& out, const float* h, size_t o_w2, size_t o_b2, size_t o_u2) {
    out.assign((size_t)4 * L2F_STREAM_BYTES, 0);
    auto split = [](float w, __half& hi, __half& lo) {
        hi = __float2half(w);
        lo = __float2half(w - __half2float(hi));
    };
    for (int dir = 0; dir < 2; ++dir)
        for (int hr = 0; hr < 2; ++hr) {
            __half* base = (__half*)(out.data() + ((size_t)dir * 2 + hr) * L2F_STREAM_BYTES);
            for (int c = 0; c < L2F_CH; ++c) {
                __half* ch = base + (size_t)c * (L2F_CHUNK_BYTES / 2);
                for (int jj = 0; jj < 64; ++jj) {
                    const int col = hr * 64 + jj, gate = col / 32, ul = col % 32;
                    const int kc = gate * U2 + c * 32 + ul;
                    const float gs = gate == 2 ? 1.0f : 0.5f;
                    for (int kb = 0; kb < 4; ++kb)
                        for (int k = 0; k < 64; ++k) {
                            __half hi, lo;
                            split(gs * h[o_w2 + (size_t)(kb * 64 + k) * 2 * G2 + dir * G2 + kc], hi, lo);
                            ch[(size_t)(2 * kb) * (L2F_IMG / 2) + ((size_t)(k / 8) * 64 * 8 + (size_t)jj * 8 + k % 8)] = hi;
                            ch[(size_t)(2 * kb + 1) * (L2F_IMG / 2) + ((size_t)(k / 8) * 64 * 8 + (size_t)jj * 8 + k % 8)] = lo;
                        }
                    for (int k = 0; k < U2; ++k) {
                        const int s = 8 + k / 64, kk = k % 64;
                        ch[(size_t)s * (L2F_IMG / 2) + ((size_t)(kk / 8) * 64 * 8 + (size_t)jj * 8 + kk % 8)] =
                            __float2half(gs * h[o_u2 + (size_t)dir * U2 * G2 + (size_t)k * G2 + kc]);
                    }
                    __half bh, bl;
                    split(gs * h[o_b2 + dir * G2 + kc], bh, bl);
                    __half* st10 = ch + (size_t)10 * (L2F_IMG / 2);
                    st10[(size_t)(32 / 8) * 64 * 8 + (size_t)jj * 8 + 0] = bh;        // k = 32, 33 of the stage: the bias block
                    st10[(size_t)(32 / 8) * 64 * 8 + (size_t)jj * 8 + 1] = bl;
                }
            }
        }
}

template <int NP, bool PROF>
inline cudaError_t launch_lstm2f_np(const Lstm2fArgs& a, int sm_count, int max_clusters, cudaStream_t st) {
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(k_lstm2_fused<NP, PROF>, cudaFuncAttributeMaxDynamicSharedMemorySize, L2F_SMEM);
        if (e != cudaSuccess) return e;
        attr = true;
    }
    const int csize = 2 * NP;
    const int tile_pairs = a.n_tiles / 2;
    // clusters come in (forward, backward) pairs; no more of them than there is work for
    int per_dir = (tile_pairs + NP - 1) / NP;
    int max_per_dir = sm_count / csize / 2;
    if (NP > 1) {
        // the GPCs may not take sm_count / csize clusters of this size: ask
        cudaLaunchConfig_t q = {};
        q.gridDim = dim3((unsigned)(sm_count / csize * csize)); q.blockDim = dim3(L2F_THREADS); q.dynamicSmemBytes = L2F_SMEM;
        cudaLaunchAttribute qa[1];
        qa[0].id = cudaLaunchAttributeClusterDimension;
        qa[0].val.clusterDim.x = csize; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
        q.attrs = qa; q.numAttrs = 1;
        int n_cl = 0;
        if (cudaOccupancyMaxActiveClusters(&n_cl, k_lstm2_fused<NP, PROF>, &q) == cudaSuccess && n_cl > 0 && n_cl / 2 < max_per_dir)
            max_per_dir = n_cl / 2;
    }
    if (max_per_dir > max_clusters) max_per_dir = max_clusters;
    if (max_per_dir < 1) max_per_dir = 1;
    if (per_dir > max_per_dir) per_dir = max_per_dir;
    if (per_dir < 1) per_dir = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(per_dir * 2 * csize));
    cfg.blockDim = dim3(L2F_THREADS);
    cfg.dynamicSmemBytes = L2F_SMEM;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = csize; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, k_lstm2_fused<NP, PROF>, a);
}

// pairs per cluster that share one copy of the weight stream (C3R_LSTM2F_NP = 1, 2 or 4)
inline int lstm2f_np() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("C3R_LSTM2F_NP");
        v = e ? atoi(e) : 1;
        if (v != 1 && v != 2 && v != 4) v = 1;
    }
    return v;
}

// max_clusters: at most this many clusters per direction (a smaller grid takes more rounds of its persistent loop)
inline cudaError_t launch_lstm2f(const Lstm2fArgs& a, int sm_count, int max_clusters, cudaStream_t st) {
    if (a.prof) return launch_lstm2f_np<1, true>(a, sm_count, max_clusters, st);       // C3R_TRACE: the instrumented build
    switch (lstm2f_np()) {
        case 2: return launch_lstm2f_np<2, false>(a, sm_count, max_clusters, st);
        case 4: return launch_lstm2f_np<4, false>(a, sm_count, max_clusters, st);
        default: return launch_lstm2f_np<1, false>(a, sm_count, max_clusters, st);
    }
}

}  // namespace c3r
