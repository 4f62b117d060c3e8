// Pileup network forward on the 5th-gen tensor cores ("nn_impl = 1").
//
//   fp16 operands, fp32 accumulation in TMEM, fp32 gate math and cell state.
//   LSTM1's input kernel is split W = W_hi + W_lo (two fp16 terms) and so is its operand, raw read counts
//   x = x_hi + x_lo (|x| up to 8000; fp16 holds integers exactly only up to 2048); everything else is single fp16.
//
// Kernels
//   k_gemm_tc   tcgen05 GEMM, cta_group::1, 128x128 tiles, bulk-async-copy (TMA unit) operand
//               pipeline.  Used for L4 (K=10560, N=128) and L5 (K=128, N=256, +SELU).
//   k_lstm_tc   LSTM1 as a persistent recurrent layer, cta_group::2: a CTA pair owns 256 sites of
//               one direction; the input and recurrent weights stay resident in shared memory
//               split across the pair; per step tcgen05.mma -> TMEM -> gates in registers -> h
//               back to shared memory as the next step's A operand.
//   LSTM2 is k_lstm2_fused (nn_lstm2f.cuh).
//
// Operand layout everywhere: K-major, no swizzle, 8x(16 B) core matrices; element (r, k) of a
// tile with R rows sits at  (k/8)*R*8 + r*8 + k%8  halfs  (LBO = R*16 B, SBO = 128 B).
// Activations are written by their producer kernel already in this layout, so every operand
// tile is one contiguous bulk copy.
//
// Math restated from /root/reference/clair3_rna/model.py:126-216 (SURVEY.md Appendix D).
#pragma once
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include "nn_fp32.cuh"
#include "nn_sched.h"
#include "tc_ptx.cuh"

namespace c3r {

constexpr int TC_TILE = 128;                 // sites per CTA tile
constexpr int TC_KB = 64;                    // K per pipeline stage
constexpr int TC_IMG = TC_TILE * TC_KB;      // halfs in one 128x64 operand image (16 KB)
// K of LSTM1's input part for C channels: [x_hi | x_hi | x_lo | 1 | 1] rounded up to whole k16 MMA steps
// (C = 18: 56 -> 64, C = 30: 92 -> 96)
constexpr int lstm1_kx(int C) { return (3 * C + 2 + 15) / 16 * 16; }
constexpr int LSTM1_KX_MAX = lstm1_kx(30);

// ================================================================== GEMM
// The GEMM runs the split-precision product  A_hi*B_hi + A_lo*B_hi + A_hi*B_lo  (A = A_hi + A_lo and
// B = B_hi + B_lo as two fp16 terms each), which removes the fp16 rounding of both operands.
struct GemmArgs {
    const __half* A;      // [m_tiles][n_kb][TC_IMG]
    const __half* B;      // [n_tiles][n_kb][TC_IMG]
    const __half* A_lo;   // same layouts, low-order terms (terms == 3)
    const __half* B_lo;
    int terms;            // split-precision products as a bit mask: 1 = A_hi*B_hi, 2 = A_lo*B_hi, 4 = A_hi*B_lo
    const float* bias;    // [n_tiles*128], GEMM column order
    float* out;           // row-major [m*128+r][n_tiles*128], + bias + SELU
    int m_tiles, n_tiles, n_kb;
    int ksplit;           // K cut into ksplit ranges, one work item each; > 1: raw partial sums (no bias, no SELU)
    size_t split_stride;  // go to out + range * split_stride and the consumer adds them up (k_l4_finish)
    int* err;
};

// One pipeline stage = one 64-wide k block of all four operand images (A_hi, A_lo, B_hi, B_lo; 64 KB), consumed by the
// three split-precision products, so every operand byte crosses L2 -> shared memory once.
constexpr int GEMM_STAGES = 3;
constexpr int GEMM_THREADS = 192;
constexpr int GEMM_STAGE_BYTES = 4 * TC_IMG * 2;
constexpr int GEMM_SMEM = GEMM_STAGES * GEMM_STAGE_BYTES + 1024;

__global__ void __launch_bounds__(GEMM_THREADS, 1) k_gemm_tc(GemmArgs g) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* bars = (uint64_t*)(smem + GEMM_STAGES * GEMM_STAGE_BYTES);
    // bars: full[4] empty[4] acc_full[2] acc_empty[2] (slots for 4 stages, GEMM_STAGES used), then tmem ptr
    uint32_t* tmem_ptr_s = (uint32_t*)(bars + 12);
    float* bias_s = (float*)(bars + 32);                    // staged per tile by the epilogue warps
    const uint32_t s_base = ptx::smem_u32(smem);
    const uint32_t b_full = ptx::smem_u32(bars), b_empty = b_full + 32, b_accf = b_full + 64, b_acce = b_full + 80;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < GEMM_STAGES; ++i) { ptx::mbar_init(b_full + 8 * i, 1); ptx::mbar_init(b_empty + 8 * i, 1); }
        for (int i = 0; i < 2; ++i) { ptx::mbar_init(b_accf + 8 * i, 1); ptx::mbar_init(b_acce + 8 * i, 4); }
        ptx::fence_barrier_init();
    }
    if (warp == 1) {
        ptx::tmem_alloc<1>(ptx::smem_u32(tmem_ptr_s), 256);
        ptx::tmem_relinquish<1>();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem = *tmem_ptr_s;
    const int n_tiles_total = g.m_tiles * g.n_tiles;
    const int ksplit = g.ksplit > 1 ? g.ksplit : 1;
    const int n_items = n_tiles_total * ksplit;
    const uint32_t idesc = ptx::make_idesc_f16(128, 128);

    if (warp == 0) {
        if (lane == 0) {
            uint32_t it = 0;
            for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
                const int tile = item % n_tiles_total, ks = item / n_tiles_total;
                const int m = tile / g.n_tiles, n = tile % g.n_tiles;
                const size_t ao = (size_t)m * g.n_kb * TC_IMG, bo = (size_t)n * g.n_kb * TC_IMG;
                const int kb0 = ks * g.n_kb / ksplit, kb1 = (ks + 1) * g.n_kb / ksplit;
                for (int kb = kb0; kb < kb1; ++kb, ++it) {        // same k order and ranges for every tile: a site's result
                                                                  // does not depend on where in the batch it sits
                    const uint32_t s = it % GEMM_STAGES, ph = (it / GEMM_STAGES) & 1;
                    const uint32_t dst = s_base + s * GEMM_STAGE_BYTES;
                    ptx::mbar_wait(b_empty + 8 * s, ph ^ 1, g.err, 101);
                    const bool a_lo = g.terms & 2;                // the low-order activation image is only read by term 2
                    ptx::mbar_arrive_expect_tx(b_full + 8 * s, a_lo ? GEMM_STAGE_BYTES : GEMM_STAGE_BYTES - TC_IMG * 2);
                    ptx::bulk_g2s(dst, g.A + ao + (size_t)kb * TC_IMG, TC_IMG * 2, b_full + 8 * s);
                    if (a_lo) ptx::bulk_g2s(dst + TC_IMG * 2, g.A_lo + ao + (size_t)kb * TC_IMG, TC_IMG * 2, b_full + 8 * s);
                    ptx::bulk_g2s(dst + 2 * TC_IMG * 2, g.B + bo + (size_t)kb * TC_IMG, TC_IMG * 2, b_full + 8 * s);
                    ptx::bulk_g2s(dst + 3 * TC_IMG * 2, g.B_lo + bo + (size_t)kb * TC_IMG, TC_IMG * 2, b_full + 8 * s);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            uint32_t it = 0, tc = 0;
            for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++tc) {
                const int ks = item / n_tiles_total;
                const int kb0 = ks * g.n_kb / ksplit, kb1 = (ks + 1) * g.n_kb / ksplit;
                const uint32_t slot = tc & 1, aph = (tc >> 1) & 1;
                ptx::mbar_wait(b_acce + 8 * slot, aph ^ 1, g.err, 102);
                ptx::tc_fence_after();
                for (int kb = kb0; kb < kb1; ++kb, ++it) {
                    const uint32_t s = it % GEMM_STAGES, ph = (it / GEMM_STAGES) & 1;
                    ptx::mbar_wait(b_full + 8 * s, ph, g.err, 103);
                    ptx::tc_fence_after();
                    const uint32_t st0 = s_base + s * GEMM_STAGE_BYTES;
#pragma unroll
                    for (int term = 0; term < 3; ++term) {              // A_hi*B_hi, A_lo*B_hi, A_hi*B_lo
                        if (!((g.terms >> term) & 1)) continue;
                        const uint32_t sa = st0 + (term == 1 ? TC_IMG * 2 : 0), sb = st0 + (term == 2 ? 3 : 2) * TC_IMG * 2;
#pragma unroll
                        for (int k4 = 0; k4 < TC_KB / 16; ++k4) {
                            const uint64_t da = ptx::make_smem_desc(sa + k4 * 2 * (TC_TILE * 16), TC_TILE * 16, 128);
                            const uint64_t db = ptx::make_smem_desc(sb + k4 * 2 * (TC_TILE * 16), TC_TILE * 16, 128);
                            ptx::mma_f16<1>(tmem + slot * 128, da, db, idesc, (kb > kb0 || term > 0 || k4 > 0) ? 1u : 0u);
                        }
                    }
                    ptx::mma_commit_1(b_empty + 8 * s);
                }
                ptx::mma_commit_1(b_accf + 8 * slot);
            }
        }
    } else {
        const int q = warp & 3;
        const int row = q * 32 + lane;
        uint32_t tc = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++tc) {
            const int tile = item % n_tiles_total, ks = item / n_tiles_total;
            const int m = tile / g.n_tiles, n = tile % g.n_tiles;
            const uint32_t slot = tc & 1, aph = (tc >> 1) & 1;
            ptx::mbar_wait(b_accf + 8 * slot, aph, g.err, 104);
            ptx::tc_fence_after();
            const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + slot * 128;
            asm volatile("bar.sync 1, 128;" ::: "memory");      // previous tile's readers are done
            bias_s[threadIdx.x - 64] = g.bias[(size_t)n * 128 + (threadIdx.x - 64)];
            asm volatile("bar.sync 1, 128;" ::: "memory");
            const float* bias = bias_s;
#pragma unroll 1
            for (int j = 0; j < 8; ++j) {
                uint32_t v[16];
                ptx::tmem_ld16(taddr + j * 16, v);
                ptx::tmem_wait_ld();
                float* o = g.out + ((size_t)m * 128 + row) * ((size_t)g.n_tiles * 128) + (size_t)n * 128 + j * 16;
                if (ksplit > 1) {
                    float4* o4 = (float4*)(o + (size_t)ks * g.split_stride);
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        o4[c] = make_float4(__uint_as_float(v[4 * c]), __uint_as_float(v[4 * c + 1]), __uint_as_float(v[4 * c + 2]), __uint_as_float(v[4 * c + 3]));
                } else {
#pragma unroll
                    for (int c = 0; c < 16; ++c) o[c] = seluf_(__uint_as_float(v[c]) + bias[j * 16 + c]);
                }
            }
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(b_acce + 8 * slot);
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) ptx::tmem_dealloc<1>(tmem, 256);
}

// ================================================================== LSTM1
// One CTA pair (cluster of 2, tcgen05 cta_group::2) = 256 sites x one direction.
//   CH      gate-column chunks per step; a chunk = 32 units x 4 gates = 128 accumulator columns
//   KX      K of the input part fused into the step MMA ([x_hi | x_hi | x_lo | 1 | 1 | 0..] against
//           [W_hi ; W_lo ; W_hi ; b_hi ; b_lo ; 0], lstm1_kx)
//   U       units (K of the recurrent part) = CH*32
template <int CH, int KX>
struct LstmCfg {
    static constexpr int U = CH * 32;
    static constexpr int KT = KX + U;                       // K per step
    static constexpr int B_BYTES = CH * 64 * KT * 2;        // this CTA's half of the weights
    static constexpr int AH_BYTES = TC_TILE * U * 2;        // h operand, one buffer
    static constexpr int AX_BYTES = TC_TILE * KX * 2;       // x operand, one buffer
    static constexpr int BAR_OFF = B_BYTES + 2 * AH_BYTES + 2 * AX_BYTES;
    static constexpr int SMEM = BAR_OFF + 256;
    static_assert(SMEM <= 232448, "LSTM1 operands exceed the shared memory of a CTA");
    static constexpr int TMEM_COLS = 512;                   // 2 accumulator slots (256) + cell state (U <= 160)
    static constexpr int C_COL = 256;
};

struct LstmArgs {
    const __half* Wimg;     // [2 dirs][2 ranks][B_BYTES/2] operand images
    const __half* xop;      // x operand images [tile][33][KX/8][128][8] (k_xop)
    __half* hout;           // packed fp16 output [tile][33][4][TC_IMG]
    int64_t n_sites;        // valid sites (tensor rows); tiles beyond are zero
    int n_tiles;            // 128-site tiles (even)
    int* err;
    long long* trace;       // optional [2 ranks][33 steps][8 chunks][8 events] SM-clock stamps of cluster 0, work item 0
};

__device__ __forceinline__ void lstm_trace(const LstmArgs& a, bool on, uint32_t rank, int step, int c, int ev) {
    if (on) a.trace[(((size_t)rank * NT + step) * 8 + c) * 8 + ev] = clock64();
}

constexpr int LSTM_GATE_WARPS = 16;          // 4 per TMEM lane quarter, 8 units of a chunk each
constexpr int LSTM_THREADS = 64 + 32 * LSTM_GATE_WARPS;   // warp 0: MMA issue, warp 1: x loader, then the gate warps

// Gate math on the SFU.  Default: tanh.approx.f32 (MUFU.TANH, max relative error 2^-11), sigmoid as
// 0.5*tanh(0.5z)+0.5 with the 0.5z folded into the packed weights - 5 SFU ops per (site, unit).  Its error is of the size of the fp16 rounding h
// already goes through as the next step's MMA operand; measured effect on the output probabilities
// versus the ex2/rcp form: none (max |dp| 2.53e-4 vs 2.55e-4 on the stress weights, tools/prec_probe.py).
// LSTM_EXACT_GATES = true selects ex2.approx / rcp.approx (<= 2 ulp each), 8 SFU ops per (site, unit):
//   sigmoid(x) = 1/(1+2^(-x log2e)),  tanh(x) = (1-b)/(1+b) with b = 2^(-2x log2e),
//   sigmoid(i)*tanh(g) and sigmoid(o)*tanh(c) share one reciprocal each, exponents clamped so
//   (1+a)(1+b) stays finite (sigmoid(-30) and 1+tanh(-15) are below fp32 eps).
#ifndef C3R_EXACT_GATES
#define C3R_EXACT_GATES 0
#endif
constexpr bool LSTM_EXACT_GATES = C3R_EXACT_GATES != 0;
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
constexpr float LOG2E = 1.4426950408889634f;
__device__ __forceinline__ float sig_times_tanh(float zs, float zt) {
    const float a = ex2_approx(-LOG2E * fmaxf(zs, -30.0f));
    const float b = ex2_approx(-2.0f * LOG2E * fmaxf(zt, -15.0f));
    return (1.0f - b) * rcp_approx((1.0f + a) * (1.0f + b));
}
__device__ __forceinline__ float sigmoid_fast(float x) { return rcp_approx(1.0f + ex2_approx(-LOG2E * x)); }
__device__ __forceinline__ float tanh_approx(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// sigmoid(z) from the pre-halved pre-activation x = 0.5 z (the i, f, o columns of every LSTM weight and bias are
// packed times 0.5 - an exact scaling - so the gate stage saves three multiplies per unit)
__device__ __forceinline__ float sigmoid_tanh(float x) { return fmaf(tanh_approx(x), 0.5f, 0.5f); }

// One LSTM cell update from the pre-activations (zi, zf, zo pre-halved, see above).
//   C3R_GATE_MODE 0: five tanh.approx                      2: ex2/rcp everywhere (8 SFU ops)
//                 1: as 0 but the forget gate by ex2/rcp (6 SFU ops): the absolute error of tanh.approx (2^-11)
//                    in f multiplies the cell state, which is not bounded by 1 - with a forget bias of 3 the state
//                    reaches ~20 and a 2.4e-4 error in f becomes 5e-3 in c per step
#ifndef C3R_GATE_MODE
#define C3R_GATE_MODE (C3R_EXACT_GATES ? 2 : 0)
#endif
__device__ __forceinline__ void lstm_cell(float zi, float zf, float zg, float zo, float cp, float& cn, float& hv) {
    if (C3R_GATE_MODE == 2) {
        cn = fmaf(sigmoid_fast(2.0f * zf), cp, sig_times_tanh(2.0f * zi, zg));
        hv = sig_times_tanh(2.0f * zo, cn);
    } else if (C3R_GATE_MODE == 1) {
        cn = fmaf(sigmoid_fast(2.0f * zf), cp, sigmoid_tanh(zi) * tanh_approx(zg));
        hv = sigmoid_tanh(zo) * tanh_approx(cn);
    } else {
        cn = fmaf(sigmoid_tanh(zf), cp, sigmoid_tanh(zi) * tanh_approx(zg));
        hv = sigmoid_tanh(zo) * tanh_approx(cn);
    }
}

template <int CH, int KX>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(LSTM_THREADS, 1) k_lstm_tc(LstmArgs a) {
    static_assert(KX > 0, "the input part is fused into the step MMA");
    typedef LstmCfg<CH, KX> Cfg;
    constexpr int U = Cfg::U, KT = Cfg::KT;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t s_base = ptx::smem_u32(smem);
    const uint32_t s_B = s_base, s_AH = s_base + Cfg::B_BYTES, s_AX = s_AH + 2 * Cfg::AH_BYTES;
    uint64_t* bars = (uint64_t*)(smem + Cfg::BAR_OFF);
    // barriers: 0 w_full | 1,2 acc_full[2] | 3,4 acc_empty[2] (local gate warps) | 5,6 x_ready[2] |
    //           7,8 step_done[2] | 9,10 acc_empty_peer[2] (leader only: one relayed arrival per use from the peer) ; tmem ptr
    // Every wait below targets the current or the immediately preceding phase of its barrier
    // (mbarrier parity waits cannot tell phases further apart).
    const uint32_t b0 = ptx::smem_u32(bars);
    const uint32_t b_w = b0, b_accf = b0 + 8, b_acce = b0 + 24, b_xr = b0 + 40, b_step = b0 + 56;
    const uint32_t b_accr = b0 + 72;
    const uint32_t b_xl = b0 + 88;                           // 11,12: this CTA's x tile landed (bulk copy tx)
    // 13: h_t complete in this CTA (its 16 gate warps, once per step) | 15: the peer's relay of the same (leader only).
    // Accumulator slots are released as soon as the gate warps hold the values in registers (acc_empty), so the MMAs
    // of the next chunks run under the gate math; only the first MMA of a step waits for h_t (these two barriers).
    const uint32_t b_hrdy = b0 + 104, b_hrdy_r = b0 + 120;
    uint32_t* tmem_ptr_s = (uint32_t*)(bars + 20);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = ptx::cluster_ctarank();
    // clusters come in (forward, backward) pairs so a cluster keeps one direction's weights resident
    const int cluster_id = blockIdx.x >> 1, n_cpairs = gridDim.x >> 2;
    const int dir = cluster_id & 1;
    const int n_tile_pairs = a.n_tiles / 2;

    if (threadIdx.x == 0) {
        ptx::mbar_init(b_w, 1);
        ptx::mbar_init(b_accf, 1); ptx::mbar_init(b_accf + 8, 1);
        ptx::mbar_init(b_acce, LSTM_GATE_WARPS); ptx::mbar_init(b_acce + 8, LSTM_GATE_WARPS);   // this CTA's gate warps
        ptx::mbar_init(b_accr, 1); ptx::mbar_init(b_accr + 8, 1);                                 // peer's relay
        ptx::mbar_init(b_xr, 1); ptx::mbar_init(b_xr + 8, 1);            // peer's x tile landed (relayed)
        ptx::mbar_init(b_xl, 1); ptx::mbar_init(b_xl + 8, 1);
        ptx::mbar_init(b_step, 1); ptx::mbar_init(b_step + 8, 1);
        ptx::mbar_init(b_hrdy, LSTM_GATE_WARPS); ptx::mbar_init(b_hrdy_r, 1);
        ptx::fence_barrier_init();
        // this CTA's half of the direction's weights: resident for the whole kernel
        ptx::mbar_arrive_expect_tx(b_w, Cfg::B_BYTES);
        const __half* wsrc = a.Wimg + ((size_t)dir * 2 + rank) * (Cfg::B_BYTES / 2);
        constexpr uint32_t PIECE = 32768;
        for (uint32_t o = 0; o < (uint32_t)Cfg::B_BYTES; o += PIECE) {
            const uint32_t nb = (uint32_t)Cfg::B_BYTES - o < PIECE ? (uint32_t)Cfg::B_BYTES - o : PIECE;
            ptx::bulk_g2s(s_B + o, (const uint8_t*)wsrc + o, nb, b_w);
        }
    }
    if (warp == 0) {
        ptx::tmem_alloc<2>(ptx::smem_u32(tmem_ptr_s), Cfg::TMEM_COLS);
        ptx::tmem_relinquish<2>();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::mbar_wait(b_w, 0, a.err, 201);                      // weights landed in this CTA ...
    ptx::cluster_sync();                                     // ... and in the peer
    ptx::tc_fence_after();
    const uint32_t tmem = *tmem_ptr_s;
    constexpr uint32_t IDESC = ptx::make_idesc_f16(256, 128);

    uint32_t work_it = 0;                                    // work items done by this cluster
    for (int tile_pair = cluster_id >> 1; tile_pair < n_tile_pairs; tile_pair += n_cpairs, ++work_it) {
        const int tile = tile_pair * 2 + (int)rank;          // this CTA's 128 sites
        const uint32_t base_use = work_it * (uint32_t)(NT * CH);     // accumulator uses before this work item
        const uint32_t base_step = work_it * (uint32_t)NT;
        const bool tr = a.trace != nullptr && cluster_id == 0 && work_it == 0 && lane == 0;

        if (warp == 0) {
            // ------------------------------------------------ MMA issue (leader CTA): one thread chosen by elect.sync, so that
            // ptxas emits straight-line UTCHMMA fed from uniform registers (a `lane == 0` test or a converged warp with
            // a per-lane predicate gets an ELECT / R2UR loop around every MMA, ~100 cycles each)
            if (rank == 0) {
                if (ptx::elect_one()) {
                for (int step = 0; step < NT; ++step) {
                    const uint32_t gstep = base_step + step;
                    const uint32_t buf = gstep & 1;
                    ptx::mbar_wait(b_xl + 8 * buf, (gstep >> 1) & 1, a.err, 202);
                    ptx::mbar_wait(b_xr + 8 * buf, (gstep >> 1) & 1, a.err, 212);
                    for (int c = 0; c < CH; ++c) {
                        const uint32_t use = base_use + step * CH + c;
                        const uint32_t slot = use & 1;
                        // slot free (its previous use drained by both CTAs)
                        ptx::mbar_wait(b_acce + 8 * slot, ((use >> 1) & 1) ^ 1, a.err, 203);
                        ptx::mbar_wait(b_accr + 8 * slot, ((use >> 1) & 1) ^ 1, a.err, 213);
                        ptx::tc_fence_after();
                        lstm_trace(a, tr, 0, step, c, 0);
                        // One thread issues every MMA, so the instructions between two issues are the critical path
                        // of the whole CTA pair: descriptors are built once per chunk and advanced by constant adds
                        // (the start-address field counts 16-byte units and cannot carry out of its 14 bits here).
                        const uint64_t dB0 = ptx::make_smem_desc(s_B + c * (64 * KT * 2), 64 * 16, 128);
                        // the input part does not need h_{t-1}: it goes first
                        const uint64_t dX0 = ptx::make_smem_desc(s_AX + buf * Cfg::AX_BYTES, TC_TILE * 16, 128);
#pragma unroll
                        for (int k = 0; k < KX / 16; ++k)
                            ptx::mma_f16<2>(tmem + slot * 128, dX0 + (uint64_t)(k * ((2 * TC_TILE * 16) >> 4)),
                                            dB0 + (uint64_t)(k * ((2 * 64 * 16) >> 4)), IDESC, k > 0 ? 1u : 0u);
                        // at the start of a step, h of the previous step must be complete in both CTAs
                        if (c == 0 && step > 0) {
                            ptx::mbar_wait(b_hrdy, (gstep - 1) & 1, a.err, 204);
                            ptx::mbar_wait(b_hrdy_r, (gstep - 1) & 1, a.err, 214);
                            ptx::tc_fence_after();
                        }
                        if (step > 0) {
                            const uint64_t dH0 = ptx::make_smem_desc(s_AH + buf * Cfg::AH_BYTES, TC_TILE * 16, 128);
#pragma unroll
                            for (int k = 0; k < U / 16; ++k)
                                ptx::mma_f16<2>(tmem + slot * 128, dH0 + (uint64_t)(k * ((2 * TC_TILE * 16) >> 4)),
                                                dB0 + (uint64_t)(((KX / 8 + k * 2) * (64 * 16)) >> 4), IDESC, 1u);
                        }
                        ptx::mma_commit_2_mcast(b_accf + 8 * slot, 3);
                        lstm_trace(a, tr, 0, step, c, 1);
                    }
                    ptx::mma_commit_2_mcast(b_step + 8 * buf, 3);
                }
                }
                __syncwarp();
            }
            if (rank == 1 && lane == 0) {
                // relay: one cluster-scope arrival per accumulator use on behalf of this CTA's 16 gate
                // warps, so the expensive cluster release fence is off their critical path
                for (int u = 0; u < NT * CH; ++u) {
                    const uint32_t use = base_use + u;
                    const uint32_t slot = use & 1;
                    ptx::mbar_wait(b_acce + 8 * slot, (use >> 1) & 1, a.err, 215);
                    ptx::mbar_arrive_cluster_relaxed(b_accr + 8 * slot, 0);
                    lstm_trace(a, tr, 1, u / CH, u % CH, 5);
                    if (u % CH == CH - 1) {                  // end of a step: h_t of this CTA is complete
                        const uint32_t gstep = base_step + u / CH;
                        ptx::mbar_wait(b_hrdy, gstep & 1, a.err, 217);
                        ptx::mbar_arrive_cluster_relaxed(b_hrdy_r, 0);
                    }
                }
            }
        } else if (warp == 1) {
            // ------------------------------------------------ x_t operand tile, one bulk copy per step
            if (lane == 0) {
                for (int step = 0; step < NT; ++step) {
                    const uint32_t gstep = base_step + step;
                    const uint32_t buf = gstep & 1;
                    // buffer `buf` was last read by the MMAs of global step gstep-2
                    if (gstep >= 2) ptx::mbar_wait(b_step + 8 * buf, ((gstep >> 1) - 1) & 1, a.err, 205);
                    lstm_trace(a, tr, rank, step, 0, 6);
                    const int t = dir == 0 ? step : NT - 1 - step;
                    ptx::mbar_arrive_expect_tx(b_xl + 8 * buf, Cfg::AX_BYTES);
                    ptx::bulk_g2s(s_AX + buf * Cfg::AX_BYTES,
                                  a.xop + ((size_t)tile * NT + t) * (size_t)(KX * TC_TILE), Cfg::AX_BYTES, b_xl + 8 * buf);
                    if (rank == 1) {                         // tell the leader this CTA's tile has landed
                        ptx::mbar_wait(b_xl + 8 * buf, (gstep >> 1) & 1, a.err, 206);
                        ptx::mbar_arrive_cluster_relaxed(b_xr + 8 * buf, 0);
                    }
                    lstm_trace(a, tr, rank, step, 0, 7);
                }
            }
        } else {
            // ------------------------------------------------ gates: TMEM -> c, h
            const int gw = warp - 2;                         // 0..15
            const int q = warp & 3;                          // TMEM lane quarter this warp may access
            const int sub = gw >> 2;                         // which 8 units of the chunk's 32
            const int row = q * 32 + lane;
            const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
            for (int step = 0; step < NT; ++step) {
                const uint32_t gstep = base_step + step;
                const uint32_t nbuf = (gstep + 1) & 1;       // h_t goes to the buffer step+1 reads
                const int t = dir == 0 ? step : NT - 1 - step;
                uint8_t* ah = smem + Cfg::B_BYTES + nbuf * Cfg::AH_BYTES;
                __half* hout_t = a.hout + ((size_t)tile * NT + t) * 4 * TC_IMG;
#pragma unroll
                for (int c = 0; c < CH; ++c) {
                    const uint32_t use = base_use + step * CH + c;
                    const uint32_t slot = use & 1;
                    ptx::mbar_wait(b_accf + 8 * slot, (use >> 1) & 1, a.err, 208);
                    ptx::tc_fence_after();
                    lstm_trace(a, tr && gw == 0, rank, step, c, 2);
                    uint32_t cprev[8];
                    uint32_t v[4][8];
#pragma unroll
                    for (int gte = 0; gte < 4; ++gte)
                        ptx::tmem_ld8(tmem + lane_addr + slot * 128 + gte * 32 + sub * 8, v[gte]);
                    if (step > 0) ptx::tmem_ld8(tmem + lane_addr + Cfg::C_COL + c * 32 + sub * 8, cprev);
                    ptx::tmem_wait_ld();
                    lstm_trace(a, tr && gw == 0, rank, step, c, 3);
                    ptx::tc_fence_before();                      // the accumulator slot is in registers: hand it back
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive(b_acce + 8 * slot);
                    lstm_trace(a, tr && gw == 0, rank, step, c, 4);
                    uint32_t cnew[8];
                    __align__(16) __half hh[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const float cp = step > 0 ? __uint_as_float(cprev[u]) : 0.0f;
                        float cn, hv;
                        lstm_cell(__uint_as_float(v[0][u]), __uint_as_float(v[1][u]), __uint_as_float(v[2][u]),
                                  __uint_as_float(v[3][u]), cp, cn, hv);
                        cnew[u] = __float_as_uint(cn);
                        hh[u] = __float2half(hv);
                    }
                    ptx::tmem_st8(tmem + lane_addr + Cfg::C_COL + c * 32 + sub * 8, cnew);
                    // h_t: next step's A operand (k index = unit)
                    const uint4 pk = *(const uint4*)hh;
                    const int k8 = c * 4 + sub;
                    *(uint4*)(ah + (size_t)k8 * (TC_TILE * 16) + row * 16) = pk;
                    ptx::tmem_wait_st();
                    if (c == CH - 1) {                           // this warp's part of h_t is in shared memory: one
                        ptx::tc_fence_before();                  // generic->async proxy fence covers all of its writes
                        ptx::fence_proxy_async();
                        __syncwarp();
                        if (lane == 0) ptx::mbar_arrive(b_hrdy);
                    }
                    // layer output goes out AFTER the arrival: the release fence of the arrival would
                    // otherwise wait for these HBM stores on the recurrence's critical path
                    {
                        const int col8 = (dir * U) / 8 + k8;                 // 8-column group in the concat [fwd | bwd]
                        const size_t oo = (size_t)(col8 / 8) * TC_IMG + (size_t)(col8 % 8) * (TC_TILE * 8) + row * 8;
                        *(uint4*)(hout_t + oo) = pk;
                    }
                }
            }
            // the step_done commits multicast to this CTA have landed before it may exit
            if (gw == 0) {
                const uint32_t g_last = base_step + NT - 1;
                ptx::mbar_wait(b_step + 8 * (g_last & 1), (g_last >> 1) & 1, a.err, 209);
                ptx::mbar_wait(b_step + 8 * ((g_last - 1) & 1), ((g_last - 1) >> 1) & 1, a.err, 210);
            }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync();
    if (warp == 0) ptx::tmem_dealloc<2>(tmem, Cfg::TMEM_COLS);
}

// int32 windows [n][33][C] -> LSTM1 x operand images [tile][33][KX/8][128 rows][8 halfs]:
//   k < C: x_hi, C <= k < 2C: x_hi again (meets W_lo), 2C <= k < 3C: x_lo (meets W_hi), k = 3C, 3C+1: 1 (meets
//   b_hi, b_lo), rest 0.  x_hi = fp16(x), x_lo = x - x_hi: exact for |x| <= 8000 (|x_lo| <= 2), so counts above 2048,
//   which fp16 cannot hold, reach the MMA unrounded (x_pack_hi_lo).
// Block = one (tile, t), thread = one site; each k-group is one coalesced 2 KB store.
__device__ __forceinline__ void x_pack_hi_lo(int32_t v, __half& hi, __half& lo) {
    hi = __float2half((float)v);
    lo = __float2half((float)v - __half2float(hi));
}
template <int C, int KX>
__global__ void __launch_bounds__(TC_TILE) k_xop(const int32_t* __restrict__ tensor, __half* __restrict__ xop, int64_t n_sites) {
    static_assert(KX >= 3 * C + 2 && KX % 16 == 0, "x_hi | x_hi | x_lo | 1 | 1 must fit the input part");
    const int tile = blockIdx.x / NT, t = blockIdx.x % NT, r = threadIdx.x;
    const int64_t site = (int64_t)tile * TC_TILE + r;
    __align__(16) __half hv[KX];
#pragma unroll
    for (int k = 0; k < KX; ++k) hv[k] = __float2half(0.0f);
    if (site < n_sites) {
        const int2* src = (const int2*)(tensor + (site * NT + t) * C);       // rows are 8-byte aligned (C even)
#pragma unroll
        for (int j = 0; j < C / 2; ++j) {
            const int2 v = src[j];
            x_pack_hi_lo(v.x, hv[2 * j], hv[2 * C + 2 * j]);
            x_pack_hi_lo(v.y, hv[2 * j + 1], hv[2 * C + 2 * j + 1]);
            hv[C + 2 * j] = hv[2 * j];
            hv[C + 2 * j + 1] = hv[2 * j + 1];
        }
    }
    hv[3 * C] = __float2half(1.0f);
    hv[3 * C + 1] = __float2half(1.0f);
    __half* dst = xop + ((size_t)tile * NT + t) * (size_t)(KX * TC_TILE) + r * 8;
#pragma unroll
    for (int k8 = 0; k8 < KX / 8; ++k8) *(uint4*)(dst + (size_t)k8 * (TC_TILE * 8)) = *(const uint4*)(&hv[k8 * 8]);
}

}  // namespace c3r
#include "nn_lstm2f.cuh"
namespace c3r {

// L4's partial sums -> l4 = selu(sum + bias): fp32 [site][128] (inspection) and the fp16 hi / lo operand images
// [tile][2 kb][128 x 64] of the L5 GEMM.  Block = 32 rows of a 128-site tile, thread = (row, 8-column cell), 4 cells each.
__global__ void __launch_bounds__(128) k_l4_finish(const float* __restrict__ part, int n_part, size_t stride,
                                                   const float* __restrict__ bias, float* __restrict__ l4,
                                                   __half* __restrict__ img, __half* __restrict__ img_lo) {
    const int tile = blockIdx.x >> 2;
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        const int e = ((blockIdx.x & 3) * 4 + it) * 128 + threadIdx.x, row = e >> 4, cell = e & 15;
        const size_t src = ((size_t)tile * 128 + row) * DENSE + cell * 8;
        float v[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) v[c] = bias[cell * 8 + c];
        for (int q = 0; q < n_part; ++q) {
            const float4 a = *(const float4*)(part + (size_t)q * stride + src), b = *(const float4*)(part + (size_t)q * stride + src + 4);
            v[0] += a.x; v[1] += a.y; v[2] += a.z; v[3] += a.w; v[4] += b.x; v[5] += b.y; v[6] += b.z; v[7] += b.w;
        }
        __align__(16) __half hi[8];
        __align__(16) __half lo[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            v[c] = seluf_(v[c]);
            hi[c] = __float2half(v[c]);
            lo[c] = __float2half(v[c] - __half2float(hi[c]));
        }
        *(float4*)(l4 + src) = make_float4(v[0], v[1], v[2], v[3]);
        *(float4*)(l4 + src + 4) = make_float4(v[4], v[5], v[6], v[7]);
        const size_t dst = ((size_t)tile * 2 + cell / 8) * TC_IMG + (size_t)(cell % 8) * (TC_TILE * 8) + row * 8;
        *(uint4*)(img + dst) = *(const uint4*)hi;
        *(uint4*)(img_lo + dst) = *(const uint4*)lo;
    }
}

// The two output layers on a5 = [selu(L5_1) | selu(L5_2)] (fp32 [site][256]): Y_gt21 (21) and Y_genotype (3), SELU,
// softmax (model.py:154-156,195-197, 213-214).  One warp per site, lane = output.
constexpr int HOUT_WARPS = 8;
__global__ void __launch_bounds__(HOUT_WARPS * 32) k_heads_out(NetF32 w, const float* __restrict__ a5, float* __restrict__ probs, int64_t n) {
    __shared__ float wy[DENSE][24];
    __shared__ float by[24];
    for (int i = threadIdx.x; i < DENSE * 24; i += blockDim.x) {
        const int k = i / 24, o = i % 24;
        wy[k][o] = o < 21 ? w.ky1[k * 21 + o] : w.ky2[k * 3 + (o - 21)];
    }
    if (threadIdx.x < 24) by[threadIdx.x] = threadIdx.x < 21 ? w.by1[threadIdx.x] : w.by2[threadIdx.x - 21];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int o = lane < 24 ? lane : 23;
    for (int64_t s = (int64_t)blockIdx.x * HOUT_WARPS + warp; s < n; s += (int64_t)gridDim.x * HOUT_WARPS) {
        const float* av = a5 + s * 256 + (o < 21 ? 0 : DENSE);
        float v0 = by[o], v1 = 0.0f, v2 = 0.0f, v3 = 0.0f;
#pragma unroll 8
        for (int k = 0; k < DENSE; k += 4) {
            const float4 a4 = *(const float4*)(av + k);
            v0 = fmaf(a4.x, wy[k][o], v0); v1 = fmaf(a4.y, wy[k + 1][o], v1);
            v2 = fmaf(a4.z, wy[k + 2][o], v2); v3 = fmaf(a4.w, wy[k + 3][o], v3);
        }
        const float y = seluf_((v0 + v1) + (v2 + v3));
        // softmax within lanes 0..20 and within lanes 21..23
        const bool g1 = lane < 21, g2 = lane >= 21 && lane < 24;
        float m1 = g1 ? y : -INFINITY, m2 = g2 ? y : -INFINITY;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) { m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, d)); m2 = fmaxf(m2, __shfl_xor_sync(0xffffffffu, m2, d)); }
        const float e = g1 ? expf(y - m1) : (g2 ? expf(y - m2) : 0.0f);
        float s1 = g1 ? e : 0.0f, s2 = g2 ? e : 0.0f;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, d); s2 += __shfl_xor_sync(0xffffffffu, s2, d); }
        if (lane < 24) probs[s * 24 + lane] = e / (g1 ? s1 : s2);
    }
}

// ================================================================== host side
constexpr int L4_KSPLIT = 3;                 // L4's K = 165 k blocks goes in 3 ranges of 55 (see tc_l4_heads)

struct TcNet {
    int ready = 0;
    int C = 18, KX = lstm1_kx(18), sm_count = 148;
    void* wbuf = nullptr;          // all fp16 images + fp32 biases
    size_t wbytes = 0;
    const __half *img1 = nullptr, *k4p = nullptr, *k4p_lo = nullptr;
    const float* b4 = nullptr;
    const uint8_t* wstream2 = nullptr;   // fused LSTM2: weight stream [2 dirs][2 halves][L2F_STREAM_BYTES]
    const __half *k5p = nullptr, *k5p_lo = nullptr;   // [L5_1 | L5_2] as one N = 256 GEMM: [2 n tiles][2 kb][TC_IMG]
    const float* b5p = nullptr;                        // [256]
    // activation scratch (sized for cap_tiles 128-site tiles)
    void* abuf = nullptr;
    size_t abytes = 0;
    int cap_tiles = 0;
    __half* h1[2] = {};            // LSTM1 output, one buffer per pass parity (tc_forward)
    __half *h2 = nullptr, *h2_lo = nullptr, *xop = nullptr;
    __half* h1_cur = nullptr;      // the h1 buffer of the pass queued last
    float *l4 = nullptr, *l4p = nullptr;                   // l4p: L4's partial sums [L4_KSPLIT][tiles*128][128]
    size_t l4_stride = 0;
    __half *l4h = nullptr, *l4h_lo = nullptr;              // l4 as fp16 operand images [tile][2 kb][TC_IMG] (hi, lo)
    float* a5 = nullptr;                                   // selu(L5_1) | selu(L5_2): [tiles*128][256]
    int* err = nullptr;
    long long* trace = nullptr;    // [LSTM1: 2 ranks][33][8][8] then the fused LSTM2 profile, filled when C3R_TRACE is set
    bool attr_set = false;
    struct TcPipe* pipe = nullptr; // second stream + events of the A/B tail overlap (tc_forward)
};

inline void tc_pipe_release(struct TcPipe* p);
inline void tc_release(TcNet& t) {
    if (t.pipe) tc_pipe_release(t.pipe);
    if (t.wbuf) cudaFree(t.wbuf);
    if (t.abuf) cudaFree(t.abuf);
    if (t.err) cudaFree(t.err);
    if (t.trace) cudaFree(t.trace);
    t = TcNet();
}

// element (r, k) of an R-row K-major no-swizzle image
inline size_t img_index(int R, int r, int k) { return (size_t)(k / 8) * R * 8 + (size_t)r * 8 + (k % 8); }

inline int tc_build(TcNet& t, const NetF32& net, const float* h, size_t o_w1, size_t o_b1, size_t o_u1, size_t o_w2,
                    size_t o_b2, size_t o_u2, size_t o_k4, size_t o_b4, size_t o_k51, size_t o_b51, size_t o_k52, size_t o_b52,
                    int sm_count, std::string* err) {
    tc_release(t);
    const int C = net.C;
    t.C = C;
    t.KX = lstm1_kx(C);
    t.sm_count = sm_count;
    const int KX = t.KX;
    const int KT1 = KX + U1;
    const size_t n_img1 = (size_t)2 * 2 * 4 * 64 * KT1;          // [dir][rank][chunk][64 x KT1]
    const size_t n_k4p = (size_t)(L4_IN / TC_KB) * TC_IMG;
    const size_t n_k5p = (size_t)2 * 2 * TC_IMG;
    std::vector<__half> hb(n_img1 + 2 * n_k4p + 2 * n_k5p);
    std::vector<float> fb(DENSE + 2 * DENSE);
    __half* img1 = hb.data();
    __half* k4p = img1 + n_img1;
    __half* k4p_lo = k4p + n_k4p;
    __half* k5p = k4p_lo + n_k4p;
    __half* k5p_lo = k5p + n_k5p;
    auto split = [](float w, __half& hi, __half& lo) {
        hi = __float2half(w);
        lo = __float2half(w - __half2float(hi));
    };
    // Keras gate column of chunk column j (gate-major inside a chunk: j = gate*32 + unit_local)
    for (int dir = 0; dir < 2; ++dir)
        for (int rank = 0; rank < 2; ++rank)
            for (int c = 0; c < 4; ++c) {
                __half* im = img1 + ((((size_t)dir * 2 + rank) * 4 + c) * 64) * KT1;
                for (int j = 0; j < 64; ++j) {
                    const int col = rank * 64 + j, gate = col / 32, ul = col % 32;
                    const int kc = gate * U1 + c * 32 + ul;                     // column in [.., 4u]
                    const float gs = gate == 2 ? 1.0f : 0.5f;                   // i, f, o columns hold 0.5 * z (see the gate math)
                    for (int k = 0; k < KT1; ++k) {
                        __half v = __float2half(0.0f);
                        if (k < 3 * C) {                // [W_hi ; W_lo ; W_hi] against [x_hi | x_hi | x_lo]
                            const int ch = k % C;
                            __half hi, lo;
                            split(gs * h[o_w1 + (size_t)ch * 2 * G1 + dir * G1 + kc], hi, lo);
                            v = k >= C && k < 2 * C ? lo : hi;
                        } else if (k == 3 * C || k == 3 * C + 1) {
                            __half hi, lo;
                            split(gs * h[o_b1 + dir * G1 + kc], hi, lo);
                            v = k == 3 * C ? hi : lo;
                        } else if (k >= KX) {
                            v = __float2half(gs * h[o_u1 + (size_t)dir * U1 * G1 + (size_t)(k - KX) * G1 + kc]);
                        }
                        im[img_index(64, j, k)] = v;
                    }
                }
            }
    for (int k = 0; k < L4_IN; ++k)
        for (int j = 0; j < DENSE; ++j)
        {
            const size_t ix = (size_t)(k / TC_KB) * TC_IMG + img_index(128, j, k % TC_KB);
            split(h[o_k4 + (size_t)k * DENSE + j], k4p[ix], k4p_lo[ix]);
        }
    for (int j = 0; j < DENSE; ++j) fb[j] = h[o_b4 + j];
    // L5_1 and L5_2 side by side: GEMM column n*128 + j = unit j of layer n; B image row = output unit, k = input
    for (int n = 0; n < 2; ++n)
        for (int k = 0; k < DENSE; ++k)
            for (int j = 0; j < DENSE; ++j) {
                const size_t ix = ((size_t)n * 2 + k / TC_KB) * TC_IMG + img_index(128, j, k % TC_KB);
                split(h[(n == 0 ? o_k51 : o_k52) + (size_t)k * DENSE + j], k5p[ix], k5p_lo[ix]);
            }
    for (int j = 0; j < DENSE; ++j) { fb[DENSE + j] = h[o_b51 + j]; fb[2 * DENSE + j] = h[o_b52 + j]; }

    std::vector<uint8_t> ws;
    lstm2f_pack(ws, h, o_w2, o_b2, o_u2);
    const size_t foff = ((hb.size() * 2 + 255) / 256) * 256;
    const size_t soff = ((foff + fb.size() * 4 + 1023) / 1024) * 1024;
    t.wbytes = soff + ws.size() + 256;
    cudaError_t e = cudaMalloc(&t.wbuf, t.wbytes);
    if (e != cudaSuccess) { *err = cudaGetErrorString(e); return -1; }
    uint8_t* d = (uint8_t*)t.wbuf;
    cudaMemcpy(d, hb.data(), hb.size() * 2, cudaMemcpyHostToDevice);
    cudaMemcpy(d + soff, ws.data(), ws.size(), cudaMemcpyHostToDevice);
    t.wstream2 = d + soff;
    e = cudaMemcpy(d + foff, fb.data(), fb.size() * 4, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { *err = cudaGetErrorString(e); return -1; }
    t.img1 = (const __half*)d;
    t.k4p = t.img1 + n_img1;
    t.k4p_lo = t.k4p + n_k4p;
    t.k5p = t.k4p_lo + n_k4p;
    t.k5p_lo = t.k5p + n_k5p;
    t.b4 = (const float*)(d + foff);
    t.b5p = t.b4 + DENSE;
    e = cudaMalloc((void**)&t.err, 64);
    if (e != cudaSuccess) { *err = cudaGetErrorString(e); return -1; }
    cudaMemset(t.err, 0, 64);
    if (getenv("C3R_TRACE")) {
        cudaMalloc((void**)&t.trace, 2 * 2 * NT * 8 * 8 * sizeof(long long));
        cudaMemset(t.trace, 0, 2 * 2 * NT * 8 * 8 * sizeof(long long));
    }
    t.ready = 1;
    return 0;
}

inline int tc_ensure(TcNet& t, int tiles, std::string* err) {
    if (tiles <= t.cap_tiles) return 0;
    if (t.abuf) cudaFree(t.abuf);
    t.abuf = nullptr;
    const size_t n_h1 = (size_t)tiles * NT * 4 * TC_IMG, n_h2 = (size_t)tiles * NT * 5 * TC_IMG;
    const size_t n_l4 = (size_t)tiles * 128 * DENSE;
    const size_t n_xop = (size_t)tiles * NT * LSTM1_KX_MAX * TC_TILE;
    t.abytes = (n_h1 + n_h2) * 2 * 2 + n_xop * 2 + n_l4 * (1 + L4_KSPLIT) * 4 + n_l4 * 2 * 2 + n_l4 * 2 * 4 + 1024;
    cudaError_t e = cudaMalloc(&t.abuf, t.abytes);
    if (e != cudaSuccess) { *err = std::string("activation scratch: ") + cudaGetErrorString(e); t.cap_tiles = 0; return -1; }
    uint8_t* p = (uint8_t*)t.abuf;
    t.l4 = (float*)p; p += n_l4 * 4;
    t.l4p = (float*)p; p += n_l4 * 4 * L4_KSPLIT;
    t.l4_stride = n_l4;
    t.a5 = (float*)p; p += n_l4 * 2 * 4;
    t.l4h = (__half*)p; p += n_l4 * 2;
    t.l4h_lo = (__half*)p; p += n_l4 * 2;
    t.h1[0] = (__half*)p; p += n_h1 * 2;
    t.h1[1] = (__half*)p; p += n_h1 * 2;
    t.h2 = (__half*)p; p += n_h2 * 2;
    t.h2_lo = (__half*)p; p += n_h2 * 2;
    t.xop = (__half*)p;
    t.cap_tiles = tiles;
    return 0;
}

// at most 40960 sites per sub-pass (tc_forward rounds it down to whole rounds of the recurrent kernels): bounds the
// activation scratch (3.4 GB) and sets how a large batch is cut into sub-passes
constexpr int TC_SUB_TILES = 320;

template <int CH, int KX>
// max_cpairs: at most this many (forward, backward) cluster pairs (a smaller grid takes more rounds of its persistent loop)
inline cudaError_t launch_lstm(const LstmArgs& a, int sm_count, int max_cpairs, cudaStream_t st) {
    typedef LstmCfg<CH, KX> Cfg;
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(k_lstm_tc<CH, KX>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
        if (e != cudaSuccess) return e;
        attr = true;
    }
    int cpairs = a.n_tiles / 2;              // (forward, backward) cluster pairs, one per tile pair at most
    if (cpairs > sm_count / 4) cpairs = sm_count / 4;
    if (cpairs > max_cpairs) cpairs = max_cpairs;
    if (cpairs < 1) cpairs = 1;
    k_lstm_tc<CH, KX><<<cpairs * 4, LSTM_THREADS, Cfg::SMEM, st>>>(a);
    return cudaGetLastError();
}

// split-precision products of the L4 GEMM as a bit mask: 1 = A_hi*B_hi, 2 = A_lo*B_hi, 4 = A_hi*B_lo.
// C3R_L4_TERMS overrides for experiments (tools/l4_terms_probe.sh).
inline int l4_terms() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("C3R_L4_TERMS");
        v = e ? atoi(e) : 7;
        if (v < 1 || v > 7 || !(v & 1)) v = 7;
    }
    return v;
}

inline cudaError_t launch_gemm(const GemmArgs& g, int sm_count, cudaStream_t st) {
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(k_gemm_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM);
        if (e != cudaSuccess) return e;
        attr = true;
    }
    int grid = g.m_tiles * g.n_tiles * (g.ksplit > 1 ? g.ksplit : 1);
    if (grid > sm_count) grid = sm_count;
    k_gemm_tc<<<grid, GEMM_THREADS, GEMM_SMEM, st>>>(g);
    return cudaGetLastError();
}

// tensor int32 [n,33,C] (device) -> probs [n,24] (device).  Returns kernel launches, <0 on error.
//
// Work items of the recurrent kernels are (256-site tile pair, direction) on one CTA pair each, so a pass whose
// item count is not a multiple of the 74 CTA pairs leaves SMs idle in its last round (116 items at 14.6 k sites:
// the second round is 57 % full).  A pass follows a plan of nn_sched.h: either rounds (LSTM1; LSTM2 as A, the full
// rounds, and B, the rest, with the L4 GEMM + heads of A on a second stream beside B: one-tile-per-CTA kernels
// that take the SMs B leaves idle) or two groups of SMs on the two streams, where LSTM1 waves of one group run
// beside LSTM2 of the other.
struct TcPipe {
    cudaStream_t s2 = nullptr;
    cudaEvent_t ev[8] = {};              // ev[i]: launch i of the pass's plan has ended
    cudaEvent_t fork = nullptr;          // the second stream starts after the buffer waits of the caller's stream
    // Passes of different tickets run on different streams but share the scratch buffers.  A pass may write h2 / l4
    // once the previous pass has ended (pass_done).  (An event that was never recorded does not block.)
    cudaEvent_t pass_done = nullptr;
    // h1 is double-buffered (TcNet::h1[2]), so LSTM1 of the NEXT pass can run on the SMs the last LSTM2 launch of
    // this pass leaves idle (its remainder round: 84 of 148 SMs at config 2).
    // h1_free2[b]: LSTM2 has read buffer b;  xop_free: LSTM1 has read the shared operand image;
    // last_ready: every LSTM2 launch of the previous pass but the one that ends last has ended;  last_done: all have;
    // last_pairs: the cluster pairs of the one that ends last;  last_split: the previous pass ran in two groups.
    cudaEvent_t h1_free2[2] = {}, xop_free = nullptr, last_ready = nullptr, last_done = nullptr;
    int last_pairs = 0, parity = 0;
    bool last_split = false;
    long n_pass = 0, n_overlap = 0;      // passes queued / passes whose LSTM1 went in pieces beside the previous pass (C3R_TIMING)
    bool ok = false;
};
inline int tc_pipe_init(TcPipe& p, std::string* err) {
    if (p.ok) return 0;
    int prio_lo = 0, prio_hi = 0;                    // the network's streams are high priority (c3r_create)
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    // the second stream (L4 + heads of the full rounds, beside LSTM2's remainder round) is high priority as well
    cudaError_t e = cudaStreamCreateWithPriority(&p.s2, cudaStreamNonBlocking, getenv("C3R_FLAT_PRIORITY") ? prio_lo : prio_hi);
    for (int i = 0; i < 8 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&p.ev[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p.fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p.pass_done, cudaEventDisableTiming);
    for (cudaEvent_t* ev : {&p.h1_free2[0], &p.h1_free2[1], &p.xop_free, &p.last_ready, &p.last_done})
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming);
    if (e != cudaSuccess) { *err = std::string("pipeline streams: ") + cudaGetErrorString(e); return -1; }
    p.ok = true;
    return 0;
}
inline void tc_pipe_release(TcPipe* p) {
    if (p->s2) cudaStreamDestroy(p->s2);
    for (cudaEvent_t e : p->ev) if (e) cudaEventDestroy(e);
    if (p->fork) cudaEventDestroy(p->fork);
    if (p->pass_done) cudaEventDestroy(p->pass_done);
    for (cudaEvent_t ev : {p->h1_free2[0], p->h1_free2[1], p->xop_free, p->last_ready, p->last_done}) if (ev) cudaEventDestroy(ev);
    delete p;
}

// tiles [t0, t0 + nt) of the pass, sites [s0, s0 + ns)
struct TcSub { int t0, nt; int64_t s0, ns; };

inline cudaError_t tc_lstm2(TcNet& t, const TcSub& b, int max_pairs, cudaStream_t st, const __half* h1buf) {
    Lstm2fArgs f;
    f.wstream = t.wstream2; f.h1 = h1buf + (size_t)b.t0 * NT * 4 * TC_IMG;
    f.hout = t.h2 + (size_t)b.t0 * NT * 5 * TC_IMG;
    f.hout_lo = (l4_terms() & 2) ? t.h2_lo + (size_t)b.t0 * NT * 5 * TC_IMG : nullptr;
    f.n_tiles = b.nt; f.err = t.err;
    f.prof = (t.trace && b.t0 == 0) ? t.trace + 2 * NT * 8 * 8 : nullptr;   // C3R_TRACE: wait-time totals of cluster 0 (LSTM2's part of the trace buffer)
    return launch_lstm2f(f, t.sm_count, max_pairs / lstm2f_np(), st);
}
inline cudaError_t tc_l4_heads(TcNet& t, const NetF32& net, const TcSub& b, float* probs, cudaStream_t st) {
    GemmArgs g4;
    g4.A = t.h2 + (size_t)b.t0 * NT * 5 * TC_IMG; g4.B = t.k4p; g4.A_lo = t.h2_lo + (size_t)b.t0 * NT * 5 * TC_IMG; g4.B_lo = t.k4p_lo;
    // K = 10560 always goes in L4_KSPLIT ranges (partial sums added up by k_l4_finish): a remainder launch of a few dozen
    // tiles still fills the SMs, and the summation order is the same whatever the batch size
    g4.terms = l4_terms(); g4.bias = t.b4; g4.out = t.l4p + (size_t)b.t0 * 128 * DENSE; g4.m_tiles = b.nt; g4.n_tiles = 1; g4.n_kb = L4_IN / TC_KB;
    g4.ksplit = L4_KSPLIT; g4.split_stride = t.l4_stride; g4.err = t.err;
    cudaError_t e = launch_gemm(g4, t.sm_count, st);
    if (e != cudaSuccess) return e;
    // l4 = selu(sum of the partial sums + bias) as fp16 operand images; [L5_1 | L5_2] as one tensor-core GEMM
    // (N = 256, K = 128, split precision, + bias + SELU); the two small output layers and the softmax per site
    k_l4_finish<<<b.nt * 4, 128, 0, st>>>(t.l4p + (size_t)b.t0 * 128 * DENSE, L4_KSPLIT, t.l4_stride, t.b4,
                                      t.l4 + (size_t)b.t0 * 128 * DENSE, t.l4h + (size_t)b.t0 * 2 * TC_IMG, t.l4h_lo + (size_t)b.t0 * 2 * TC_IMG);
    GemmArgs g5;
    g5.A = t.l4h + (size_t)b.t0 * 2 * TC_IMG; g5.A_lo = t.l4h_lo + (size_t)b.t0 * 2 * TC_IMG; g5.B = t.k5p; g5.B_lo = t.k5p_lo;
    g5.terms = 7; g5.bias = t.b5p; g5.out = t.a5 + (size_t)b.t0 * 128 * 256; g5.m_tiles = b.nt; g5.n_tiles = 2; g5.n_kb = 2;
    g5.ksplit = 1; g5.split_stride = 0; g5.err = t.err;
    e = launch_gemm(g5, t.sm_count, st);
    if (e != cudaSuccess) return e;
    {
        int64_t blocks = (b.ns + HOUT_WARPS - 1) / HOUT_WARPS;
        if (blocks > (int64_t)t.sm_count * 4) blocks = (int64_t)t.sm_count * 4;
        if (blocks > 0) k_heads_out<<<(unsigned)blocks, HOUT_WARPS * 32, 0, st>>>(net, t.a5 + (size_t)b.t0 * 128 * 256, probs + b.s0 * 24, b.ns);
    }
    return cudaGetLastError();
}

// `xop_ready`: LSTM1's operand images of all n sites, already built by k_window_xop (then `tensor` is not read)
inline int tc_forward(TcNet& t, const NetF32& net, const int32_t* tensor, int64_t n, float* probs, cudaStream_t st,
                      std::string* err, const __half* xop_ready = nullptr) {
    if (!t.ready) { *err = "weights not packed"; return -1; }
    if (!t.pipe) t.pipe = new TcPipe();
    if (tc_pipe_init(*t.pipe, err)) return -1;
    TcPipe& P = *t.pipe;
    int launches = 0;
#define TCK(call, what) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { *err = std::string(what) + ": " + cudaGetErrorString(e__); return -1; } } while (0)
    // a batch larger than the scratch goes through in sub-passes of whole rounds of the recurrent kernels
    // (sm_count / 4 cluster pairs x 2 tiles each), so that only the last sub-pass has a partly filled round
    const int round_tiles = 2 * (t.sm_count / 4) > 0 ? 2 * (t.sm_count / 4) : 2;
    const int sub_tiles = TC_SUB_TILES >= round_tiles ? (TC_SUB_TILES / round_tiles) * round_tiles : TC_SUB_TILES;
    for (int64_t o = 0; o < n; o += (int64_t)sub_tiles * TC_TILE) {
        const int64_t m = n - o < (int64_t)sub_tiles * TC_TILE ? n - o : (int64_t)sub_tiles * TC_TILE;
        int tiles = (int)((m + TC_TILE - 1) / TC_TILE);
        tiles += tiles & 1;                  // CTA pairs
        if (tc_ensure(t, tiles, err)) return -1;
        const int hb = P.parity;                                    // h1 buffer of this pass
        P.parity ^= 1;
        __half* const h1buf = t.h1[hb];
        t.h1_cur = h1buf;
        TCK(cudaStreamWaitEvent(st, P.h1_free2[hb], 0), "wait");   // LSTM2 of the pass before the previous one has read this buffer
        if (!xop_ready) TCK(cudaStreamWaitEvent(st, P.xop_free, 0), "wait");   // LSTM1 of the previous pass has read the shared image
        const __half* xop_in = t.xop;
        if (xop_ready) xop_in = xop_ready + (size_t)(o / TC_TILE) * NT * (size_t)(t.KX * TC_TILE);
        else {
            if (t.C == 18) k_xop<18, lstm1_kx(18)><<<tiles * NT, TC_TILE, 0, st>>>(tensor + o * NT * t.C, t.xop, m);
            else k_xop<30, lstm1_kx(30)><<<tiles * NT, TC_TILE, 0, st>>>(tensor + o * NT * t.C, t.xop, m);
            ++launches;
        }
        const int pairs = tiles / 2;
        const int slots = t.sm_count / 4 > 0 ? t.sm_count / 4 : 1;          // tile pairs the recurrent kernels hold at once
        // tile pairs one round of the LSTM2 kernel takes (clusters of 2*NP CTAs, half of them per direction)
        const int per_round = (t.sm_count / (2 * lstm2f_np()) / 2) * lstm2f_np();
        auto lstm1 = [&](const TcSub& b, int cap, cudaStream_t s) -> cudaError_t {
            LstmArgs a1;
            a1.Wimg = t.img1; a1.xop = xop_in + (size_t)b.t0 * NT * t.KX * TC_TILE;
            a1.hout = h1buf + (size_t)b.t0 * NT * 4 * TC_IMG;
            a1.n_sites = b.ns; a1.n_tiles = b.nt; a1.err = t.err; a1.trace = b.t0 == 0 ? t.trace : nullptr;
            return t.C == 18 ? launch_lstm<4, lstm1_kx(18)>(a1, t.sm_count, cap, s) : launch_lstm<4, lstm1_kx(30)>(a1, t.sm_count, cap, s);
        };
        // The last LSTM2 launch of the pass before this one leaves sm_count - 4 x last_pairs SMs idle: while it is
        // still ahead of us, LSTM1 of THIS pass goes beside it.  After a pass of rounds (its remainder round, or its
        // only round) LSTM1 goes in pieces that fit - two pieces (an LSTM1 round takes less than half an LSTM2
        // round), then the rest once it has ended.  At config 2 (37 + 21 tile pairs): 16 + 16 pairs of LSTM1 run
        // under the previous pass's remainder round and the remaining 26 are ONE round instead of two; a 5 Mb chunk
        // of config 5 (20 pairs, one partly filled round) puts all of its LSTM1 beside the previous chunk's LSTM2.
        // After a pass in two groups, the last LSTM2 launch ends soon after the other group's: LSTM1 goes as one
        // launch that starts on the SMs that group released and takes the rest as the last launch ends.
        // Such a pass runs its LSTM2 in rounds.
        const int ip = (t.sm_count - 4 * P.last_pairs) / 4;         // tile pairs (both directions) that fit beside it
        bool overlap = o == 0 && P.last_pairs > 0 && ip >= 8 && getenv("C3R_NO_LSTM1_OVERLAP") == nullptr;
        if (overlap) {
            overlap = cudaEventQuery(P.last_done) == cudaErrorNotReady;
            (void)cudaGetLastError();
        }
        auto piece = [&](int p0, int np) {
            TcSub b; b.t0 = 2 * p0; b.nt = 2 * np; b.s0 = (int64_t)b.t0 * TC_TILE;
            const int64_t left = m - b.s0;
            b.ns = left < 0 ? 0 : left < (int64_t)b.nt * TC_TILE ? left : (int64_t)b.nt * TC_TILE;
            return b;
        };
        // C3R_PASS_SCHEDULE=rounds: every pass in rounds
        const char* ps = getenv("C3R_PASS_SCHEDULE");
        const SchedPlan plan = overlap || (ps && strcmp(ps, "rounds") == 0) ? sched_rounds(pairs, slots, per_round)
                                                                            : sched_plan(pairs, slots, per_round, lstm2f_np());
        ++P.n_pass;
        int first = 0;                                                  // plan launches already issued
        if (overlap) {
            ++P.n_overlap;
            TCK(cudaStreamWaitEvent(st, P.last_ready, 0), "wait");
            if (P.last_split) {
                TCK(lstm1(piece(0, pairs), slots, st), "lstm1");
            } else {
                int done = 0;
                for (int c = 0; c < 2 && done < pairs; ++c) {
                    const int np = pairs - done < ip ? pairs - done : ip;
                    TCK(lstm1(piece(done, np), slots, st), "lstm1");
                    done += np; ++launches;
                }
                if (done < pairs) {
                    TCK(cudaStreamWaitEvent(st, P.last_done, 0), "wait");
                    TCK(lstm1(piece(done, pairs - done), slots, st), "lstm1");
                } else --launches;                                      // (counted with the plan's launch below)
            }
            TCK(cudaEventRecord(P.ev[0], st), "event");
            first = 1;                                                  // in place of the plan's LSTM1 (launch 0)
            ++launches;
        }
        cudaStream_t ss[2] = {st, P.s2};
        TCK(cudaEventRecord(P.fork, st), "event");
        TCK(cudaStreamWaitEvent(P.s2, P.fork, 0), "wait");
        // the last launch of `kind` on stream `s` listed before launch i, or -1
        auto last_of = [&](int kind, int s, int i) {
            int r = -1;
            for (int j = 0; j < i; ++j) if (plan.l[j].kind == kind && plan.l[j].stream == s) r = j;
            return r;
        };
        int l1_last = -1, l2_last = -1, l2_prev = -1, s2_last = -1;
        for (int i = 0; i < plan.n; ++i) {
            if (plan.l[i].kind == SCHED_LSTM1) l1_last = i;
            if (plan.l[i].kind == SCHED_LSTM2) { l2_prev = l2_last; l2_last = i; }
            if (plan.l[i].stream == 1) s2_last = i;
        }
        bool h2_free[2] = {false, false};                               // stream waited for pass_done
        float* pr = probs + o * 24;
        for (int i = 0; i < plan.n; ++i) {
            const SchedLaunch& L = plan.l[i];
            cudaStream_t s = ss[L.stream];
            const int other = L.stream ^ 1;
            if (L.wait >= 0) TCK(cudaStreamWaitEvent(s, P.ev[L.wait], 0), "wait");
            if (L.kind == SCHED_LSTM2 && !h2_free[L.stream]) {
                TCK(cudaStreamWaitEvent(s, P.pass_done, 0), "wait");   // the previous pass no longer reads h2 / l4
                h2_free[L.stream] = true;
            }
            if (i == l2_last && l2_prev < 0) TCK(cudaEventRecord(P.last_ready, s), "event");
            if (i >= first) {
                if (L.kind == SCHED_LSTM1) TCK(lstm1(piece(L.p0, L.np), L.cap, s), "lstm1");
                else if (L.kind == SCHED_LSTM2) TCK(tc_lstm2(t, piece(L.p0, L.np), L.cap, s, h1buf), "lstm2");
                else { TCK(tc_l4_heads(t, net, piece(L.p0, L.np), pr, s), "l4/heads"); launches += 3; }
                ++launches;
                TCK(cudaEventRecord(P.ev[i], s), "event");
            }
            // the shared operand image is free once every LSTM1 launch has read it; LSTM2 of the pass has read h1
            // (and its last launch has ended) once every LSTM2 launch has ended
            const int kind_last = i == l1_last ? SCHED_LSTM1 : i == l2_last || i == l2_prev ? SCHED_LSTM2 : -1;
            if (kind_last >= 0) {
                const int j = last_of(kind_last, other, i);
                if (j >= 0) TCK(cudaStreamWaitEvent(s, P.ev[j], 0), "wait");
            }
            if (i == l1_last) TCK(cudaEventRecord(P.xop_free, s), "event");
            if (i == l2_prev) TCK(cudaEventRecord(P.last_ready, s), "event");
            if (i == l2_last) {
                TCK(cudaEventRecord(P.last_done, s), "event");
                TCK(cudaEventRecord(P.h1_free2[hb], s), "event");
                P.last_pairs = L.np < L.cap ? L.np : L.cap;
                P.last_split = plan.split != 0;
            }
        }
        if (s2_last >= 0) TCK(cudaStreamWaitEvent(st, P.ev[s2_last], 0), "wait");   // the caller's stream ends after everything
        TCK(cudaEventRecord(P.pass_done, st), "event");
    }
#undef TCK
    return launches;
}

// device-side protocol errors (bounded mbarrier waits) surface here
inline int tc_check_error(TcNet& t, cudaStream_t st, int* code) {
    int h[1] = {0};
    if (!t.err) { *code = 0; return 0; }
    cudaError_t e = cudaMemcpyAsync(h, t.err, 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return -1;
    *code = h[0];
    if (h[0]) cudaMemsetAsync(t.err, 0, 4, st);
    return 0;
}

}  // namespace c3r
