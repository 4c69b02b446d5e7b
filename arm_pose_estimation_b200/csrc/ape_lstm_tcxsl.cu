// Stage 2, SPLIT PRECISION for a SMALL batch at H = 256: all L layers of the MC-dropout LSTM in ONE launch, one cluster of 16 CTAs
// per 128 rows with the hidden units split across the cluster - the structure of ape_lstm_tcxl.cu (H = 128) with the arithmetic of the
// H = 256 split layer kernel (ape_lstm_tcxs.cu).
//
// A watch-only or pocket model whose weights fail the single-pass probe runs on the split layer kernels, where one CTA pair walks all
// eight 32-unit chunks of a layer, T x L dependent steps in a row, 776 MMAs per step.  Here CTA k owns the 16 units [16 k, 16 k + 16)
// of every layer - slot (k & 1, k >> 1) of the tcx blob (slot (r, c) holds the units 32 c + 16 r .. + 15), its four pieces Wx_hi
// (+ the bias K step), Wx_lo, Wh_hi, Wh_lo resident in shared memory for the layer (130 KB for a layer >= 1).  The 8-CTA plan of
// tcxl does not fit at H = 256 (one CTA's weights alone would be 256 KB); with 16 CTAs the weights and h_hi / h_lo still come to
// 258 KB of shared memory, so one operand tile moves to tensor memory:
//   * shared memory: the weight slot 130 KB + h_hi of all units 64 KB (pulled each step from the L2 exchange buffer with one bulk
//     copy) + the ones tile of the bias K step 4 KB + the barrier block = 198 KB;
//   * tensor memory (512 columns): accumulator 64, x_hi / x_lo SINGLE-buffered 2 x 128, h_lo 128, output product 64.  x_{t+1} is built
//     as soon as the x-part MMAs of step t have completed (BAR_XFREE: every x-part MMA of a step precedes its h-part); h_lo of h_{t-1}
//     is written by the loader warps (ld.global.cg + tcgen05.st, k-groups 0..15 first: the MMA order reads them first) after the
//     cluster barrier that ends step t-1 - by then the accumulator of step t-1 was drained, so every MMA that read h_{t-2} has retired;
//   * per accumulator the MMAs run in tcxs's order, 16-k-group pieces: x_hi[0:16], x_lo[0:16] x Wx_hi piece 0; x_hi[16:32], ones,
//     x_lo[16:32] x Wx_hi piece 1; x_hi x Wx_lo; then h_hi[0:16], h_lo[0:16], h_hi[16:32], h_lo[16:32] x Wh_hi; h_hi x Wh_lo
//     (cta_group::1 with M = 128, N = 64), and the epilogue is tcxs's (ex2 / rcp cell, the same split points, the output layer as hi
//     product + remainder product + b_o), so the results are bit-identical to the layer kernels.
// Cluster c takes rows [128 c, 128 c + 128) of the layers >= 1 and layer 0 of the estimates those rows belong to (an estimate that
// straddles two clusters has its layer 0 computed by both).  A 16-CTA cluster is a non-portable size: the launch opts in.
#include "ape_common.cuh"
#include "ape_lstm_pack.h"
#include "ape_lstm_tc_args.cuh"
#include "ape_umma.cuh"
#include "ape_f32x2.cuh"

#include <atomic>

namespace ape {
namespace tcxsl {

constexpr int H = 256, KG = H / 8, NCHL = H / 32, NCTA = 16, NU = H / NCTA, NCOL = 4 * NU, ROWS = 128, MAX_L = 4, MAX_CLUSTERS = 64;
// 8 epilogue warps (two per TMEM lane quarter, one k-group = 8 units each), 12 loader warps (three per quarter), one controller warp
constexpr int EPI_WARPS = 8, LOAD_PARTS = 3, LOAD_WARPS = 4 * LOAD_PARTS, THREADS = (EPI_WARPS + LOAD_WARPS + 1) * 32;
constexpr int CTRL_WARP = EPI_WARPS + LOAD_WARPS;
constexpr int PIECE_KG = 16;                               // tcxs's weight pieces: the unit of its MMA order
constexpr uint32_t KG_BYTES_B = NCOL * 16;                 // one k-group of a 64-column weight piece
constexpr uint32_t PH_BYTES = KG * KG_BYTES_B;             // Wh_hi or Wh_lo
__host__ __device__ constexpr uint32_t p0_bytes(int kgx) { return (uint32_t)(kgx + 2) * KG_BYTES_B; }   // Wx_hi + bias K step
__host__ __device__ constexpr uint32_t p1_bytes(int kgx) { return (uint32_t)kgx * KG_BYTES_B; }         // Wx_lo
__host__ __device__ constexpr uint32_t chunk_bytes(int kgx) { return p0_bytes(kgx) + p1_bytes(kgx) + 2 * PH_BYTES; }
constexpr uint32_t W_BYTES = chunk_bytes(KG);              // 130 KB: a slot of a layer >= 1 (the largest)
constexpr uint32_t H_BYTES = KG * ROWS * 16;               // one h operand tile (64 KB)
constexpr uint32_t ONES_BYTES = 2 * ROWS * 16;             // A operand of the bias K step
constexpr int NO = 32;                                     // columns of an output tile (O <= 32)
constexpr uint32_t OT_BYTES = KG * NO * 16;
constexpr uint32_t BAR_BLOCK_BYTES = 128;                 // the mbarriers, then the TMEM base address tcgen05.alloc writes
constexpr uint32_t SMEM = W_BYTES + H_BYTES + ONES_BYTES + BAR_BLOCK_BYTES;
constexpr uint32_t ACC_COL = 0, XH_COL = 64, XL_COL = XH_COL + H / 2, HL_COL = XL_COL + H / 2, OUT_COL = HL_COL + H / 2, TMEM_COLS = 512;
static_assert(SMEM <= 227 * 1024, "shared memory budget");
static_assert(ACC_COL + NCOL <= XH_COL && OUT_COL + 2 * NO <= TMEM_COLS, "tensor memory plan");
static_assert(2 * OT_BYTES <= W_BYTES, "the output tiles take the weights' place");
constexpr float NEG2LOG2E = -2.0f * 1.4426950408889634f;   // accumulator -> ex2 argument (i, f, o weights are stored halved)

struct Args {
    const uint8_t* W[MAX_L];        // layer l of the split blob: [pair cta 2][chunk H/32][Wx_hi + bias | Wx_lo | Wh_hi | Wh_lo]
    int kgx[MAX_L];
    int L, T, I, E, n, nF, frame0, feat_ring, dense;
    const float* in;                // feature ring [B][feat_ring][I] or dense windows [E][T][I]
    const int32_t* stream_frames;
    int mask_mode;
    const uint8_t* masks;           // injected: [E][L-1][T][n][H]
    PhiloxRoundKeys rk;
    uint32_t stream_id0, keep_thr16;
    float scale;                    // 1 / (1 - p) (1 with no dropout): applied to a layer's output sequence BEFORE the split
    uint4* hx;                      // [2][hi | lo][H/8][128] exchange buffer of h_t (operand layout), by step parity
    uint4* seq;                     // [2][T][hi | lo][H/8][128] a layer's output sequence (the next layer's input), by layer parity
    size_t ws_stride;               // uint4s between the hx / seq buffers of consecutive clusters
    const uint8_t* Wo16;            // [2][H/8][32][8]: fp16(W_o), remainder
    const float* bo;
    int O;
    float* preds;
    int pred_ring;
};

enum { BAR_W = 0, BAR_X = 1, BAR_XFREE = 2, BAR_ACC = 3, BAR_H = 4, BAR_HLO = 5, BAR_OUT = 7, BAR_COUNT = 8 };   // BAR_HLO + half
static_assert(BAR_COUNT * 8 + 16 <= BAR_BLOCK_BYTES, "barrier block too small");

// v -> fp16 pair: hi = fp16(v), lo = fp16(v - hi), for two values at once (ape_lstm_tcxs.cu)
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn(a, b);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

__device__ __forceinline__ uint4 and4(uint4 v, uint4 m) { return make_uint4(v.x & m.x, v.y & m.y, v.z & m.z, v.w & m.w); }

__global__ void __launch_bounds__(THREADS, 1) lstm_small_tcxs_kernel(const __grid_constant__ Args a) {
    using namespace umma;
    constexpr uint32_t LBO_A = ROWS * 16, LBO_B = KG_BYTES_B, SBO = 128;

    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* sW = smem;                                  // this CTA's slot of the layer (the output tiles at the very end)
    uint8_t* sH = sW + W_BYTES;                          // [KG][ROWS] units: h_hi of h_{t-1}, ALL units
    uint8_t* sOnes = sH + H_BYTES;                       // [2][ROWS] units
    uint64_t* bars = reinterpret_cast<uint64_t*>(sOnes + ONES_BYTES);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + BAR_COUNT);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    const int T = a.T, L = a.L;
    const int cid = (int)(blockIdx.x / NCTA);
    const int r0 = cid * ROWS;
    const int rows1 = min(ROWS, a.E * a.n - r0);
    const int e_lo = r0 / a.n, rows0 = (r0 + rows1 - 1) / a.n - e_lo + 1;
    uint4* const hx = a.hx + (size_t)cid * a.ws_stride;
    uint4* const seq = a.seq + (size_t)cid * a.ws_stride;

    for (int i = tid; i < 2 * ROWS; i += THREADS)
        reinterpret_cast<uint4*>(sOnes)[i] = make_uint4(i < ROWS ? 0x3C003C00u : 0u, 0u, 0u, 0u);
    if (warp == CTRL_WARP) {
        tmem_alloc<1>(tmem_slot, TMEM_COLS);
        tmem_relinquish<1>();
    }
    if (tid == 0) {
        mbar_init(&bars[BAR_W], 1);
        mbar_init(&bars[BAR_X], LOAD_WARPS);
        mbar_init(&bars[BAR_XFREE], 1);
        mbar_init(&bars[BAR_ACC], 1);
        mbar_init(&bars[BAR_H], 1);
        mbar_init(&bars[BAR_HLO], LOAD_WARPS);
        mbar_init(&bars[BAR_HLO + 1], LOAD_WARPS);
        mbar_init(&bars[BAR_OUT], 1);
        mbar_init_fence();
    }
    fence_proxy_async_smem();
    fence_before_sync();
    cluster_sync();
    fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    uint32_t ph_w = 0, ph_x = 0, ph_xf = 0, ph_acc = 0, ph_h = 0, ph_hlo = 0;

    for (int l = 0; l < L; ++l) {
        const int kgx = a.kgx[l];
        const bool last_layer = l == L - 1;
        const int rows = l == 0 ? rows0 : rows1;
        // after step t, h_t goes on to the other CTAs (the last step's h only feeds the output layer, on CTA 0)
        auto pull = [&](int t) { return t + 1 < T || (last_layer && a.preds && rank == 0); };
        // ---- this CTA's slot of layer l -> shared memory (every MMA of the previous layer has completed: see the barrier below) ----
        if (warp == CTRL_WARP && lane == 0) {
            const uint32_t cb = chunk_bytes(kgx);
            mbar_arrive_expect_tx(&bars[BAR_W], cb);
            bulk_g2s(sW, a.W[l] + ((size_t)(rank & 1) * NCHL + (rank >> 1)) * cb, cb, &bars[BAR_W]);
        }

        if (warp < EPI_WARPS) {
            // =================================== epilogue warps: row = TMEM lane = 32 (warp & 3) + lane, k-group b8 = warp >> 2 ===
            const int row = 32 * (warp & 3) + lane, b8 = warp >> 2;
            const uint32_t t_lane = (uint32_t)(32 * (warp & 3)) << 16;
            float cst[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) cst[u] = 0.0f;
            for (int t = 0; t < T; ++t) {
                mbar_wait_wd(&bars[BAR_ACC], ph_acc); ph_acc ^= 1;
                fence_after_sync();
                const bool exchange = t + 1 < T || (last_layer && a.preds);
                const size_t kg = (size_t)(rank * (NU / 8) + b8);                 // this warp's k-group of h_t
                uint4* hx_dst = hx + (size_t)(t & 1) * 2 * KG * ROWS + kg * ROWS + row;
                uint4* seq_dst = seq + ((size_t)(l & 1) * T + t) * 2 * KG * ROWS + kg * ROWS + row;
                uint32_t r[32];
                tmem_ld_x32(tmem + t_lane + ACC_COL + 32 * b8, r);
                tmem_ld_wait();
                float hv[8];
#pragma unroll
                for (int u = 0; u < 8; u += 2) {
                    // ex2 arguments of units u, u + 1 (the bias is in the accumulator), gate g of both in one pair
                    auto arg = [&](int g) { return pk(__uint_as_float(r[4 * u + g]), __uint_as_float(r[4 * u + 4 + g])) * splat(NEG2LOG2E); };
                    F2 c2 = pk(cst[u], cst[u + 1]), h2;
                    tc::lstm_cell2(arg(0), arg(1), arg(2), arg(3), c2, h2);
                    cst[u] = lo(c2); cst[u + 1] = hi(c2);
                    hv[u] = lo(h2); hv[u + 1] = hi(h2);
                }
                // h_t as fp16 pairs: as is for the recurrence, scaled by the consumer's 1 / (1 - p) BEFORE the split for the next layer
                if (exchange) {
                    uint32_t hi[4], lo[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) split2(hv[2 * k], hv[2 * k + 1], hi[k], lo[k]);
                    hx_dst[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                    hx_dst[(size_t)KG * ROWS] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                }
                if (!last_layer) {
                    uint32_t hi[4], lo[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) split2(hv[2 * k] * a.scale, hv[2 * k + 1] * a.scale, hi[k], lo[k]);
                    seq_dst[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                    seq_dst[(size_t)KG * ROWS] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                }
                fence_before_sync();
                cluster_sync();                            // every slice of h_t (and of the layer's sequence) is written, every MMA of step t done
            }
            if (last_layer && a.preds && rank == 0 && b8 == 0) {      // output_layer (nn_models.py:189) on the last step, CTA 0
                mbar_wait_wd(&bars[BAR_OUT], 0);
                fence_after_sync();
                const bool valid = row < rows;
                const int e = valid ? (r0 + row) / a.n : 0, smp = r0 + row - e * a.n;
                const int bb = e / a.nF, fb = valid ? stream_frame0(a.stream_frames, a.frame0, bb) : -1, f = fb + e % a.nF;
                float* dst = a.preds + (fb >= 0 ? ((((size_t)bb * a.pred_ring + f % a.pred_ring) * a.n) + smp) * a.O : 0);
#pragma unroll
                for (int k0 = 0; k0 < NO; k0 += 16) {      // outputs k0 .. k0 + 15
                    uint32_t oh[16], orem[16];             // h_T(hi, lo) x fp16(W_o)^T, h_T(hi, lo) x (W_o - fp16(W_o))^T
                    tmem_ld_x16(tmem + t_lane + OUT_COL + k0, oh);
                    tmem_ld_x16(tmem + t_lane + OUT_COL + NO + k0, orem);
                    tmem_ld_wait();
                    if (fb >= 0) {                         // (an inactive stream keeps its prediction ring untouched)
#pragma unroll
                        for (int k = 0; k < 16; ++k)
                            if (k0 + k < a.O) dst[k0 + k] = __uint_as_float(oh[k]) + __uint_as_float(orem[k]) + __ldg(a.bo + k0 + k);
                    }
                }
                fence_before_sync();
            }
        } else if (warp < CTRL_WARP) {
            // =================================== loader warps: x_hi, x_lo and h_lo of every row -> TMEM ======================
            const int lw = warp & 3, part = (warp - EPI_WARPS) >> 2, row = 32 * lw + lane;
            const uint32_t t_lane = (uint32_t)(32 * lw) << 16;
            const bool valid = row < rows;
            const int e = valid ? (l == 0 ? e_lo + row : (r0 + row) / a.n) : 0, smp = (valid && l > 0) ? r0 + row - e * a.n : 0;
            const int bidx = e / a.nF, f = stream_frame0(a.stream_frames, a.frame0, bidx) + e % a.nF;
            const uint32_t stream = a.stream_id0 + (uint32_t)bidx;
            constexpr int NJ = (PIECE_KG + LOAD_PARTS - 1) / LOAD_PARTS;    // this warp's k-groups of a 16-k-group half: part, part + 3, ...
            // x_t -> the x buffer (single: its previous contents, x_{t-1}, were read by the x-part MMAs of step t-1, complete by now)
            auto build_x = [&](int t) {
                const uint32_t xh = tmem + t_lane + XH_COL, xl = tmem + t_lane + XL_COL;
                if (l == 0) {
                    const float* src = nullptr;
                    if (valid) {
                        if (a.dense) src = a.in + ((size_t)e * T + t) * a.I;
                        else {                             // sliding window, clamped at frame 0 (estimator.py:96-97)
                            int fw = f - T + 1 + t;
                            fw = fw < 0 ? 0 : fw;
                            src = a.in + ((size_t)bidx * a.feat_ring + fw % a.feat_ring) * a.I;
                        }
                    }
                    for (int j = part; j < kgx; j += LOAD_PARTS) {
                        float v[8];
#pragma unroll
                        for (int k = 0; k < 8; ++k) v[k] = (valid && 8 * j + k < a.I) ? __ldg(src + 8 * j + k) : 0.0f;
                        uint32_t hi[4], lo[4];
#pragma unroll
                        for (int k = 0; k < 4; ++k) split2(v[2 * k], v[2 * k + 1], hi[k], lo[k]);
                        tmem_st_x4(xh + 4 * j, hi[0], hi[1], hi[2], hi[3]);
                        tmem_st_x4(xl + 4 * j, lo[0], lo[1], lo[2], lo[3]);
                    }
                } else {
                    // the previous layer's h_t (hi, lo: scaled by 1 / (1 - p)) of this row's estimate, one dropout mask ANDed into both
                    const uint4* src = seq + ((size_t)((l - 1) & 1) * T + t) * 2 * KG * ROWS + (l == 1 ? e - e_lo : row);
#pragma unroll
                    for (int half = 0; half < 2; ++half) {
                        uint4 vh[NJ], vl[NJ];
#pragma unroll
                        for (int jj = 0; jj < NJ; ++jj) {                        // every L2 load of the half goes out first
                            const int j = PIECE_KG * half + LOAD_PARTS * jj + part;
                            const bool ld = valid && LOAD_PARTS * jj + part < PIECE_KG;
                            vh[jj] = ld ? __ldcg(src + (size_t)j * ROWS) : make_uint4(0, 0, 0, 0);
                            vl[jj] = ld ? __ldcg(src + (size_t)(KG + j) * ROWS) : make_uint4(0, 0, 0, 0);
                        }
#pragma unroll
                        for (int jj = 0; jj < NJ; ++jj) {
                            if (LOAD_PARTS * jj + part >= PIECE_KG) break;
                            const int j = PIECE_KG * half + LOAD_PARTS * jj + part;
                            uint4 m = make_uint4(~0u, ~0u, ~0u, ~0u);
                            if (a.mask_mode == APE_MASK_PHILOX) {
                                m = philox_keep_halfmask_rk(a.rk, stream, (uint32_t)f, (uint32_t)smp, (uint32_t)(l - 1), (uint32_t)t, (uint32_t)j,
                                                            a.keep_thr16);
                            } else if (a.mask_mode == APE_MASK_INJECTED && valid) {
                                const uint2 mm = __ldg(reinterpret_cast<const uint2*>(
                                    a.masks + ((((size_t)e * (L - 1) + (l - 1)) * T + t) * a.n + smp) * H + j * 8));
                                m.x = ((mm.x & 0xFFu) ? 0xFFFFu : 0u) | ((mm.x & 0xFF00u) ? 0xFFFF0000u : 0u);
                                m.y = ((mm.x & 0xFF0000u) ? 0xFFFFu : 0u) | ((mm.x & 0xFF000000u) ? 0xFFFF0000u : 0u);
                                m.z = ((mm.y & 0xFFu) ? 0xFFFFu : 0u) | ((mm.y & 0xFF00u) ? 0xFFFF0000u : 0u);
                                m.w = ((mm.y & 0xFF0000u) ? 0xFFFFu : 0u) | ((mm.y & 0xFF000000u) ? 0xFFFF0000u : 0u);
                            }
                            const uint4 h = and4(vh[jj], m), o = and4(vl[jj], m);
                            tmem_st_x4(xh + 4 * j, h.x, h.y, h.z, h.w);
                            tmem_st_x4(xl + 4 * j, o.x, o.y, o.z, o.w);
                        }
                    }
                }
                tmem_st_wait();
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars[BAR_X]);
            };
            // h_lo of h_t (all units, this row) from the exchange buffer -> TMEM, in two halves of 16 k-groups, each published on its
            // own barrier (the h-part MMAs read k-groups 0..15 first)
            auto load_hlo = [&](int t) {
                const uint4* src = hx + (size_t)(t & 1) * 2 * KG * ROWS + (size_t)KG * ROWS + row;
                const uint32_t hl = tmem + t_lane + HL_COL;
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    uint4 v[NJ];
#pragma unroll
                    for (int jj = 0; jj < NJ; ++jj) {
                        const int j = PIECE_KG * half + LOAD_PARTS * jj + part;
                        v[jj] = LOAD_PARTS * jj + part < PIECE_KG ? __ldcg(src + (size_t)j * ROWS) : make_uint4(0, 0, 0, 0);
                    }
#pragma unroll
                    for (int jj = 0; jj < NJ; ++jj) {
                        if (LOAD_PARTS * jj + part >= PIECE_KG) break;
                        tmem_st_x4(hl + 4 * (PIECE_KG * half + LOAD_PARTS * jj + part), v[jj].x, v[jj].y, v[jj].z, v[jj].w);
                    }
                    tmem_st_wait();
                    fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars[BAR_HLO + half]);
                }
            };
            // (the loaders publish nothing through the step barrier: they arrive at the barrier of step t+1 as soon as they have passed
            // the one of step t - ape_lstm_tcl.cu)
            build_x(0);
            cluster_arrive();
            for (int t = 0; t < T; ++t) {
                if (t + 1 < T) {                           // x_{t+1} once the x-part MMAs of step t have read x_t
                    mbar_wait_wd(&bars[BAR_XFREE], ph_xf); ph_xf ^= 1;
                    fence_after_sync();
                    build_x(t + 1);
                }
                cluster_wait();                            // the barrier that ends step t: h_t is in the exchange buffer
                if (t + 1 < T) cluster_arrive();
                if (pull(t)) load_hlo(t);
            }
        } else {
            // =================================== controller warp: MMA issue, h_hi pull ========================================
            const uint32_t idesc = make_idesc_f16(128, NCOL), idesc_out = make_idesc_f16(128, NO);
            const uint64_t dHh = make_desc(smem_u32(sH), LBO_A, SBO);
            const uint64_t dOnes = make_desc(smem_u32(sOnes), LBO_A, SBO);
            const uint64_t dWxh = make_desc(smem_u32(sW), LBO_B, SBO);                         // Wx_hi, then the bias K step
            const uint64_t dWxl = desc_advance(dWxh, p0_bytes(kgx));                              // Wx_lo
            const uint64_t dWhh = desc_advance(dWxl, p1_bytes(kgx)), dWhl = desc_advance(dWhh, PH_BYTES);   // Wh_hi, Wh_lo
            const uint32_t xh = tmem + XH_COL, xl = tmem + XL_COL, hl = tmem + HL_COL;
            const uint32_t nxp = (uint32_t)(kgx + PIECE_KG - 1) / PIECE_KG;
            constexpr uint32_t KS_B = 2 * LBO_B >> 4, KS_A = 2 * LBO_A >> 4;                      // descriptor steps of one K = 16
            constexpr uint32_t MP = PIECE_KG / 2;                                                 // K = 16 MMAs of a piece
            auto wait_hlo = [&](int half) {
                mbar_wait_wd(&bars[BAR_HLO + half], ph_hlo);
                if (half == 1) ph_hlo ^= 1;
                fence_after_sync();
            };
            mbar_wait_wd(&bars[BAR_W], ph_w); ph_w ^= 1;   // the layer's weights have landed
            fence_after_sync();
            for (int t = 0; t < T; ++t) {
                mbar_wait_wd(&bars[BAR_X], ph_x); ph_x ^= 1;
                fence_after_sync();
                if (elect_one()) {
                    for (uint32_t p = 0; p < nxp; ++p) {                   // Wx_hi piece p: x_hi, (last piece: ones), x_lo
                        const uint32_t m0 = p * MP, nm = min((uint32_t)kgx / 2 - m0, MP);
                        for (uint32_t m = 0; m < nm; ++m)
                            mma_f16_ts<1>(tmem + ACC_COL, xh + 8 * (m0 + m), dWxh + (m0 + m) * KS_B, idesc, (p > 0 || m > 0) ? 1u : 0u);
                        if (p == nxp - 1) mma_f16<1>(tmem + ACC_COL, dOnes, dWxh + (uint32_t)kgx / 2 * KS_B, idesc, 1u);
                        for (uint32_t m = 0; m < nm; ++m) mma_f16_ts<1>(tmem + ACC_COL, xl + 8 * (m0 + m), dWxh + (m0 + m) * KS_B, idesc, 1u);
                    }
                    for (uint32_t m = 0; m < (uint32_t)kgx / 2; ++m)     // Wx_lo: x_hi
                        mma_f16_ts<1>(tmem + ACC_COL, xh + 8 * m, dWxl + m * KS_B, idesc, 1u);
                    if (t + 1 < T) commit(&bars[BAR_XFREE]);           // x_t is no longer read: the loaders may build x_{t+1}
                }
                __syncwarp();
                if (t > 0) {
                    mbar_wait_wd(&bars[BAR_H], ph_h); ph_h ^= 1;             // h_hi of h_{t-1} is in sH
                    wait_hlo(0);                                             // h_lo k-groups 0..15 are in TMEM
                    if (elect_one()) {                                       // Wh_hi piece 0: h_hi, h_lo; piece 1: h_hi
#pragma unroll
                        for (uint32_t m = 0; m < MP; ++m) mma_f16<1>(tmem + ACC_COL, dHh + m * KS_A, dWhh + m * KS_B, idesc, 1u);
#pragma unroll
                        for (uint32_t m = 0; m < MP; ++m) mma_f16_ts<1>(tmem + ACC_COL, hl + 8 * m, dWhh + m * KS_B, idesc, 1u);
#pragma unroll
                        for (uint32_t m = MP; m < KG / 2; ++m) mma_f16<1>(tmem + ACC_COL, dHh + m * KS_A, dWhh + m * KS_B, idesc, 1u);
                    }
                    __syncwarp();
                    wait_hlo(1);                                             // h_lo k-groups 16..31
                    if (elect_one()) {                                       // Wh_hi piece 1: h_lo; then Wh_lo: h_hi
#pragma unroll
                        for (uint32_t m = MP; m < KG / 2; ++m) mma_f16_ts<1>(tmem + ACC_COL, hl + 8 * m, dWhh + m * KS_B, idesc, 1u);
#pragma unroll
                        for (uint32_t m = 0; m < KG / 2; ++m) mma_f16<1>(tmem + ACC_COL, dHh + m * KS_A, dWhl + m * KS_B, idesc, 1u);
                    }
                    __syncwarp();
                }
                if (elect_one()) commit(&bars[BAR_ACC]);
                __syncwarp();
                fence_before_sync();
                cluster_sync();                            // end of step t: every CTA's slice of h_t is in the exchange buffer
                // pull h_hi of h_t (a copy nobody waits for must not be in flight at exit)
                if (pull(t) && lane == 0) {
                    asm volatile("fence.proxy.async;" ::: "memory");        // generic-proxy writes of the other SMs -> this bulk copy
                    mbar_arrive_expect_tx(&bars[BAR_H], H_BYTES);
                    bulk_g2s(sH, hx + (size_t)(t & 1) * 2 * KG * ROWS, H_BYTES, &bars[BAR_H]);
                }
                __syncwarp();
            }
            if (last_layer && a.preds && rank == 0) {
                // h_T(hi, lo) x [fp16(W_o) | W_o - fp16(W_o)]^T: the two output tiles take the weights' place (every MMA that read them is done)
                if (lane == 0) {
                    mbar_arrive_expect_tx(&bars[BAR_W], 2 * OT_BYTES);
                    bulk_g2s(sW, a.Wo16, 2 * OT_BYTES, &bars[BAR_W]);
                }
                mbar_wait_wd(&bars[BAR_H], ph_h); ph_h ^= 1;
                mbar_wait_wd(&bars[BAR_W], ph_w); ph_w ^= 1;
                wait_hlo(0);
                wait_hlo(1);
                if (elect_one()) {
                    for (int half = 0; half < 2; ++half) {
                        const uint64_t dO = make_desc(smem_u32(sW) + half * OT_BYTES, NO * 16, SBO);
#pragma unroll
                        for (int m = 0; m < KG / 2; ++m)
                            mma_f16<1>(tmem + OUT_COL + half * NO, dHh + m * KS_A, dO + m * (2 * NO * 16 >> 4), idesc_out, m > 0 ? 1u : 0u);
#pragma unroll
                        for (int m = 0; m < KG / 2; ++m)
                            mma_f16_ts<1>(tmem + OUT_COL + half * NO, hl + 8 * m, dO + m * (2 * NO * 16 >> 4), idesc_out, 1u);
                    }
                    commit(&bars[BAR_OUT]);
                }
                __syncwarp();
            }
        }
    }
    __syncwarp();
    fence_before_sync();
    cluster_sync();
    if (warp == CTRL_WARP) tmem_dealloc<1>(tmem, TMEM_COLS);
}

bool supported(int Hh, int I, int L, int T, int O, long long E, int n) {
    return Hh == H && L >= 2 && L <= MAX_L && T >= 1 && T <= 40 && I >= 1 && ape_pack_kin_pad(0, I, H) <= H && O >= 1 && O <= NO &&
           E >= 0 && n >= 1 && E * n <= (long long)ROWS * MAX_CLUSTERS;
}

static size_t cluster_ws_bytes(int T) { return (size_t)(2 + 2 * T) * 2 * KG * ROWS * 16; }      // hx + seq (hi and lo) of one cluster
size_t workspace_bytes(int T, long long rows) {
    const long long clusters = rows <= 0 ? 1 : (rows + ROWS - 1) / ROWS;
    return cluster_ws_bytes(T) * (size_t)clusters + 256;
}

static size_t layer_bytes(int layer, int I) { return (size_t)2 * NCHL * chunk_bytes(layer == 0 ? ape_pack_kin_pad(0, I, H) / 8 : KG); }

// the launch configuration of `clusters` clusters (a 16-CTA cluster is a non-portable size: the kernel opts in first)
static cudaError_t launch_config(int clusters, cudaStream_t st, cudaLaunchConfig_t& cfg, cudaLaunchAttribute* attr) {
    cudaError_t e = cudaFuncSetAttribute(lstm_small_tcxs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(lstm_small_tcxs_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    cfg = cudaLaunchConfig_t{};
    cfg.gridDim = dim3(NCTA * clusters); cfg.blockDim = dim3(THREADS); cfg.dynamicSmemBytes = SMEM; cfg.stream = st;
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = NCTA; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return e;
}

// clusters of this launch the current device can hold at once (cudaOccupancyMaxActiveClusters), cached per device; 0 = none
int max_active_clusters(int* clusters) {
    constexpr int MAX_DEVICES = 64;
    static std::atomic<int> cache[MAX_DEVICES];               // (zero-initialised: 0 = not asked yet, else clusters + 1)
    int dev = 0;
    APE_CUDA_TRY(cudaGetDevice(&dev));
    if (dev >= 0 && dev < MAX_DEVICES && cache[dev].load() > 0) { *clusters = cache[dev].load() - 1; return APE_OK; }
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr[1];
    APE_CUDA_TRY(launch_config(1, nullptr, cfg, attr));
    int n = 0;
    APE_CUDA_TRY(cudaOccupancyMaxActiveClusters(&n, lstm_small_tcxs_kernel, &cfg));
    if (dev >= 0 && dev < MAX_DEVICES) cache[dev].store(n + 1);
    *clusters = n;
    return APE_OK;
}

// all layers of the call `g` (ape_mc_lstm_tcxsl) from the split blob `blob` (weights_tcx); shapes already checked
int run(const ape_lstm_args* g, const uint8_t* blob, void* workspace, cudaStream_t st) {
    Args a{};
    const uint8_t* p = blob;
    for (int l = 0; l < g->L; ++l) {
        a.W[l] = p;
        a.kgx[l] = l == 0 ? ape_pack_kin_pad(0, g->I, H) / 8 : KG;
        p += layer_bytes(l, g->I);
    }
    const long long E = (long long)g->B * g->nF;
    a.L = g->L; a.T = g->T; a.I = g->I; a.E = (int)E; a.n = g->n_samples; a.nF = g->nF; a.frame0 = g->frame0; a.feat_ring = g->feat_ring;
    a.dense = g->x_dense != nullptr;
    a.in = g->x_dense ? g->x_dense : g->feat_ring_buf;
    a.stream_frames = g->stream_frames;
    a.mask_mode = g->mask_mode; a.masks = g->masks;
    a.rk = philox_round_keys(g->philox_seed);
    a.stream_id0 = g->stream_id0;
    a.keep_thr16 = keep_threshold16(g->dropout_p);
    a.scale = g->mask_mode == APE_MASK_NONE ? 1.0f : 1.0f / (1.0f - g->dropout_p);
    char* ws = (char*)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    a.hx = (uint4*)ws;
    a.seq = (uint4*)(ws + (size_t)2 * 2 * KG * ROWS * 16);
    a.ws_stride = cluster_ws_bytes(g->T) / 16;
    const int clusters = (int)((E * g->n_samples + ROWS - 1) / ROWS);
    a.Wo16 = p;                                          // the output-layer tiles follow the last layer
    a.bo = g->weights + ape_pack_out_offset(g->I, g->H, g->L) + (size_t)g->O * g->H;
    a.O = g->O;
    a.preds = g->preds; a.pred_ring = g->pred_ring;
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr[1];
    APE_CUDA_TRY(launch_config(clusters, st, cfg, attr));
    APE_CUDA_TRY(cudaLaunchKernelEx(&cfg, lstm_small_tcxs_kernel, a));
    return check_launch();
}

}  // namespace tcxsl
}  // namespace ape
