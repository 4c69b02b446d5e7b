// Stage 2, SPLIT PRECISION for a SMALL batch at H = 128: all L layers of the MC-dropout LSTM in ONE launch, one cluster of 8 CTAs
// per 128 rows with the hidden units split across the cluster - the structure of the single-pass cluster kernel (ape_lstm_tcl.cu)
// with the arithmetic of the split-precision layer kernel (ape_lstm_tcx.cu).
//
// A model whose weights fail the single-pass probe runs on the split layer kernels, which give a 256-row tile to one CTA pair that
// walks every gate column of a layer, T steps in a row, 49 MMAs per 32-unit chunk.  For a real-time call (one stream x 100 MC
// samples) that is T x L dependent passes over whole layers on two SMs.  Here CTA k owns the 16 units [16 k, 16 k + 16) of every
// layer - one (pair-CTA, chunk) slot of the tcx blob: slot (r, c) holds the units 32 c + 16 r .. + 15, so CTA k takes slot
// (k & 1, k >> 1), its four pieces Wx_hi (+ the bias K step), Wx_lo, Wh_hi, Wh_lo resident in shared memory for the layer - and:
//   * x_hi / x_lo (layer 0: split from the fp32 feature window; layers >= 1: the previous layer's hi / lo units, one dropout mask
//     ANDed into both) are built by the loader warps one step ahead in TENSOR MEMORY (tcgen05.st), double-buffered by step parity;
//   * h_hi / h_lo of all units sit in shared memory: each step the epilogue warps write their slice to an L2 exchange buffer
//     [2 parities][hi | lo][H/8][128] -> ONE cluster barrier -> every CTA pulls the whole 64 KB with one bulk copy;
//   * per accumulator the MMAs run in tcx's order (Wx_hi x_hi, bias step against a ones tile, Wx_hi x_lo, Wx_lo x_hi, then
//     Wh_hi h_hi, Wh_hi h_lo, Wh_lo h_hi), cta_group::1 with M = 128, N = 64, and the epilogue is tcx's (ex2 / rcp cell, the same
//     split points), so the results are bit-identical to the layer kernels.
// Shared memory per CTA: weights <= 66 KB + h_hi / h_lo 64 KB + ones tile 4 KB; tensor memory: accumulator 64 columns, x_hi / x_lo
// 2 x 128, output 32 (of 512).  Cluster c takes rows [128 c, 128 c + 128) of the layers >= 1 and layer 0 of the estimates those rows
// belong to (an estimate that straddles two clusters has its layer 0 computed by both).
#include "ape_common.cuh"
#include "ape_lstm_pack.h"
#include "ape_lstm_tc_args.cuh"
#include "ape_umma.cuh"
#include "ape_f32x2.cuh"

namespace ape {
namespace tcxl {

constexpr int H = 128, KG = H / 8, NCHL = H / 32, NCTA = 8, NU = H / NCTA, NCOL = 4 * NU, ROWS = tc::CLUSTER_ROWS;
// 8 epilogue warps (two per TMEM lane quarter, one k-group = 8 units each), 12 loader warps (three per quarter), one controller warp
constexpr int EPI_WARPS = 8, LOAD_PARTS = 3, LOAD_WARPS = 4 * LOAD_PARTS, THREADS = (EPI_WARPS + LOAD_WARPS + 1) * 32;
constexpr int CTRL_WARP = EPI_WARPS + LOAD_WARPS;
constexpr uint32_t KG_BYTES_B = NCOL * 16;                 // one k-group of a 64-column weight piece
constexpr uint32_t W_BYTES = tcx_blob::chunk_bytes(H, KG); // 66 KB: a slot of a layer >= 1 (the largest)
constexpr uint32_t H_BYTES = KG * ROWS * 16;               // one h operand tile (32 KB)
constexpr uint32_t ONES_BYTES = 2 * ROWS * 16;             // A operand of the bias K step
constexpr int NO = 16;                                     // columns of an output tile
constexpr uint32_t OT_BYTES = tc::wo16_bytes(H) / 2;
constexpr uint32_t SMEM = W_BYTES + 2 * H_BYTES + ONES_BYTES + 64;
constexpr uint32_t ACC_COL = 0, X_COL = 128, X_COLS = 2 * (H / 2), OUT_COL = 384, TMEM_COLS = 512;   // x buffer p: hi at X_COL + p X_COLS, lo + 64
static_assert(SMEM <= 227 * 1024, "shared memory budget");
static_assert(ACC_COL + NCOL <= X_COL && X_COL + 2 * X_COLS <= OUT_COL && OUT_COL + 2 * NO <= TMEM_COLS, "tensor memory plan");
static_assert(2 * OT_BYTES <= W_BYTES, "the output tiles take the weights' place");
using tc::NEG2LOG2E;
using tc::split2;

enum { BAR_W = 0, BAR_X = 1, BAR_ACC = 3, BAR_H = 4, BAR_OUT = 5, BAR_COUNT = 6 };

__global__ void __cluster_dims__(NCTA, 1, 1) __launch_bounds__(THREADS, 1) lstm_small_tcx_kernel(const __grid_constant__ tc::ClusterArgs a) {
    using namespace umma;
    constexpr uint32_t LBO_A = ROWS * 16, LBO_B = KG_BYTES_B, SBO = 128;

    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* sW = smem;                                  // this CTA's slot of the layer (the output tiles at the very end)
    uint8_t* sH = sW + W_BYTES;                          // [hi | lo][KG][ROWS] units: h_{t-1} of ALL units
    uint8_t* sOnes = sH + 2 * H_BYTES;                   // [2][ROWS] units
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
        mbar_init(&bars[BAR_X + 1], LOAD_WARPS);
        mbar_init(&bars[BAR_ACC], 1);
        mbar_init(&bars[BAR_H], 1);
        mbar_init(&bars[BAR_OUT], 1);
        mbar_init_fence();
    }
    fence_proxy_async_smem();
    fence_before_sync();
    cluster_sync();
    fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    uint32_t ph_w = 0, ph_x[2] = {0, 0}, ph_acc = 0, ph_h = 0;

    for (int l = 0; l < L; ++l) {
        const int kgx = a.kgx[l];
        const bool last_layer = l == L - 1;
        const int rows = l == 0 ? rows0 : rows1;
        // ---- this CTA's slot of layer l -> shared memory (every MMA of the previous layer has completed: see the barrier below) ----
        if (warp == CTRL_WARP && lane == 0) {
            const uint32_t cb = tcx_blob::chunk_bytes(H, kgx);
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
                const bool exchange = t + 1 < T || (last_layer && a.preds);      // the last step's h only feeds the output layer
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
                uint32_t o[2 * NO];                        // [h_T(hi, lo) x fp16(W_o)^T | h_T(hi, lo) x (W_o - fp16(W_o))^T]
                tmem_ld_x32(tmem + t_lane + OUT_COL, o);
                tmem_ld_wait();
                if (row < rows) {
                    const int e = (r0 + row) / a.n, smp = r0 + row - e * a.n;
                    const int bb = e / a.nF, fb = stream_frame0(a.stream_frames, a.frame0, bb), f = fb + e % a.nF;
                    if (fb >= 0) {
                        float* dst = a.preds + ((((size_t)bb * a.pred_ring + f % a.pred_ring) * a.n) + smp) * a.O;
#pragma unroll
                        for (int k = 0; k < NO; ++k)
                            if (k < a.O) dst[k] = __uint_as_float(o[k]) + __uint_as_float(o[NO + k]) + __ldg(a.bo + k);
                    }
                }
                fence_before_sync();
            }
        } else if (warp < CTRL_WARP) {
            // =================================== loader warps: x_hi, x_lo of every row -> TMEM, one step ahead =============
            const int lw = warp & 3, part = (warp - EPI_WARPS) >> 2, row = 32 * lw + lane;
            const uint32_t t_lane = (uint32_t)(32 * lw) << 16;
            const bool valid = row < rows;
            const int e = valid ? (l == 0 ? e_lo + row : (r0 + row) / a.n) : 0, smp = (valid && l > 0) ? r0 + row - e * a.n : 0;
            const int bidx = e / a.nF, f = stream_frame0(a.stream_frames, a.frame0, bidx) + e % a.nF;
            const uint32_t stream = a.stream_id0 + (uint32_t)bidx;
            // x_t goes into X buffer t & 1, which the x-part MMAs of step t-2 read: complete once the barrier ending step t-2 has passed
            auto build_x = [&](int t) {
                const uint32_t xh = tmem + t_lane + X_COL + (uint32_t)(t & 1) * X_COLS, xl = xh + H / 2;
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
                    constexpr int NJ = (KG + LOAD_PARTS - 1) / LOAD_PARTS;       // this warp's k-groups: part, part + 3, ...
                    uint4 vh[NJ], vl[NJ];
#pragma unroll
                    for (int jj = 0; jj < NJ; ++jj) {                            // every L2 load of the step goes out first
                        const int j = LOAD_PARTS * jj + part;
                        const bool ld = valid && j < KG;
                        vh[jj] = ld ? __ldcg(src + (size_t)j * ROWS) : make_uint4(0, 0, 0, 0);
                        vl[jj] = ld ? __ldcg(src + (size_t)(KG + j) * ROWS) : make_uint4(0, 0, 0, 0);
                    }
#pragma unroll
                    for (int jj = 0; jj < NJ; ++jj) {
                        const int j = LOAD_PARTS * jj + part;
                        if (j >= KG) break;
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
                        tmem_st_x4(xh + 4 * j, vh[jj].x & m.x, vh[jj].y & m.y, vh[jj].z & m.z, vh[jj].w & m.w);
                        tmem_st_x4(xl + 4 * j, vl[jj].x & m.x, vl[jj].y & m.y, vl[jj].z & m.z, vl[jj].w & m.w);
                    }
                }
                tmem_st_wait();
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars[BAR_X + (t & 1)]);
            };
            // (the loaders publish nothing through the step barrier: they arrive at the barrier of step t+1 as soon as they have passed
            // the one of step t, and only then build x_{t+2}, so the cluster does not wait for a build every step - ape_lstm_tcl.cu)
            build_x(0);
            if (T > 1) build_x(1);
            cluster_arrive();
            for (int t = 0; t < T; ++t) {
                cluster_wait();                            // the barrier that ends step t
                if (t + 1 < T) cluster_arrive();
                if (t + 2 < T) build_x(t + 2);
            }
        } else {
            // =================================== controller warp: MMA issue, h_t pull ========================================
            const uint32_t idesc = make_idesc_f16(128, NCOL), idesc_out = make_idesc_f16(128, NO);
            const uint64_t dHh = make_desc(smem_u32(sH), LBO_A, SBO), dHl = make_desc(smem_u32(sH) + H_BYTES, LBO_A, SBO);
            const uint64_t dOnes = make_desc(smem_u32(sOnes), LBO_A, SBO);
            const uint64_t dWxh = make_desc(smem_u32(sW), LBO_B, SBO);                         // Wx_hi, then the bias K step
            const uint64_t dWxl = desc_advance(dWxh, tcx_blob::p0_bytes(kgx));                              // Wx_lo
            const uint64_t dWhh = desc_advance(dWxl, tcx_blob::p1_bytes(kgx)), dWhl = desc_advance(dWhh, tcx_blob::ph_bytes(H));   // Wh_hi, Wh_lo
            const uint32_t nx = (uint32_t)kgx / 2;                                                 // K = 16 MMAs of an x-part
            constexpr uint32_t KS_B = 2 * LBO_B >> 4, KS_A = 2 * LBO_A >> 4;                      // descriptor steps of one K = 16
            mbar_wait_wd(&bars[BAR_W], ph_w); ph_w ^= 1;   // the layer's weights have landed
            fence_after_sync();
            for (int t = 0; t < T; ++t) {
                mbar_wait_wd(&bars[BAR_X + (t & 1)], ph_x[t & 1]); ph_x[t & 1] ^= 1;
                fence_after_sync();
                if (elect_one()) {
                    const uint32_t xh = tmem + X_COL + (uint32_t)(t & 1) * X_COLS, xl = xh + H / 2;
                    for (uint32_t m = 0; m < nx; ++m) mma_f16_ts<1>(tmem + ACC_COL, xh + 8 * m, dWxh + m * KS_B, idesc, m > 0 ? 1u : 0u);
                    mma_f16<1>(tmem + ACC_COL, dOnes, dWxh + nx * KS_B, idesc, 1u);
                    for (uint32_t m = 0; m < nx; ++m) mma_f16_ts<1>(tmem + ACC_COL, xl + 8 * m, dWxh + m * KS_B, idesc, 1u);
                    for (uint32_t m = 0; m < nx; ++m) mma_f16_ts<1>(tmem + ACC_COL, xh + 8 * m, dWxl + m * KS_B, idesc, 1u);
                }
                __syncwarp();
                if (t > 0) {
                    mbar_wait_wd(&bars[BAR_H], ph_h); ph_h ^= 1;             // h_{t-1} (hi, lo) of all units is in sH
                    fence_after_sync();
                    if (elect_one()) {
#pragma unroll
                        for (uint32_t m = 0; m < KG / 2; ++m) mma_f16<1>(tmem + ACC_COL, dHh + m * KS_A, dWhh + m * KS_B, idesc, 1u);
#pragma unroll
                        for (uint32_t m = 0; m < KG / 2; ++m) mma_f16<1>(tmem + ACC_COL, dHl + m * KS_A, dWhh + m * KS_B, idesc, 1u);
#pragma unroll
                        for (uint32_t m = 0; m < KG / 2; ++m) mma_f16<1>(tmem + ACC_COL, dHh + m * KS_A, dWhl + m * KS_B, idesc, 1u);
                    }
                    __syncwarp();
                }
                if (elect_one()) commit(&bars[BAR_ACC]);
                __syncwarp();
                fence_before_sync();
                cluster_sync();                            // end of step t: every CTA's slice of h_t is in the exchange buffer
                // pull the whole h_t tile (after the last step only CTA 0 needs h_T - for the output product - and a copy nobody waits
                // for must not be in flight at exit)
                const bool pull = t + 1 < T || (last_layer && a.preds && rank == 0);
                if (pull && lane == 0) {
                    asm volatile("fence.proxy.async;" ::: "memory");        // generic-proxy writes of the other SMs -> this bulk copy
                    mbar_arrive_expect_tx(&bars[BAR_H], 2 * H_BYTES);
                    bulk_g2s(sH, hx + (size_t)(t & 1) * 2 * KG * ROWS, 2 * H_BYTES, &bars[BAR_H]);
                }
                __syncwarp();
            }
            if (last_layer && a.preds && rank == 0) {
                // h_T(hi, lo) x [fp16(W_o) | W_o - fp16(W_o)]^T: the two output tiles take the weights' place (every MMA that read them is done)
                mbar_wait_wd(&bars[BAR_H], ph_h); ph_h ^= 1;
                if (lane == 0) {
                    mbar_arrive_expect_tx(&bars[BAR_W], 2 * OT_BYTES);
                    bulk_g2s(sW, a.Wo16, 2 * OT_BYTES, &bars[BAR_W]);
                }
                mbar_wait_wd(&bars[BAR_W], ph_w); ph_w ^= 1;
                fence_after_sync();
                if (elect_one()) {
                    for (int half = 0; half < 2; ++half) {
                        const uint64_t dO = make_desc(smem_u32(sW) + half * OT_BYTES, NO * 16, SBO);
#pragma unroll
                        for (int m = 0; m < KG / 2; ++m)
                            mma_f16<1>(tmem + OUT_COL + half * NO, dHh + m * KS_A, dO + m * (2 * NO * 16 >> 4), idesc_out, m > 0 ? 1u : 0u);
#pragma unroll
                        for (int m = 0; m < KG / 2; ++m)
                            mma_f16<1>(tmem + OUT_COL + half * NO, dHl + m * KS_A, dO + m * (2 * NO * 16 >> 4), idesc_out, 1u);
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

int run(const tc::ClusterArgs& a, int clusters, cudaStream_t st) {
    APE_CUDA_TRY(cudaFuncSetAttribute(lstm_small_tcx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
    lstm_small_tcx_kernel<<<NCTA * clusters, THREADS, SMEM, st>>>(a);
    return check_launch();
}

}  // namespace tcxl
}  // namespace ape
