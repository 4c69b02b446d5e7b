// Stage 2 for a SMALL batch (<= 128 rows: the single-stream real-time case, BASELINE configs[1] - one stream x 100 MC samples):
// all L layers of the MC-dropout LSTM in ONE launch of ONE cluster of 8 CTAs, the hidden units split across the cluster.
//
// The layer kernels (ape_lstm_tc / tcs / tcw) give a 256-row tile to one CTA pair, which then walks ALL 4H gate columns every step: for
// one stream that is T x L dependent passes over a whole layer's weights on two SMs - 0.07 ms for layer 0 (ONE row) and 0.09 ms for
// layer 1 (100 rows) of the 0.19 ms frame - while 146 SMs idle.  A recurrence cannot be split over time, but it splits over hidden
// units: here CTA k of the cluster owns the units [k H/8, (k+1) H/8) of every layer (its 64 or 128 gate columns of the fp16 weights
// stay resident in shared memory for the whole layer), computes their gates for all rows with tcgen05 MMAs (cta_group::1, M = 128,
// fp16 operands, fp32 accumulate in TMEM), updates their cells, and the eight slices of h_t are exchanged once per step:
//     epilogue warps write their slice of h_t (fp16 operand units) to an L2-resident exchange buffer -> ONE cluster barrier ->
//     every CTA pulls the whole h_t tile into its shared-memory A operand with one bulk asynchronous copy (cp.async.bulk).
//     (Pushing the slices into the eight h tiles with shared-to-distributed-shared bulk copies instead was measured SLOWER: 0.114 vs
//     0.095 ms per launch - 64 KB of distributed-shared-memory traffic per CTA and step.)
// x_t (the previous layer's h sequence with this layer's dropout mask, or the feature window for layer 0) is built per row by four
// loader warps straight into TENSOR MEMORY one step ahead (tcgen05.st; the x-part MMAs take their A operand from TMEM), so shared
// memory only holds the weights and the h tile.  Same operand rounding points, gate arithmetic (tanh form) and Philox keys as the
// layer kernels; the fp16 weight blob is theirs (a CTA's slice = one or two of its 64-column tiles).
// A call of more than 128 rows runs as SEVERAL clusters in the same launch, cluster c taking rows [128 c, 128 c + 128) of the layers >= 1 and
// layer 0 of the estimates those rows belong to (rows are independent; an estimate that straddles two clusters has its layer 0 computed by
// both): up to a few thousand rows - a few dozen real-time streams - this is faster than the layer kernels, which give every 256-row tile to
// one CTA pair for T x L dependent passes over whole layers.
#include "ape_common.cuh"
#include "ape_lstm_pack.h"
#include "ape_lstm_tc_args.cuh"
#include "ape_umma.cuh"
#include "ape_f32x2.cuh"

namespace ape {
namespace tcl {

using tc::tanh_approx;

constexpr int NCTA = 8, ROWS = tc::CLUSTER_ROWS;
// 12 loader warps: three per TMEM lane quarter, each taking every third k-group of its 32 rows (building x_t for a layer >= 1 is 32 L2
// loads + 32 Philox draws per row at H = 256; with one warp per quarter it took 7.5 - 12 us, twice the rest of a step)
// 8 epilogue warps: two per TMEM lane quarter, each taking every second k-group (8 units) of its 32 rows' cells
constexpr int EPI_WARPS = 8, EPI_PARTS = EPI_WARPS / 4, LOAD_PARTS = 3, LOAD_WARPS = 4 * LOAD_PARTS, THREADS = (EPI_WARPS + LOAD_WARPS + 1) * 32;   // + the controller warp
constexpr int CTRL_WARP = EPI_WARPS + LOAD_WARPS;
constexpr uint32_t BLK_COLS = 64, KG_BYTES_B = BLK_COLS * 16;    // a weight tile of the blob: [k-group][64 gate columns][8 halfs]
constexpr uint32_t ACC_COL = 0, X_COL = 128, OUT_COL = 384, TMEM_COLS = 512;

__device__ __forceinline__ void stamp(long long* st, int step, int ev) {
    if (st) st[step * 8 + ev] = tc::globaltimer_ns();
}

enum { BAR_W = 0, BAR_X = 1, BAR_ACC = 3, BAR_H = 4, BAR_OUT = 5, BAR_COUNT = 6 };

template <int H>
__global__ void __cluster_dims__(NCTA, 1, 1) __launch_bounds__(THREADS, 1) lstm_small_kernel(const __grid_constant__ tc::ClusterArgs a) {
    using namespace umma;
    constexpr int KG = H / 8, NU = H / NCTA, NB = NU / 16, NCOL = 4 * NU;       // this CTA: NU units = NB weight tiles = NCOL gate columns
    constexpr int NO = H > 128 ? 32 : 16;                                      // columns of an output tile
    constexpr uint32_t LBO_A = ROWS * 16, LBO_B = KG_BYTES_B, SBO = 128, H_BYTES = KG * ROWS * 16;
    constexpr uint32_t BLK_BYTES = 2 * KG * KG_BYTES_B;                        // room of one weight tile (x k-groups then h k-groups)
    static_assert(NB * BLK_BYTES + H_BYTES + NCOL * 4 + 64 <= 227 * 1024, "shared memory budget");
    static_assert(X_COL + 2 * (H / 2) <= OUT_COL && NCOL <= (int)X_COL, "tensor memory plan");

    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* sW = smem;                                  // [NB][kgx + KG k-groups][64][8]   (the output tiles at the very end)
    uint8_t* sH = sW + NB * BLK_BYTES;                   // [KG][ROWS] units: h_{t-1} of ALL units, A operand of the recurrent MMAs
    float* sBias = reinterpret_cast<float*>(sH + H_BYTES);  // [NCOL] this CTA's bias columns of the current layer
    uint64_t* bars = reinterpret_cast<uint64_t*>(sBias + NCOL);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + BAR_COUNT);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    const int T = a.T, L = a.L;
    // this cluster's slab: rows [r0, r0 + rows1) of the layers >= 1 = (estimate, sample) pairs, and layer 0 of the estimates e_lo .. e_hi they belong to
    const int cid = (int)(blockIdx.x / NCTA);
    const int r0 = cid * ROWS;
    const int rows1 = min(ROWS, a.E * a.n - r0);
    const int e_lo = r0 / a.n, rows0 = (r0 + rows1 - 1) / a.n - e_lo + 1;
    uint4* const hx = a.hx + (size_t)cid * a.ws_stride;  // [2][H/8][128] exchange buffer of h_t, by step parity
    uint4* const seq = a.seq + (size_t)cid * a.ws_stride; // [2][T][H/8][128] a layer's output sequence, by layer parity
    long long* const stamps = cid == 0 ? a.stamps : nullptr;

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
    // barrier phases: each is tracked by the ONE role that waits on that barrier (controller: W, X, H; epilogue warps: ACC)
    uint32_t ph_w = 0, ph_x[2] = {0, 0}, ph_acc = 0, ph_h = 0;

    for (int l = 0; l < L; ++l) {
        const int kgx = a.kgx[l];
        const bool last_layer = l == L - 1;
        const int rows = l == 0 ? rows0 : rows1;
        // ---- this CTA's weight tiles of layer l -> shared memory (all MMAs of the previous layer have completed: see the barrier below) ----
        const uint32_t tile_bytes = (uint32_t)(kgx + KG) * KG_BYTES_B;
        if (warp == CTRL_WARP && lane == 0) {
            mbar_arrive_expect_tx(&bars[BAR_W], NB * tile_bytes);
            for (int b = 0; b < NB; ++b) {
                // tile (r, c) of the blob holds the units 32 c + 16 r .. + 15: H = 128: CTA k = tile (k & 1, k >> 1); H = 256: CTA k = tiles (0, k), (1, k)
                const int r = NB == 1 ? (int)(rank & 1) : b, c = NB == 1 ? (int)(rank >> 1) : (int)rank;
                const uint8_t* src = a.W[l] + ((size_t)r * (H / 32) + c) * tile_bytes;
                bulk_g2s(sW + b * BLK_BYTES, src, tile_bytes, &bars[BAR_W]);
            }
        }

        if (warp < EPI_WARPS) {
            // =================================== epilogue warps: row = TMEM lane = 32 (warp & 3) + lane ====================
            const int row = 32 * (warp & 3) + lane, epart = warp >> 2;       // epart: which k-groups of the CTA's units this warp updates
            const uint32_t t_lane = (uint32_t)(32 * (warp & 3)) << 16;
            constexpr int NB8 = NU / 8 / EPI_PARTS;                          // k-groups (8 units) per warp: b8 = EPI_PARTS * i + epart
            static_assert(NB8 >= 1 && NB8 * EPI_PARTS * 8 == NU, "epilogue split");
            float cst[8 * NB8];
#pragma unroll
            for (int u = 0; u < 8 * NB8; ++u) cst[u] = 0.0f;
            // this CTA's bias columns in shared memory (a global load per unit and step sat in front of every gate)
            for (int i = tid; i < NCOL; i += EPI_WARPS * 32) sBias[i] = __ldg(a.bias_s[l] + (size_t)rank * NCOL + i);
            asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
            const float4* sBias4 = reinterpret_cast<const float4*>(sBias);
            for (int t = 0; t < T; ++t) {
                mbar_wait_wd(&bars[BAR_ACC], ph_acc); ph_acc ^= 1;
                fence_after_sync();
                if (rank == 0 && tid == 0) stamp(stamps, l * T + t, 3);        // accumulators ready
                const bool exchange = t + 1 < T || (last_layer && a.preds);      // the last step's h only feeds the output layer
                // this CTA's k-groups of the h_t tile / of the layer's output sequence: [k-group rank NU/8 + b8][row]
                uint4* hx_dst = hx + (size_t)(t & 1) * KG * ROWS + (size_t)(rank * (NU / 8)) * ROWS + row;
                uint4* seq_dst = seq + ((size_t)(l & 1) * T + t) * KG * ROWS + (size_t)(rank * (NU / 8)) * ROWS + row;
#pragma unroll
                for (int i8 = 0; i8 < NB8; ++i8) {         // 8 units = 32 accumulator columns = one k-group at a time
                    const int b8 = EPI_PARTS * i8 + epart;
                    uint32_t r[32];
                    tmem_ld_x32(tmem + t_lane + ACC_COL + 32 * b8, r);
                    tmem_ld_wait();
                    float hv[8];
#pragma unroll
                    for (int u = 0; u < 8; u += 2) {                               // two units per instruction (packed fp32 pairs, ape_f32x2.cuh: the scalar operations bit for bit)
                        float tg[8];
#pragma unroll
                        for (int v = 0; v < 2; ++v) {
                            const float4 bs = sBias4[8 * b8 + u + v];              // 0.5 b (i, f, o), b (g)
                            const F2 aif = fma2(pk(__uint_as_float(r[4 * (u + v) + 0]), __uint_as_float(r[4 * (u + v) + 1])), splat(0.5f), pk(bs.x, bs.y));
                            const F2 ago = fma2(pk(__uint_as_float(r[4 * (u + v) + 2]), __uint_as_float(r[4 * (u + v) + 3])), pk(1.0f, 0.5f), pk(bs.z, bs.w));
                            tg[4 * v + 0] = tanh_approx(lo(aif)); tg[4 * v + 1] = tanh_approx(hi(aif));
                            tg[4 * v + 2] = tanh_approx(lo(ago)); tg[4 * v + 3] = tanh_approx(hi(ago));
                        }
                        const F2 h2c = splat(0.5f);
                        const F2 gi = fma2(pk(tg[0], tg[4]), h2c, h2c), gf = fma2(pk(tg[1], tg[5]), h2c, h2c);
                        const F2 c2 = fma2(gf, pk(cst[8 * i8 + u], cst[8 * i8 + u + 1]), gi * pk(tg[2], tg[6]));
                        cst[8 * i8 + u] = lo(c2); cst[8 * i8 + u + 1] = hi(c2);
                        const F2 h2 = fma2(pk(tg[3], tg[7]), h2c, h2c) * pk(tanh_approx(lo(c2)), tanh_approx(hi(c2)));
                        hv[u] = lo(h2); hv[u + 1] = hi(h2);
                    }
                    // h_t as fp16 units: as is for the recurrence, scaled by the consumer's 1 / (1 - p) (before the rounding) for the next layer
                    if (exchange)
                        hx_dst[(size_t)b8 * ROWS] = make_uint4(pack_half2(hv[0], hv[1]), pack_half2(hv[2], hv[3]), pack_half2(hv[4], hv[5]), pack_half2(hv[6], hv[7]));
                    if (!last_layer)
                        seq_dst[(size_t)b8 * ROWS] = make_uint4(pack_half2(hv[0] * a.scale, hv[1] * a.scale), pack_half2(hv[2] * a.scale, hv[3] * a.scale),
                                                                pack_half2(hv[4] * a.scale, hv[5] * a.scale), pack_half2(hv[6] * a.scale, hv[7] * a.scale));
                }
                if (rank == 0 && tid == 0) stamp(stamps, l * T + t, 4);        // cell update done, slice written
                fence_before_sync();
                cluster_sync();                            // every slice of h_t (and of the layer's sequence) is written, every MMA of step t done
                                                           // (release / acquire at cluster scope covers the global writes of the sequence)
            }
            if (last_layer && a.preds && rank == 0 && epart == 0) {      // output_layer (nn_models.py:189) on the last step, CTA 0
                mbar_wait_wd(&bars[BAR_OUT], 0);
                fence_after_sync();
                uint32_t o[2 * NO];                        // [h_T x fp16(W_o)^T | h_T x (W_o - fp16(W_o))^T]
                if (NO == 16) tmem_ld_x32(tmem + t_lane + OUT_COL, o);
                else { tmem_ld_x32(tmem + t_lane + OUT_COL, o); tmem_ld_x32(tmem + t_lane + OUT_COL + 32, o + 32); }
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
            // =================================== loader warps: x_t of every row -> TMEM, one step ahead =====================
            const int lw = warp & 3, part = (warp - EPI_WARPS) >> 2, row = 32 * lw + lane;   // (warp % 4 == lw: its TMEM lane quarter)
            const uint32_t t_lane = (uint32_t)(32 * lw) << 16;
            const bool valid = row < rows;
            const int e = valid ? (l == 0 ? e_lo + row : (r0 + row) / a.n) : 0, smp = (valid && l > 0) ? r0 + row - e * a.n : 0;
            const int bidx = e / a.nF, f = stream_frame0(a.stream_frames, a.frame0, bidx) + e % a.nF;
            const uint32_t stream = a.stream_id0 + (uint32_t)bidx;
            // x_t goes into X buffer t & 1, which the x-part MMAs of step t-2 read: those are complete once the cluster barrier that ends
            // step t-2 has been passed.  So x_0 and x_1 are built up front and x_{t+2} right behind the barrier that ends step t.
            auto build_x = [&](int t) {
                const uint32_t xcol = tmem + t_lane + X_COL + (uint32_t)(t & 1) * (H / 2);
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
                        tmem_st_x4(xcol + 4 * j, pack_half2(v[0], v[1]), pack_half2(v[2], v[3]), pack_half2(v[4], v[5]), pack_half2(v[6], v[7]));
                    }
                } else {
                    // the previous layer's h_t (fp16 units scaled by 1 / (1 - p)) of this row's estimate, dropout mask of gap l - 1 ANDed in
                    const uint4* src = seq + ((size_t)((l - 1) & 1) * T + t) * KG * ROWS + (l == 1 ? e - e_lo : row);
                    // all KG loads of the step go out before anything else: they come from L2 (written by other SMs), and two at a time
                    // had been the longest chain of a step (16 L2 round trips: 7.9 us per step for the whole kernel)
                    constexpr int NJ = (KG + LOAD_PARTS - 1) / LOAD_PARTS;       // this warp's k-groups: part, part + 3, ...
                    uint4 xv[NJ];
#pragma unroll
                    for (int jj = 0; jj < NJ; ++jj) {
                        const int j = LOAD_PARTS * jj + part;
                        xv[jj] = (valid && j < KG) ? __ldcg(src + (size_t)j * ROWS) : make_uint4(0, 0, 0, 0);
                    }
#pragma unroll
                    for (int jj = 0; jj < NJ; ++jj) {
                        const int j = LOAD_PARTS * jj + part;
                        if (j >= KG) break;
                        uint4 v = xv[jj];
                        if (a.mask_mode == APE_MASK_PHILOX) {
                            const uint4 m = philox_keep_halfmask_rk(a.rk, stream, (uint32_t)f, (uint32_t)smp, (uint32_t)(l - 1), (uint32_t)t,
                                                                    (uint32_t)j, a.keep_thr16);
                            v.x &= m.x; v.y &= m.y; v.z &= m.z; v.w &= m.w;
                        } else if (a.mask_mode == APE_MASK_INJECTED && valid) {
                            const uint2 mm = __ldg(reinterpret_cast<const uint2*>(
                                a.masks + ((((size_t)e * (L - 1) + (l - 1)) * T + t) * a.n + smp) * H + j * 8));
                            v.x &= ((mm.x & 0xFFu) ? 0xFFFFu : 0u) | ((mm.x & 0xFF00u) ? 0xFFFF0000u : 0u);
                            v.y &= ((mm.x & 0xFF0000u) ? 0xFFFFu : 0u) | ((mm.x & 0xFF000000u) ? 0xFFFF0000u : 0u);
                            v.z &= ((mm.y & 0xFFu) ? 0xFFFFu : 0u) | ((mm.y & 0xFF00u) ? 0xFFFF0000u : 0u);
                            v.w &= ((mm.y & 0xFF0000u) ? 0xFFFFu : 0u) | ((mm.y & 0xFF000000u) ? 0xFFFF0000u : 0u);
                        }
                        tmem_st_x4(xcol + 4 * j, v.x, v.y, v.z, v.w);
                    }
                }
                tmem_st_wait();
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars[BAR_X + (t & 1)]);
            };
            // The loader warps publish nothing through the step barrier, so they ARRIVE at the barrier of step t+1 as soon as they have
            // passed the one of step t, and only then build x_{t+2}: a build (32 L2 loads + 32 Philox draws per row at H = 256) is
            // longer than a step, and with arrive + wait in one place the whole cluster waited for it every step.
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
            const uint32_t idesc = make_idesc_f16(128, BLK_COLS), idesc_out = make_idesc_f16(128, NO);
            const uint64_t dH = make_desc(smem_u32(sH), LBO_A, SBO), dW0 = make_desc(smem_u32(sW), LBO_B, SBO);
            mbar_wait_wd(&bars[BAR_W], ph_w); ph_w ^= 1;   // the layer's weights have landed
            fence_after_sync();
            for (int t = 0; t < T; ++t) {
                mbar_wait_wd(&bars[BAR_X + (t & 1)], ph_x[t & 1]); ph_x[t & 1] ^= 1;
                fence_after_sync();
                if (rank == 0 && lane == 0) stamp(stamps, l * T + t, 0);       // x_t ready
                if (elect_one()) {
                    const uint32_t xa = tmem + X_COL + (uint32_t)(t & 1) * (H / 2);
#pragma unroll
                    for (int b = 0; b < NB; ++b) {
                        const uint64_t dW = dW0 + b * (BLK_BYTES >> 4);
                        if (kgx == KG) {                   // layers >= 1: full width, unrolled (the issuing thread is on the step's critical path)
#pragma unroll
                            for (int m = 0; m < KG / 2; ++m)
                                mma_f16_ts<1>(tmem + ACC_COL + b * BLK_COLS, xa + 8 * m, dW + m * (2 * LBO_B >> 4), idesc, m > 0 ? 1u : 0u);
                        } else {
                            for (int m = 0; m < kgx / 2; ++m)
                                mma_f16_ts<1>(tmem + ACC_COL + b * BLK_COLS, xa + 8 * m, dW + m * (2 * LBO_B >> 4), idesc, m > 0 ? 1u : 0u);
                        }
                    }
                }
                __syncwarp();
                if (t > 0) {
                    mbar_wait_wd(&bars[BAR_H], ph_h); ph_h ^= 1;             // h_{t-1} of all units is in sH
                    fence_after_sync();
                    if (rank == 0 && lane == 0) stamp(stamps, l * T + t, 1);   // h_{t-1} landed
                    if (elect_one()) {
#pragma unroll
                        for (int b = 0; b < NB; ++b) {
                            const uint64_t dW = dW0 + b * (BLK_BYTES >> 4) + (uint32_t)kgx * (KG_BYTES_B >> 4);
#pragma unroll
                            for (int m = 0; m < KG / 2; ++m)
                                mma_f16<1>(tmem + ACC_COL + b * BLK_COLS, dH + m * (2 * LBO_A >> 4), dW + m * (2 * LBO_B >> 4), idesc, 1u);
                        }
                    }
                    __syncwarp();
                }
                if (elect_one()) commit(&bars[BAR_ACC]);
                __syncwarp();
                if (rank == 0 && lane == 0) stamp(stamps, l * T + t, 2);       // MMAs issued + committed
                fence_before_sync();
                cluster_sync();                            // end of step t: every CTA's slice of h_t is in the exchange buffer
                if (rank == 0 && lane == 0) stamp(stamps, l * T + t, 5);       // barrier passed
                // pull the whole h_t tile (after the last step only CTA 0 needs h_T - for the output product - and a copy nobody waits for
                // must not be in flight at exit)
                const bool pull = t + 1 < T || (last_layer && a.preds && rank == 0);
                if (pull && lane == 0) {
                    asm volatile("fence.proxy.async;" ::: "memory");        // generic-proxy writes of the other SMs -> this bulk copy
                    mbar_arrive_expect_tx(&bars[BAR_H], H_BYTES);
                    bulk_g2s(sH, hx + (size_t)(t & 1) * KG * ROWS, H_BYTES, &bars[BAR_H]);
                }
                __syncwarp();
            }
            if (last_layer && a.preds && rank == 0) {
                // h_T x [fp16(W_o) | W_o - fp16(W_o)]^T: the two output tiles take the weight tiles' place (every MMA that read them is done)
                constexpr uint32_t OT_BYTES = KG * NO * 16;
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
                            mma_f16<1>(tmem + OUT_COL + half * NO, dH + m * (2 * LBO_A >> 4), dO + m * (2 * NO * 16 >> 4), idesc_out, m > 0 ? 1u : 0u);
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

template <int H> static int launch_t(const tc::ClusterArgs& a, int clusters, cudaStream_t st) {
    constexpr int KG = H / 8, NB = H / NCTA / 16;
    const size_t smem = (size_t)NB * 2 * KG * KG_BYTES_B + (size_t)KG * ROWS * 16 + (size_t)4 * (H / NCTA) * 4 + 64;
    APE_CUDA_TRY(cudaFuncSetAttribute(lstm_small_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    lstm_small_kernel<H><<<NCTA * clusters, THREADS, smem, st>>>(a);
    return check_launch();
}

int run(int H, const tc::ClusterArgs& a, int clusters, cudaStream_t st) {
    return H == 256 ? launch_t<256>(a, clusters, st) : launch_t<128>(a, clusters, st);
}

}  // namespace tcl
}  // namespace ape
