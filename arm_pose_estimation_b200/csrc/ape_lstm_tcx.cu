// Stage 2, SPLIT-PRECISION tensor-core variant for H = 128 (one layer per launch): the tcgen05 path for models whose weights the
// single-pass fp16 kernels cannot carry (large weight scales, saturating gates - `BatchedEstimator`'s probe decides).
//
// The single-pass kernels round every operand to fp16 (2^-11) and evaluate the gates with tanh.approx (2^-11); a recurrent net
// amplifies both by ||W|| per step and layer, so at 2x / 4x / 8x the default weight scale the position error is 2.5e-4 / 6.6e-4 /
// 1.7e-2 m (tests/test_gpu_tc.py::test_weight_scale_sweep_against_oracle) against the 1e-4 m bound.  Here every operand is an fp16
// PAIR v = hi + lo (hi = fp16(v), lo = fp16(v - hi): ~22 bits) and a product is three tensor-core passes into the same fp32
// accumulator - a_hi b_hi + a_lo b_hi + a_hi b_lo (the lo x lo term is below fp32 resolution) - i.e. a 3x longer K loop, and the
// cell update uses ex2 / rcp (2^-22) instead of tanh.approx.  Same arithmetic as torch's fp32 LSTM to ~1e-6 relative.
//
// Structure = the wavefront kernel (ape_lstm_tcw.cu) with its second layer's resources given to the lo halves:
//   * a CTA pair (cta_group::2, M = 256) owns a 256-row tile for all T steps; items (tile, t) run on across tile boundaries;
//   * weights stream from L2 through a ring of 18 KB slots (cp.async.bulk): per 32-unit chunk four pieces - Wx_hi (+ the bias K step:
//     the bias enters as an fp16 pair against a tile of ones, i / f / o columns halved so the accumulator is the ex2 argument
//     up to one constant factor), Wx_lo, Wh_hi, Wh_lo; Wx_hi and Wh_hi are used twice (against the hi and the lo operand);
//   * x_hi, x_lo: shared-memory operand tiles written by the loader warps (layer 0: split from the fp32 feature window; layers >= 1:
//     the previous layer's hi / lo fp16 units with the dropout mask ANDed into both);
//   * h_hi, h_lo: packed fp16 pairs in TMEM (tcgen05.st), double-buffered by step parity, A operands of the recurrent MMAs;
//   * accumulators: two 128-column TMEM slots used alternately by the chunk sequence; fp32 cell state in an L2-resident scratch;
//   * the output layer (last step of the last layer) as a tensor-core product h_T(hi, lo) x [fp16(W_o) | W_o - fp16(W_o)]^T.
// Per chunk 49 MMAs instead of 17: the kernel is tensor-pipe-bound (3x the passes of the single-pass kernels), which still is an
// order of magnitude above the fp32 FFMA kernel it replaces as the fallback.
#include "ape_common.cuh"
#include "ape_lstm_pack.h"
#include "ape_lstm_tc_args.cuh"
#include "ape_umma.cuh"

namespace ape {
namespace tcx {

using tc::TcLayerArgs;

constexpr int H = 128, NCHL = H / 32, KG = H / 8;
constexpr int EPI_WARPS = 16, LOAD_WARPS = 8, N_ISSUERS = 2;
constexpr int THREADS = (EPI_WARPS + LOAD_WARPS + 4) * 32;       // 896 = 7 warpgroups
constexpr int MMA_WARP = 0, TMA_WARP = 2, LOAD_WARP0 = 4, EPI_WARP0 = 12;   // epilogue warps on the highest ids (scheduler priority)
constexpr int REGS_EPI = 96, REGS_LOAD = 40, REGS_MMA = 40;
static_assert(EPI_WARPS * 32 * REGS_EPI + LOAD_WARPS * 32 * REGS_LOAD + 128 * REGS_MMA <= THREADS * 72, "register file");
#define TCX_REG_INC(n) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(n))
#define TCX_REG_DEC(n) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(n))
constexpr int ROWS = 128;
constexpr uint32_t KG_BYTES_B = 64 * 16;                   // one k-group of a 64-column weight tile
constexpr uint32_t SLOT_BYTES = (KG + 2) * KG_BYTES_B;     // 18 KB: the largest piece (Wx_hi of a layer >= 1 + the bias K step)
constexpr uint32_t A_BYTES = KG * ROWS * 16;               // one operand tile (32 KB)
constexpr uint32_t ONES_BYTES = 2 * ROWS * 16;             // constant A tile of the bias K step
constexpr int NP = 8, NFULL = 16;                          // ring depth; "piece landed" barriers by piece number (> NP: never alias)
constexpr uint32_t OUT_N = 32;
constexpr uint32_t OUT_BYTES = KG * (OUT_N / 2) * 16;
constexpr uint32_t BAR_BLOCK_BYTES = 512;
constexpr uint32_t SMEM = 2 * A_BYTES + NP * SLOT_BYTES + ONES_BYTES + BAR_BLOCK_BYTES;
constexpr uint32_t HH_COL = 256, HL_COL = 384, H_COLS = H / 2, TMEM_COLS = 512;
constexpr size_t CSTATE_FLOATS = (size_t)H * ROWS;         // per CTA: [k-group * 2 + half][row] float4
static_assert(SMEM <= 227 * 1024, "shared memory budget");
using tc::NEG2LOG2E;
using tc::split2;
static_assert(2 * OUT_BYTES == tc::wo16_bytes(H), "the output-layer tiles of the tcx blob");

enum {
    BAR_X_READY = 0, BAR_X_DONE = 1, BAR_ACC_READY = 2, BAR_SLOT_FREE = 4, BAR_H_READY = 6, BAR_W_FULL = BAR_H_READY + NCHL,
    BAR_W_EMPTY = BAR_W_FULL + NFULL, BAR_OUT_READY = BAR_W_EMPTY + NP, BAR_COUNT = BAR_OUT_READY + 1
};
static_assert(BAR_COUNT * 8 + 16 <= BAR_BLOCK_BYTES, "barrier block too small");

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
lstm_layer_tcx_kernel(const __grid_constant__ TcLayerArgs a) {
    using namespace umma;
    constexpr uint32_t LBO_A = ROWS * 16, LBO_B = KG_BYTES_B, SBO = 128;
    const int T = a.T, kgx = a.kgx;

    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* sXh = smem;                                       // [A_BYTES] x_hi of the current item
    uint8_t* sXl = sXh + A_BYTES;                              // [A_BYTES] x_lo
    uint8_t* sW = sXl + A_BYTES;                               // [NP][SLOT_BYTES] weight ring
    uint8_t* sOnes = sW + NP * SLOT_BYTES;                     // [2][ROWS] units: A operand of the bias K step
    uint64_t* bars = reinterpret_cast<uint64_t*>(sOnes + ONES_BYTES);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + BAR_COUNT);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    const int n_my_tiles = (a.n_pair_tiles - cluster_id + n_clusters - 1) / n_clusters;
    const int NI = n_my_tiles * T;                             // items (tile, step) of this pair
    const bool has_out = a.preds != nullptr;

    tc::timeline_stamp(a.timeline, 0);
    for (int i = tid; i < 2 * ROWS; i += THREADS)
        reinterpret_cast<uint4*>(sOnes)[i] = make_uint4(i < ROWS ? 0x3C003C00u : 0u, 0u, 0u, 0u);
    // (k-groups of the x tiles beyond kgx are never read: the x-part has kgx / 2 MMAs)
    if (warp == MMA_WARP) {
        tmem_alloc<2>(tmem_slot, TMEM_COLS);
        tmem_relinquish<2>();
    }
    if (tid == 0) {
        mbar_init(&bars[BAR_X_READY], 2 * LOAD_WARPS);
        mbar_init(&bars[BAR_X_DONE], N_ISSUERS);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bars[BAR_ACC_READY + i], 1);
            mbar_init(&bars[BAR_SLOT_FREE + i], 2 * EPI_WARPS);
        }
        for (int c = 0; c < NCHL; ++c) mbar_init(&bars[BAR_H_READY + c], 2 * EPI_WARPS);
        for (int p = 0; p < NFULL; ++p) mbar_init(&bars[BAR_W_FULL + p], rank == 0 ? 2 : 1);   // leader: own copy + the peer's forward
        for (int p = 0; p < NP; ++p) mbar_init(&bars[BAR_W_EMPTY + p], 1);
        mbar_init(&bars[BAR_OUT_READY], 1);
        mbar_init_fence();
    }
    fence_proxy_async_smem();
    fence_before_sync();
    cluster_sync();
    fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    tc::timeline_stamp(a.timeline, 1);

    if (warp >= EPI_WARP0 && warp < EPI_WARP0 + EPI_WARPS) {
        TCX_REG_INC(REGS_EPI);
        // =================================== epilogue warps ===========================================================
        // warp (q, s): rows 32q..32q+31 (its TMEM lane quarter) x the 8 hidden units 8s..8s+7 of every 32-unit chunk
        const int q = warp & 3, s = (warp - EPI_WARP0) >> 2;
        const int row_l = 32 * q + lane;
        const uint32_t t_lane = (uint32_t)(32 * q) << 16;
        unsigned long long cst_base = reinterpret_cast<unsigned long long>(
            reinterpret_cast<float4*>(a.cstate + (size_t)blockIdx.x * CSTATE_FLOATS) + (size_t)(2 * s) * ROWS + row_l);
        uint32_t acc0 = tmem + t_lane + (uint32_t)(32 * s);
        uint32_t hst0 = tmem + t_lane + (uint32_t)(4 * s);     // this thread's 4 columns of an h buffer (+ 16 per chunk)
        uint32_t bars_local = smem_u32(bars), bars_leader;
        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(bars_leader) : "r"(bars_local), "r"(0));
        asm volatile("" : "+l"(cst_base), "+r"(acc0), "+r"(hst0), "+r"(bars_local), "+r"(bars_leader));
        float4* const cst0 = reinterpret_cast<float4*>(cst_base);
        auto arrive_leader = [&](int bar) {
            asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bars_leader + (uint32_t)bar * 8u) : "memory");
        };
        auto wait_bar = [&](int bar, uint32_t parity) {
            uint32_t spins = 0;
            while (!mbar_try_wait_addr(bars_local + (uint32_t)bar * 8u, parity)) { if (++spins > MBAR_WD_SPINS) __trap(); }
        };
        auto cst_at = [&](int hp) { return cst0 + (size_t)(8 * (hp >> 1) + (hp & 1)) * ROWS; };   // [k-group 4 cl + s][half][row]
        int npt = a.n_pair_tiles;
        asm volatile("" : "+r"(npt));
        const int NIe = ((npt - cluster_id + n_clusters - 1) / n_clusters) * T;
        uint32_t ph_out = 0;
        int t = -1, tile = cluster_id - n_clusters;

        for (int w = 0; w < NIe; ++w) {
            if (++t == T) t = 0;
            if (t == 0) tile += n_clusters;
            const bool final_out = has_out && t == T - 1;
            const bool keep_h = t + 1 < T || final_out;
            uint32_t r[16];
            float4 cbuf[2];
            float hq[4];
            cbuf[0] = cbuf[1] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            if (t > 0) cbuf[0] = __ldcg(cst_at(0));
            wait_bar(BAR_ACC_READY + 0, 0);                     // each slot is used twice per item: parity = (chunk >> 1) & 1
            fence_after_sync();
            tmem_ld_x16(acc0, r);
#pragma unroll
            for (int hp = 0; hp < 2 * NCHL; ++hp) {
                const int cl = hp >> 1, half = hp & 1, slot = cl & 1;
                tmem_ld_wait();
                float pa[16];                                  // ex2 arguments (bias is in the accumulator); two columns per multiply
#pragma unroll
                for (int i = 0; i < 16; i += 2) {
                    const F2 v = pk(__uint_as_float(r[i]), __uint_as_float(r[i + 1])) * splat(NEG2LOG2E);
                    pa[i] = lo(v); pa[i + 1] = hi(v);
                }
                if (half == 1) {                               // chunk drained: its issuer may refill the slot
                    fence_before_sync();
                    __syncwarp();
                    if (lane == 0) arrive_leader(BAR_SLOT_FREE + slot);
                }
                const float cp[4] = {cbuf[hp & 1].x, cbuf[hp & 1].y, cbuf[hp & 1].z, cbuf[hp & 1].w};
                if (hp + 1 < 2 * NCHL) cbuf[(hp + 1) & 1] = t > 0 ? __ldcg(cst_at(hp + 1)) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                if (half == 0) tmem_ld_x16(acc0 + (uint32_t)(slot * 128 + 16), r);
                float hv[4], cn[4];
#pragma unroll
                for (int u = 0; u < 4; u += 2) {               // two cells per instruction stream (packed fp32 pairs)
                    F2 c2 = pk(cp[u], cp[u + 1]), h2;
                    tc::lstm_cell2(pk(pa[4 * u + 0], pa[4 * u + 4]), pk(pa[4 * u + 1], pa[4 * u + 5]), pk(pa[4 * u + 2], pa[4 * u + 6]),
                                   pk(pa[4 * u + 3], pa[4 * u + 7]), c2, h2);
                    cn[u] = lo(c2); cn[u + 1] = hi(c2);
                    hv[u] = lo(h2); hv[u + 1] = hi(h2);
                }
                if (t + 1 < T) __stcg(cst_at(hp), make_float4(cn[0], cn[1], cn[2], cn[3]));
                if (half == 0) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) hq[u] = hv[u];
                } else {
                    if (keep_h) {                              // h_t as fp16 pairs hi + lo: operands of the next step / of the output product
                        uint32_t hi[4], lo[4];
                        split2(hq[0], hq[1], hi[0], lo[0]); split2(hq[2], hq[3], hi[1], lo[1]);
                        split2(hv[0], hv[1], hi[2], lo[2]); split2(hv[2], hv[3], hi[3], lo[3]);
                        const uint32_t col = (uint32_t)((t + 1) & 1) * H_COLS + (uint32_t)(16 * cl);
                        tmem_st_x4(hst0 + HH_COL + col, hi[0], hi[1], hi[2], hi[3]);
                        tmem_st_x4(hst0 + HL_COL + col, lo[0], lo[1], lo[2], lo[3]);
                        tmem_st_wait();
                    }
                    if (a.out_units) {                         // the next layer's input: scaled by its 1/(1-p) BEFORE the split
                        const float os = a.out_scale;
                        uint32_t hi[4], lo[4];
                        split2(hq[0] * os, hq[1] * os, hi[0], lo[0]); split2(hq[2] * os, hq[3] * os, hi[1], lo[1]);
                        split2(hv[0] * os, hv[1] * os, hi[2], lo[2]); split2(hv[2] * os, hv[3] * os, hi[3], lo[3]);
                        const size_t at = ((((size_t)tile * T + t) * 2 + rank) * KG + 4 * cl + s) * ROWS + row_l;
                        a.out_units[at] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                        a.out_units_lo[at] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                    }
                    fence_before_sync();
                    __syncwarp();
                    if (lane == 0) arrive_leader(BAR_H_READY + cl);
                }
                if (half == 1 && hp + 1 < 2 * NCHL) {          // the next chunk's first half
                    wait_bar(BAR_ACC_READY + ((slot + 1) & 1), (uint32_t)(((hp + 1) >> 1) >> 1));
                    fence_after_sync();
                    tmem_ld_x16(acc0 + (uint32_t)(((slot + 1) & 1) * 128), r);
                }
            }
            if (final_out) {                                   // output_layer (nn_models.py:189), last step of the last layer only
                wait_bar(BAR_OUT_READY, ph_out);
                ph_out ^= 1;
                fence_after_sync();
                uint32_t o32[32];                              // columns 0..15: h_T x fp16(W_o)^T, 16..31: h_T x (W_o - fp16(W_o))^T
                tmem_ld_x32(tmem + t_lane + HH_COL + (uint32_t)((T & 1) ^ 1) * H_COLS, o32);
                tmem_ld_wait();
                const int row = (tile * 2 + (int)rank) * ROWS + row_l;
                if (row < a.rows) {
                    const int e = row / a.n, smp = row - e * a.n;
                    const int bb = e / a.nF, fb = stream_frame0(a.stream_frames, a.frame0, bb), f = fb + e % a.nF;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int o = s + 4 * i;
                        if (o < a.O && fb >= 0) {
                            const float y = __uint_as_float(tc::pick4(o32, i, s)) + __uint_as_float(tc::pick4(o32, 4 + i, s)) + __ldg(a.bo + o);
                            a.preds[((((size_t)bb * a.pred_ring + f % a.pred_ring) * a.n_out) + smp) * a.O + o] = y;
                        }
                    }
                }
                fence_before_sync();
            }
        }
    } else if (warp >= LOAD_WARP0 && warp < LOAD_WARP0 + LOAD_WARPS) {
        TCX_REG_DEC(REGS_LOAD);
        // =================================== loader warps: x_hi, x_lo of item i ==========================================
        const int lt = tid - LOAD_WARP0 * 32, row_l = lt & (ROWS - 1), half = lt >> 7;
        const bool unit_mode = a.in_mode == tc::IN_UNITS || a.in_mode == tc::IN_SHARED_UNITS;
        int t = -1, tile = cluster_id - n_clusters;
        int e = 0, smp = 0, bidx = 0, f = 0, row = 0;
        bool valid = false;
        for (int i = 0; i < NI; ++i) {
            if (++t == T) t = 0;
            if (t == 0) {
                tile += n_clusters;
                row = (tile * 2 + (int)rank) * ROWS + row_l;
                valid = row < a.rows;
                e = valid ? row / a.n : 0; smp = valid ? row - e * a.n : 0;
                bidx = e / a.nF; f = stream_frame0(a.stream_frames, a.frame0, bidx) + e % a.nF;
            }
            if (unit_mode) {
                const uint32_t stream = a.stream_id0 + (uint32_t)bidx;
                size_t off;
                if (a.in_mode == tc::IN_UNITS) off = ((((size_t)tile * T + t) * 2 + rank) * KG) * ROWS + row_l;
                else off = ((((size_t)(e >> 8) * T + t) * 2 + ((e >> 7) & 1)) * KG) * ROWS + (e & 127);   // one row per estimate, 128-row CTAs
                const uint4* src_hi = reinterpret_cast<const uint4*>(a.in) + off;
                const uint4* src_lo = reinterpret_cast<const uint4*>(a.in_lo) + off;
                const int j0 = half * (KG / 2);
#pragma unroll 1
                for (int b0 = j0; b0 < j0 + KG / 2; b0 += 2) {
                    uint4 vh[2], vl[2];
#pragma unroll
                    for (int jj = 0; jj < 2; ++jj) {
                        vh[jj] = valid ? __ldg(src_hi + (size_t)(b0 + jj) * ROWS) : make_uint4(0, 0, 0, 0);
                        vl[jj] = valid ? __ldg(src_lo + (size_t)(b0 + jj) * ROWS) : make_uint4(0, 0, 0, 0);
                    }
                    if (a.mask_mode == APE_MASK_PHILOX) {
#pragma unroll
                        for (int jj = 0; jj < 2; ++jj) {
                            const uint4 m = APE_PHILOX_DRAW(a, stream, (uint32_t)f, (uint32_t)smp, (uint32_t)a.gap, (uint32_t)t,
                                                            (uint32_t)(b0 + jj), a.keep_thr16);
                            vh[jj].x &= m.x; vh[jj].y &= m.y; vh[jj].z &= m.z; vh[jj].w &= m.w;
                            vl[jj].x &= m.x; vl[jj].y &= m.y; vl[jj].z &= m.z; vl[jj].w &= m.w;
                        }
                    } else if (a.mask_mode == APE_MASK_INJECTED && valid) {
#pragma unroll
                        for (int jj = 0; jj < 2; ++jj) {
                            const uint2 mm = __ldg(reinterpret_cast<const uint2*>(
                                a.masks + ((((size_t)e * a.n_gaps + a.gap) * T + t) * a.n + smp) * H + (b0 + jj) * 8));
                            uint4 m;
                            m.x = ((mm.x & 0xFFu) ? 0xFFFFu : 0u) | ((mm.x & 0xFF00u) ? 0xFFFF0000u : 0u);
                            m.y = ((mm.x & 0xFF0000u) ? 0xFFFFu : 0u) | ((mm.x & 0xFF000000u) ? 0xFFFF0000u : 0u);
                            m.z = ((mm.y & 0xFFu) ? 0xFFFFu : 0u) | ((mm.y & 0xFF00u) ? 0xFFFF0000u : 0u);
                            m.w = ((mm.y & 0xFF0000u) ? 0xFFFFu : 0u) | ((mm.y & 0xFF000000u) ? 0xFFFF0000u : 0u);
                            vh[jj].x &= m.x; vh[jj].y &= m.y; vh[jj].z &= m.z; vh[jj].w &= m.w;
                            vl[jj].x &= m.x; vl[jj].y &= m.y; vl[jj].z &= m.z; vl[jj].w &= m.w;
                        }
                    }
                    if (b0 == j0 && i >= 1) mbar_wait_wd(&bars[BAR_X_DONE], ((uint32_t)(i - 1)) & 1u);
#pragma unroll
                    for (int jj = 0; jj < 2; ++jj) {
                        *reinterpret_cast<uint4*>(sXh + unit_offset(ROWS, row_l, b0 + jj)) = vh[jj];
                        *reinterpret_cast<uint4*>(sXl + unit_offset(ROWS, row_l, b0 + jj)) = vl[jj];
                    }
                }
            } else {                                           // layer 0: fp32 features (window of the ring, or dense rows)
                if (i >= 1) mbar_wait_wd(&bars[BAR_X_DONE], ((uint32_t)(i - 1)) & 1u);
                const float* src = nullptr;
                if (valid) {
                    if (a.in_mode == tc::IN_DENSE_F32) {
                        src = reinterpret_cast<const float*>(a.in) + ((size_t)row * T + t) * a.Kin;
                    } else {                                   // sliding window, clamped at frame 0 (estimator.py:96-97)
                        int fw = f - T + 1 + t;
                        fw = fw < 0 ? 0 : fw;
                        src = reinterpret_cast<const float*>(a.in) + ((size_t)bidx * a.feat_ring + fw % a.feat_ring) * a.Kin;
                    }
                }
                for (int j = half; j < kgx; j += 2) {
                    float v[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) v[k] = (valid && 8 * j + k < a.Kin) ? __ldg(src + 8 * j + k) : 0.0f;
                    uint32_t hi[4], lo[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) split2(v[2 * k], v[2 * k + 1], hi[k], lo[k]);
                    *reinterpret_cast<uint4*>(sXh + unit_offset(ROWS, row_l, j)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                    *reinterpret_cast<uint4*>(sXl + unit_offset(ROWS, row_l, j)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive_leader(&bars[BAR_X_READY], rank);
        }
    } else {
      TCX_REG_DEC(REGS_MMA);
      if (warp >= MMA_WARP && warp < MMA_WARP + N_ISSUERS) {
        if (rank == 0) {
            // =============================== MMA issuers (leader CTA): issuer k owns accumulator slot k ========================
            const uint32_t my_slot = (uint32_t)(warp - MMA_WARP);
            const uint32_t idesc = make_idesc_f16(256, 128), idesc_out = make_idesc_f16(256, OUT_N);
            const uint64_t dXh = make_desc(smem_u32(sXh), LBO_A, SBO), dXl = make_desc(smem_u32(sXl), LBO_A, SBO);
            const uint64_t dW = make_desc(smem_u32(sW), LBO_B, SBO), dOnes = make_desc(smem_u32(sOnes), LBO_A, SBO);
            const uint32_t bar_full = smem_u32(&bars[BAR_W_FULL]), bar_empty = smem_u32(&bars[BAR_W_EMPTY]);
            const uint32_t d_tmem = tmem + my_slot * 128u;
            const uint32_t nx = (uint32_t)kgx / 2;             // K = 16 MMAs of an x-part
            uint32_t wslot = 0, gpiece = 0, uses = 0;
            auto ring_next = [&]() { wslot = wslot + 1 == NP ? 0 : wslot + 1; ++gpiece; };
            auto wait_full = [&]() {
                uint32_t spins = 0;
                while (!mbar_try_wait_addr(bar_full + (gpiece & (NFULL - 1)) * 8, (gpiece / NFULL) & 1)) { if (++spins > MBAR_WD_SPINS) __trap(); }
                fence_after_sync();
            };
            auto chunk = [&](int cl, bool mine, int t, int w) {
                if (!mine) { ring_next(); ring_next(); if (t > 0) { ring_next(); ring_next(); } return; }
                if (uses >= 1) mbar_wait_wd(&bars[BAR_SLOT_FREE + my_slot], (uses & 1) ^ 1);
                ++uses;
                wait_full();                                   // Wx_hi (+ bias rows): x_hi, ones, x_lo
                if (elect_one()) {
                    const uint64_t bd = dW + wslot * (SLOT_BYTES >> 4);
                    for (uint32_t m = 0; m < nx; ++m) mma_f16<2>(d_tmem, dXh + m * (2 * LBO_A >> 4), bd + m * (2 * LBO_B >> 4), idesc, m > 0 ? 1u : 0u);
                    mma_f16<2>(d_tmem, dOnes, bd + nx * (2 * LBO_B >> 4), idesc, 1u);
                    for (uint32_t m = 0; m < nx; ++m) mma_f16<2>(d_tmem, dXl + m * (2 * LBO_A >> 4), bd + m * (2 * LBO_B >> 4), idesc, 1u);
                    commit_pair_addr(bar_empty + wslot * 8, 0x3);
                }
                __syncwarp();
                ring_next();
                wait_full();                                   // Wx_lo: x_hi
                if (elect_one()) {
                    const uint64_t bd = dW + wslot * (SLOT_BYTES >> 4);
                    for (uint32_t m = 0; m < nx; ++m) mma_f16<2>(d_tmem, dXh + m * (2 * LBO_A >> 4), bd + m * (2 * LBO_B >> 4), idesc, 1u);
                    commit_pair_addr(bar_empty + wslot * 8, 0x3);
                    if (t == 0) commit_pair(&bars[BAR_ACC_READY + my_slot], 0x3);
                    if (cl >= NCHL - 2) commit_pair(&bars[BAR_X_DONE], 0x3);      // this issuer's last x-part of the item
                }
                __syncwarp();
                ring_next();
                if (t > 0) {
                    mbar_wait_wd(&bars[BAR_H_READY + NCHL - 1], ((uint32_t)(w - 1)) & 1u);    // all of h_{t-1} (slices are published in order)
                    fence_after_sync();
                    const uint32_t hh = tmem + HH_COL + (uint32_t)(t & 1) * H_COLS, hl = tmem + HL_COL + (uint32_t)(t & 1) * H_COLS;
                    wait_full();                               // Wh_hi: h_hi, h_lo
                    if (elect_one()) {
                        const uint64_t bd = dW + wslot * (SLOT_BYTES >> 4);
#pragma unroll
                        for (uint32_t m = 0; m < KG / 2; ++m) mma_f16_ts<2>(d_tmem, hh + 8 * m, bd + m * (2 * LBO_B >> 4), idesc, 1u);
#pragma unroll
                        for (uint32_t m = 0; m < KG / 2; ++m) mma_f16_ts<2>(d_tmem, hl + 8 * m, bd + m * (2 * LBO_B >> 4), idesc, 1u);
                        commit_pair_addr(bar_empty + wslot * 8, 0x3);
                    }
                    __syncwarp();
                    ring_next();
                    wait_full();                               // Wh_lo: h_hi
                    if (elect_one()) {
                        const uint64_t bd = dW + wslot * (SLOT_BYTES >> 4);
#pragma unroll
                        for (uint32_t m = 0; m < KG / 2; ++m) mma_f16_ts<2>(d_tmem, hh + 8 * m, bd + m * (2 * LBO_B >> 4), idesc, 1u);
                        commit_pair_addr(bar_empty + wslot * 8, 0x3);
                        commit_pair(&bars[BAR_ACC_READY + my_slot], 0x3);
                    }
                    __syncwarp();
                    ring_next();
                }
            };
            // output layer of a finished tile: h_T (hi, then lo; TMEM buffers T & 1) x [fp16(W_o) | W_o - fp16(W_o)]^T into the other h_hi buffer
            auto out_piece = [&](uint32_t item_parity) {
                if (my_slot == 0) {
                    mbar_wait_wd(&bars[BAR_H_READY + NCHL - 1], item_parity);
                    wait_full();
                    if (elect_one()) {
                        const uint64_t bd = make_desc(smem_u32(sW) + wslot * SLOT_BYTES, (OUT_N / 2) * 16, SBO);
                        const uint32_t ah = tmem + HH_COL + (uint32_t)(T & 1) * H_COLS, al = tmem + HL_COL + (uint32_t)(T & 1) * H_COLS;
                        const uint32_t dt = tmem + HH_COL + (uint32_t)((T & 1) ^ 1) * H_COLS;
#pragma unroll
                        for (uint32_t m = 0; m < KG / 2; ++m) mma_f16_ts<2>(dt, ah + 8 * m, bd + m * (2 * (OUT_N / 2) * 16 >> 4), idesc_out, m > 0 ? 1u : 0u);
#pragma unroll
                        for (uint32_t m = 0; m < KG / 2; ++m) mma_f16_ts<2>(dt, al + 8 * m, bd + m * (2 * (OUT_N / 2) * 16 >> 4), idesc_out, 1u);
                        commit_pair_addr(bar_empty + wslot * 8, 0x3);
                        commit_pair(&bars[BAR_OUT_READY], 0x3);
                    }
                    __syncwarp();
                }
                ring_next();
            };
            int t = -1;
            for (int w = 0; w < NI; ++w) {
                if (++t == T) t = 0;
                mbar_wait_wd(&bars[BAR_X_READY], (uint32_t)w & 1u);
                fence_after_sync();
                for (int cl = 0; cl < NCHL; ++cl) {
                    if (cl == 2 && has_out && t == 0 && w >= 1) out_piece(((uint32_t)(w - 1)) & 1u);   // the previous tile's output layer
                    chunk(cl, (uint32_t)(cl & 1) == my_slot, t, w);
                }
            }
            if (has_out) out_piece(((uint32_t)(NI - 1)) & 1u);
        } else if (warp == MMA_WARP && lane == 0) {
            // =============================== peer CTA: forward "piece landed in my ring" to the leader ==================
            uint32_t gpiece = 0;
            auto forward = [&]() {
                mbar_wait_wd(&bars[BAR_W_FULL + (gpiece & (NFULL - 1))], (gpiece / NFULL) & 1);
                mbar_arrive_remote(&bars[BAR_W_FULL + (gpiece & (NFULL - 1))], 0);
                ++gpiece;
            };
            int t = -1;
            for (int w = 0; w < NI; ++w) {
                if (++t == T) t = 0;
                for (int cl = 0; cl < NCHL; ++cl) {
                    if (cl == 2 && has_out && t == 0 && w >= 1) forward();
                    forward(); forward();
                    if (t > 0) { forward(); forward(); }
                }
            }
            if (has_out) forward();
        }
      } else if (warp == TMA_WARP && lane == 0) {
        // =================================== weight-ring producer (one lane per CTA) =====================================
        const uint32_t p0b = tcx_blob::p0_bytes(kgx), p1b = tcx_blob::p1_bytes(kgx), phb = tcx_blob::ph_bytes(H), cb = tcx_blob::chunk_bytes(H, kgx);
        const uint8_t* Wl = a.Ww + (size_t)rank * NCHL * cb;   // this CTA's half of the layer's pieces
        uint32_t wslot = 0, wphase = 0, gpiece = 0;
        bool wrapped = false;
        auto put = [&](const uint8_t* src, uint32_t bytes) {
            uint64_t* full = &bars[BAR_W_FULL + (gpiece & (NFULL - 1))];
            if (wrapped) mbar_wait_wd(&bars[BAR_W_EMPTY + wslot], wphase ^ 1);
            mbar_arrive_expect_tx(full, bytes);
            bulk_g2s(sW + wslot * SLOT_BYTES, src, bytes, full);
            if (++wslot == NP) { wslot = 0; wphase ^= 1; wrapped = true; }
            ++gpiece;
        };
        int t = -1;
        for (int w = 0; w < NI; ++w) {
            if (++t == T) t = 0;
            for (int cl = 0; cl < NCHL; ++cl) {
                if (cl == 2 && has_out && t == 0 && w >= 1) put(a.Wo16 + (size_t)rank * OUT_BYTES, OUT_BYTES);
                const uint8_t* c0 = Wl + (size_t)cl * cb;
                put(c0, p0b);
                put(c0 + p0b, p1b);
                if (t > 0) { put(c0 + p0b + p1b, phb); put(c0 + p0b + p1b + phb, phb); }
            }
        }
        if (has_out) put(a.Wo16 + (size_t)rank * OUT_BYTES, OUT_BYTES);
      }
    }
    __syncwarp();
    fence_before_sync();
    cluster_sync();
    tc::timeline_stamp(a.timeline, 2);
    if (warp == MMA_WARP) tmem_dealloc<2>(tmem, TMEM_COLS);
}

bool supported(int Hh, int I, int O) { return Hh == H && ape_pack_kin_pad(0, I, Hh) <= Hh && O <= (int)OUT_N / 2; }

size_t scratch_bytes(int sm_count) { return (size_t)sm_count * CSTATE_FLOATS * sizeof(float); }

int launch_layer(const TcLayerArgs& a, int sm_count, cudaStream_t st) {
    if (a.kgx < 2 || a.kgx > KG || (a.kgx & 1) || a.rpc != ROWS || !a.cstate || !a.Ww || a.T < 1) return APE_ERR_UNSUPPORTED;
    const bool unit_mode = a.in_mode == tc::IN_UNITS || a.in_mode == tc::IN_SHARED_UNITS;
    if (unit_mode && (!a.in_lo || a.kgx != KG)) return APE_ERR_BAD_ARG;
    if (a.out_units && !a.out_units_lo) return APE_ERR_BAD_ARG;
    if (a.preds && (!a.Wo16 || a.O > (int)OUT_N / 2)) return APE_ERR_UNSUPPORTED;
    APE_CUDA_TRY(cudaFuncSetAttribute(lstm_layer_tcx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
    int clusters = sm_count / 2;
    if (clusters > a.n_pair_tiles) clusters = a.n_pair_tiles;
    lstm_layer_tcx_kernel<<<2 * clusters, THREADS, SMEM, st>>>(a);
    return check_launch();
}

}  // namespace tcx
}  // namespace ape
