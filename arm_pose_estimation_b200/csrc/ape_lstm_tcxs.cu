// Stage 2, SPLIT-PRECISION tensor-core variant for H = 256 (one layer per launch): the watch-only and pocket models' tcgen05 path
// when the single-pass fp16 kernel (ape_lstm_tcs.cu) fails BatchedEstimator's probe.  Arithmetic of ape_lstm_tcx.cu: every operand
// an fp16 pair v = hi + lo, a product is three tensor-core passes a_hi b_hi + a_lo b_hi + a_hi b_lo into one fp32 accumulator, the
// bias enters as an fp16 pair against a tile of ones, ex2 / rcp cell update.  Same weight blob layout as ape_lstm_tcx.cu, at H = 256.
//
// Memory plan.  A CTA owns 128 rows (= TMEM lanes); one fp16 operand tile of 256 K-values is 64 KB of shared memory or 128 TMEM
// columns.  ape_lstm_tcx.cu keeps h_hi and h_lo double-buffered in TMEM (4 x 128 columns at H = 256) next to two accumulator slots
// (256 columns) - 768 of the 512 columns.  Here:
//   * TMEM: two 128-column accumulator slots (one 32-unit chunk x 4 gates each, used alternately by the chunk sequence) + h_hi and
//     h_lo SINGLE-buffered (2 x 128 columns): the A operands of the recurrent MMAs;
//   * h_t cannot go to TMEM while the later chunks of step t still multiply h_{t-1}: each epilogue thread stages its h_t slices
//     (hi and lo words) in a per-CTA scratch next to the cell state (L2-resident, 128 KB per CTA each) and moves them into TMEM
//     (tcgen05.st) once chunk NCH - 1's accumulator is ready - at that point every MMA that reads h_{t-1} has retired - then
//     publishes h_t.  The x-parts of the next step's chunks 0 and 1 can run before that point;
//   * shared memory: x_hi and x_lo single-buffered (2 x 64 KB), the bias tile of ones (4 KB), and a ring of 5 slots of 18 KB that
//     cp.async.bulk fills from L2.  Each chunk's four weight parts (Wx_hi + the bias K step, Wx_lo, Wh_hi, Wh_lo) travel in pieces
//     of at most 16 k-groups (the bias k-groups ride with the last Wx_hi piece);
//   * the output layer of the last layer: h_T(hi, lo) x [fp16(W_o) | W_o - fp16(W_o)]^T (N = 64, O <= 32) into accumulator slot 1.
// Per step and CTA pair 776 K = 16 MMAs (layer >= 1) against 256 in ape_lstm_tcs.cu, and ~1 MB of weights per CTA from L2.
#include "ape_common.cuh"
#include "ape_lstm_pack.h"
#include "ape_lstm_tc_args.cuh"
#include "ape_umma.cuh"

namespace ape {
namespace tcxs {

using tc::TcLayerArgs;

constexpr int H = 256, NCH = H / 32, KG = H / 8;
constexpr int EPI_WARPS = 16, LOAD_WARPS = 8, N_ISSUERS = 2;
constexpr int THREADS = (EPI_WARPS + LOAD_WARPS + 4) * 32;       // 896 = 7 warpgroups
constexpr int MMA_WARP = 0, TMA_WARP = 2, LOAD_WARP0 = 4, EPI_WARP0 = 12;   // epilogue warps on the highest ids (scheduler priority)
constexpr int REGS_EPI = 96, REGS_LOAD = 40, REGS_MMA = 40;
static_assert(EPI_WARPS * 32 * REGS_EPI + LOAD_WARPS * 32 * REGS_LOAD + 128 * REGS_MMA <= THREADS * 72, "register file");
#define TCXS_REG_INC(n) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(n))
#define TCXS_REG_DEC(n) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(n))
constexpr int ROWS = 128;
constexpr uint32_t KG_BYTES_B = 64 * 16;                   // one k-group of a 64-column weight tile
constexpr int PIECE_KG = 16;                               // weight k-groups per ring piece (8 K = 16 steps)
constexpr uint32_t SLOT_BYTES = (PIECE_KG + 2) * KG_BYTES_B;   // 18 KB: a piece + the bias K step
constexpr uint32_t A_BYTES = KG * ROWS * 16;               // one operand tile (64 KB)
constexpr uint32_t ONES_BYTES = 2 * ROWS * 16;             // constant A tile of the bias K step
constexpr uint32_t OUT_N = 64;                             // output product: 32 outputs x {fp16(W_o), remainder}
constexpr uint32_t OUT_BYTES = KG * (OUT_N / 2) * 16;      // this CTA's tile of it (16 KB)
static_assert(OUT_BYTES <= SLOT_BYTES, "the output-layer tile must fit a ring slot");
constexpr uint32_t BAR_BLOCK_BYTES = 512;
constexpr int NP = (int)((227 * 1024 - 2 * A_BYTES - ONES_BYTES - BAR_BLOCK_BYTES) / SLOT_BYTES);   // ring depth: 5
constexpr int NFULL = 8;                                   // "piece landed" barriers by piece number (> NP: never alias)
static_assert(NP >= 4 && NP < NFULL, "weight ring depth");
constexpr uint32_t SMEM = 2 * A_BYTES + NP * SLOT_BYTES + ONES_BYTES + BAR_BLOCK_BYTES;
static_assert(SMEM <= 227 * 1024, "shared memory budget");
constexpr uint32_t HH_COL = 256, HL_COL = 384, TMEM_COLS = 512;
static_assert(HL_COL + H / 2 <= TMEM_COLS, "two accumulator slots + h_hi + h_lo");
constexpr size_t CSTATE_FLOATS = (size_t)H * ROWS;         // per CTA: cell state [k-group * 2 + half][row] float4
constexpr size_t SCRATCH_FLOATS = 2 * CSTATE_FLOATS;       // ... followed by the h_t staging area [chunk][hi, lo][s][row] uint4
using tc::NEG2LOG2E;
using tc::split2;
static_assert(2 * OUT_BYTES == tc::wo16_bytes(H), "the output-layer tiles of the tcx blob");

enum {
    BAR_X_READY = 0, BAR_X_DONE = 1, BAR_ACC_READY = 2, BAR_SLOT_FREE = 4, BAR_H_READY = 6, BAR_OUT_READY = 7, BAR_W_FULL = 8,
    BAR_W_EMPTY = BAR_W_FULL + NFULL, BAR_H0_READY = BAR_W_EMPTY + NP, BAR_COUNT = BAR_H0_READY + 1
};
static_assert(BAR_COUNT * 8 + 16 <= BAR_BLOCK_BYTES, "barrier block too small");

// ring pieces per chunk: x-part pieces (Wx_hi, then the same count of Wx_lo) and, for a step with a recurrent half, 2 Wh_hi + 2 Wh_lo
__host__ __device__ constexpr int x_pieces(int kgx) { return (kgx + PIECE_KG - 1) / PIECE_KG; }
constexpr int H_PIECES = KG / PIECE_KG;
// Ring pieces of one chunk of step t.  A step has a recurrent half when t > 0 or, with a caller-supplied initial state, at t = 0
// too (on h_0).  The producer, both issuers and the peer's forwarder walk the ring by this one count.
__host__ __device__ constexpr int chunk_pieces(int kgx, int t, bool state) { return 2 * x_pieces(kgx) + (t > 0 || state ? 2 * H_PIECES : 0); }

// STATE: a caller-supplied initial state (a.h0, a.c0).  At the start of every tile the epilogue writes h_0 as fp16 pairs into the h
// buffers step 0 reads and publishes it on BAR_H0_READY; the cell starts from c_0; step 0 runs its recurrent half after the
// x-part, whose MMAs keep the stateless order and accumulate flags - so h_0 = c_0 = 0 reproduces the stateless kernel bit for bit.
// h_0 has a barrier of its own (one phase per tile): BAR_H_READY keeps one phase per item, the parity the issuers derive from the
// item index.  Sharing it, the epilogue could complete the h_T and h_0 phases before issuer 0 (which never waits for h_T) had
// consumed h_T, and a parity wait can only name the current or the previous phase.
template <bool STATE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
lstm_layer_tcxs_kernel(const __grid_constant__ TcLayerArgs a) {
    using namespace umma;
    constexpr uint32_t LBO_A = ROWS * 16, LBO_B = KG_BYTES_B, SBO = 128;
    const int T = a.T, kgx = a.kgx, nxp = x_pieces(kgx);

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
        mbar_init(&bars[BAR_H_READY], 2 * EPI_WARPS);
        mbar_init(&bars[BAR_OUT_READY], 1);
        if (STATE) mbar_init(&bars[BAR_H0_READY], 2 * EPI_WARPS);
        for (int p = 0; p < NFULL; ++p) mbar_init(&bars[BAR_W_FULL + p], rank == 0 ? 2 : 1);   // leader: own copy + the peer's forward
        for (int p = 0; p < NP; ++p) mbar_init(&bars[BAR_W_EMPTY + p], 1);
        mbar_init_fence();
    }
    fence_proxy_async_smem();
    fence_before_sync();
    cluster_sync();
    fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    tc::timeline_stamp(a.timeline, 1);

    if (warp >= EPI_WARP0 && warp < EPI_WARP0 + EPI_WARPS) {
        TCXS_REG_INC(REGS_EPI);
        // =================================== epilogue warps ===========================================================
        // warp (q, s): rows 32q..32q+31 (its TMEM lane quarter) x the 8 hidden units 8s..8s+7 of every 32-unit chunk
        const int q = warp & 3, s = (warp - EPI_WARP0) >> 2;
        const int row_l = 32 * q + lane;
        const uint32_t t_lane = (uint32_t)(32 * q) << 16;
        float* const scr = a.cstate + (size_t)blockIdx.x * SCRATCH_FLOATS;
        unsigned long long cst_base = reinterpret_cast<unsigned long long>(reinterpret_cast<float4*>(scr) + (size_t)(2 * s) * ROWS + row_l);
        unsigned long long hsg_base = reinterpret_cast<unsigned long long>(
            reinterpret_cast<uint4*>(scr + CSTATE_FLOATS) + (size_t)s * ROWS + row_l);
        uint32_t acc0 = tmem + t_lane + (uint32_t)(32 * s);
        uint32_t hst0 = tmem + t_lane + (uint32_t)(4 * s);     // this thread's 4 columns of an h buffer (+ 16 per chunk)
        uint32_t bars_local = smem_u32(bars), bars_leader;
        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(bars_leader) : "r"(bars_local), "r"(0));
        asm volatile("" : "+l"(cst_base), "+l"(hsg_base), "+r"(acc0), "+r"(hst0), "+r"(bars_local), "+r"(bars_leader));
        float4* const cst0 = reinterpret_cast<float4*>(cst_base);
        uint4* const hsg0 = reinterpret_cast<uint4*>(hsg_base);
        auto arrive_leader = [&](int bar) {
            asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bars_leader + (uint32_t)bar * 8u) : "memory");
        };
        auto wait_bar = [&](int bar, uint32_t parity) {
            uint32_t spins = 0;
            while (!mbar_try_wait_addr(bars_local + (uint32_t)bar * 8u, parity)) { if (++spins > MBAR_WD_SPINS) __trap(); }
        };
        auto cst_at = [&](int hp) { return cst0 + (size_t)(8 * (hp >> 1) + (hp & 1)) * ROWS; };   // [k-group 4 cl + s][half][row]
        auto hsg_at = [&](int cl, int part) { return hsg0 + (size_t)(8 * cl + 4 * part) * ROWS; };  // [chunk][hi, lo][s][row]
        int npt = a.n_pair_tiles;
        asm volatile("" : "+r"(npt));
        const int NIe = ((npt - cluster_id + n_clusters - 1) / n_clusters) * T;
        uint32_t ph_out = 0;
        int t = -1, tile = cluster_id - n_clusters;
        const float4* c0r = nullptr;                           // STATE: this row's c_0 (valid rows only)

        for (int w = 0; w < NIe; ++w) {
            if (++t == T) t = 0;
            if (t == 0) tile += n_clusters;
            if constexpr (STATE) {
                if (t == 0) {
                    // h_0 as fp16 pairs into h_hi / h_lo (this thread: its row, units 32 cl + 8 s + [0, 8) of every chunk).  Nothing
                    // reads them any more: this warp has drained every accumulator of the previous tile's last step and, on the last
                    // layer, waited for its output product (BAR_OUT_READY).
                    const int row = (tile * 2 + (int)rank) * ROWS + row_l;
                    const bool valid = row < a.rows;
                    const float4* h0r = reinterpret_cast<const float4*>(a.h0 + (size_t)(valid ? row : 0) * H) + 2 * s;
                    c0r = valid ? reinterpret_cast<const float4*>(a.c0 + (size_t)row * H) + 2 * s : nullptr;
                    const float4 z = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll
                    for (int cl = 0; cl < NCH; ++cl) {
                        const float4 h_a = valid ? __ldg(h0r + 8 * cl) : z, h_b = valid ? __ldg(h0r + 8 * cl + 1) : z;
                        uint32_t hi[4], lo[4];
                        split2(h_a.x, h_a.y, hi[0], lo[0]); split2(h_a.z, h_a.w, hi[1], lo[1]);
                        split2(h_b.x, h_b.y, hi[2], lo[2]); split2(h_b.z, h_b.w, hi[3], lo[3]);
                        tmem_st_x4(hst0 + HH_COL + (uint32_t)(16 * cl), hi[0], hi[1], hi[2], hi[3]);
                        tmem_st_x4(hst0 + HL_COL + (uint32_t)(16 * cl), lo[0], lo[1], lo[2], lo[3]);
                    }
                    tmem_st_wait();
                    fence_before_sync();
                    __syncwarp();
                    if (lane == 0) arrive_leader(BAR_H0_READY);
                }
            }
            const bool final_out = has_out && t == T - 1;
            const bool keep_h = t + 1 < T || final_out;
            uint32_t r[16];
            float4 cbuf[2];
            float hq[4];
            uint32_t hlast[4], llast[4];
            cbuf[0] = cbuf[1] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            if (t > 0) cbuf[0] = __ldcg(cst_at(0));
            else if (STATE && c0r) cbuf[0] = __ldg(c0r);         // c_0 of units 8 s + [0, 4) of chunk 0
            wait_bar(BAR_ACC_READY + 0, 0);                     // slot k serves chunks k, k+2, ...: parity = (chunk >> 1) & 1
            fence_after_sync();
            tmem_ld_x16(acc0, r);
#pragma unroll
            for (int hp = 0; hp < 2 * NCH; ++hp) {
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
                if (hp + 1 < 2 * NCH)                          // (c_0: units 32 cl + 8 s + 4 half + [0, 4))
                    cbuf[(hp + 1) & 1] = t > 0 ? __ldcg(cst_at(hp + 1))
                                               : (STATE && c0r) ? __ldg(c0r + 8 * ((hp + 1) >> 1) + ((hp + 1) & 1))
                                                                : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
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
                    if (keep_h) {                              // h_t as fp16 pairs hi + lo: staged until h_{t-1} is no longer read
                        uint32_t hi[4], lo[4];
                        split2(hq[0], hq[1], hi[0], lo[0]); split2(hq[2], hq[3], hi[1], lo[1]);
                        split2(hv[0], hv[1], hi[2], lo[2]); split2(hv[2], hv[3], hi[3], lo[3]);
                        if (cl + 1 < NCH) {
                            __stcg(hsg_at(cl, 0), make_uint4(hi[0], hi[1], hi[2], hi[3]));
                            __stcg(hsg_at(cl, 1), make_uint4(lo[0], lo[1], lo[2], lo[3]));
                        } else {
#pragma unroll
                            for (int k = 0; k < 4; ++k) { hlast[k] = hi[k]; llast[k] = lo[k]; }
                        }
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
                }
                if (half == 1 && hp + 1 < 2 * NCH) {          // the next chunk's first half
                    wait_bar(BAR_ACC_READY + ((slot + 1) & 1), (uint32_t)(((hp + 1) >> 1) >> 1) & 1u);
                    fence_after_sync();
                    tmem_ld_x16(acc0 + (uint32_t)(((slot + 1) & 1) * 128), r);
                }
            }
            // Chunk NCH - 1's accumulator was ready: every MMA of this step (all of which precede it or chunk NCH - 2 in their issuer's
            // order) has retired, so h_{t-1} is no longer read and h_t replaces it in TMEM (this thread: its row, 4 columns per chunk).
            if (keep_h) {
                tmem_st_x4(hst0 + HH_COL + (uint32_t)(16 * (NCH - 1)), hlast[0], hlast[1], hlast[2], hlast[3]);
                tmem_st_x4(hst0 + HL_COL + (uint32_t)(16 * (NCH - 1)), llast[0], llast[1], llast[2], llast[3]);
#pragma unroll
                for (int part = 0; part < 2; ++part) {
                    uint4 v[NCH - 1];
#pragma unroll
                    for (int cl = 0; cl + 1 < NCH; ++cl) v[cl] = __ldcg(hsg_at(cl, part));
#pragma unroll
                    for (int cl = 0; cl + 1 < NCH; ++cl)
                        tmem_st_x4(hst0 + (part ? HL_COL : HH_COL) + (uint32_t)(16 * cl), v[cl].x, v[cl].y, v[cl].z, v[cl].w);
                }
                tmem_st_wait();
            }
            fence_before_sync();
            __syncwarp();
            if (lane == 0) arrive_leader(BAR_H_READY);         // every item publishes (the issuers count items)
            if (final_out) {                                   // output_layer (nn_models.py:189), last step of the last layer only
                wait_bar(BAR_OUT_READY, ph_out);
                ph_out ^= 1;
                fence_after_sync();
                uint32_t v[32];
                float y[8];
                tmem_ld_x32(tmem + t_lane + 128u, v);          // h_T x fp16(W_o)^T, outputs 0..31
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 8; ++i) y[i] = __uint_as_float(tc::pick4(v, i, s));
                tmem_ld_x32(tmem + t_lane + 128u + 32u, v);    // h_T x (W_o - fp16(W_o))^T
                tmem_ld_wait();
                fence_before_sync();
                __syncwarp();
                if (lane == 0) arrive_leader(BAR_SLOT_FREE + 1);   // slot 1 may be refilled for the next tile
                const int row = (tile * 2 + (int)rank) * ROWS + row_l;
                if (row < a.rows) {
                    const int e = row / a.n, smp = row - e * a.n;
                    const int bb = e / a.nF, fb = stream_frame0(a.stream_frames, a.frame0, bb), f = fb + e % a.nF;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int o = s + 4 * i;
                        if (o < a.O && fb >= 0) {              // (an inactive stream keeps its prediction ring untouched)
                            const float yo = y[i] + __uint_as_float(tc::pick4(v, i, s)) + __ldg(a.bo + o);
                            a.preds[((((size_t)bb * a.pred_ring + f % a.pred_ring) * a.n_out) + smp) * a.O + o] = yo;
                        }
                    }
                }
            }
        }
    } else if (warp >= LOAD_WARP0 && warp < LOAD_WARP0 + LOAD_WARPS) {
        TCXS_REG_DEC(REGS_LOAD);
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
                    if (a.mask_mode == APE_MASK_PHILOX) {      // one draw masks both halves (the keys of every other stage)
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
      TCXS_REG_DEC(REGS_MMA);
      // The ring's piece sequence, walked identically by the producer, both issuers and the forwarder: per item (tile, t) and chunk
      // nxp Wx_hi pieces (the last with the bias K step), nxp Wx_lo pieces, then (t > 0, or STATE) H_PIECES Wh_hi and H_PIECES Wh_lo
      // pieces (chunk_pieces); after the last step of the last layer's tile, one W_o piece.
      if (warp >= MMA_WARP && warp < MMA_WARP + N_ISSUERS) {
        if (rank == 0) {
            // =============================== MMA issuers (leader CTA): issuer k owns accumulator slot k ========================
            const uint32_t my_slot = (uint32_t)(warp - MMA_WARP);
            const uint32_t idesc = make_idesc_f16(256, 128), idesc_out = make_idesc_f16(256, OUT_N);
            const uint64_t dXh = make_desc(smem_u32(sXh), LBO_A, SBO), dXl = make_desc(smem_u32(sXl), LBO_A, SBO);
            const uint64_t dW = make_desc(smem_u32(sW), LBO_B, SBO), dOnes = make_desc(smem_u32(sOnes), LBO_A, SBO);
            const uint32_t bar_full = smem_u32(&bars[BAR_W_FULL]), bar_empty = smem_u32(&bars[BAR_W_EMPTY]);
            const uint32_t d_tmem = tmem + my_slot * 128u;
            const uint32_t hh = tmem + HH_COL, hl = tmem + HL_COL;
            uint32_t wslot = 0, gpiece = 0, uses = 0, h0_par = 1;   // h0_par: parity of this tile's BAR_H0_READY phase (STATE)
            auto ring_next = [&]() { wslot = wslot + 1 == NP ? 0 : wslot + 1; ++gpiece; };
            auto wait_full = [&]() {
                uint32_t spins = 0;
                while (!mbar_try_wait_addr(bar_full + (gpiece & (NFULL - 1)) * 8, (gpiece / NFULL) & 1)) { if (++spins > MBAR_WD_SPINS) __trap(); }
                fence_after_sync();
            };
            auto wait_slot = [&]() {                           // the epilogue has drained what this slot held before
                if (uses >= 1) mbar_wait_wd(&bars[BAR_SLOT_FREE + my_slot], (uses & 1) ^ 1);
                ++uses;
            };
            auto chunk = [&](int cl, bool mine, int t, int w) {
                const int n_pieces = chunk_pieces(kgx, t, STATE);
                const bool recurrent = n_pieces > 2 * nxp;
                if (!mine) { for (int p = 0; p < n_pieces; ++p) ring_next(); return; }
                wait_slot();
                for (int p = 0; p < nxp; ++p) {                // Wx_hi (+ bias rows): x_hi, ones, x_lo
                    const uint32_t kg0 = (uint32_t)(p * PIECE_KG), nm = (uint32_t)((kgx - p * PIECE_KG < PIECE_KG ? kgx - p * PIECE_KG : PIECE_KG) / 2);
                    wait_full();
                    if (elect_one()) {
                        const uint64_t bd = dW + wslot * (SLOT_BYTES >> 4);
                        for (uint32_t m = 0; m < nm; ++m)
                            mma_f16<2>(d_tmem, dXh + (kg0 / 2 + m) * (2 * LBO_A >> 4), bd + m * (2 * LBO_B >> 4), idesc, (p > 0 || m > 0) ? 1u : 0u);
                        if (p == nxp - 1) mma_f16<2>(d_tmem, dOnes, bd + nm * (2 * LBO_B >> 4), idesc, 1u);
                        for (uint32_t m = 0; m < nm; ++m)
                            mma_f16<2>(d_tmem, dXl + (kg0 / 2 + m) * (2 * LBO_A >> 4), bd + m * (2 * LBO_B >> 4), idesc, 1u);
                        commit_pair_addr(bar_empty + wslot * 8, 0x3);
                    }
                    __syncwarp();
                    ring_next();
                }
                for (int p = 0; p < nxp; ++p) {                // Wx_lo: x_hi
                    const uint32_t kg0 = (uint32_t)(p * PIECE_KG), nm = (uint32_t)((kgx - p * PIECE_KG < PIECE_KG ? kgx - p * PIECE_KG : PIECE_KG) / 2);
                    wait_full();
                    if (elect_one()) {
                        const uint64_t bd = dW + wslot * (SLOT_BYTES >> 4);
                        for (uint32_t m = 0; m < nm; ++m)
                            mma_f16<2>(d_tmem, dXh + (kg0 / 2 + m) * (2 * LBO_A >> 4), bd + m * (2 * LBO_B >> 4), idesc, 1u);
                        commit_pair_addr(bar_empty + wslot * 8, 0x3);
                        if (p == nxp - 1) {
                            if (!recurrent) commit_pair(&bars[BAR_ACC_READY + my_slot], 0x3);
                            if (cl >= NCH - 2) commit_pair(&bars[BAR_X_DONE], 0x3);   // this issuer's last x-part of the item
                        }
                    }
                    __syncwarp();
                    ring_next();
                }
                if (recurrent) {
                    if (STATE && t == 0) mbar_wait_wd(&bars[BAR_H0_READY], h0_par);  // all of h_0 is in TMEM
                    else mbar_wait_wd(&bars[BAR_H_READY], ((uint32_t)(w - 1)) & 1u);  // all of h_{t-1} is in TMEM
                    fence_after_sync();
                    for (int p = 0; p < 2 * H_PIECES; ++p) {   // Wh_hi: h_hi, h_lo; then Wh_lo: h_hi
                        const uint32_t c0 = (uint32_t)((p % H_PIECES) * PIECE_KG * 4);   // TMEM column of the piece's first k-group
                        wait_full();
                        if (elect_one()) {
                            const uint64_t bd = dW + wslot * (SLOT_BYTES >> 4);
#pragma unroll
                            for (uint32_t m = 0; m < PIECE_KG / 2; ++m) mma_f16_ts<2>(d_tmem, hh + c0 + 8 * m, bd + m * (2 * LBO_B >> 4), idesc, 1u);
                            if (p < H_PIECES) {
#pragma unroll
                                for (uint32_t m = 0; m < PIECE_KG / 2; ++m) mma_f16_ts<2>(d_tmem, hl + c0 + 8 * m, bd + m * (2 * LBO_B >> 4), idesc, 1u);
                            }
                            commit_pair_addr(bar_empty + wslot * 8, 0x3);
                            if (p == 2 * H_PIECES - 1) commit_pair(&bars[BAR_ACC_READY + my_slot], 0x3);
                        }
                        __syncwarp();
                        ring_next();
                    }
                }
            };
            // output layer of a finished tile: h_T (hi, then lo) x [fp16(W_o) | W_o - fp16(W_o)]^T into accumulator slot 1 (issuer 1)
            auto out_piece = [&](int w) {
                if (my_slot == 1) {
                    wait_slot();
                    mbar_wait_wd(&bars[BAR_H_READY], (uint32_t)w & 1u);   // h_T is in TMEM
                    wait_full();
                    if (elect_one()) {
                        const uint64_t bd = make_desc(smem_u32(sW) + wslot * SLOT_BYTES, (OUT_N / 2) * 16, SBO);
#pragma unroll
                        for (uint32_t m = 0; m < KG / 2; ++m) mma_f16_ts<2>(d_tmem, hh + 8 * m, bd + m * (2 * (OUT_N / 2) * 16 >> 4), idesc_out, m > 0 ? 1u : 0u);
#pragma unroll
                        for (uint32_t m = 0; m < KG / 2; ++m) mma_f16_ts<2>(d_tmem, hl + 8 * m, bd + m * (2 * (OUT_N / 2) * 16 >> 4), idesc_out, 1u);
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
                if (STATE && t == 0) h0_par ^= 1;
                mbar_wait_wd(&bars[BAR_X_READY], (uint32_t)w & 1u);
                fence_after_sync();
                for (int cl = 0; cl < NCH; ++cl) chunk(cl, (uint32_t)(cl & 1) == my_slot, t, w);
                if (has_out && t == T - 1) out_piece(w);
            }
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
                const int n_pieces = NCH * chunk_pieces(kgx, t, STATE) + (has_out && t == T - 1 ? 1 : 0);
                for (int p = 0; p < n_pieces; ++p) forward();
            }
        }
      } else if (warp == TMA_WARP && lane == 0) {
        // =================================== weight-ring producer (one lane per CTA) =====================================
        const uint32_t p0b = tcx_blob::p0_bytes(kgx), p1b = tcx_blob::p1_bytes(kgx), cb = tcx_blob::chunk_bytes(H, kgx);
        const uint8_t* Wl = a.Ww + (size_t)rank * NCH * cb;    // this CTA's half of the layer's pieces
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
            for (int cl = 0; cl < NCH; ++cl) {
                const uint8_t* c0 = Wl + (size_t)cl * cb;
                for (int p = 0; p < nxp; ++p) {                // Wx_hi in pieces of PIECE_KG k-groups, the last one with the bias K step
                    const int nkg = kgx - p * PIECE_KG < PIECE_KG ? kgx - p * PIECE_KG : PIECE_KG;
                    put(c0 + (size_t)p * PIECE_KG * KG_BYTES_B, (uint32_t)(nkg + (p == nxp - 1 ? 2 : 0)) * KG_BYTES_B);
                }
                for (int p = 0; p < nxp; ++p) {
                    const int nkg = kgx - p * PIECE_KG < PIECE_KG ? kgx - p * PIECE_KG : PIECE_KG;
                    put(c0 + p0b + (size_t)p * PIECE_KG * KG_BYTES_B, (uint32_t)nkg * KG_BYTES_B);
                }
                if (chunk_pieces(kgx, t, STATE) > 2 * nxp)      // the recurrent half: Wh_hi, Wh_lo
                    for (int p = 0; p < 2 * H_PIECES; ++p) put(c0 + p0b + p1b + (size_t)p * PIECE_KG * KG_BYTES_B, PIECE_KG * KG_BYTES_B);
            }
            if (has_out && t == T - 1) put(a.Wo16 + (size_t)rank * OUT_BYTES, OUT_BYTES);
        }
      }
    }
    __syncwarp();
    fence_before_sync();
    cluster_sync();
    tc::timeline_stamp(a.timeline, 2);
    if (warp == MMA_WARP) tmem_dealloc<2>(tmem, TMEM_COLS);
}

bool supported(int Hh, int I, int O) { return Hh == H && I >= 1 && ape_pack_kin_pad(0, I, Hh) <= Hh && O >= 1 && O <= (int)OUT_N / 2; }

size_t scratch_bytes(int sm_count) { return (size_t)sm_count * SCRATCH_FLOATS * sizeof(float); }

int launch_layer(const TcLayerArgs& a, int sm_count, cudaStream_t st) {
    if (a.kgx < 2 || a.kgx > KG || (a.kgx & 1) || a.rpc != ROWS || !a.cstate || !a.Ww || a.T < 1) return APE_ERR_UNSUPPORTED;
    const bool unit_mode = a.in_mode == tc::IN_UNITS || a.in_mode == tc::IN_SHARED_UNITS;
    if (unit_mode && (!a.in_lo || a.kgx != KG)) return APE_ERR_BAD_ARG;
    if (a.out_units && !a.out_units_lo) return APE_ERR_BAD_ARG;
    if (a.preds && (!a.Wo16 || a.O > (int)OUT_N / 2)) return APE_ERR_UNSUPPORTED;
    if ((a.h0 != nullptr) != (a.c0 != nullptr)) return APE_ERR_BAD_ARG;
    auto kernel = a.h0 ? lstm_layer_tcxs_kernel<true> : lstm_layer_tcxs_kernel<false>;
    APE_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
    int clusters = sm_count / 2;
    if (clusters > a.n_pair_tiles) clusters = a.n_pair_tiles;
    kernel<<<2 * clusters, THREADS, SMEM, st>>>(a);
    return check_launch();
}

}  // namespace tcxs
}  // namespace ape
