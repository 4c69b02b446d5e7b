// Stage 2, tensor-core variant for H = 256 (the watch-only and pocket models): the same CTA-pair tcgen05 design as
// ape_lstm_tc.cu, re-balanced for a layer whose fp16 gate weights (1 MB) no longer fit the pair's shared memory.
//
//   * A CTA PAIR (cluster of 2, cta_group::2, M = 256) owns 256 (estimate, MC-sample) rows for all T steps of a layer.
//   * Gate WEIGHTS STREAM from L2 through a shared-memory ring of 32 KB slots, filled by one thread per CTA with bulk
//     asynchronous copies (cp.async.bulk, mbarrier complete_tx).  A piece is up to 32 k-groups (256 K-values: a whole x- or
//     recurrent part) x this CTA's 64 gate columns of a 32-unit chunk = up to 16 K=16 MMAs.  The MMA issuer consumes pieces in a fixed per-step order
//     (walk_step below, evaluated on the host into a table that travels as a kernel parameter), the producer walks the
//     same table, and every slot is released by a tcgen05.commit once its MMAs have retired.  The peer CTA forwards its
//     ring's "full" events to the leader, because the leader's MMAs read both CTAs' halves of B.
//   * To make room for a ring deep enough to cover the L2 latency, the recurrent operand does NOT live in shared memory:
//     h_t is written by the epilogue warps straight into TENSOR MEMORY as packed fp16 pairs (tcgen05.st, lane = row) and
//     the recurrent MMAs take their A operand from there (the [a_tmem] form of tcgen05.mma).  TMEM holds two 128-column
//     accumulator slots (one 32-unit chunk x 4 gates each, ping-pong) and two 128-column h buffers (h_{t-1} / h_t).
//     Only x_t (streamed in by the loader warps, dropout applied on the way) is a shared-memory operand tile.
//   * The fp32 CELL STATE c (64 values per epilogue thread - too many for the register file next to the epilogue's
//     working set) lives in a per-CTA 128 KB scratch in global memory that never leaves L2: each thread prefetches the
//     4 values of its next half-pass while it computes the current one (coalesced 512 B per warp and access).
//   * The OUTPUT LAYER of the last layer is one more tensor-core product: h_T stays in TMEM like every other h_t and is multiplied
//     by [fp16(W_o) | W_o - fp16(W_o)]^T (one extra 16 KB ring piece, N = 64) into accumulator slot 1 where that slot would be
//     refilled for the next tile; the epilogue sums the two halves (W_o enters with ~22 bits) and adds the bias.
//   * Schedule: chunk 0 of step t+1 is issued into its slot as soon as the epilogue of step t has drained chunk NCH - 2
//     from it - the x-part, then the recurrent K-slices already published - and chunk 1's x-part follows when chunk
//     NCH - 1 is drained, so when the last slice of h_t lands only one small piece (2 MMAs) stands between it and the first
//     accumulator of step t+1; chunk 1's recurrent part runs under the epilogue's first pass.
// Per step and CTA the tensor pipe needs 256 MMAs x 64 cycles = 16.4 k cycles; the cell update of 128 rows x 256 units
// needs 14.3 k cycles of the 16-lane MUFU pipe: the two are balanced, unlike H = 128 where the cell update binds.
// L2 -> SM traffic per CTA and step: 512 KB of weights + 256 KB of cell state.
// Precision and dropout keying are those of ape_lstm_tc.cu (fp16 operands rounded once, fp32 accumulate and state).
#include "ape_common.cuh"
#include "ape_lstm_pack.h"
#include "ape_lstm_tc_args.cuh"
#include "ape_umma.cuh"
#include "ape_f32x2.cuh"
#ifndef APE_TCS_F32X2
#define APE_TCS_F32X2 1
#endif

namespace ape {
namespace tcs {

using tc::TcLayerArgs;
using tc::ex2_approx;
using tc::rcp_approx;
using tc::LOG2E;
using tc::EX2_CLAMP;

using tc::tanh_approx;

constexpr int EPI_WARPS = 16, LOAD_WARPS = 4;
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int N_ISSUERS = 2;                       // leader CTA: MMA issuers (MMA_WARP + k issues the chunks of accumulator slot k);
                                                   //   peer CTA: the first of them forwards "piece landed" to the leader
// Which warps play which role: epilogue 0..15, loaders 16..19, issuers 20..21, producer 22.  APE_TCS_EPI_HIGH = 1 is the layout that
// gained 1.3 % in ape_lstm_tcw.cu (epilogue warps on the highest ids, which the scheduler prefers among eligible warps: issuers 0..1,
// producer 2, one idle warp, loaders 4..7, epilogue 8..23); here it measured 3.7 % SLOWER (layer-1 launch 0.652 against 0.628 ms: the CTA
// grows to 768 threads = 80 registers instead of 88, and this kernel waits for its issuers rather than for its epilogue) and stays off.
#ifndef APE_TCS_EPI_HIGH
#define APE_TCS_EPI_HIGH 0
#endif
#if APE_TCS_EPI_HIGH
constexpr int MMA_WARP = 0, TMA_WARP = MMA_WARP + N_ISSUERS, LOAD_WARP0 = 4, EPI_WARP0 = LOAD_WARP0 + LOAD_WARPS;
constexpr int THREADS = (EPI_WARP0 + EPI_WARPS) * 32;   // 768: 80 registers per thread
#else
constexpr int EPI_WARP0 = 0, LOAD_WARP0 = EPI_WARPS, MMA_WARP = EPI_WARPS + LOAD_WARPS, TMA_WARP = MMA_WARP + N_ISSUERS;
constexpr int THREADS = (TMA_WARP + 1) * 32;       // 736: 88 registers per thread
#endif
static_assert(EPI_WARP0 % 4 == 0 && LOAD_WARP0 % 4 == 0, "TMEM lane quarter = warp % 4; loader rows = thread index within the role");
constexpr int ROWS = 128;                          // rows per CTA = TMEM lanes
constexpr int NSLOT = 2;                           // accumulator slots of 128 TMEM columns
constexpr int SLICE_KG = 4;                        // k-groups (of 8 K-values) per published K-slice of h_t (one chunk's 32 units)
constexpr int SLOT_KG = 16;                        // k-groups per ring slot (8 MMAs)
constexpr int PIECE_KG = 32;                       // largest piece: 32 k-groups = 16 MMAs = two consecutive ring slots
constexpr uint32_t KG_BYTES_B = 64 * 16;           // one k-group of a 64-column weight tile
constexpr uint32_t SLOT_BYTES = SLOT_KG * KG_BYTES_B;    // ring slot = 16 KB
constexpr uint32_t BAR_BLOCK_BYTES = 512;
constexpr uint32_t SMEM_LIMIT = 227 * 1024;
#ifndef APE_TCS_TRACE
#define APE_TCS_TRACE 0      // 1: all roles stamp SM clocks into args.trace (tools/tcs_trace.py); compiled out by default: costs issue slots
#endif
#if APE_TCS_TRACE
#define TCS_TR(...) __VA_ARGS__
constexpr int TRACE_T = 3;                         // the step of the first tile of CTA 0 that is stamped
#else
#define TCS_TR(...)
#endif

template <int H> struct Cfg {
    static constexpr int NCH = H / 32, KG = H / 8;
    static constexpr uint32_t A_BYTES = KG * ROWS * 16;                // one x operand tile (two: x_t is double-buffered)
    static constexpr uint32_t FIXED = 2 * A_BYTES + BAR_BLOCK_BYTES;
    static constexpr int NP = (SMEM_LIMIT - FIXED) / SLOT_BYTES;      // ring depth (slots)
    static constexpr uint32_t SMEM = FIXED + NP * SLOT_BYTES;
    // "piece landed" barriers are indexed by the piece's sequence number (a piece may span two slots): at most NP pieces are
    // in flight, so NFULL > NP barriers never alias
    static constexpr int NFULL = 8;
    static constexpr uint32_t H_COL = NSLOT * 128;                    // first TMEM column of the two h buffers
    static constexpr uint32_t H_COLS = H / 2;                         // fp16 pairs: one buffer
    static constexpr uint32_t TMEM_COLS = 512;
    static constexpr size_t CSTATE_BYTES = (size_t)H * ROWS * 4;      // per-CTA cell-state scratch (global, L2-resident)
    static constexpr uint32_t OUT_N = 64;                             // output product: 32 outputs x {fp16(W_o), remainder}
    static constexpr uint32_t OUT_BYTES = KG * (OUT_N / 2) * 16;      // this CTA's tile of it: one ring slot
    static_assert(OUT_BYTES <= SLOT_BYTES, "the output-layer tile must fit a ring slot");
    enum {
        BAR_X_READY = 0, BAR_X_DONE = 2, BAR_ACC_READY = 4, BAR_SLOT_FREE = BAR_ACC_READY + NSLOT,
        BAR_H_READY = BAR_SLOT_FREE + NSLOT, BAR_W_FULL = BAR_H_READY + NCH, BAR_W_EMPTY = BAR_W_FULL + NFULL,
        BAR_OUT_READY = BAR_W_EMPTY + NP, BAR_OUT_DONE = BAR_OUT_READY + 1, BAR_COUNT = BAR_OUT_DONE + 1
    };
    static_assert(NSLOT == 2 && NCH % 2 == 0 && NCH > NSLOT, "chunks alternate between the two accumulator slots");
    static_assert(H_COL + 2 * H_COLS <= TMEM_COLS, "accumulator slots + two h buffers must fit the 512 TMEM columns");
    static_assert(NP >= 3 && NP < NFULL, "weight ring depth");
    static_assert(BAR_COUNT * 8 + 16 <= BAR_BLOCK_BYTES, "barrier block too small");
};

// The order in which ONE step consumes weight pieces and signals its hand-offs.  Evaluated on the host (Recorder below).
//   chunk_begin(c)                      slot c & 1 is about to be refilled
//   piece(c, is_h, kg0, nkg, first)     chunk c (+)= A[:, k-groups kg0 .. kg0+nkg) x W_c[k-groups]^T  (x-part or recurrent part);
//                                       a recurrent piece needs the K-slices (of SLICE_KG k-groups) it covers published
//   acc_done(c) / x_done()              chunk c complete / this slot's share of the x tile has been consumed
//   out_point()                         (first step of a tile) before the next piece: the output layer of the PREVIOUS tile, one
//                                       extra ring piece (the W_o tile) multiplied by that tile's h_T into accumulator slot 1
// Three kinds of step, which index the schedule table: the first step of a tile without an initial state (h_{-1} = 0), a later
// step, and the first step of a tile with a caller-supplied h_0.
enum StepKind { STEP_FIRST = 0, STEP_LATER = 1, STEP_FIRST_STATE = 2, N_STEP_KINDS = 3 };
template <int NCH, class V>
static void walk_step(int kind, int kgx, V& v) {
    const int KG = NCH * SLICE_KG;
    const bool first_step = kind == STEP_FIRST;
    auto range = [&](int c, bool is_h, int kg_lo, int kg_hi, bool first) {      // [kg_lo, kg_hi) in pieces of <= PIECE_KG
        for (int kg0 = kg_lo; kg0 < kg_hi; kg0 += PIECE_KG)
            v.piece(c, is_h, kg0, kg_hi - kg0 < PIECE_KG ? kg_hi - kg0 : PIECE_KG, first && kg0 == kg_lo);
    };
    if (kind == STEP_FIRST_STATE) {
        // Every chunk takes its x-part exactly as in STEP_FIRST, then the whole recurrent part on h_0.  The epilogue publishes h_0
        // only after it has read the previous tile's outputs, so the output piece and both x-parts it sits between go ahead of
        // the first recurrent piece, in the ring as in the issue order.
        for (int c = 0; c < NCH; ++c) {
            v.chunk_begin(c);
            if (c == 1) v.out_point();
            range(c, false, 0, kgx, true);
            if (c >= NCH - NSLOT) v.x_done();
            if (c == 1) { range(0, true, 0, KG, false); v.acc_done(0); }
            if (c >= 1) { range(c, true, 0, KG, false); v.acc_done(c); }
        }
        return;
    }
    for (int c = 0; c < NCH; ++c) {
        v.chunk_begin(c);
        if (first_step && c == 1) v.out_point();               // slot 1 is free and the previous tile's h_T is complete by now
        range(c, false, 0, kgx, true);
        if (c >= NCH - NSLOT) v.x_done();                      // the last x-part of each accumulator slot (= of each issuer)
        if (first_step) {                                      // h_{-1} = 0: no recurrent half
            v.acc_done(c);
        } else if (c >= NSLOT) {                               // refilled inside the step: all of h_{t-1} is there
            range(c, true, 0, KG, false);
            v.acc_done(c);
        } else if (c == 0) {                                   // refilled under the tail of the previous step's epilogue:
            range(0, true, 0, (NCH - 2) * SLICE_KG, false);    //   K-slices published before slot 0 was drained,
            v.piece(0, true, (NCH - 2) * SLICE_KG, SLICE_KG, false);   // then the slice that lands at the end of that pass
        } else {                                               // c == 1: only its x-part goes ahead of chunk 0's last slice, so
            v.piece(0, true, (NCH - 1) * SLICE_KG, SLICE_KG, false);   // that ONE small piece separates h_t from the next step
            v.acc_done(0);
            range(1, true, 0, KG, false);                      // (chunk 1's recurrent part has all of pass 0 to finish)
            v.acc_done(1);
        }
    }
}

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory"); }

// ---- the step schedule as a table ----------------------------------------------------------------------------------
// walk_step is evaluated on the HOST into a table that travels as a kernel parameter (constant bank): the issuer, the
// producer and the forwarder run short table-driven loops.  (Inlining the walk - straight-line code for every piece of a
// step - or reading the table from shared memory made the single issuing thread far slower than the tensor pipe.)
enum : uint32_t {
    E_SLOT1 = 1u << 0,        // accumulator slot (chunk & 1)
    E_IS_H = 1u << 1,         // recurrent piece: A = h_{t-1} from TMEM (else x_t from shared memory)
    E_FIRST = 1u << 2,        // first MMA of the chunk: overwrite the accumulator
    E_PRE_SLOT = 1u << 3,     // before: wait until the epilogue has drained this slot
    E_POST_ACC = 1u << 4,     // after: the chunk is complete
    E_POST_X = 1u << 5,       // after: the x tile has been consumed
    E_OUT_BEFORE = 1u << 6,   // before (and before the slot wait's refill): the previous tile's output-layer piece, if there is one
    E_NMMA_SHIFT = 8,         // [8, 13)   K=16 MMAs in the piece (1..16)
    E_HNEED_SHIFT = 13,       // [13, 17)  K-slices of h_{t-1} that must have been published (0..NCH)
    E_SRC_SHIFT = 17          // [17, 32)  k-group offset of the piece inside this CTA's weight tiles (1 KB units)
};
constexpr int MAX_ENTRIES = 48;

struct Schedule {                                              // indexed by StepKind
    uint2 e[N_STEP_KINDS][MAX_ENTRIES];                        // .x see above; .y A-operand offset (x: descriptor units, h: TMEM columns)
    uint32_t n[N_STEP_KINDS];
};

struct Recorder {
    uint2* tab;
    int n, kgx, KG;
    uint32_t pre;
    bool overflow;
    void chunk_begin(int) { pre |= E_PRE_SLOT; }
    void out_point() { pre |= E_OUT_BEFORE; }
    void piece(int c, bool is_h, int kg0, int nkg, bool first) {
        if (n >= MAX_ENTRIES) { overflow = true; return; }
        const uint32_t src_kg = (uint32_t)c * (uint32_t)(kgx + KG) + (is_h ? (uint32_t)kgx : 0u) + (uint32_t)kg0;
        const uint32_t hneed = is_h ? (uint32_t)((kg0 + nkg + SLICE_KG - 1) / SLICE_KG) : 0u;
        tab[n].x = (uint32_t)(c & 1) | (is_h ? E_IS_H : 0u) | (first ? E_FIRST : 0u) | pre | ((uint32_t)(nkg / 2) << E_NMMA_SHIFT) |
                   (hneed << E_HNEED_SHIFT) | (src_kg << E_SRC_SHIFT);
        tab[n].y = is_h ? (uint32_t)kg0 * 4u : ((uint32_t)kg0 * (ROWS * 16)) >> 4;
        ++n;
        pre = 0;
    }
    void acc_done(int) { if (n > 0) tab[n - 1].x |= E_POST_ACC; }
    void x_done() { if (n > 0) tab[n - 1].x |= E_POST_X; }
};

// STATE: a caller-supplied initial state (a.h0, a.c0): h_0 goes into the h buffer step 0 reads, the cell starts from c_0 and step 0
// follows the STEP_FIRST_STATE schedule; h_0 = c_0 = 0 reproduces the stateless kernel bit for bit.
template <int H, bool STATE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1) lstm_layer_tcs_kernel(const __grid_constant__ TcLayerArgs a, const __grid_constant__ Schedule sched) {
    using namespace umma;
    using C = Cfg<H>;
    constexpr int NCH = C::NCH, KG = C::KG, NP = C::NP;
    constexpr uint32_t LBO_A = ROWS * 16, LBO_B = KG_BYTES_B, SBO = 128;
    constexpr uint32_t H_COL = C::H_COL, H_COLS = C::H_COLS;

    const int kgx = a.kgx, T = a.T;
    const uint32_t chunk_bytes = (uint32_t)(kgx + KG) * KG_BYTES_B;   // x k-groups then h k-groups of one chunk
    const uint32_t w_bytes = NCH * chunk_bytes;                       // one CTA's half of the layer

    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* sAx = smem;                                       // [2][A_BYTES] x_t operand tiles (kgx k-groups used), by step parity
    uint8_t* sW = sAx + 2 * C::A_BYTES;                        // [NP][SLOT_BYTES] weight ring
    uint64_t* bars = reinterpret_cast<uint64_t*>(sW + NP * SLOT_BYTES);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + C::BAR_COUNT);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;

    // ---- one-time set-up: TMEM, barriers ------------------------------------------------------------------------------
    tc::timeline_stamp(a.timeline, 0);
    if (warp == MMA_WARP) {
        tmem_alloc<2>(tmem_slot, C::TMEM_COLS);
        tmem_relinquish<2>();
    }
    if (tid == 0) {
        for (int b = 0; b < 2; ++b) {
            mbar_init(&bars[C::BAR_X_READY + b], 2 * LOAD_WARPS);
            mbar_init(&bars[C::BAR_X_DONE + b], N_ISSUERS);    // each issuer commits after ITS last x-part of the step
        }
        for (int s = 0; s < NSLOT; ++s) {
            mbar_init(&bars[C::BAR_ACC_READY + s], 1);
            mbar_init(&bars[C::BAR_SLOT_FREE + s], 2 * EPI_WARPS);
        }
        for (int c = 0; c < NCH; ++c) mbar_init(&bars[C::BAR_H_READY + c], 2 * EPI_WARPS);
        // leader: its own copy (arrive.expect_tx + bytes) and the peer's "my copy landed" arrival; peer: its own copy
        for (int p = 0; p < C::NFULL; ++p) mbar_init(&bars[C::BAR_W_FULL + p], rank == 0 ? 2 : 1);
        for (int p = 0; p < NP; ++p) mbar_init(&bars[C::BAR_W_EMPTY + p], 1);
        mbar_init(&bars[C::BAR_OUT_READY], 1);
        mbar_init(&bars[C::BAR_OUT_DONE], 2 * EPI_WARPS);
        mbar_init_fence();
    }
    fence_proxy_async_smem();
    fence_before_sync();
    cluster_sync();
    fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    tc::timeline_stamp(a.timeline, 1);

    if (warp >= EPI_WARP0 && warp < EPI_WARP0 + EPI_WARPS) {
        // =================================== epilogue warps ===========================================================
        // warp (q, s): rows 32q..32q+31 (its TMEM lane quarter) x the 8 hidden units 8s..8s+7 of EVERY 32-unit chunk.
        const int q = warp & 3, s = (warp - EPI_WARP0) >> 2;
        const int row_l = 32 * q + lane;                       // local row == TMEM lane
        const uint32_t t_lane = (uint32_t)(32 * q) << 16;
        const bool warp_live = 32 * q < a.rpc;                 // a quarter without rows only keeps the barrier protocol going
        // this thread's cell state: float4 (4 units) per half-pass at [(k-group j = 4c + s) * 2 + half][row]
        float4* cst = reinterpret_cast<float4*>(a.cstate + (size_t)blockIdx.x * (C::CSTATE_BYTES / 4)) + row_l;
        uint32_t gstep = 0, ph_out = 0;

        for (int tile = cluster_id; tile < a.n_pair_tiles; tile += n_clusters) {
            const int row = (tile * 2 + (int)rank) * a.rpc + row_l;
            const bool valid = row_l < a.rpc && row < a.rows;
            const float4* c0r = STATE ? reinterpret_cast<const float4*>(a.c0 + (size_t)(valid ? row : 0) * H) : nullptr;
            if constexpr (STATE) {
                // h_0 as fp16 pairs into buffer 0 (the one step 0 reads).  Every MMA that read the buffer has retired: this warp has
                // drained every accumulator of the previous tile's last step and waited for its output product.
                if (warp_live) {
                    const float4* h0r = reinterpret_cast<const float4*>(a.h0 + (size_t)(valid ? row : 0) * H);
                    const float4 z = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll
                    for (int c = 0; c < NCH; ++c) {
                        const int j = 4 * c + s;
                        const float4 h_a = valid ? __ldg(h0r + 2 * j) : z, h_b = valid ? __ldg(h0r + 2 * j + 1) : z;
                        tmem_st_x4(tmem + t_lane + H_COL + (uint32_t)(4 * j), pack_half2(h_a.x, h_a.y), pack_half2(h_a.z, h_a.w),
                                   pack_half2(h_b.x, h_b.y), pack_half2(h_b.z, h_b.w));
                    }
                    tmem_st_wait();
                }
                fence_before_sync();
                __syncwarp();
                if (lane == 0)
#pragma unroll
                    for (int c = 0; c < NCH; ++c) mbar_arrive_leader(&bars[C::BAR_H_READY + c], rank);
            }

            for (int t = 0; t < T; ++t, ++gstep) {
                const uint32_t h_next = H_COL + (uint32_t)((t + 1) & 1) * H_COLS;     // TMEM columns that receive h_t
                const bool final_out = a.preds != nullptr && t == T - 1;
                // chunk c uses slot c & 1 for the (gstep * NCH/2 + c/2)-th time
                const uint32_t par0 = (gstep * (uint32_t)(NCH / 2)) & 1u;
                if (!warp_live) {
#pragma unroll
                    for (int c = 0; c < NCH; ++c) {
                        mbar_wait_wd(&bars[C::BAR_ACC_READY + (c & 1)], par0 ^ ((c >> 1) & 1));
                        if (lane == 0) {
                            mbar_arrive_leader(&bars[C::BAR_SLOT_FREE + (c & 1)], rank);
                            if (t + 1 < T || final_out) mbar_arrive_leader(&bars[C::BAR_H_READY + c], rank);
                        }
                    }
                } else {
                    // Half-passes of 4 hidden units (16 accumulator columns + one float4 of cell state), double-buffered:
                    // the loads of half-pass hp+1 are in flight while the cells of half-pass hp are computed.
                    uint32_t rbuf[2][16];
                    float4 cbuf[2];
                    bool prefetched = true;
                    float hlo[4];
                    cbuf[0] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                    cbuf[1] = cbuf[0];
                    if (t > 0 && APE_EXP != 8) cbuf[0] = __ldcg(cst + (size_t)((4 * 0 + s) * 2 + 0) * ROWS);
                    else if (STATE && valid) cbuf[0] = __ldg(c0r + 2 * s);
                    // The bias of half-pass hp+1 is requested at the end of half-pass hp's arithmetic, where few registers are live:
                    // its ~40 cycles of L1 latency used to sit in front of the first FMA of every half-pass (ncu: a fifth of the
                    // kernel's stall samples).
                    float4 bnext[4];
                    auto request_bias = [&](int hp1) {
                        const float4* bias4 = reinterpret_cast<const float4*>(a.bias_s + ((hp1 >> 1) * 32 + 8 * s + 4 * (hp1 & 1)) * 4);
                        bnext[0] = __ldg(bias4); bnext[1] = __ldg(bias4 + 1); bnext[2] = __ldg(bias4 + 2); bnext[3] = __ldg(bias4 + 3);
                    };
                    request_bias(0);
                    mbar_wait_wd(&bars[C::BAR_ACC_READY + 0], par0);
                    fence_after_sync();
                    tmem_ld_x16(tmem + t_lane + (uint32_t)(32 * s), rbuf[0]);
#pragma unroll
                    for (int hp = 0; hp < 2 * NCH; ++hp) {
                        const int c = hp >> 1, half = hp & 1;
                        const uint32_t* r = rbuf[hp & 1];
                        // this half-pass's bias (warp-uniform addresses, L1-resident) was requested in the tail of the previous one
#if APE_EXP == 10
                        const float4 bsv[4] = {make_float4(0.1f, 0.2f, 0.3f, 0.4f), make_float4(0.1f, 0.2f, 0.3f, 0.4f), make_float4(0.1f, 0.2f, 0.3f, 0.4f), make_float4(0.1f, 0.2f, 0.3f, 0.4f)};
#else
                        const float4 bsv[4] = {bnext[0], bnext[1], bnext[2], bnext[3]};
#endif
                        if (half == 0 && hp > 0 && !prefetched) {      // the chunk was not complete yet when the last half-pass looked
                            mbar_wait_wd(&bars[C::BAR_ACC_READY + (c & 1)], par0 ^ ((c >> 1) & 1));
                            fence_after_sync();
                            tmem_ld_x16(tmem + t_lane + (uint32_t)((c & 1) * 128 + 32 * s), rbuf[hp & 1]);
                        }
                        tmem_ld_wait();                        // this half-pass's columns have landed
                        TCS_TR(if (a.trace && blockIdx.x == 0 && tile == cluster_id && warp == 0 && lane == 0 && (t == TRACE_T || t == TRACE_T - 1))
                                   a.trace[512 + (t - TRACE_T + 1) * 16 + hp] = clock64();)
                        if (half == 1) {                       // chunk c fully drained: the issuer may refill its slot
                            fence_before_sync();
                            __syncwarp();
                            if (lane == 0) mbar_arrive_leader(&bars[C::BAR_SLOT_FREE + (c & 1)], rank);
                        }
                        if (hp + 1 < 2 * NCH) {
                            const int c1 = (hp + 1) >> 1, h1 = (hp + 1) & 1;
                            if (t > 0 && APE_EXP != 8) cbuf[(hp + 1) & 1] = __ldcg(cst + (size_t)((4 * c1 + s) * 2 + h1) * ROWS);
                            else if (STATE && valid) cbuf[(hp + 1) & 1] = __ldg(c0r + 2 * (4 * c1 + s) + h1);
                            // Next chunk: its accumulators are prefetched under this half-pass IF the chunk is already complete -
                            // waiting for it here would tie the pass period to the refill latency of the two-slot ring (drain of
                            // chunk c -> chunk c+2 complete), so an unfinished chunk is waited for at the top of its own pass.
                            prefetched = true;
                            if (half == 1) {
                                prefetched = __all_sync(0xffffffffu, mbar_test_wait_addr(smem_u32(&bars[C::BAR_ACC_READY + (c1 & 1)]), par0 ^ ((c1 >> 1) & 1)));
                                if (prefetched) fence_after_sync();
                            }
                            if (prefetched) tmem_ld_x16(tmem + t_lane + (uint32_t)((c1 & 1) * 128 + 32 * s + 16 * h1), rbuf[(hp + 1) & 1]);
                        }
                        // the 4 cells advance in lock-step through the transcendental stages (independent MUFU ops back to back):
                        //   e = 2^-(gate+bias)  ->  i*g~ and f share one reciprocal  ->  2^(-2c)  ->  h = o * tanh(c)
                        float hv[4], cn[4];
                        const float cp[4] = {cbuf[hp & 1].x, cbuf[hp & 1].y, cbuf[hp & 1].z, cbuf[hp & 1].w};
#if APE_TC_TANH
                        // 5 MUFU per cell: sigmoid(x) = 0.5 + 0.5 tanh(x / 2) with the hardware tanh (tanh.approx.f32)
                        float tg[16];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const float4 bs = bsv[u];              // 0.5 b (i, f, o), b (g)
#if APE_EXP == 7      // timing experiment: half of the epilogue warps skip the MUFU work (results wrong) - is the cell phase XU-contention bound?
                            if (s & 1) {
                                tg[4 * u + 0] = fmaf(__uint_as_float(r[4 * u + 0]), 0.5f, bs.x) * 0.1f;
                                tg[4 * u + 1] = fmaf(__uint_as_float(r[4 * u + 1]), 0.5f, bs.y) * 0.1f;
                                tg[4 * u + 2] = (__uint_as_float(r[4 * u + 2]) + bs.z) * 0.1f;
                                tg[4 * u + 3] = fmaf(__uint_as_float(r[4 * u + 3]), 0.5f, bs.w) * 0.1f;
                                continue;
                            }
#endif
#if APE_TCS_F32X2 && APE_EXP != 7
                            // tanh arguments in packed fp32 pairs (ape_f32x2.cuh): (i, f) and (g, o) sit in adjacent accumulator registers and
                            // adjacent bias words, r * (0.5, 0.5) + b and r * (1, 0.5) + b are the scalar operations bit for bit
                            const F2 aif = fma2(pk(__uint_as_float(r[4 * u + 0]), __uint_as_float(r[4 * u + 1])), splat(0.5f), pk(bs.x, bs.y));
                            const F2 ago = fma2(pk(__uint_as_float(r[4 * u + 2]), __uint_as_float(r[4 * u + 3])), pk(1.0f, 0.5f), pk(bs.z, bs.w));
                            tg[4 * u + 0] = tanh_approx(lo(aif)); tg[4 * u + 1] = tanh_approx(hi(aif));
                            tg[4 * u + 2] = tanh_approx(lo(ago)); tg[4 * u + 3] = tanh_approx(hi(ago));
#else
                            tg[4 * u + 0] = tanh_approx(fmaf(__uint_as_float(r[4 * u + 0]), 0.5f, bs.x));
                            tg[4 * u + 1] = tanh_approx(fmaf(__uint_as_float(r[4 * u + 1]), 0.5f, bs.y));
                            tg[4 * u + 2] = tanh_approx(__uint_as_float(r[4 * u + 2]) + bs.z);
                            tg[4 * u + 3] = tanh_approx(fmaf(__uint_as_float(r[4 * u + 3]), 0.5f, bs.w));
#endif
                        }
#if APE_TCS_F32X2 && APE_EXP != 7
#pragma unroll
                        for (int u = 0; u < 4; u += 2) {               // the cell update of two units per instruction (as in ape_lstm_tcw.cu)
                            const F2 h2c = splat(0.5f);
                            const F2 gi = fma2(pk(tg[4 * u + 0], tg[4 * u + 4]), h2c, h2c), gf = fma2(pk(tg[4 * u + 1], tg[4 * u + 5]), h2c, h2c);
                            const F2 c2 = fma2(gf, pk(cp[u], cp[u + 1]), gi * pk(tg[4 * u + 2], tg[4 * u + 6]));
                            cn[u] = lo(c2); cn[u + 1] = hi(c2);
                            const F2 h2 = fma2(pk(tg[4 * u + 3], tg[4 * u + 7]), h2c, h2c) * pk(tanh_approx(cn[u]), tanh_approx(cn[u + 1]));
                            hv[u] = lo(h2); hv[u + 1] = hi(h2);
                        }
#else
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const float gi = fmaf(tg[4 * u + 0], 0.5f, 0.5f), gf = fmaf(tg[4 * u + 1], 0.5f, 0.5f);
                            cn[u] = fmaf(gf, cp[u], gi * tg[4 * u + 2]);
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) hv[u] = fmaf(tg[4 * u + 3], 0.5f, 0.5f) * ((APE_EXP == 7 && (s & 1)) ? cn[u] * 0.1f : tanh_approx(cn[u]));
#endif
#else
                        float ev[16], num[4], den[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const float4 bs = bsv[u];              // 0.5 b (i, f, o), b (g) -> -log2e (gate + b), g: -2 log2e (gate + b)
                            ev[4 * u + 0] = ex2_approx(fminf(fmaf(__uint_as_float(r[4 * u + 0]), -LOG2E, bs.x * (-2.0f * LOG2E)), EX2_CLAMP));
                            ev[4 * u + 1] = ex2_approx(fminf(fmaf(__uint_as_float(r[4 * u + 1]), -LOG2E, bs.y * (-2.0f * LOG2E)), EX2_CLAMP));
                            ev[4 * u + 2] = ex2_approx(fminf(fmaf(__uint_as_float(r[4 * u + 2]), -2.0f * LOG2E, bs.z * (-2.0f * LOG2E)), EX2_CLAMP));
                            // (o gate unclamped: an infinite e_o only makes the reciprocal below 0; e_c is finite since |c| <= T)
                            ev[4 * u + 3] = ex2_approx(fmaf(__uint_as_float(r[4 * u + 3]), -LOG2E, bs.w * (-2.0f * LOG2E)));
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const float ab = (1.0f + ev[4 * u + 0]) * (1.0f + ev[4 * u + 2]), cf = 1.0f + ev[4 * u + 1];
                            num[u] = fmaf(cp[u], ab, (1.0f - ev[4 * u + 2]) * cf);
                            den[u] = rcp_approx(ab * cf);
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            cn[u] = num[u] * den[u];
                            // e_c = 2^(-2c log2e): |c| <= T, no overflow; with a state |c| <= |c_0| + T, clamped
                            num[u] = ex2_approx(STATE ? fminf(cn[u] * (-2.0f * LOG2E), EX2_CLAMP) : cn[u] * (-2.0f * LOG2E));
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) hv[u] = (1.0f - num[u]) * rcp_approx((1.0f + ev[4 * u + 3]) * (1.0f + num[u]));
#endif
                        if (hp + 1 < 2 * NCH && APE_EXP != 10) request_bias(hp + 1);
                        // cell state back to its scratch line (not needed after the last step)
                        if (t + 1 < T && APE_EXP != 8) __stcg(cst + (size_t)((4 * c + s) * 2 + half) * ROWS, make_float4(cn[0], cn[1], cn[2], cn[3]));
                        const int j = 4 * c + s;               // k-group of units 32c + 8s .. + 7
                        if (half == 1) {
                            if (t + 1 < T || final_out) {
                                // h_t as fp16 pairs into the TMEM operand buffer of the next step (lane = row, 4 columns = this
                                // k-group), then publish this chunk's K-slice: its piece of the next recurrent product can be
                                // issued while later chunks still run (last step of the last layer: h_T feeds the output product)
                                if (APE_EXP != 9) {
                                tmem_st_x4(tmem + t_lane + h_next + (uint32_t)(4 * j), pack_half2(hlo[0], hlo[1]), pack_half2(hlo[2], hlo[3]),
                                           pack_half2(hv[0], hv[1]), pack_half2(hv[2], hv[3]));
                                tmem_st_wait();
                                }
                                fence_before_sync();
                                __syncwarp();
                                if (lane == 0) mbar_arrive_leader(&bars[C::BAR_H_READY + c], rank);
                            }
                            if (a.out_units) {
                                const float os = a.out_scale;
                                a.out_units[((((size_t)tile * T + t) * 2 + rank) * KG + j) * ROWS + row_l] =
                                    make_uint4(pack_half2(hlo[0] * os, hlo[1] * os), pack_half2(hlo[2] * os, hlo[3] * os),
                                               pack_half2(hv[0] * os, hv[1] * os), pack_half2(hv[2] * os, hv[3] * os));
                            }
                        } else {
#pragma unroll
                            for (int u = 0; u < 4; ++u) hlo[u] = hv[u];
                        }
                    }
                }
                if (final_out) {                               // output_layer (nn_models.py:189), last step only
                    // Issuer 1 multiplies the published h_T (TMEM) by [fp16(W_o) | W_o - fp16(W_o)]^T - one extra ring piece - into
                    // the first 64 columns of accumulator slot 1 once chunk NCH-1 has been drained from it.  Every warp waits for
                    // the product: that is also the guarantee that h_T has been consumed before the next tile rewrites the buffer.
                    mbar_wait_wd(&bars[C::BAR_OUT_READY], ph_out);
                    ph_out ^= 1;
                    fence_after_sync();
                    if (warp_live) {
                        uint32_t v[32];
                        float y[8];
                        tmem_ld_x32(tmem + t_lane + 128u, v);                  // h_T x fp16(W_o)^T, outputs 0..31
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 8; ++i) y[i] = __uint_as_float(tc::pick4(v, i, s));
                        tmem_ld_x32(tmem + t_lane + 128u + 32u, v);            // h_T x (W_o - fp16(W_o))^T
                        tmem_ld_wait();
                        if (valid) {
                            const int e = row / a.n, smp = row - e * a.n;
                            const int b = e / a.nF, fb = stream_frame0(a.stream_frames, a.frame0, b), f = fb + e % a.nF;
#pragma unroll
                            for (int i = 0; i < 8; ++i) {      // this thread: outputs o = s, s+4, ... of its row (O <= 32)
                                const int o = s + 4 * i;
                                if (o < a.O && fb >= 0) {      // (an inactive stream keeps its prediction ring untouched)
                                    const float yo = y[i] + __uint_as_float(tc::pick4(v, i, s)) + __ldg(a.bo + o);
                                    float* dst = a.preds + (((size_t)b * a.pred_ring + f % a.pred_ring) * a.n_out) * a.O + o;
                                    if (a.n == 1 && a.n_out > 1) for (int s2 = 0; s2 < a.n_out; ++s2) dst[(size_t)s2 * a.O] = yo;
                                    else dst[(size_t)smp * a.O] = yo;
                                }
                            }
                        }
                    }
                    fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_leader(&bars[C::BAR_OUT_DONE], rank);   // slot 1 may be refilled for the next tile
                }
            }
        }
    } else if (warp >= LOAD_WARP0 && warp < LOAD_WARP0 + LOAD_WARPS) {
        // =================================== operand-loader warps: x_t -> sAx ===========================================
        constexpr int TPR = LOAD_WARPS * 32 / ROWS;            // loader threads per row, each an equal share of the x k-groups
        const int row_l = (tid - LOAD_WARP0 * 32) & (ROWS - 1);
        const int part = (tid - LOAD_WARP0 * 32) / ROWS;
        uint32_t gl = 0;                                       // steps loaded so far: step gl goes to x buffer gl & 1
        for (int tile = cluster_id; tile < a.n_pair_tiles; tile += n_clusters) {
            const int row = (tile * 2 + (int)rank) * a.rpc + row_l;
            const bool valid = row_l < a.rpc && row < a.rows;
            const int e = valid ? row / a.n : 0, smp = valid ? row - e * a.n : 0;
            const int b = e / a.nF, f = stream_frame0(a.stream_frames, a.frame0, b) + e % a.nF;
            for (int t = 0; t < T; ++t, ++gl) {
                uint8_t* sX = sAx + (gl & 1) * C::A_BYTES;
                // the tile written two steps ago has been consumed (the loader may run up to two steps ahead of the MMAs)
                auto wait_buffer = [&]() { if (gl >= 2) mbar_wait_wd(&bars[C::BAR_X_DONE + (gl & 1)], ((gl >> 1) & 1) ^ 1); };
                TCS_TR(const bool trl = a.trace && blockIdx.x == 0 && tile == cluster_id && t == TRACE_T && tid == LOAD_WARP0 * 32;)
                if (a.in_mode == tc::IN_UNITS || a.in_mode == tc::IN_SHARED_UNITS) {
                    // The first batch of 8 k-groups is fetched and masked before anything waits; only the shared-memory
                    // stores (and the remaining batches, which would not fit the register file) sit behind "the previous
                    // x tile has been consumed".
                    const uint4* src = reinterpret_cast<const uint4*>(a.in);
                    if (a.in_mode == tc::IN_UNITS) src += ((((size_t)tile * T + t) * 2 + rank) * KG) * ROWS + row_l;
                    else src += ((((size_t)(e >> (a.in_rpc_shift + 1)) * T + t) * 2 + ((e >> a.in_rpc_shift) & 1)) * KG) * ROWS +
                                (e & ((1 << a.in_rpc_shift) - 1));
                    constexpr int KH = KG / TPR, BK = 8;        // k-groups per loader thread, in batches of 8 (register budget)
                    static_assert(KH % BK == 0, "whole batches");
                    const int j0 = part * KH;
                    src += (size_t)j0 * ROWS;
                    const uint32_t stream = a.stream_id0 + (uint32_t)b;
                    // x_t is double-buffered, so the loader runs a step ahead of the MMAs and none of this (Philox draws included)
                    // sits on the step boundary; only the first store of a step waits for "the tile of two steps ago is consumed".
#pragma unroll 1
                    for (int b0 = 0; b0 < KH; b0 += BK) {
                        uint4 pre[BK];
#pragma unroll
                        for (int jj = 0; jj < BK; ++jj) pre[jj] = valid ? __ldg(src + (size_t)(b0 + jj) * ROWS) : make_uint4(0, 0, 0, 0);
                        if (a.mask_mode == APE_MASK_PHILOX) {
#pragma unroll
                            for (int jj = 0; jj < BK; ++jj) {
                                const uint4 m = APE_PHILOX_DRAW(a, stream, (uint32_t)f, (uint32_t)smp, (uint32_t)a.gap, (uint32_t)t,
                                                                     (uint32_t)(j0 + b0 + jj), a.keep_thr16);
                                pre[jj].x &= m.x; pre[jj].y &= m.y; pre[jj].z &= m.z; pre[jj].w &= m.w;
                            }
                        } else if (a.mask_mode == APE_MASK_INJECTED && valid) {
#pragma unroll
                            for (int jj = 0; jj < BK; ++jj) {
                                const uint2 m = __ldg(reinterpret_cast<const uint2*>(
                                    a.masks + ((((size_t)e * a.n_gaps + a.gap) * T + t) * a.n + smp) * H + (j0 + b0 + jj) * 8));
                                pre[jj].x &= ((m.x & 0xFFu) ? 0xFFFFu : 0u) | ((m.x & 0xFF00u) ? 0xFFFF0000u : 0u);
                                pre[jj].y &= ((m.x & 0xFF0000u) ? 0xFFFFu : 0u) | ((m.x & 0xFF000000u) ? 0xFFFF0000u : 0u);
                                pre[jj].z &= ((m.y & 0xFFu) ? 0xFFFFu : 0u) | ((m.y & 0xFF00u) ? 0xFFFF0000u : 0u);
                                pre[jj].w &= ((m.y & 0xFF0000u) ? 0xFFFFu : 0u) | ((m.y & 0xFF000000u) ? 0xFFFF0000u : 0u);
                            }
                        }
                        if (b0 == 0) {
                            TCS_TR(if (trl) a.trace[580] = clock64();)
                            wait_buffer();
                            TCS_TR(if (trl) a.trace[581] = clock64();)
                        }
#pragma unroll
                        for (int jj = 0; jj < BK; ++jj) *reinterpret_cast<uint4*>(sX + unit_offset(ROWS, row_l, j0 + b0 + jj)) = pre[jj];
                    }
                } else {                                       // layer 0: fp32 features (window of the ring, or dense rows)
                    wait_buffer();
                    const float* src = nullptr;
                    if (valid) {
                        if (a.in_mode == tc::IN_DENSE_F32) {
                            src = reinterpret_cast<const float*>(a.in) + ((size_t)row * T + t) * a.Kin;
                        } else {                               // sliding window, clamped at frame 0 (estimator.py:96-97)
                            int fw = f - T + 1 + t;
                            fw = fw < 0 ? 0 : fw;
                            src = reinterpret_cast<const float*>(a.in) + ((size_t)b * a.feat_ring + fw % a.feat_ring) * a.Kin;
                        }
                    }
                    for (int j = part; j < kgx; j += TPR) {
                        float v[8];
#pragma unroll
                        for (int k = 0; k < 8; ++k) v[k] = (valid && 8 * j + k < a.Kin) ? __ldg(src + 8 * j + k) : 0.0f;
                        *reinterpret_cast<uint4*>(sX + unit_offset(ROWS, row_l, j)) =
                            make_uint4(pack_half2(v[0], v[1]), pack_half2(v[2], v[3]), pack_half2(v[4], v[5]), pack_half2(v[6], v[7]));
                    }
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(&bars[C::BAR_X_READY + (gl & 1)], rank);
                TCS_TR(if (trl) a.trace[582] = clock64();)
            }
        }
    } else if (warp >= MMA_WARP && warp < MMA_WARP + N_ISSUERS) {
        if (rank == 0) {
            // =============================== MMA issuers (leader CTA; the whole warp runs, one elected lane issues) =====
            // Issuer k owns the chunks of accumulator slot k: a single issuing thread spends ~650 cycles of waits and table
            // handling per piece plus ~34 cycles per MMA and was the bottleneck of the step (82 % busy).  Both issuers walk
            // the whole table (the ring position and the piece sequence number advance with every entry) and act on their own
            // entries only; tcgen05.commit covers the issuing thread's own MMAs, which is exactly what each hand-off needs.
            const uint32_t my_slot = (uint32_t)(warp - MMA_WARP);
            const uint32_t idesc = make_idesc_f16(256, 128);
            const uint64_t dX0 = make_desc(smem_u32(sAx), LBO_A, SBO), dW = make_desc(smem_u32(sW), LBO_B, SBO);
            const uint32_t bar_full = smem_u32(&bars[C::BAR_W_FULL]), bar_empty = smem_u32(&bars[C::BAR_W_EMPTY]);
            uint32_t gl = 0, wslot = 0, gpiece = 0, gchunk = 0, hphase = 0, ph_outdone = 0;
            // Output layer of the last layer (nn_models.py:189, last step only): h_T (TMEM) x [fp16(W_o) | W_o - fp16(W_o)]^T, one extra
            // ring piece of KG/2 MMAs with N = 64 into the first 64 columns of accumulator slot 1.  It is issued by issuer 1 where
            // that slot would be refilled for the next tile (or after the last tile); every role advances its ring position and
            // piece number by one there.  slot_waited: chunk NCH-1's drain has been waited for.
            const uint32_t idesc_out = make_idesc_f16(256, C::OUT_N);
            auto out_piece = [&](bool slot_waited) {
                if (my_slot == 1) {
                    if (!slot_waited) mbar_wait_wd(&bars[C::BAR_SLOT_FREE + 1], (gchunk & 1) ^ 1);
                    uint32_t spins = 0;
                    while (!mbar_try_wait_addr(bar_full + (gpiece & (C::NFULL - 1)) * 8, (gpiece / C::NFULL) & 1)) { if (++spins > MBAR_WD_SPINS) __trap(); }
                    mbar_wait_wd(&bars[C::BAR_H_READY + NCH - 1], hphase);             // all of h_T (slices are published in order)
                    fence_after_sync();
                    if (elect_one()) {
                        const uint64_t bd = make_desc(smem_u32(sW) + wslot * SLOT_BYTES, (C::OUT_N / 2) * 16, SBO);
                        const uint32_t at = tmem + H_COL + (uint32_t)(T & 1) * H_COLS;   // step T-1 wrote h_T into buffer T & 1
#pragma unroll
                        for (uint32_t m = 0; m < KG / 2; ++m)
                            mma_f16_ts<2>(tmem + 128, at + 8 * m, bd + m * (2 * (C::OUT_N / 2) * 16 >> 4), idesc_out, m > 0 ? 1u : 0u);
                        commit_pair_addr(bar_empty + wslot * 8, 0x3);
                        commit_pair(&bars[C::BAR_OUT_READY], 0x3);
                    }
                    __syncwarp();
                    mbar_wait_wd(&bars[C::BAR_OUT_DONE], ph_outdone);                  // every epilogue warp has read its outputs
                    ph_outdone ^= 1;
                    fence_after_sync();
                } else if (STATE) {
                    // Issuer 0's next H_READY wait (step 0 with a state) is for h_0, whose phase has the parity of the phase BEFORE h_T:
                    // while h_T is still being published that wait would pass at once and the recurrent MMAs would read the h buffer
                    // before h_0 is in it.  So it waits for h_T here as issuer 1 does.
                    mbar_wait_wd(&bars[C::BAR_H_READY + NCH - 1], hphase);
                }
                hphase ^= 1;                                   // the last step of a final layer publishes h_T: one more H_READY phase
                wslot = wslot + 1 == NP ? 0 : wslot + 1;
                ++gpiece;
            };
            bool out_pending = false;
            for (int tile = cluster_id; tile < a.n_pair_tiles; tile += n_clusters) {
                for (int t = 0; t < T; ++t, ++gl) {
                    TCS_TR(long long* tr = (a.trace && blockIdx.x == 0 && tile == cluster_id && t == TRACE_T && lane == 0) ? a.trace : nullptr;)
                    const uint32_t xb = gl & 1;                // x_t's buffer
                    mbar_wait_wd(&bars[C::BAR_X_READY + xb], (gl >> 1) & 1);
                    TCS_TR(if (tr) tr[576] = clock64();)
                    const uint64_t dX = dX0 + xb * (C::A_BYTES >> 4);
                    const uint32_t h_prev = tmem + H_COL + (uint32_t)(t & 1) * H_COLS;   // TMEM columns of h_{t-1}
                    const int which = t > 0 ? STEP_LATER : STATE ? STEP_FIRST_STATE : STEP_FIRST;
                    const uint32_t n_ent = sched.n[which];
                    uint32_t h_waited = 0;                     // K-slices of h_{t-1} seen so far in this step
                    uint2 e = sched.e[which][0];
#pragma unroll 1
                    for (uint32_t i = 0; i < n_ent; ++i) {
                        const uint2 e_next = sched.e[which][i + 1 < n_ent ? i + 1 : i];   // fetched under this piece's waits
                        const uint32_t nmma = (e.x >> E_NMMA_SHIFT) & 0x1F;
                        bool slot_waited = false;
                        if ((e.x & E_OUT_BEFORE) && out_pending) {     // (first step of a tile) the previous tile's output layer
                            if (my_slot == 1) {                // this entry's own slot wait, taken first: chunk NCH-1 has been drained
                                mbar_wait_wd(&bars[C::BAR_SLOT_FREE + 1], (gchunk & 1) ^ 1);
                                ++gchunk;
                                slot_waited = true;
                            }
                            out_piece(true);
                            out_pending = false;
                        }
                        const uint32_t slot_b = wslot + 1 == NP ? 0 : wslot + 1;
                        if ((e.x & E_SLOT1) != my_slot) {      // the other issuer's piece: only the ring bookkeeping advances
                            wslot = nmma > SLOT_KG / 2 ? slot_b : wslot;
                            wslot = wslot + 1 == NP ? 0 : wslot + 1;
                            ++gpiece;
                            e = e_next;
                            continue;
                        }
                        if ((e.x & E_PRE_SLOT) && !slot_waited) {   // the epilogue has drained the chunk that used this slot before
                            if (gchunk >= 1) mbar_wait_wd(&bars[C::BAR_SLOT_FREE + my_slot], (gchunk & 1) ^ 1);
                            ++gchunk;                          // (this issuer's count = uses of its slot so far)
                            TCS_TR(if (tr) tr[560 + ((2 * (gchunk - 1) + my_slot) & 7)] = clock64();)
                        }
                        // the piece is in BOTH CTAs' rings (one slot, or two consecutive ones for > 8 MMAs): one barrier per piece
                        uint32_t spins = 0;
                        while (!mbar_try_wait_addr(bar_full + (gpiece & (C::NFULL - 1)) * 8, (gpiece / C::NFULL) & 1)) { if (++spins > MBAR_WD_SPINS) __trap(); }
                        // LAST, because it is what the step boundary waits for: the K-slices of h_{t-1} this piece multiplies have
                        // been published.  Every epilogue warp publishes its slices in order, so slice k complete implies k-1, ...
                        const uint32_t hneed = (e.x >> E_HNEED_SHIFT) & 0xF;
                        if (hneed > h_waited) {
                            mbar_wait_wd(&bars[C::BAR_H_READY + hneed - 1], hphase);
                            TCS_TR(if (tr) tr[568 + hneed - 1] = clock64();)
                            h_waited = hneed;
                        }
                        fence_after_sync();
                        TCS_TR(if (tr && i < 48) { tr[2 * i] = clock64(); tr[600 + i] = spins; })
                        if (elect_one()) {
                            const uint64_t bd = dW + wslot * (SLOT_BYTES >> 4), bd_b = dW + slot_b * (SLOT_BYTES >> 4);
                            const uint32_t d_tmem = tmem + (e.x & E_SLOT1) * 128;
                            // fully unrolled with uniform predicates: operand addresses advance by constants in uniform registers
                            if (e.x & E_IS_H) {
                                const uint32_t at = h_prev + e.y;
#pragma unroll
                                for (uint32_t m = 0; m < SLOT_KG / 2; ++m)
                                    if (m < nmma) mma_f16_ts<2>(d_tmem, at + 8 * m, bd + m * (2 * LBO_B >> 4), idesc, 1u);
                                commit_pair_addr(bar_empty + wslot * 8, 0x3);          // both CTAs' producers may refill this slot
                                if (nmma > SLOT_KG / 2) {
#pragma unroll
                                    for (uint32_t m = 0; m < SLOT_KG / 2; ++m)
                                        if (m + SLOT_KG / 2 < nmma) mma_f16_ts<2>(d_tmem, at + 8 * (m + SLOT_KG / 2), bd_b + m * (2 * LBO_B >> 4), idesc, 1u);
                                    commit_pair_addr(bar_empty + slot_b * 8, 0x3);
                                }
                            } else {
                                const uint64_t ad = dX + e.y;
                                mma_f16<2>(d_tmem, ad, bd, idesc, (e.x & E_FIRST) ? 0u : 1u);
#pragma unroll
                                for (uint32_t m = 1; m < SLOT_KG / 2; ++m)
                                    if (m < nmma) mma_f16<2>(d_tmem, ad + m * (2 * LBO_A >> 4), bd + m * (2 * LBO_B >> 4), idesc, 1u);
                                commit_pair_addr(bar_empty + wslot * 8, 0x3);
                                if (nmma > SLOT_KG / 2) {
#pragma unroll
                                    for (uint32_t m = 0; m < SLOT_KG / 2; ++m)
                                        if (m + SLOT_KG / 2 < nmma)
                                            mma_f16<2>(d_tmem, ad + (m + SLOT_KG / 2) * (2 * LBO_A >> 4), bd_b + m * (2 * LBO_B >> 4), idesc, 1u);
                                    commit_pair_addr(bar_empty + slot_b * 8, 0x3);
                                }
                            }
                            if (e.x & E_POST_ACC) commit_pair(&bars[C::BAR_ACC_READY + (e.x & E_SLOT1)], 0x3);
                            if (e.x & E_POST_X) commit_pair(&bars[C::BAR_X_DONE + xb], 0x3);
                        }
                        __syncwarp();
                        TCS_TR(if (tr && i < 48) tr[2 * i + 1] = clock64();)
                        wslot = nmma > SLOT_KG / 2 ? slot_b : wslot;
                        wslot = wslot + 1 == NP ? 0 : wslot + 1;
                        ++gpiece;
                        e = e_next;
                    }
                    if (t > 0 || STATE) hphase ^= 1;
                }
                out_pending = a.preds != nullptr;
            }
            if (out_pending) out_piece(false);                 // the last tile's output layer
        } else if (warp == MMA_WARP && lane == 0) {
            // =============================== peer CTA: forward "piece landed in my ring" to the leader ==================
            uint32_t gpiece = 0;
            auto forward = [&]() {
                mbar_wait_wd(&bars[C::BAR_W_FULL + (gpiece & (C::NFULL - 1))], (gpiece / C::NFULL) & 1);
                mbar_arrive_remote(&bars[C::BAR_W_FULL + (gpiece & (C::NFULL - 1))], 0);
                ++gpiece;
            };
            bool out_pending = false;
            for (int tile = cluster_id; tile < a.n_pair_tiles; tile += n_clusters) {
                for (int t = 0; t < T; ++t) {
                    const int which = t > 0 ? STEP_LATER : STATE ? STEP_FIRST_STATE : STEP_FIRST;
                    const uint32_t n_ent = sched.n[which];
#pragma unroll 1
                    for (uint32_t i = 0; i < n_ent; ++i) {
                        if (out_pending && (sched.e[which][i].x & E_OUT_BEFORE)) { forward(); out_pending = false; }   // the W_o piece
                        forward();
                    }
                }
                out_pending = a.preds != nullptr;
            }
            if (out_pending) forward();
        }
    } else if (warp == TMA_WARP && lane == 0) {
        // =================================== weight-ring producer (one lane per CTA) =====================================
        const uint8_t* Wc = a.W + (size_t)rank * w_bytes;      // this CTA's half of the layer's weight tiles
        uint32_t wslot = 0, wphase = 0, gpiece = 0;
        bool wrapped = false, out_pending = false;
        auto out_piece = [&]() {                               // this CTA's tile of the output-layer operand: one ring slot
            uint64_t* full = &bars[C::BAR_W_FULL + (gpiece & (C::NFULL - 1))];
            if (wrapped) mbar_wait_wd(&bars[C::BAR_W_EMPTY + wslot], wphase ^ 1);
            mbar_arrive_expect_tx(full, C::OUT_BYTES);
            bulk_g2s(sW + wslot * SLOT_BYTES, a.Wo16 + (size_t)rank * C::OUT_BYTES, C::OUT_BYTES, full);
            if (++wslot == NP) { wslot = 0; wphase ^= 1; wrapped = true; }
            ++gpiece;
        };
        for (int tile = cluster_id; tile < a.n_pair_tiles; tile += n_clusters) {
            for (int t = 0; t < T; ++t) {
                TCS_TR(long long* tr = (a.trace && blockIdx.x == 0 && tile == cluster_id && t == TRACE_T) ? a.trace : nullptr;)
                const int which = t > 0 ? STEP_LATER : STATE ? STEP_FIRST_STATE : STEP_FIRST;
                const uint32_t n_ent = sched.n[which];
#pragma unroll 1
                for (uint32_t i = 0; i < n_ent; ++i, ++gpiece) {
                    const uint32_t ex = sched.e[which][i].x;
                    if (out_pending && (ex & E_OUT_BEFORE)) { out_piece(); out_pending = false; }
                    uint32_t kg_left = ((ex >> E_NMMA_SHIFT) & 0x1F) * 2, src_kg = ex >> E_SRC_SHIFT;
                    uint64_t* full = &bars[C::BAR_W_FULL + (gpiece & (C::NFULL - 1))];      // one "landed" barrier per piece
                    TCS_TR(if (tr && i < 48) tr[256 + 2 * i] = clock64();)
                    bool first = true;
                    while (kg_left > 0) {                      // one or two slots
                        const uint32_t kg = kg_left < (uint32_t)SLOT_KG ? kg_left : (uint32_t)SLOT_KG, bytes = kg * KG_BYTES_B;
                        if (wrapped) mbar_wait_wd(&bars[C::BAR_W_EMPTY + wslot], wphase ^ 1);   // previous occupant consumed
                        if (first) mbar_arrive_expect_tx(full, kg_left * KG_BYTES_B);           // all bytes of the piece
                        first = false;
                        bulk_g2s(sW + wslot * SLOT_BYTES, Wc + (size_t)src_kg * KG_BYTES_B, bytes, full);
                        kg_left -= kg; src_kg += kg;
                        if (++wslot == NP) { wslot = 0; wphase ^= 1; wrapped = true; }
                    }
                    TCS_TR(if (tr && i < 48) tr[257 + 2 * i] = clock64();)
                }
            }
            out_pending = a.preds != nullptr;
        }
        if (out_pending) out_piece();
    }
    __syncwarp();
    fence_before_sync();
    cluster_sync();
    tc::timeline_stamp(a.timeline, 2);
    if (warp == MMA_WARP) tmem_dealloc<2>(tmem, C::TMEM_COLS);
}

bool supported(int H) { return H == 256; }

size_t scratch_bytes(int H, int sm_count) { return H == 256 ? (size_t)sm_count * Cfg<256>::CSTATE_BYTES : 0; }

int launch_layer(int H, const TcLayerArgs& a, int sm_count, cudaStream_t st) {
    if (H != 256) return APE_ERR_UNSUPPORTED;
    using C = Cfg<256>;
    if (a.kgx < 2 || a.kgx > C::KG || (a.kgx & 1) || !a.cstate) return APE_ERR_UNSUPPORTED;
    if (a.preds && (!a.Wo16 || a.O > (int)C::OUT_N / 2)) return APE_ERR_UNSUPPORTED;
    if ((a.h0 != nullptr) != (a.c0 != nullptr)) return APE_ERR_BAD_ARG;
    Schedule sched{};
    for (int which = 0; which < N_STEP_KINDS; ++which) {
        Recorder r{sched.e[which], 0, a.kgx, C::KG, 0u, false};
        walk_step<C::NCH>(which, a.kgx, r);
        if (r.overflow) return APE_ERR_UNSUPPORTED;
        sched.n[which] = (uint32_t)r.n;
    }
    const size_t smem = C::SMEM;
    auto kernel = a.h0 ? lstm_layer_tcs_kernel<256, true> : lstm_layer_tcs_kernel<256, false>;
    APE_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int clusters = sm_count / 2;
    if (clusters > a.n_pair_tiles) clusters = a.n_pair_tiles;
    kernel<<<2 * clusters, THREADS, smem, st>>>(a, sched);
    return check_launch();
}

}  // namespace tcs
}  // namespace ape

// Host self-check hook (tests only): the step schedule of the streamed-weights kernel for an x-part of kgx k-groups.
// first_step: 0 = a later step, 1 = the first step of a tile, 2 = the first step of a tile with a caller-supplied initial state.
// entries: [n][2] words (.x flags / MMAs / K-slices needed / weight offset, .y A-operand offset), see the E_* bits above.
extern "C" int ape_selfcheck_tcs_schedule(int kgx, int first_step, uint32_t* entries, int max_entries, int* n_entries) {
    using namespace ape::tcs;
    using C = Cfg<256>;
    if (!entries || !n_entries || kgx < 2 || kgx > C::KG || (kgx & 1) || first_step < 0 || first_step > 2) return APE_ERR_BAD_ARG;
    Schedule sched{};
    Recorder r{sched.e[0], 0, kgx, C::KG, 0u, false};
    walk_step<C::NCH>(first_step == 0 ? STEP_LATER : first_step == 1 ? STEP_FIRST : STEP_FIRST_STATE, kgx, r);
    if (r.overflow || r.n > max_entries) return APE_ERR_UNSUPPORTED;
    for (int i = 0; i < r.n; ++i) { entries[2 * i] = sched.e[0][i].x; entries[2 * i + 1] = sched.e[0][i].y; }
    *n_entries = r.n;
    return APE_OK;
}
