// Stage 2, tensor-core variant: layers >= 1 of the MC-dropout LSTM on tcgen05 with TMEM accumulators.
//
// One CTA PAIR (cluster of 2, tcgen05 cta_group::2) owns a tile of 256 (estimate, MC-sample) rows - 128 per CTA,
// one row per TMEM lane - for all T steps of one layer.  Everything the recurrence needs stays on chip:
//   * the layer's gate weights as fp16 in shared memory, split by gate column across the pair (each CTA holds
//     64 of every 128-column chunk; the hardware shares the halves), loaded once per CTA;
//   * x_t and h_{t-1} as fp16 A-operand tiles in shared memory (K-major no-swizzle, see ape_umma.cuh): h_t is
//     written by the epilogue warps themselves and never goes through global memory inside a layer, x_t is
//     streamed in by dedicated loader warps that apply the dropout mask as a bitwise AND on the fp16 units;
//   * the 128 x 4H fp32 gate pre-activations in TMEM (H/32 chunks of 32 hidden units x 4 gates = 128 columns);
//   * the fp32 cell state c in registers (8 units x H/32 chunks per thread).
// Warp roles per CTA: 16 epilogue warps (TMEM -> registers, bias, sigmoid/tanh cell update, operand packing,
// output layer), 4 operand-loader warps (x_{t+1} under the epilogue of step t: inter-layer fp16 units or layer 0's
// feature window, Philox / injected dropout) and one MMA-issue warp; only the leader CTA's issuer runs.  Hand-offs go
// through mbarriers: tcgen05.commit (multicast to both CTAs) publishes accumulators, the epilogue warps of both
// CTAs arrive on the leader's barriers to publish operands / free accumulator chunks.  The x-part of step t+1
// is issued into a chunk as soon as the epilogue has drained it, so the tensor pipe runs under the epilogue of
// step t; only the recurrent half waits for h_t.
// All layers run here (layer 0 once per estimate, layers >= 1 per MC sample); between layers h_t travels as fp16
// units pre-scaled by the consumer's 1/(1-p) so every operand is rounded to fp16 exactly once.
// Precision: fp16 operands, fp32 accumulate and state.  The fp32 FFMA kernel remains the exact path; the host
// API picks per model with a probe (see estimate/batched.py).
#include "ape_common.cuh"
#include "ape_lstm_pack.h"
#include "ape_lstm_plan.cuh"
#include "ape_umma.cuh"
#include "ape_f32x2.cuh"
#include "ape_lstm_tc_args.cuh"

namespace ape {
namespace tc {

#ifndef APE_TC_LOAD_WARPS
#define APE_TC_LOAD_WARPS 8
#endif
constexpr int EPI_WARPS = 16, LOAD_WARPS = APE_TC_LOAD_WARPS;
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int MMA_WARP = EPI_WARPS + LOAD_WARPS;
// APE_TC_SETMAXNREG = 1 (default): the CTA is padded to whole warpgroups (3 idle warps next to the MMA issuer) and the roles re-balance
// the register file with setmaxnreg: epilogue warps 88 registers, loaders 56, the issuer's warpgroup 40 (896 x 72 = 512 x 88 + 256 x 56 +
// 128 x 40) - the epilogue's working set (cell state, two accumulator buffers, the gate values) spills less: +3 % on B200.  (96 / 48 / 24
// spills in the loaders and the issuer instead; 0 = the 800-thread CTA with a uniform 72.)
#ifndef APE_TC_SETMAXNREG
#define APE_TC_SETMAXNREG 1
#endif
#ifndef APE_TC_REGS_EPI
#define APE_TC_REGS_EPI 88
#define APE_TC_REGS_LOAD 56
#define APE_TC_REGS_MMA 40
#endif
#if APE_TC_SETMAXNREG
static_assert(512 * APE_TC_REGS_EPI + 256 * APE_TC_REGS_LOAD + 128 * APE_TC_REGS_MMA <= 896 * 72, "the re-balanced register file must fit the launch allocation");
constexpr int THREADS = (MMA_WARP + 4) * 32;       // 16 epilogue + 8 operand-loader + 1 MMA-issue + 3 idle warps = 896
#define APE_REG_INC(n) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(n))
#define APE_REG_DEC(n) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(n))
#else
constexpr int THREADS = (MMA_WARP + 1) * 32;       // 16 epilogue + 8 operand-loader + 1 MMA-issue warps = 800
#define APE_REG_INC(n)
#define APE_REG_DEC(n)
#endif
constexpr int ROWS = 128;                          // rows per CTA = TMEM lanes

enum { BAR_X_READY = 0, BAR_X_DONE = 1, BAR_ACC_READY = 2, BAR_SLOT_FREE = 6, BAR_H_READY = 10, BAR_OUT_READY = 14, BAR_OUT_DONE = 15, BAR_COUNT = 16 };
constexpr uint32_t BAR_BLOCK_BYTES = 256;          // barriers + the TMEM base slot

// Tracing (tools/tc_trace.py) is a compile-time option: even predicated off, the stamps cost every epilogue warp ~40 issue slots per
// chunk.  Build with -DAPE_TC_TRACE=1 to get them: role 0 = epilogue warp 0 (chunk 0), role 1 = loader warp 16, role 2 = MMA issuer;
// only block 0, first tile, lane 0.
#ifndef APE_TC_TRACE
#define APE_TC_TRACE 0
#endif
#if APE_TC_TRACE
#define APE_TRACE(role, t, ev) do { if (a.trace && blockIdx.x == 0 && tile == cluster_id && lane == 0 && (t) < 16) \
    a.trace[((role) * 16 + (t)) * 16 + (ev)] = clock64(); } while (0)
#else
#define APE_TRACE(role, t, ev) do { } while (0)
#endif

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory"); }

// STATE: a caller-supplied initial state (a.h0, a.c0).  Step 0 of every tile then runs like every later step - x-part, then the
// recurrent half on h_0 - and the cell starts from c_0; the x-part MMAs keep their order, so h_0 = c_0 = 0 reproduces the
// stateless kernel bit for bit (the recurrent products only add +0 to the fp32 accumulators).
template <int H, bool STATE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1) lstm_layer_tc_kernel(TcLayerArgs a) {
    using namespace umma;
    constexpr int NCH = H / 32, KG = H / 8;
    constexpr uint32_t KG_BYTES_B = 64 * 16;                   // one k-group of a 64-column weight tile
    constexpr uint32_t A_BYTES = KG * ROWS * 16;               // one A-operand tile
    constexpr uint32_t LBO_A = ROWS * 16, LBO_B = 64 * 16, SBO = 128;
    constexpr uint32_t TMEM_COLS = NCH * 128 <= 32 ? 32 : NCH * 128 <= 64 ? 64 : NCH * 128 <= 128 ? 128 : NCH * 128 <= 256 ? 256 : 512;

    const int kgx = a.kgx, T = a.T;
    const uint32_t chunk_bytes = (uint32_t)(kgx + KG) * KG_BYTES_B;   // x k-groups then h k-groups of one chunk
    const uint32_t w_bytes = NCH * chunk_bytes;

    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* sAh = smem;                                       // [2][A_BYTES]
    uint8_t* sAx = sAh + 2 * A_BYTES;                          // [A_BYTES] (kgx k-groups used)
    float* sBias = reinterpret_cast<float*>(sAx + A_BYTES);    // [4H]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sBias + 4 * H);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + BAR_COUNT);
    uint8_t* sW = reinterpret_cast<uint8_t*>(bars) + BAR_BLOCK_BYTES; // [w_bytes], after the barrier block

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;

    // ---- one-time set-up: weights + bias -> smem, TMEM, barriers ------------------------------------------------
    timeline_stamp(a.timeline, 0);
    {
        const uint4* src = reinterpret_cast<const uint4*>(a.W + (size_t)rank * w_bytes);
        uint4* dst = reinterpret_cast<uint4*>(sW);
        for (uint32_t i = tid; i < w_bytes / 16; i += THREADS) dst[i] = __ldg(src + i);
        for (int i = tid; i < 4 * H; i += THREADS) sBias[i] = a.bias_s[i];
    }
    if (warp == MMA_WARP) {
        tmem_alloc<2>(tmem_slot, TMEM_COLS);
        tmem_relinquish<2>();
    }
    if (tid == 0) {
        mbar_init(&bars[BAR_X_READY], 2 * LOAD_WARPS);
        mbar_init(&bars[BAR_X_DONE], 1);
        for (int c = 0; c < 4; ++c) {
            mbar_init(&bars[BAR_ACC_READY + c], 1);
            mbar_init(&bars[BAR_SLOT_FREE + c], 2 * EPI_WARPS);
            mbar_init(&bars[BAR_H_READY + c], 2 * EPI_WARPS);   // the 32 hidden units of chunk c of h_t are in both CTAs' tiles
        }
        mbar_init(&bars[BAR_OUT_READY], 1);
        mbar_init(&bars[BAR_OUT_DONE], 2 * EPI_WARPS);
        mbar_init_fence();
    }
    fence_proxy_async_smem();
    fence_before_sync();
    cluster_sync();
    fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    timeline_stamp(a.timeline, 1);

    if (warp < EPI_WARPS) {
        APE_REG_INC(APE_TC_REGS_EPI);
        // =================================== epilogue warps ===========================================================
        // warp (q, s): rows 32q..32q+31 (its TMEM lane quarter) x the 8 hidden units 8s..8s+7 of EVERY 32-unit chunk.  Chunk c
        // of the accumulator is drained by all warps at the start of pass c, so the issuer can refill it (x-part of the next
        // step, then the recurrent pieces whose K-slices are already published) while passes c+1.. are still computing.
        const int q = warp & 3, s = warp >> 2;
        const int row_l = 32 * q + lane;                       // local row == TMEM lane
        const uint32_t t_lane = (uint32_t)(32 * q) << 16;
        const bool warp_live = 32 * q < a.rpc;                 // a quarter without rows only keeps the barrier protocol going
        uint32_t ph_acc = 0, ph_out = 0;
        float cst[NCH][8];

        for (int tile = cluster_id; tile < a.n_pair_tiles; tile += n_clusters) {
            const int row = (tile * 2 + (int)rank) * a.rpc + row_l;
            const bool valid = row_l < a.rpc && row < a.rows;
#pragma unroll
            for (int c = 0; c < NCH; ++c)
#pragma unroll
                for (int u = 0; u < 8; ++u) cst[c][u] = 0.0f;
            if constexpr (STATE) {
                // h_0 into the operand tile step 0 reads (tile 0), c_0 into the registers.  The tile is free: this warp has drained
                // every accumulator of the previous tile's last step (and waited for its output product), so every MMA that read
                // an h tile of that tile has retired.
                if (warp_live) {
                    const float4* h0r = reinterpret_cast<const float4*>(a.h0 + (size_t)(valid ? row : 0) * H);
                    const float4* c0r = reinterpret_cast<const float4*>(a.c0 + (size_t)(valid ? row : 0) * H);
#pragma unroll
                    for (int c = 0; c < NCH; ++c) {
                        const int j = 4 * c + s;
                        const float4 z = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                        const float4 h_a = valid ? __ldg(h0r + 2 * j) : z, h_b = valid ? __ldg(h0r + 2 * j + 1) : z;
                        const float4 c_a = valid ? __ldg(c0r + 2 * j) : z, c_b = valid ? __ldg(c0r + 2 * j + 1) : z;
                        cst[c][0] = c_a.x; cst[c][1] = c_a.y; cst[c][2] = c_a.z; cst[c][3] = c_a.w;
                        cst[c][4] = c_b.x; cst[c][5] = c_b.y; cst[c][6] = c_b.z; cst[c][7] = c_b.w;
                        *reinterpret_cast<uint4*>(sAh + unit_offset(ROWS, row_l, j)) =
                            make_uint4(pack_half2(h_a.x, h_a.y), pack_half2(h_a.z, h_a.w), pack_half2(h_b.x, h_b.y), pack_half2(h_b.z, h_b.w));
                    }
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0)
#pragma unroll
                    for (int c = 0; c < NCH; ++c) mbar_arrive_leader(&bars[BAR_H_READY + c], rank);
            }

            for (int t = 0; t < T; ++t) {
                uint8_t* sAh_next = sAh + ((t + 1) & 1) * A_BYTES;
                // last step of the last layer: h_T is published like every other h_t - the output layer is one more (small)
                // tensor-core product  h_T x W_o^T  issued into the last accumulator chunk once that chunk has been drained
                const bool final_out = a.preds != nullptr && t == T - 1;
                if (warp == 0) APE_TRACE(0, t, 0);
                if (!warp_live) {
#pragma unroll
                    for (int c = 0; c < NCH; ++c) {
                        mbar_wait(&bars[BAR_ACC_READY + c], ph_acc);
                        if (lane == 0) {
                            mbar_arrive_leader(&bars[BAR_SLOT_FREE + c], rank);
                            if (t + 1 < T || final_out) mbar_arrive_leader(&bars[BAR_H_READY + c], rank);
                        }
                    }
                } else {
                    // Half-passes of 4 hidden units (16 accumulator columns), double-buffered: the TMEM load of half-pass
                    // hp+1 is in flight while the cells of half-pass hp are computed.
                    uint32_t rbuf[2][16];
                    float hlo[4];
                    mbar_wait(&bars[BAR_ACC_READY + 0], ph_acc);
                    fence_after_sync();
                    tmem_ld_x16(tmem + t_lane + (uint32_t)(32 * s), rbuf[0]);
#pragma unroll
                    for (int hp = 0; hp < 2 * NCH; ++hp) {
                        const int c = hp >> 1, half = hp & 1;
                        uint32_t* r = rbuf[hp & 1];
                        tmem_ld_wait();                        // this half-pass's columns have landed
                        if (half == 1) {                       // chunk c fully drained: the issuer may refill it
                            fence_before_sync();
                            __syncwarp();
                            if (lane == 0) mbar_arrive_leader(&bars[BAR_SLOT_FREE + c], rank);
                            if (warp == 0) APE_TRACE(0, t, 2 + 3 * c);
                        }
                        if (hp + 1 < 2 * NCH) {
                            if (half == 1) {
                                mbar_wait(&bars[BAR_ACC_READY + c + 1], ph_acc);
                                fence_after_sync();
                                if (warp == 0) APE_TRACE(0, t, 1 + 3 * (c + 1));
                            }
                            tmem_ld_x16(tmem + t_lane + (uint32_t)(((hp + 1) >> 1) * 128 + 32 * s + 16 * ((hp + 1) & 1)), rbuf[(hp + 1) & 1]);
                        }
                        const float4* bias4 = reinterpret_cast<const float4*>(sBias + (c * 32 + 8 * s + 4 * half) * 4);
                        // the 4 cells advance in lock-step through the transcendental stages (independent MUFU ops back to back):
                        //   e = 2^-(gate+bias)  ->  i*g~ and f share one reciprocal  ->  2^(-2c)  ->  h = o * tanh(c)
                        float hv[4];
#if APE_TC_TANH
                        // 5 MUFU per cell: sigmoid(x) = 0.5 + 0.5 tanh(x / 2) with the hardware tanh (see ape_lstm_tc_args.cuh)
                        float tg[16];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const float4 bs = bias4[u];            // 0.5 b (i, f, o), b (g)
                            // tanh arguments in packed fp32 pairs (ape_f32x2.cuh): (i, f) and (g, o) sit in adjacent accumulator registers and
                            // adjacent bias words; r * (0.5, 0.5) + b and r * (1, 0.5) + b are the scalar operations bit for bit
                            const F2 aif = fma2(pk(__uint_as_float(r[4 * u + 0]), __uint_as_float(r[4 * u + 1])), splat(0.5f), pk(bs.x, bs.y));
                            const F2 ago = fma2(pk(__uint_as_float(r[4 * u + 2]), __uint_as_float(r[4 * u + 3])), pk(1.0f, 0.5f), pk(bs.z, bs.w));
                            tg[4 * u + 0] = tanh_approx(lo(aif)); tg[4 * u + 1] = tanh_approx(hi(aif));
                            tg[4 * u + 2] = tanh_approx(lo(ago)); tg[4 * u + 3] = tanh_approx(hi(ago));
                        }
#pragma unroll
                        for (int u = 0; u < 4; u += 2) {               // the cell update of two units per instruction (as in ape_lstm_tcw.cu)
                            const F2 h2c = splat(0.5f);
                            const F2 gi = fma2(pk(tg[4 * u + 0], tg[4 * u + 4]), h2c, h2c), gf = fma2(pk(tg[4 * u + 1], tg[4 * u + 5]), h2c, h2c);
                            const F2 c2 = fma2(gf, pk(cst[c][4 * half + u], cst[c][4 * half + u + 1]), gi * pk(tg[4 * u + 2], tg[4 * u + 6]));
                            cst[c][4 * half + u] = lo(c2); cst[c][4 * half + u + 1] = hi(c2);
                            const F2 h2 = fma2(pk(tg[4 * u + 3], tg[4 * u + 7]), h2c, h2c) * pk(tanh_approx(lo(c2)), tanh_approx(hi(c2)));
                            hv[u] = lo(h2); hv[u + 1] = hi(h2);
                        }
#else
                        float ev[16], num[4], den[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const float4 bs = bias4[u];            // 0.5 b (i, f, o), b (g) -> -log2e (gate + b), g: -2 log2e (gate + b)
                            ev[4 * u + 0] = ex2_approx(fminf(fmaf(__uint_as_float(r[4 * u + 0]), -LOG2E, bs.x * (-2.0f * LOG2E)), EX2_CLAMP));
                            ev[4 * u + 1] = ex2_approx(fminf(fmaf(__uint_as_float(r[4 * u + 1]), -LOG2E, bs.y * (-2.0f * LOG2E)), EX2_CLAMP));
                            ev[4 * u + 2] = ex2_approx(fminf(fmaf(__uint_as_float(r[4 * u + 2]), -2.0f * LOG2E, bs.z * (-2.0f * LOG2E)), EX2_CLAMP));
                            // (o gate unclamped: an infinite e_o only makes the reciprocal below 0; e_c is finite since |c| <= T)
                            ev[4 * u + 3] = ex2_approx(fmaf(__uint_as_float(r[4 * u + 3]), -LOG2E, bs.w * (-2.0f * LOG2E)));
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const float ab = (1.0f + ev[4 * u + 0]) * (1.0f + ev[4 * u + 2]), cf = 1.0f + ev[4 * u + 1];
                            num[u] = fmaf(cst[c][4 * half + u], ab, (1.0f - ev[4 * u + 2]) * cf);
                            den[u] = rcp_approx(ab * cf);
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            cst[c][4 * half + u] = num[u] * den[u];
                            // e_c = 2^(-2c log2e): |c| <= T, no overflow; with a state |c| <= |c_0| + T, clamped
                            const float pc = cst[c][4 * half + u] * (-2.0f * LOG2E);
                            num[u] = ex2_approx(STATE ? fminf(pc, EX2_CLAMP) : pc);
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) hv[u] = (1.0f - num[u]) * rcp_approx((1.0f + ev[4 * u + 3]) * (1.0f + num[u]));
#endif

                        const int j = 4 * c + s;               // k-group of units 32c + 8s .. + 7
                        if (half == 1) {
                            *reinterpret_cast<uint4*>(sAh_next + unit_offset(ROWS, row_l, j)) =
                                make_uint4(pack_half2(hlo[0], hlo[1]), pack_half2(hlo[2], hlo[3]), pack_half2(hv[0], hv[1]), pack_half2(hv[2], hv[3]));
                        }
                        if (half == 1) {
                            if (final_out && c == NCH - 1 && warp == 0) {
                                // Output layer: this CTA's 16 of the 32 columns of the fp16 W_o tile (the leader holds the fp16 ROUNDING of
                                // W_o for the 16 outputs, the peer the fp16 REMAINDER W_o - fp16(W_o): their products are summed, so only
                                // h_T carries an fp16 rounding) go where h_{T-1} was - that tile is dead: this pass started after the LAST
                                // accumulator of the step was complete, i.e. after every MMA that reads it had retired, and shared memory
                                // has no room for a dedicated copy.  It is in place before this warp publishes the last slice of h_T.
                                const uint4* wo = reinterpret_cast<const uint4*>(a.Wo16) + (size_t)rank * KG * 16;
                                uint4* dst = reinterpret_cast<uint4*>(sAh + (t & 1) * A_BYTES);
#pragma unroll
                                for (int i = 0; i < KG * 16 / 32; ++i) dst[i * 32 + lane] = __ldg(wo + i * 32 + lane);
                            }
                            if (t + 1 < T || final_out) {      // publish this chunk's slice of h_t: its K-slice of the next recurrent
                                fence_proxy_async_smem();      // product can be issued while later chunks still run
                                __syncwarp();
                                if (lane == 0) mbar_arrive_leader(&bars[BAR_H_READY + c], rank);
                            }
                            if (warp == 0) APE_TRACE(0, t, 3 + 3 * c);
                            if (a.out_units && APE_EXP != 4) {
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
                ph_acc ^= 1;
                if (final_out) {                               // output_layer (nn_models.py:189), last step only
                    if (warp == 0) APE_TRACE(0, t, 13);
                    // the issuer multiplies the published h_T by W_o^T (fp16 operands, fp32 accumulate) into the first 16 columns
                    // of the last accumulator chunk; every warp waits for it - also the guarantee that h_T has been consumed
                    // before the next tile's cell updates rewrite the operand tiles
                    mbar_wait(&bars[BAR_OUT_READY], ph_out);
                    ph_out ^= 1;
                    fence_after_sync();
                    if (warp_live) {
                        uint32_t o32[32];                      // columns 0..15: h_T x fp16(W_o)^T, 16..31: h_T x (W_o - fp16(W_o))^T
                        tmem_ld_x32(tmem + t_lane + (uint32_t)((NCH - 1) * 128), o32);
                        tmem_ld_wait();
                        if (valid) {
                            const int e = row / a.n, smp = row - e * a.n;
                            const int b = e / a.nF, fb = stream_frame0(a.stream_frames, a.frame0, b), f = fb + e % a.nF;
#pragma unroll
                            for (int i = 0; i < 4; ++i) {      // this thread: outputs o = s, s+4, ... of its row (O <= 16)
                                const int o = s + 4 * i;
                                if (o < a.O && fb >= 0) {      // (an inactive stream keeps its prediction ring untouched)
                                    const float y = __uint_as_float(pick4(o32, i, s)) + __uint_as_float(pick4(o32, 4 + i, s)) + __ldg(a.bo + o);
                                    float* dst = a.preds + (((size_t)b * a.pred_ring + f % a.pred_ring) * a.n_out) * a.O + o;
                                    if (a.n == 1 && a.n_out > 1) for (int s2 = 0; s2 < a.n_out; ++s2) dst[(size_t)s2 * a.O] = y;
                                    else dst[(size_t)smp * a.O] = y;
                                }
                            }
                        }
                    }
                    fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_leader(&bars[BAR_OUT_DONE], rank);   // the chunk may be refilled for the next tile
                    if (warp == 0) APE_TRACE(0, t, 14);
                }
            }
        }
    } else if (warp < MMA_WARP) {
        APE_REG_DEC(APE_TC_REGS_LOAD);
        // =================================== operand-loader warps: x_t -> sAx ===========================================
        constexpr int TPR = LOAD_WARPS * 32 / ROWS;            // loader threads per row, each an equal share of the x k-groups
        const int row_l = (tid - EPI_THREADS) & (ROWS - 1);
        const int half = (tid - EPI_THREADS) >> 7;
        uint32_t ph_xdone = 0;
        bool first = true;
        for (int tile = cluster_id; tile < a.n_pair_tiles; tile += n_clusters) {
            const int row = (tile * 2 + (int)rank) * a.rpc + row_l;
            const bool valid = row_l < a.rpc && row < a.rows;
            const int e = valid ? row / a.n : 0, smp = valid ? row - e * a.n : 0;
            const int b = e / a.nF, f = stream_frame0(a.stream_frames, a.frame0, b) + e % a.nF;
            for (int t = 0; t < T; ++t) {
                if (a.in_mode == IN_UNITS || a.in_mode == IN_SHARED_UNITS) {
                    // all loads of the step go out before anything waits; masks are ANDed in as the data lands; only the
                    // shared-memory stores sit behind "the previous x tile has been consumed"
                    const uint4* src = reinterpret_cast<const uint4*>(a.in);
                    if (a.in_mode == IN_UNITS) src += ((((size_t)tile * T + t) * 2 + rank) * KG) * ROWS + row_l;
                    else src += ((((size_t)(e >> (a.in_rpc_shift + 1)) * T + t) * 2 + ((e >> a.in_rpc_shift) & 1)) * KG) * ROWS +
                                (e & ((1 << a.in_rpc_shift) - 1));
                    if (warp == EPI_WARPS) APE_TRACE(1, t, 0);
                    constexpr int KH = KG / TPR;
                    const int j0 = half * KH;
                    src += (size_t)j0 * ROWS;
                    uint4 pre[KH];
#pragma unroll
                    for (int jj = 0; jj < KH; ++jj) pre[jj] = valid ? __ldg(src + (size_t)jj * ROWS) : make_uint4(0, 0, 0, 0);
#pragma unroll
                    for (int jj = 0; jj < KH; ++jj) {
                        const int j = j0 + jj;
                        if (a.mask_mode == APE_MASK_PHILOX && APE_EXP != 3) {
                            const uint4 m = APE_PHILOX_DRAW(a, a.stream_id0 + (uint32_t)b, (uint32_t)f, (uint32_t)smp,
                                                                 (uint32_t)a.gap, (uint32_t)t, (uint32_t)j, a.keep_thr16);
                            pre[jj].x &= m.x; pre[jj].y &= m.y; pre[jj].z &= m.z; pre[jj].w &= m.w;
                        } else if (a.mask_mode == APE_MASK_INJECTED && valid) {
                            const uint2 m = __ldg(reinterpret_cast<const uint2*>(
                                a.masks + ((((size_t)e * a.n_gaps + a.gap) * T + t) * a.n + smp) * H + j * 8));
                            pre[jj].x &= ((m.x & 0xFFu) ? 0xFFFFu : 0u) | ((m.x & 0xFF00u) ? 0xFFFF0000u : 0u);
                            pre[jj].y &= ((m.x & 0xFF0000u) ? 0xFFFFu : 0u) | ((m.x & 0xFF000000u) ? 0xFFFF0000u : 0u);
                            pre[jj].z &= ((m.y & 0xFFu) ? 0xFFFFu : 0u) | ((m.y & 0xFF00u) ? 0xFFFF0000u : 0u);
                            pre[jj].w &= ((m.y & 0xFF0000u) ? 0xFFFFu : 0u) | ((m.y & 0xFF000000u) ? 0xFFFF0000u : 0u);
                        }
                    }
                    if (warp == EPI_WARPS) APE_TRACE(1, t, 1);
                    if (!first) { mbar_wait(&bars[BAR_X_DONE], ph_xdone); ph_xdone ^= 1; }
                    first = false;
                    if (warp == EPI_WARPS) APE_TRACE(1, t, 2);
#pragma unroll
                    for (int jj = 0; jj < KH; ++jj) *reinterpret_cast<uint4*>(sAx + unit_offset(ROWS, row_l, j0 + jj)) = pre[jj];
                } else {                                       // layer 0: fp32 features (window of the ring, or dense rows)
                    if (!first) { mbar_wait(&bars[BAR_X_DONE], ph_xdone); ph_xdone ^= 1; }
                    first = false;
                    const float* src = nullptr;
                    if (valid) {
                        if (a.in_mode == IN_DENSE_F32) {
                            src = reinterpret_cast<const float*>(a.in) + ((size_t)row * T + t) * a.Kin;
                        } else {                               // sliding window, clamped at frame 0 (estimator.py:96-97)
                            int fw = f - T + 1 + t;
                            fw = fw < 0 ? 0 : fw;
                            src = reinterpret_cast<const float*>(a.in) + ((size_t)b * a.feat_ring + fw % a.feat_ring) * a.Kin;
                        }
                    }
                    for (int j = half; j < kgx; j += TPR) {
                        float v[8];
#pragma unroll
                        for (int k = 0; k < 8; ++k) v[k] = (valid && 8 * j + k < a.Kin) ? __ldg(src + 8 * j + k) : 0.0f;
                        *reinterpret_cast<uint4*>(sAx + unit_offset(ROWS, row_l, j)) =
                            make_uint4(pack_half2(v[0], v[1]), pack_half2(v[2], v[3]), pack_half2(v[4], v[5]), pack_half2(v[6], v[7]));
                    }
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(&bars[BAR_X_READY], rank);
                if (warp == EPI_WARPS) APE_TRACE(1, t, 3);
            }
        }
    } else {
      APE_REG_DEC(APE_TC_REGS_MMA);     // (with setmaxnreg, 3 idle warps pad the issuer's warpgroup: they only take part in this and the final barrier)
      if (warp == MMA_WARP && rank == 0) {
        // =================================== MMA issuer (leader CTA; the whole warp runs, one elected lane issues) ======
        const uint32_t idesc = make_idesc_f16(256, 128);
        const uint64_t dX = make_desc(smem_u32(sAx), LBO_A, SBO), dH0 = make_desc(smem_u32(sAh), LBO_A, SBO);
        const uint64_t dW = make_desc(smem_u32(sW), LBO_B, SBO);
        // Issue order inside a step follows the order in which the epilogue of the PREVIOUS step releases things:
        //   SLOT_FREE[c]  (chunk c of the accumulator drained)      -> x-part of chunk c, then its recurrent pieces for the
        //                                                              K-slices already published
        //   H_READY[c']   (units 32c'..32c'+31 of h_{t-1} published) -> recurrent pieces (c, c') of every chunk c <= c'
        // so when the last slice arrives only 2 MMAs stand between it and ACC_READY[0].
        uint32_t ph_xready = 0, ph_hready = 0, ph_slot = 0, ph_outdone = 0;
        bool first = true;
        constexpr int KS2 = 2;                                  // K=16 MMAs per 32-unit K-slice (4 k-groups)
        // Output layer of the last layer (nn_models.py:189, last step only): h_T x [fp16(W_o) | W_o - fp16(W_o)]^T as KG/2 MMAs of
        // N = 32 into the first columns of the LAST accumulator chunk, once that chunk has been drained and all of h_T has been
        // published.  It is issued where the chunk would be refilled for the next tile (or after the last tile); the epilogue
        // reads the 32 columns and hands the chunk back (OUT_DONE).
        const uint32_t idesc_out = make_idesc_f16(256, 32);
        const uint64_t dWo = make_desc(smem_u32(sAh + ((T - 1) & 1) * A_BYTES), 16 * 16, SBO);  // over the dead h_{T-1} tile
        bool out_pending = false;
        auto issue_output = [&]() {
            for (int c = 0; c < NCH; ++c) mbar_wait(&bars[BAR_H_READY + c], ph_hready);
            ph_hready ^= 1;
            fence_after_sync();
            if (elect_one()) {
                const uint64_t dHT = desc_advance(dH0, (uint32_t)(T & 1) * A_BYTES);      // step T-1 wrote h_T into tile (T & 1)
#pragma unroll
                for (int k2 = 0; k2 < KG / 2; ++k2)
                    mma_f16<2>(tmem + (NCH - 1) * 128, desc_advance(dHT, k2 * 2 * LBO_A), desc_advance(dWo, k2 * 2 * (16 * 16)), idesc_out, k2 > 0 ? 1u : 0u);
                commit_pair(&bars[BAR_OUT_READY], 0x3);
            }
            __syncwarp();
            mbar_wait(&bars[BAR_OUT_DONE], ph_outdone);         // every epilogue warp has read its outputs
            ph_outdone ^= 1;
            fence_after_sync();
            out_pending = false;
        };
        for (int tile = cluster_id; tile < a.n_pair_tiles; tile += n_clusters) {
            for (int t = 0; t < T; ++t) {
                APE_TRACE(2, t, 0);
                mbar_wait(&bars[BAR_X_READY], ph_xready);
                ph_xready ^= 1;
                fence_after_sync();
                APE_TRACE(2, t, 1);
                if (STATE && out_pending) {                     // (t == 0) the previous tile's output layer goes first: the
                    mbar_wait(&bars[BAR_SLOT_FREE + NCH - 1], ph_slot);   // epilogue publishes h_0 only after it has read those outputs
                    fence_after_sync();
                    issue_output();
                }
                const uint64_t dH = desc_advance(dH0, (t & 1) * A_BYTES);
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    if (!first) { mbar_wait(&bars[BAR_SLOT_FREE + c], ph_slot); fence_after_sync(); }
                    if (c == NCH - 1 && out_pending) issue_output();             // (t == 0: the previous tile's output layer)
                    APE_TRACE(2, t, 2 + 3 * c);
                    if (elect_one()) {
                        const uint64_t wx = desc_advance(dW, c * chunk_bytes);
                        for (int k2 = 0; k2 < kgx / 2; ++k2)
                            mma_f16<2>(tmem + c * 128, desc_advance(dX, k2 * 2 * LBO_A), desc_advance(wx, k2 * 2 * LBO_B), idesc, k2 > 0 ? 1u : 0u);
                        if (t == 0 && !STATE) commit_pair(&bars[BAR_ACC_READY + c], 0x3);  // h_{-1} = 0: no recurrent half
                        if (c == NCH - 1) commit_pair(&bars[BAR_X_DONE], 0x3);
                        if (t > 0 || STATE) {
                            const uint64_t wh = desc_advance(wx, (uint32_t)kgx * KG_BYTES_B);
#pragma unroll
                            for (int cs = 0; cs < c; ++cs)                       // slices published before this chunk drained
#pragma unroll
                                for (int k2 = cs * KS2; k2 < (cs + 1) * KS2; ++k2)
                                    mma_f16<2>(tmem + c * 128, desc_advance(dH, k2 * 2 * LBO_A), desc_advance(wh, k2 * 2 * LBO_B), idesc, 1u);
                        }
                    }
                    __syncwarp();
                    APE_TRACE(2, t, 3 + 3 * c);
                    if (t > 0 || STATE) {
                        mbar_wait(&bars[BAR_H_READY + c], ph_hready);           // slice c of h_{t-1}
                        fence_after_sync();
                        APE_TRACE(2, t, 4 + 3 * c);
                        if (elect_one()) {
#pragma unroll
                            for (int cc = 0; cc <= c; ++cc) {                    // chunks whose x-part is already in flight
                                const uint64_t wh = desc_advance(dW, cc * chunk_bytes + (uint32_t)kgx * KG_BYTES_B);
#pragma unroll
                                for (int k2 = c * KS2; k2 < (c + 1) * KS2; ++k2)
                                    mma_f16<2>(tmem + cc * 128, desc_advance(dH, k2 * 2 * LBO_A), desc_advance(wh, k2 * 2 * LBO_B), idesc, 1u);
                                if (c == NCH - 1) commit_pair(&bars[BAR_ACC_READY + cc], 0x3);
                            }
                        }
                        __syncwarp();
                    }
                }
                APE_TRACE(2, t, 14);
                if (!first) ph_slot ^= 1;
                if (t > 0 || STATE) ph_hready ^= 1;
                first = false;
            }
            out_pending = a.preds != nullptr;
        }
        if (out_pending) {                                      // the last tile's output layer
            mbar_wait(&bars[BAR_SLOT_FREE + NCH - 1], ph_slot);
            fence_after_sync();
            issue_output();
        }
      }
    }
    __syncwarp();
    fence_before_sync();
    cluster_sync();
    timeline_stamp(a.timeline, 2);
    if (warp == MMA_WARP) tmem_dealloc<2>(tmem, TMEM_COLS);
}

// all_steps (the model API, DropoutLSTM.forward / monte_carlo_predictions): the output layer on EVERY step of the last layer's
// sequence.  units: [pair tile][T][cta][H/8][128 rows] 16-byte units of fp16 h_t (unscaled); Wo: [O][H] then bias [O];
// preds: [row][T][O] float32.  One thread per output value; rows x T x O x H multiply-adds, negligible next to the layers.
// units_lo (the split-precision kernels, else null): the lo halves of the same units; h = hi + lo is exact in fp32 (the pair
// carries ~22 bits) and enters the same FMA chain.
__global__ void units_output_kernel(const uint4* __restrict__ units, const uint4* __restrict__ units_lo, const float* __restrict__ Wo,
                                    float* __restrict__ preds, int rows, int T, int H, int O) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)rows * T * O) return;
    const int o = (int)(idx % O), t = (int)((idx / O) % T), row = (int)(idx / ((long long)O * T));
    const int tile = row >> 8, cta = (row >> 7) & 1, r = row & 127, KG = H / 8;
    const size_t at = ((((size_t)tile * T + t) * 2 + cta) * KG) * ROWS + r;
    const uint4* src = units + at;
    const float* w = Wo + (size_t)o * H;
    float sum = __ldg(Wo + (size_t)O * H + o);
    for (int j = 0; j < KG; ++j) {
        const uint4 u = __ldg(src + (size_t)j * ROWS);
        const uint4 ul = units_lo ? __ldg(units_lo + at + (size_t)j * ROWS) : make_uint4(0, 0, 0, 0);
        const uint32_t v[4] = {u.x, u.y, u.z, u.w}, vl[4] = {ul.x, ul.y, ul.z, ul.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float2 f = __half22float2(*reinterpret_cast<const __half2*>(&v[k]));
            if (units_lo) {
                const float2 fl = __half22float2(*reinterpret_cast<const __half2*>(&vl[k]));
                f.x += fl.x; f.y += fl.y;
            }
            sum = fmaf(__ldg(w + 8 * j + 2 * k), f.x, sum);
            sum = fmaf(__ldg(w + 8 * j + 2 * k + 1), f.y, sum);
        }
    }
    preds[idx] = sum;
}

int launch_units_output(const uint4* units, const uint4* units_lo, const float* Wo, float* preds, long long rows, int T, int H, int O,
                        cudaStream_t st) {
    const long long total = rows * T * O;
    const int threads = 256;
    units_output_kernel<<<(unsigned)((total + threads - 1) / threads), threads, 0, st>>>(units, units_lo, Wo, preds, (int)rows, T, H, O);
    return check_launch();
}

template <int H> static size_t smem_bytes(int kgx) {
    return 3 * (size_t)(H / 8) * ROWS * 16 + 4 * H * sizeof(float) + BAR_BLOCK_BYTES + (size_t)(H / 32) * (kgx + H / 8) * 64 * 16;
}

template <int H> static int launch(const TcLayerArgs& a, int sm_count, cudaStream_t st) {
    const size_t smem = smem_bytes<H>(a.kgx);
    auto kernel = a.h0 ? lstm_layer_tc_kernel<H, true> : lstm_layer_tc_kernel<H, false>;
    APE_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int clusters = sm_count / 2;
    if (clusters > a.n_pair_tiles) clusters = a.n_pair_tiles;
    kernel<<<2 * clusters, THREADS, smem, st>>>(a);
    return check_launch();
}

}  // namespace tc
}  // namespace ape

constexpr int TC_MAX_SMS = 160;                    // cell-state scratch is sized for this many CTAs (B200: 148)
// rows per CTA of layer 0 (one row per estimate): a small batch is spread over more CTA pairs, 32 rows each; the split-precision
// kernels (tc_flags == 3) take 128 rows always
// (128 rows from 512 estimates on: a 32-row CTA takes as long per step as a full one - its 4 live epilogue warps share one SM quarter -
// so spreading layer 0 of a large batch over 4x the SMs only takes them away from the big layers that run beside it: +1 % per step)
static int tc_rpc0(bool split, long long E) { return split || E >= 512 ? 128 : 32; }
static int tc_kgx(int layer, int I, int H) { return layer == 0 ? ape_pack_kin_pad(0, I, H) / 8 : H / 8; }
static size_t tc_layer_bytes(int layer, int I, int H) {
    return (size_t)2 * (H / 32) * (tc_kgx(layer, I, H) + H / 8) * 64 * 16 + (size_t)4 * H * 4;
}
// bytes of layer l in the single-pass blob (weights_tc) or in the split-precision blob (weights_tcx, ape_lstm_tc_args.cuh: tcx_blob)
static size_t blob_layer_bytes(bool split, int layer, int I, int H) {
    return split ? ape::tcx_blob::layer_bytes(H, layer, I) : tc_layer_bytes(layer, I, H);
}

// bytes of the fp16 weight blob of the tensor-core path: per layer the two CTAs' weight tiles, then the scaled bias; then the
// output-layer tiles and (L >= 3) the wavefront kernel's pieces of layers >= 1
extern "C" int ape_lstm_tc_blob_bytes(int I, int H, int L, int64_t* bytes) {
    if (!bytes || I < 1 || H < 32 || H % 32 != 0 || L < 1) return APE_ERR_BAD_ARG;
    int64_t total = 0;
    for (int l = 0; l < L; ++l) total += (int64_t)tc_layer_bytes(l, I, H);
    total += (int64_t)ape::tc::wo16_bytes(H);
    if (L >= 3) total += (int64_t)(L - 1) * (int64_t)ape::tcw::layer_bytes(H);   // wavefront kernel's pieces of layers >= 1 (H = 128)
    *bytes = total;
    return APE_OK;
}

extern "C" int ape_mc_lstm_tc_supported(int I, int H, int L, int O) {
    // (H <= 128: the output layer is one N = 16 tensor-core product, so O <= 16; the H = 256 kernel takes O <= 20)
    return ((((H == 64 || H == 128) && O <= 16) || (ape::tcs::supported(H) && O <= 20)) && L >= 2 && I >= 1 &&
            ape_pack_kin_pad(0, I, H) <= H && O >= 1) ? 1 : 0;
}

// shapes of the split-precision kernels (tc_flags == 3)
static bool split_supported(int I, int H, int L, int O) {
    return L >= 2 && I >= 1 && O >= 1 && (H == 256 ? ape::tcxs::supported(H, I, O) : ape::tcx::supported(H, I, O));
}

// The small-batch cluster kernels (tc_flags == 4: ape_lstm_tcl.cu; tc_flags == 5: ape_lstm_tcxl.cu at H = 128, ape_lstm_tcxsl.cu at
// H = 256) run every layer of a call in one launch, one cluster per 128 rows (E x n_samples), up to 64 clusters.
constexpr long long CLUSTER_MAX_ROWS = (long long)ape::tc::CLUSTER_ROWS * 64;
static bool cluster_rows_fit(int H, long long E, int n_samples) {
    return (H == 128 || H == 256) && E >= 0 && n_samples >= 1 && E * n_samples <= CLUSTER_MAX_ROWS;
}
static bool cluster_supported(int I, int H, int L, int T, int O, long long E, int n_samples) {
    return cluster_rows_fit(H, E, n_samples) && L >= 2 && L <= ape::tc::CLUSTER_MAX_L && T >= 1 && T <= 40 && I >= 1 &&
           ape_pack_kin_pad(0, I, H) <= H && O >= 1 && O <= (H > 128 ? 32 : 16);
}
// Workspace of a cluster launch: per cluster the exchange buffer of h_t [2][planes][H/8][128] and two layer sequences
// [2][T][planes][H/8][128] (planes: 1, split precision 2 - hi and lo), for every cluster of the largest call (rows), + 256 for the alignment
static size_t cluster_bytes(int H, int T, size_t planes) { return (size_t)(2 + 2 * T) * planes * (H / 8) * ape::tc::CLUSTER_ROWS * 16; }
static size_t cluster_workspace_bytes(int H, int T, long long rows, size_t planes) {
    const long long clusters = rows <= 0 ? 1 : (rows + ape::tc::CLUSTER_ROWS - 1) / ape::tc::CLUSTER_ROWS;
    return cluster_bytes(H, T, planes) * (size_t)clusters + 256;
}

// Workspace layout of the tensor-core path, computed from the LARGEST call that will use the workspace (ws_E) so that calls of
// different sizes in flight on different streams agree on every offset:
//   [2 x scratch region][layer 0 output, copy 0][copy 1][units of layers >= 1, up to 2 buffers (+ 1 for all_steps)]
// Split precision: every units buffer is a (hi, lo) pair, the lo halves behind the hi halves.
struct TcWsLayout { size_t scratch_region, u0, u1, total; };
static size_t tc_u0_bytes(bool split, long long E, int T, int H) {
    const unsigned long long rpc0 = tc_rpc0(split, E), tiles0 = ((unsigned long long)E + 2 * rpc0 - 1) / (2 * rpc0);
    return (size_t)((tiles0 * 256 * T * H * 2 + 255) & ~(unsigned long long)255);
}
static TcWsLayout tc_ws_layout(bool split, int H, int L, int T, long long E, int n_samples, bool all_steps) {
    TcWsLayout w{};
    // a short call (< 512 estimates) spreads layer 0 over 32-row CTAs and needs up to 4x the row slots per estimate (single pass)
    w.u0 = tc_u0_bytes(split, E, T, H);
    if (E > 511) { const size_t small = tc_u0_bytes(split, 511, T, H); if (small > w.u0) w.u0 = small; }
    const unsigned long long tiles1 = ((unsigned long long)E * n_samples + 255) / 256;
    w.u1 = (size_t)((tiles1 * 256 * T * H * 2 + 255) & ~(unsigned long long)255);
    // per-CTA cell-state scratch: two regions (layer 0 of the next call may run on a side stream under a layer >= 1 of this one);
    // streamed-weights kernel (H = 256), two-layer wavefront kernel (H = 128, L >= 3) and split-precision kernels
    if (split) {
        w.scratch_region = H == 256 ? ape::tcxs::scratch_bytes(TC_MAX_SMS) : ape::tcx::scratch_bytes(TC_MAX_SMS);
    } else {
        w.scratch_region = ape::tcs::scratch_bytes(H, TC_MAX_SMS);
        if (L >= 3) { const size_t s2 = ape::tcw::scratch_bytes(H, TC_MAX_SMS); if (s2 > w.scratch_region) w.scratch_region = s2; }
    }
    const int n_u1 = L - 2 + (all_steps ? 1 : 0);
    const size_t planes = split ? 2 : 1;
    w.total = 2 * w.scratch_region + 2 * planes * w.u0 + (size_t)(n_u1 > 2 ? 2 : (n_u1 < 0 ? 0 : n_u1)) * planes * w.u1 + 512;
    // the small-batch cluster kernel (tc_flags == 4) keeps its exchange buffers where the layer kernels keep their units: one set per
    // cluster (sized for every call whose rows fit a launch: the query's other arguments do not enter)
    if (!split && !all_steps && cluster_rows_fit(H, E, n_samples)) {
        const size_t need = 2 * w.scratch_region + cluster_workspace_bytes(H, T, E * n_samples, 1) + 512;
        if (need > w.total) w.total = need;
    }
    return w;
}

extern "C" int ape_mc_lstm_tc_workspace_bytes(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes) {
    if (!bytes || I < 1 || H < 1 || L < 1 || T < 1 || O < 1 || E < 0 || n_samples < 1) return APE_ERR_BAD_ARG;
    if (!ape_mc_lstm_tc_supported(I, H, L, O)) return APE_ERR_UNSUPPORTED;
    *bytes = tc_ws_layout(false, H, L, T, E, n_samples, false).total;
    return APE_OK;
}

// the same for a call with all_steps != 0 (the model API: the last layer's sequence is kept for the per-step output layer)
extern "C" int ape_mc_lstm_tc_workspace_bytes_all_steps(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes) {
    if (!bytes || I < 1 || H < 1 || L < 1 || T < 1 || O < 1 || E < 0 || n_samples < 1) return APE_ERR_BAD_ARG;
    if (!ape_mc_lstm_tc_supported(I, H, L, O)) return APE_ERR_UNSUPPORTED;
    *bytes = tc_ws_layout(false, H, L, T, E, n_samples, true).total;
    return APE_OK;
}

// The split-precision queries: the tcx_* symbols answer for the H = 128 kernel, the tcxs_* symbols for the H = 256 one.
static int split_blob_query(int kernel_H, int I, int H, int L, int64_t* bytes) {
    if (!bytes || H != kernel_H || !split_supported(I, H, L, 1)) return APE_ERR_BAD_ARG;
    int64_t total = (int64_t)ape::tc::wo16_bytes(H);
    for (int l = 0; l < L; ++l) total += (int64_t)blob_layer_bytes(true, l, I, H);
    *bytes = total;
    return APE_OK;
}
static int split_workspace_query(int kernel_H, int I, int H, int L, int T, int O, int E, int n_samples, bool all_steps, uint64_t* bytes) {
    if (!bytes || T < 1 || E < 0 || n_samples < 1) return APE_ERR_BAD_ARG;
    if (H != kernel_H || !split_supported(I, H, L, O)) return APE_ERR_UNSUPPORTED;
    *bytes = tc_ws_layout(true, H, L, T, E, n_samples, all_steps).total;
    return APE_OK;
}
extern "C" int ape_mc_lstm_tcx_supported(int I, int H, int L, int O) { return H == 128 && split_supported(I, H, L, O); }
extern "C" int ape_mc_lstm_tcxs_supported(int I, int H, int L, int O) { return H == 256 && split_supported(I, H, L, O); }
extern "C" int ape_lstm_tcx_blob_bytes(int I, int H, int L, int64_t* bytes) { return split_blob_query(128, I, H, L, bytes); }
extern "C" int ape_lstm_tcxs_blob_bytes(int I, int H, int L, int64_t* bytes) { return split_blob_query(256, I, H, L, bytes); }
extern "C" int ape_mc_lstm_tcx_workspace_bytes(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes) {
    return split_workspace_query(128, I, H, L, T, O, E, n_samples, false, bytes);
}
extern "C" int ape_mc_lstm_tcx_workspace_bytes_all_steps(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes) {
    return split_workspace_query(128, I, H, L, T, O, E, n_samples, true, bytes);
}
extern "C" int ape_mc_lstm_tcxs_workspace_bytes(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes) {
    return split_workspace_query(256, I, H, L, T, O, E, n_samples, false, bytes);
}
extern "C" int ape_mc_lstm_tcxs_workspace_bytes_all_steps(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes) {
    return split_workspace_query(256, I, H, L, T, O, E, n_samples, true, bytes);
}

// Two consecutive layers >= 1 of an H = 128 model run as ONE wavefront launch (ape_lstm_tcw.cu) when the batch gives every CTA pair
// at least one tile (below that a lone tile is faster through two one-layer launches: its two layers cannot overlap on the epilogue
// warps of one pair); tc_flags 1 / 2 force either way.  (A caller-supplied initial state runs on the one-layer kernels: the wavefront
// kernel takes none; the split-precision kernels have no wavefront form.)
static bool tc_pairs_layers(const ape_lstm_args* g, long long tiles1, int sm_count) {
    return ape::tcw::supported(g->H, g->T, g->O) && g->tc_flags != 1 && g->tc_flags != 3 && g->h0 == nullptr &&
           (g->tc_flags == 2 || tiles1 >= sm_count / 2);
}
// layers of the launch that starts at layer l of the range [.., l_end)
static int layers_in_launch(bool pair_ok, int l, int l_end) { return pair_ok && l >= 1 && l + 1 < l_end ? 2 : 1; }

// kernels ape_mc_lstm_tc will launch for these arguments (bench.py's gpu_launches)
extern "C" int ape_mc_lstm_tc_launch_count(const ape_lstm_args* g, int* launches) {
    if (!g || !launches) return APE_ERR_BAD_ARG;
    int dev = 0, sm_count = 0;
    APE_CUDA_TRY(cudaGetDevice(&dev));
    APE_CUDA_TRY(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev));
    const long long rows = (long long)g->B * g->nF * g->n_samples;
    const int l_begin = (g->layer_begin == 0 && g->layer_end == 0) ? 0 : g->layer_begin;
    const int l_end = (g->layer_begin == 0 && g->layer_end == 0) ? g->L : g->layer_end;
    if (g->tc_flags == 4 || g->tc_flags == 5) { *launches = 1; return APE_OK; }
    const bool pair_ok = tc_pairs_layers(g, (rows + 255) / 256, sm_count);
    int n = 0;
    for (int l = l_begin; l < l_end; l += layers_in_launch(pair_ok, l, l_end)) ++n;
    *launches = n + (g->all_steps ? 1 : 0);
    return APE_OK;
}

// Workspace of the split-precision small-batch kernels (tc_flags == 5): the exchange buffer and layer sequences (hi and lo) of one
// cluster per 128 rows of the largest call.  The tcxl symbol answers for the H = 128 kernel, the tcxsl symbol for the H = 256 one.
static int cluster_workspace_query(int kernel_H, int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes) {
    if (!bytes || T < 1 || E < 0 || n_samples < 1) return APE_ERR_BAD_ARG;
    if (H != kernel_H || !cluster_supported(I, H, L, T, O, E, n_samples)) return APE_ERR_UNSUPPORTED;
    *bytes = cluster_workspace_bytes(H, T, (long long)E * n_samples, 2);
    return APE_OK;
}
extern "C" int ape_mc_lstm_tcxl_workspace_bytes(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes) {
    return cluster_workspace_query(128, I, H, L, T, O, E, n_samples, bytes);
}
extern "C" int ape_mc_lstm_tcxsl_workspace_bytes(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes) {
    return cluster_workspace_query(256, I, H, L, T, O, E, n_samples, bytes);
}

// The argument block of a cluster kernel for the call `g`: the layers of `blob` (single pass: weights_tc, each layer closed by its
// scaled bias; split: weights_tcx) and the exchange buffers of every cluster in `workspace`
static ape::tc::ClusterArgs cluster_args(const ape_lstm_args* g, bool split, const uint8_t* blob, void* workspace) {
    ape::tc::ClusterArgs a{};
    const int H = g->H;
    const uint8_t* p = blob;
    for (int l = 0; l < g->L; ++l) {
        a.W[l] = p;
        a.kgx[l] = tc_kgx(l, g->I, H);
        p += blob_layer_bytes(split, l, g->I, H);
        if (!split) a.bias_s[l] = (const float*)(p - (size_t)4 * H * 4);
    }
    const long long E = (long long)g->B * g->nF;
    a.L = g->L; a.T = g->T; a.I = g->I; a.E = (int)E; a.n = g->n_samples; a.nF = g->nF; a.frame0 = g->frame0; a.feat_ring = g->feat_ring;
    a.dense = g->x_dense != nullptr;
    a.in = g->x_dense ? g->x_dense : g->feat_ring_buf;
    a.stream_frames = g->stream_frames;
    a.mask_mode = g->mask_mode; a.masks = g->masks;
    a.rk = ape::philox_round_keys(g->philox_seed);
    a.stream_id0 = g->stream_id0;
    a.keep_thr16 = ape::keep_threshold16(g->dropout_p);
    a.scale = g->mask_mode == APE_MASK_NONE ? 1.0f : 1.0f / (1.0f - g->dropout_p);
    const size_t planes = split ? 2 : 1;
    char* ws = (char*)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    a.hx = (uint4*)ws;
    a.seq = (uint4*)(ws + 2 * planes * (H / 8) * ape::tc::CLUSTER_ROWS * 16);
    a.ws_stride = cluster_bytes(H, g->T, planes) / 16;
    a.Wo16 = p;                                                // the output-layer tiles follow the last layer
    a.bo = g->weights + ape_pack_out_offset(g->I, H, g->L) + (size_t)g->O * H;
    a.O = g->O;
    a.preds = g->preds; a.pred_ring = g->pred_ring;
    a.stamps = (!split && g->trace && g->trace_layer == -2) ? (long long*)g->trace : nullptr;
    return a;
}

// one launch of a cluster kernel for all layers of the call `g`, reported as layer 0's time
static int cluster_launch(const ape_lstm_args* g, bool split, const uint8_t* blob, void* workspace, cudaStream_t st) {
    const ape::tc::ClusterArgs a = cluster_args(g, split, blob, workspace);
    const int clusters = (int)(((long long)a.E * a.n + ape::tc::CLUSTER_ROWS - 1) / ape::tc::CLUSTER_ROWS);
    ape::LayerTimer timer(g->layer_ms, g->L, st);
    int rc = timer.start();
    if (rc == APE_OK) rc = !split ? ape::tcl::run(g->H, a, clusters, st) : g->H == 256 ? ape::tcxsl::run(a, clusters, st)
                                                                                       : ape::tcxl::run(a, clusters, st);
    if (rc == APE_OK) rc = timer.mark(g->L);
    return rc == APE_OK ? timer.finish() : rc;
}

// tc_flags == 5: every layer of a call of <= 8192 rows of a split-precision model in ONE launch of the small-batch kernel for kernel_H
// (ape_lstm_tcxl.cu: ape_mc_lstm_tc, H = 128; ape_lstm_tcxsl.cu: ape_mc_lstm_tcxsl, H = 256).  Every refusal comes before the first
// CUDA call; then `available` (or null) may refuse a device that cannot run the kernel.
static int split_cluster_call(const ape_lstm_args* g, int kernel_H, cudaStream_t st, int (*available)()) {
    const long long E = (long long)g->B * g->nF;
    if (g->h0 || g->all_steps || g->layer_begin != 0 || g->layer_end != 0) return APE_ERR_UNSUPPORTED;
    if (g->H != kernel_H || !cluster_supported(g->I, g->H, g->L, g->T, g->O, E, g->n_samples)) return APE_ERR_UNSUPPORTED;
    if (!g->weights_tcx || !g->workspace || (g->ws_E != 0 && g->ws_E < E)) return APE_ERR_BAD_ARG;
    if (E == 0) return APE_OK;
    const int rc = available ? available() : APE_OK;
    return rc == APE_OK ? cluster_launch(g, true, (const uint8_t*)g->weights_tcx, g->workspace, st) : rc;
}

extern "C" int ape_mc_lstm_tc(const ape_lstm_args* g, void* stream) {
    using namespace ape;
    int rc = check_lstm_args(g);                               // (h0 / c0: both or neither, and n_samples == 1)
    if (rc != APE_OK) return rc;
    if (g->tc_flags == 5) return split_cluster_call(g, 128, (cudaStream_t)stream, nullptr);
    // an initial state runs on the one-layer kernels (tc_flags 0 and 1) and on the H = 256 split-precision kernel; the wavefront,
    // small-batch and H = 128 split-precision kernels take none
    if (g->h0 && (g->tc_flags == 2 || (g->tc_flags == 3 && g->H != 256) || g->tc_flags == 4)) return APE_ERR_UNSUPPORTED;
    // the state kernels read h_0 / c_0 rows as float4 (H is a multiple of 32, so every layer's block keeps the base alignment)
    if (((uintptr_t)g->h0 | (uintptr_t)g->c0) & 15) return APE_ERR_BAD_ARG;
    // tc_flags == 3: the split-precision kernels (csrc/ape_lstm_tcx.cu, H = 256: ape_lstm_tcxs.cu) and their blob, weights_tcx
    const bool split = g->tc_flags == 3;
    if (!(split ? split_supported(g->I, g->H, g->L, g->O) : ape_mc_lstm_tc_supported(g->I, g->H, g->L, g->O))) return APE_ERR_UNSUPPORTED;
    if (g->all_steps && (g->layer_begin != 0 || g->layer_end != 0)) return APE_ERR_UNSUPPORTED;
    if (g->T > 40) return APE_ERR_UNSUPPORTED;                 // |c_t| <= t keeps 2^(2 c log2e) finite in fp32 only for T <= 44
                                                               // (with a state |c_t| <= |c_0| + t: the state kernels clamp it)
    const uint8_t* blob = (const uint8_t*)(split ? g->weights_tcx : g->weights_tc);
    if (!blob || (split && !g->workspace)) return APE_ERR_BAD_ARG;     // (a split call needs the workspace even when it is empty)
    const long long E = (long long)g->B * g->nF;
    if (E == 0) return APE_OK;
    if (!g->workspace || (g->ws_E != 0 && g->ws_E < E)) return APE_ERR_BAD_ARG;
    const int l_begin = (g->layer_begin == 0 && g->layer_end == 0) ? 0 : g->layer_begin;
    const int l_end = (g->layer_begin == 0 && g->layer_end == 0) ? g->L : g->layer_end;
    if (l_begin < 0 || l_end > g->L || l_begin >= l_end) return APE_ERR_BAD_ARG;
    if (g->tc_flags < 0 || g->tc_flags > 5) return APE_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const bool all_steps = g->all_steps != 0;
    const TcWsLayout wl = tc_ws_layout(split, g->H, g->L, g->T, g->ws_E > 0 ? g->ws_E : E, g->n_samples, all_steps);
    char* wsp = (char*)(((uintptr_t)g->workspace + 255) & ~(uintptr_t)255);
    if (g->tc_flags == 4) {
        // small-batch kernel: every layer of a call of <= 8192 rows in ONE launch, one 8-CTA cluster per 128 rows (csrc/ape_lstm_tcl.cu),
        // its buffers behind the scratch regions
        if (l_begin != 0 || l_end != g->L || all_steps || !cluster_supported(g->I, g->H, g->L, g->T, g->O, E, g->n_samples))
            return APE_ERR_UNSUPPORTED;
        return cluster_launch(g, false, blob, wsp + 2 * wl.scratch_region, st);
    }
    int dev = 0, sm_count = 0;
    APE_CUDA_TRY(cudaGetDevice(&dev));
    APE_CUDA_TRY(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev));

    const int H = g->H;
    const long long rows = E * g->n_samples;
    const int rpc0 = tc_rpc0(split, E);
    const int tiles0 = (int)((E + 2 * rpc0 - 1) / (2 * rpc0)), tiles1 = (int)((rows + 255) / 256);
    // per-CTA cell-state scratch at the front (a position that does not depend on the call's size)
    char* scratch = wsp;
    if (wl.scratch_region && sm_count > TC_MAX_SMS) return APE_ERR_UNSUPPORTED;
    wsp += 2 * wl.scratch_region;
    // SMs the launches of layers >= 1 leave free (a whole number of SM pairs): a concurrent stage 1 + layer 0 of the NEXT call - a few
    // CTAs on a high-priority stream - then never has to wait for a persistent launch to retire CTAs
    if (g->reserve_sms < 0 || g->reserve_sms > sm_count - 2) return APE_ERR_BAD_ARG;
    const int sm_big = sm_count - ((g->reserve_sms + 1) & ~1);

    // units between layers: layer 0's output (two copies, one row per estimate), the outputs of layers >= 1 (one row per (estimate,
    // sample); all_steps: the last layer's sequence is kept too, for the per-step output layer); split: the lo halves behind the hi
    struct Units { uint4 *hi, *lo; };
    const size_t planes = split ? 2 : 1;
    auto units_at = [&](char* p, size_t bytes) { return Units{(uint4*)p, split ? (uint4*)(p + bytes) : nullptr}; };
    const Units units0 = units_at(wsp + (g->ws_parity & 1) * planes * wl.u0, wl.u0);
    const Units units[2] = {units_at(wsp + 2 * planes * wl.u0, wl.u1), units_at(wsp + 2 * planes * wl.u0 + planes * wl.u1, wl.u1)};
    auto layer_w = [&](int l) {                                            // layer l's weights inside the blob
        const uint8_t* p = blob;
        for (int k = 0; k < l; ++k) p += blob_layer_bytes(split, k, g->I, H);
        return p;
    };
    const uint8_t* wo16 = layer_w(g->L);                                    // the fp16 output-layer tile sits after all layers,
    const size_t ww_layer = !split && g->L >= 3 ? tcw::layer_bytes(H) : 0;  // ... then the wavefront kernel's pieces of layers 1 .. L-1
    const uint8_t* ww = wo16 + tc::wo16_bytes(H);
    const float scale = g->mask_mode == APE_MASK_NONE ? 1.0f : 1.0f / (1.0f - g->dropout_p);
    auto layer_args = [&](int l) {
        const bool last = l == g->L - 1;
        tc::TcLayerArgs a{};
        if (split) {
            a.Ww = layer_w(l);                                              // the split kernels stream all of a layer's pieces
        } else {
            a.W = layer_w(l);
            a.bias_s = (const float*)(a.W + tc_layer_bytes(l, g->I, H) - (size_t)4 * H * 4);
            a.Ww = (ww_layer && l >= 1) ? ww + (size_t)(l - 1) * ww_layer : nullptr;
        }
        a.T = g->T;
        a.kgx = tc_kgx(l, g->I, H);
        a.Kin = l == 0 ? g->I : H;
        a.feat_ring = g->feat_ring; a.nF = g->nF; a.frame0 = g->frame0; a.stream_frames = g->stream_frames;
        if (l == 0) {
            a.in_mode = g->x_dense ? tc::IN_DENSE_F32 : tc::IN_WINDOW_F32;
            a.in = g->x_dense ? (const void*)g->x_dense : (const void*)g->feat_ring_buf;
            a.rows = (int)E; a.n = 1;
            a.rpc = rpc0;
            a.n_pair_tiles = tiles0;
            a.mask_mode = APE_MASK_NONE;
            a.out_units = units0.hi; a.out_units_lo = units0.lo;
        } else {
            const Units& in = l == 1 ? units0 : units[(l - 2) & 1];
            a.in_mode = l == 1 ? tc::IN_SHARED_UNITS : tc::IN_UNITS;
            a.in = in.hi; a.in_lo = in.lo;
            a.rows = (int)rows; a.n = g->n_samples;
            a.rpc = 128;
            a.in_rpc_shift = rpc0 == 128 ? 7 : 5;
            a.n_pair_tiles = tiles1;
            a.mask_mode = g->mask_mode;
            if (!last || all_steps) { a.out_units = units[(l - 1) & 1].hi; a.out_units_lo = units[(l - 1) & 1].lo; }
        }
        a.masks = g->masks; a.gap = l - 1; a.n_gaps = g->L - 1;
        a.seed = g->philox_seed; a.stream_id0 = g->stream_id0;
        a.rk = philox_round_keys(g->philox_seed);
        a.keep_thr16 = keep_threshold16(g->dropout_p);
        // the next layer's dropout scale, applied before the fp16 rounding (all_steps: the last layer's sequence feeds the output layer as is)
        a.out_scale = last ? 1.0f : scale;
        a.Wo = g->weights + ape_pack_out_offset(g->I, g->H, g->L);
        a.bo = a.Wo + (size_t)g->O * g->H;
        a.O = g->O;
        a.Wo16 = wo16;
        a.preds = (last && !all_steps) ? g->preds : nullptr;
        a.pred_ring = g->pred_ring; a.n_out = g->n_samples;
        a.cstate = wl.scratch_region ? (float*)(scratch + (l == 0 ? 0 : wl.scratch_region)) : nullptr;
        a.h0 = g->h0 ? g->h0 + (size_t)l * E * H : nullptr;   // [L][E][H]: with a state every layer has E rows (n_samples == 1)
        a.c0 = g->c0 ? g->c0 + (size_t)l * E * H : nullptr;
        a.trace = (g->trace && l == g->trace_layer) ? (long long*)g->trace : nullptr;
        // trace_layer < 0: the CTA timeline of every layer instead, [layer][TC_MAX_SMS CTAs][4]
        a.timeline = (g->trace && g->trace_layer < 0) ? (long long*)g->trace + (size_t)l * TC_MAX_SMS * 4 : nullptr;
        return a;
    };
    const bool pair_ok = tc_pairs_layers(g, tiles1, sm_count);
    LayerTimer timer(l_begin == 0 && l_end == g->L ? g->layer_ms : nullptr, g->L, st);   // (a pair's time goes to its first layer)
    rc = timer.start();
    for (int l = l_begin, n; l < l_end && rc == APE_OK; l += n) {
        n = layers_in_launch(pair_ok, l, l_end);
        const tc::TcLayerArgs a = layer_args(l);
        const int sms = l == 0 ? sm_count : sm_big;
        if (n == 2)     rc = tcw::launch_pair(a, layer_args(l + 1), sm_big, st);
        else if (split) rc = H == 256 ? tcxs::launch_layer(a, sms, st) : tcx::launch_layer(a, sms, st);
        else            rc = H == 128 ? tc::launch<128>(a, sms, st) : H == 64 ? tc::launch<64>(a, sms, st) : tcs::launch_layer(H, a, sms, st);
        if (rc == APE_OK) rc = timer.mark(l + n);
    }
    if (rc == APE_OK && all_steps) {                           // output layer on every step (nn_models.py:189: output_layer(all)); split: hi + lo
        const Units& seq = units[(g->L - 2) & 1];
        rc = tc::launch_units_output(seq.hi, seq.lo, g->weights + ape_pack_out_offset(g->I, g->H, g->L), g->preds, rows, g->T, H, g->O, st);
    }
    return rc == APE_OK ? timer.finish() : rc;
}

extern "C" int ape_mc_lstm_tcxsl_max_active_clusters(int* clusters) {
    if (!clusters) return APE_ERR_BAD_ARG;
    *clusters = 0;
    return ape::tcxsl::max_active_clusters(clusters);
}

// a device that cannot hold one 16-CTA cluster of the H = 256 split-precision small-batch kernel refuses the call
static int tcxsl_available() {
    int clusters = 0;
    const int rc = ape::tcxsl::max_active_clusters(&clusters);
    return rc != APE_OK ? rc : clusters < 1 ? APE_ERR_UNSUPPORTED : APE_OK;
}

// Every layer of a call of <= 8192 rows of a split-precision H = 256 model in ONE launch (csrc/ape_lstm_tcxsl.cu), tc_flags == 5.
extern "C" int ape_mc_lstm_tcxsl(const ape_lstm_args* g, void* stream) {
    const int rc = ape::check_lstm_args(g);
    if (rc != APE_OK) return rc;
    if (g->tc_flags != 5) return APE_ERR_BAD_ARG;
    return split_cluster_call(g, 256, (cudaStream_t)stream, tcxsl_available);
}
