// Shared by the tensor-core MC-LSTM kernels and by ape_mc_lstm_tc (ape_lstm_tc.cu), whose one host-side layer walk launches them:
// the per-layer argument block, the input modes, the transcendental helpers of the cell update, and each kernel's host entry
// points - ape_lstm_tc.cu (gate weights resident in shared memory, H <= 128), ape_lstm_tcs.cu (gate weights streamed from L2
// through a TMA ring, H = 256), ape_lstm_tcw.cu (two layers per launch, H = 128), ape_lstm_tcx.cu / ape_lstm_tcxs.cu (split
// precision, H = 128 / 256), ape_lstm_tcl.cu (all layers of a small call in one launch) and ape_lstm_tcxl.cu / ape_lstm_tcxsl.cu (the
// same at split precision, H = 128 / 256).
#pragma once
#include "ape_f32x2.cuh"
#include "ape_common.cuh"
#include "ape_umma.cuh"

namespace ape {
namespace tc {

constexpr float LOG2E = 1.4426950408889634f;
constexpr float EX2_CLAMP = 40.0f;                 // (1 + 2^40)^3 still fits fp32

enum { IN_WINDOW_F32 = 0, IN_DENSE_F32 = 1, IN_SHARED_UNITS = 2, IN_UNITS = 3 };

struct TcLayerArgs {
    const uint8_t* W;          // this layer: [cta 2][chunk][x k-groups then h k-groups][64 gate columns][8 halfs]
    const float* bias_s;       // [4H] column c = 4u+g, scaled for the tanh form: 0.5 b (i, f, o), b (g)
    const uint8_t* Ww;         // wavefront kernel (H = 128, layers >= 1 of an L >= 3 model), else null: [cta 2][chunk 4][x-piece | h-piece]:
                               // x-piece [16 + 2 k-groups][64][8] (i, f, o columns halved; k-group 16 rows 0, 1 = fp16(bias_s), remainder),
                               // h-piece [16 k-groups][64][8] (i, f, o columns halved)
    int T, kgx, Kin;           // x-part: kgx k-groups (layer 0: ceil16(I)/8, else H/8) of which Kin columns are real
    int rpc;                   // rows per CTA actually used (128, or 32 to spread a small layer 0 over more SMs)
    int in_rpc_shift;          // IN_SHARED_UNITS: log2(rpc) of the producing layer
    int in_mode;
    const void* in;
    const void* in_lo;         // split-precision kernel (ape_lstm_tcx.cu): the lo halves of the input units (in = the hi halves)
    int feat_ring, nF, frame0, rows, n;
    const int32_t* stream_frames;   // per-stream frame counters (null: frame0 for all); < 0: the stream sits this call out
    int mask_mode;
    const uint8_t* masks;
    int gap, n_gaps;
    uint64_t seed;
    PhiloxRoundKeys rk;        // philox_round_keys(seed)
    uint32_t stream_id0;
    uint32_t keep_thr16;
    uint4* out_units;          // [pair tile][T][cta][k-group][128 rows] 16-byte units of fp16 (h_t * out_scale), or null
    uint4* out_units_lo;       // split-precision kernel: the lo halves (fp16(v - fp16(v))) of the same units
    float out_scale;           // the consumer's 1/(1-p): scaling BEFORE the fp16 rounding keeps it a single rounding
    const float* Wo;
    const float* bo;
    const uint8_t* Wo16;       // fp16 output-layer tiles [cta 2][H/8 k-groups][16 outputs (H = 256: 32)][8 halfs]: cta 0 fp16(W_o),
                               // cta 1 the remainder W_o - fp16(W_o) as fp16 (outputs >= O are zero rows)
    int O;
    float* preds;
    int pred_ring, n_out;
    int n_pair_tiles;
    float* cstate;             // streamed-weights kernel (H = 256): per-CTA cell-state scratch, tcs::scratch_bytes() bytes
    const float* h0;           // caller-supplied initial state of THIS layer, [rows][H] float32 each (n == 1), or both null:
    const float* c0;           //   step 0 of every tile then also runs the recurrent half on h_0 and starts the cell from c_0
    long long* trace;          // debugging: null, or [3 roles][16 steps][16 events] SM-clock stamps of the first tile of CTA 0
    long long* timeline;       // debugging: null, or [CTA][4] = {globaltimer at entry, after the set-up, at exit; SM id} (tools/lanes_timeline.py)
};

__device__ __forceinline__ long long globaltimer_ns() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ void timeline_stamp(long long* tl, int slot) {
    if (tl && threadIdx.x == 0) {
        tl[blockIdx.x * 4 + slot] = globaltimer_ns();
        if (slot == 0) { uint32_t sm; asm volatile("mov.u32 %0, %%smid;" : "=r"(sm)); tl[blockIdx.x * 4 + 3] = sm; }
    }
}

// Cell-update arithmetic of both tensor-core kernels.  APE_TC_TANH = 1 (default): every gate through the hardware tanh
// (tanh.approx.f32; sigmoid(x) = 0.5 + 0.5 tanh(x / 2)) - 5 MUFU and ~10 FP32 ops per cell.  0: the exp2 / reciprocal form
// (7 MUFU, ~19 FP32 ops; i * g~ and f share one reciprocal), kept for A/B measurements.  Measured on B200: the tanh form is
// 6 % (H = 256) faster per layer and the position error against the fp32 kernel is unchanged (it is set by
// the fp16 operand rounding).  The bias in the fp16 blob is stored ready for the tanh form: 0.5 b (i, f, o), b (g).
#ifndef APE_TC_TANH
#define APE_TC_TANH 1
#endif
__device__ __forceinline__ float tanh_approx(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// v[4 * i + s] for a warp-uniform s in 0..3 without dynamic register indexing (which would put v in local memory)
__device__ __forceinline__ uint32_t pick4(const uint32_t* v, int i, int s) {
    const uint32_t a = (s & 1) ? v[4 * i + 1] : v[4 * i + 0], b = (s & 1) ? v[4 * i + 3] : v[4 * i + 2];
    return (s & 2) ? b : a;
}

#ifndef APE_PHILOX_RK
#define APE_PHILOX_RK 1      // 1: host-evaluated Philox round keys (constant-bank operands); 0: key schedule on the device (A/B only)
#endif
#if APE_PHILOX_RK
#define APE_PHILOX_DRAW(a, ...) philox_keep_halfmask_rk((a).rk, __VA_ARGS__)
#else
#define APE_PHILOX_DRAW(a, ...) philox_keep_halfmask((a).seed, __VA_ARGS__)
#endif

#ifndef APE_EXP
#define APE_EXP 0            // timing experiments only (tools/tc_experiments.sh); 0 = the real kernel
#endif
#if APE_EXP == 2
__device__ __forceinline__ float ex2_approx(float x) { return x * 0.99f; }
__device__ __forceinline__ float rcp_approx(float x) { return x * 1.01f; }
#else
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
#endif

// One LSTM cell from the four ex2 ARGUMENTS  p = -(gate + bias) * log2e  (g gate: * 2 log2e):
//   i*g~ = (1 - e_g) / ((1 + e_i)(1 + e_g)),  f = 1 / (1 + e_f)  share one reciprocal; h = o * tanh(c) another.
__device__ __forceinline__ void lstm_cell(float pi, float pf, float pg, float po, float& c, float& h) {
    const float ei = ex2_approx(fminf(pi, EX2_CLAMP)), ef = ex2_approx(fminf(pf, EX2_CLAMP));
    const float eg = ex2_approx(fminf(pg, EX2_CLAMP)), eo = ex2_approx(fminf(po, EX2_CLAMP));
    const float ab = (1.0f + ei) * (1.0f + eg), cf = 1.0f + ef;
    const float num = fmaf(c, ab, (1.0f - eg) * cf);
    c = num * rcp_approx(ab * cf);
    const float ec = ex2_approx(fminf(c * (-2.0f * LOG2E), EX2_CLAMP));
    h = (1.0f - ec) * rcp_approx((1.0f + eo) * (1.0f + ec));
}

// Two cells at once in packed fp32 pairs (ape_f32x2.cuh): the same operations as lstm_cell component by component (the clamps and the
// MUFU calls stay scalar), 15 issue slots for the arithmetic of two cells instead of 30.
__device__ __forceinline__ void lstm_cell2(F2 pi, F2 pf, F2 pg, F2 po, F2& c, F2& h) {
    const F2 ei = pk(ex2_approx(fminf(lo(pi), EX2_CLAMP)), ex2_approx(fminf(hi(pi), EX2_CLAMP)));
    const F2 ef = pk(ex2_approx(fminf(lo(pf), EX2_CLAMP)), ex2_approx(fminf(hi(pf), EX2_CLAMP)));
    const F2 eg = pk(ex2_approx(fminf(lo(pg), EX2_CLAMP)), ex2_approx(fminf(hi(pg), EX2_CLAMP)));
    const F2 eo = pk(ex2_approx(fminf(lo(po), EX2_CLAMP)), ex2_approx(fminf(hi(po), EX2_CLAMP)));
    const F2 one = splat(1.0f);
    const F2 ab = (one + ei) * (one + eg), cf = one + ef;
    const F2 num = fma2(c, ab, (one - eg) * cf), d = ab * cf;
    c = num * pk(rcp_approx(lo(d)), rcp_approx(hi(d)));
    const F2 pc = c * splat(-2.0f * LOG2E);
    const F2 ec = pk(ex2_approx(fminf(lo(pc), EX2_CLAMP)), ex2_approx(fminf(hi(pc), EX2_CLAMP)));
    const F2 d2 = (one + eo) * (one + ec);
    h = (one - ec) * pk(rcp_approx(lo(d2)), rcp_approx(hi(d2)));
}

// all_steps: the fp32 output layer on every step of the last layer's kept sequence (units [pair tile][T][cta][H/8][128 rows]);
// units_lo: the split-precision kernels' lo halves of the same units, or null (ape_lstm_tc.cu)
int launch_units_output(const uint4* units, const uint4* units_lo, const float* Wo, float* preds, long long rows, int T, int H, int O,
                        cudaStream_t st);

}  // namespace tc

namespace tcs {
// streamed-weights kernel (ape_lstm_tcs.cu)
bool supported(int H);
size_t scratch_bytes(int H, int sm_count);      // one region of per-CTA cell-state scratch (a launch needs one)
int launch_layer(int H, const tc::TcLayerArgs& a, int sm_count, cudaStream_t st);    // a.h0 / a.c0: the state variant
}  // namespace tcs

namespace tcw {
// two-layer wavefront kernel (ape_lstm_tcw.cu): layers a and b = a + 1 of an H = 128 model in one launch
bool supported(int H, int T, int O);
size_t layer_bytes(int H);                      // bytes of one layer's pieces (TcLayerArgs::Ww)
size_t scratch_bytes(int H, int sm_count);      // per-CTA cell-state scratch of one launch
int launch_pair(const tc::TcLayerArgs& a, const tc::TcLayerArgs& b, int sm_count, cudaStream_t st);
}  // namespace tcw

namespace tcl {
// small-batch kernel (ape_lstm_tcl.cu): all layers of a call in one launch, one cluster of 8 CTAs per 128 rows (hidden units split
// across the cluster, h_t exchanged once per step); up to 64 clusters
bool supported(int H, int I, int L, int O, long long E, int n);
size_t workspace_bytes(int H, int T, long long rows);     // rows = E * n_samples of the largest call (one cluster per 128 rows)
int run(const ape_lstm_args* g, const uint8_t* const* layer_w, const float* const* layer_bias, const uint8_t* wo16, void* workspace,
        cudaStream_t st);
}  // namespace tcl

namespace tcx {
// split-precision kernel (ape_lstm_tcx.cu): every operand an fp16 pair hi + lo, three tensor-core passes per product, ex2 / rcp cell
bool supported(int H, int I, int O);
size_t layer_bytes(int layer, int I);            // bytes of one layer's pieces (TcLayerArgs::Ww), both CTAs
size_t wo16_bytes();                             // bytes of the output-layer tiles after the last layer (TcLayerArgs::Wo16), both CTAs
size_t scratch_bytes(int sm_count);              // per-CTA cell-state scratch of one launch
int launch_layer(const tc::TcLayerArgs& a, int sm_count, cudaStream_t st);
}  // namespace tcx

namespace tcxs {
// split-precision kernel for H = 256 (ape_lstm_tcxs.cu): the arithmetic and blob layout of tcx, h_t staged through L2 into
// single-buffered TMEM operands
bool supported(int H, int I, int O);
size_t layer_bytes(int layer, int I);
size_t wo16_bytes();
size_t scratch_bytes(int sm_count);              // per-CTA cell state and h_t staging of one launch
int launch_layer(const tc::TcLayerArgs& a, int sm_count, cudaStream_t st);    // a.h0 / a.c0: the state variant
}  // namespace tcxs

namespace tcxl {
// split-precision small-batch kernel (ape_lstm_tcxl.cu, H = 128): all layers of a call in one launch, one 8-CTA cluster per 128 rows,
// the arithmetic of tcx on the tcx blob
bool supported(int H, int I, int L, int T, int O, long long E, int n);
size_t workspace_bytes(int T, long long rows);             // rows = E * n_samples of the largest call (one cluster per 128 rows)
int run(const ape_lstm_args* g, const uint8_t* blob, void* workspace, cudaStream_t st);
}  // namespace tcxl

namespace tcxsl {
// split-precision small-batch kernel for H = 256 (ape_lstm_tcxsl.cu): all layers of a call in one launch, one 16-CTA cluster per
// 128 rows, the arithmetic of tcxs on the tcx blob
bool supported(int H, int I, int L, int T, int O, long long E, int n);
size_t workspace_bytes(int T, long long rows);             // rows = E * n_samples of the largest call (one cluster per 128 rows)
int max_active_clusters(int* clusters);                    // 16-CTA clusters of this launch the current device holds at once
int run(const ape_lstm_args* g, const uint8_t* blob, void* workspace, cudaStream_t st);
}  // namespace tcxsl
}  // namespace ape
