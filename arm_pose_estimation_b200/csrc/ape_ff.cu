// MC-dropout feed-forward regressors (DropoutFF / DropoutFF2D, nn_models.py:252-370 of the reference): Linear + leaky_relu
// stack, dropout ONLY in front of the output layer.  The hidden stack therefore does not depend on the MC sample: it is
// evaluated once per input row, and only  y_s = W_o (mask_s * h) / (1 - p) + b_o  runs per sample.  fp32 FFMA throughout.
// Two kernels: the batched one (8 rows per CTA, below) for the usual shapes, and a generic one-CTA-per-row kernel (threads over output
// units for the dense layers, then one warp per MC sample with a warp-shuffle reduction per output) for everything else.
// ape_mc_ff_ring runs the batched kernel on the rings of the batched path (BatchedEstimator with a feed-forward state dict).
// Not on the deployed models' path.
#include "ape_common.cuh"

namespace ape {

constexpr int FF_THREADS = 256;

struct FfArgs {
    const float* blob;       // layer 0: W^T [I][H], b [H]; hidden l: W^T [H][H], b [H]; output: W [O][H], b [O]
    int I, H, Lh, O;
    const float* x;          // [rows][I]
    int rows, n;
    int mask_mode;
    const uint8_t* masks;    // APE_MASK_INJECTED: [rows][n][H] of {0,1}
    uint64_t seed;
    uint32_t stream_id0, frame0, keep_thr16;
    float keep_scale;
    float* preds;            // [rows][n][O]; ring mode: [B][pred_ring][n][O]
    // ring mode (ape_mc_ff_ring): row e = b * nF + j is frame f = stream_frame0(stream_frames, frame0, b) + j of stream b, its input
    // the window of frames f - T + 1 .. f (time-major, I = T * Ifr) of the feature ring x = [B][feat_ring][Ifr]
    const int32_t* stream_frames;
    int Ifr, T, feat_ring, nF, pred_ring;
};

__global__ void __launch_bounds__(FF_THREADS) mc_ff_row_kernel(FfArgs a) {
    extern __shared__ float sh[];                      // [2][max(I, H)]
    const int K0 = a.I > a.H ? a.I : a.H;
    float* cur = sh;
    float* nxt = sh + K0;
    const int row = blockIdx.x, tid = threadIdx.x;
    for (int k = tid; k < a.I; k += FF_THREADS) cur[k] = a.x[(size_t)row * a.I + k];
    __syncthreads();
    const float* w = a.blob;
    int K = a.I;
    for (int l = 0; l <= a.Lh; ++l) {                  // input layer + Lh hidden layers, leaky_relu(0.01) after each
        const float* bias = w + (size_t)K * a.H;
        for (int j = tid; j < a.H; j += FF_THREADS) {
            float acc = bias[j];
            for (int k = 0; k < K; ++k) acc = fmaf(__ldg(w + (size_t)k * a.H + j), cur[k], acc);
            nxt[j] = acc > 0.0f ? acc : 0.01f * acc;
        }
        __syncthreads();
        float* t = cur; cur = nxt; nxt = t;
        w = bias + a.H;
        K = a.H;
    }
    const float* wo = w;
    const float* bo = wo + (size_t)a.O * a.H;
    const int warp = tid >> 5, lane = tid & 31;
    for (int s = warp; s < a.n; s += FF_THREADS / 32) {
        float acc[20];
#pragma unroll
        for (int o = 0; o < 20; ++o) acc[o] = 0.0f;
        for (int k0 = 0; k0 < a.H; k0 += 32) {
            const int k = k0 + lane;
            float v = 0.0f;
            if (k < a.H) {
                bool keep = true;
                if (a.mask_mode == APE_MASK_INJECTED) {
                    keep = a.masks[((size_t)row * a.n + s) * a.H + k] != 0;
                } else if (a.mask_mode == APE_MASK_PHILOX) {       // gap id 15 is reserved for the feed-forward output dropout
                    const uint32_t bits = philox_keep8(a.seed, a.stream_id0 + (uint32_t)row, a.frame0, (uint32_t)s, 15u, 0u,
                                                       (uint32_t)(k >> 3), a.keep_thr16);
                    keep = (bits >> (k & 7)) & 1u;
                }
                v = keep ? cur[k] * a.keep_scale : 0.0f;
            }
#pragma unroll
            for (int o = 0; o < 20; ++o)
                if (o < a.O && k < a.H) acc[o] = fmaf(__ldg(wo + (size_t)o * a.H + k), v, acc[o]);
        }
#pragma unroll
        for (int o = 0; o < 20; ++o) {
            if (o < a.O) {
                float v = acc[o];
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
                if (lane == 0) a.preds[((size_t)row * a.n + s) * a.O + o] = v + __ldg(bo + o);
            }
        }
    }
}

// ---- the batched kernel -----------------------------------------------------------------------------------------------------
// FF_TR input rows per CTA.  Hidden stack: a [FF_TR x 128-unit] output tile per pass, W^T streamed through shared memory in chunks of
// FF_KC k-rows (each weight is read from L2 once per CTA and used for FF_TR rows; thread = 4 consecutive units of one row: 16 FMAs per
// two 16-byte shared-memory loads), activations ping-pong between two shared-memory tiles.  Output layer: thread = one (row, MC sample)
// pair, its 8-unit keep flags drawn with the precomputed Philox round keys (the same counters as the row kernel: gap id 15), the masked
// hidden vector swept against W_o^T in shared memory (every lane reads the same weights: broadcast loads, OP FMAs per unit).
// The row kernel above re-read every weight per row and left half of its threads idle in the hidden stack: 0.252 ms for 1024 rows x 100
// samples (I = 110, H = 128, two hidden layers) against 0.050 ms here (8192 rows: 0.21 ms = 0.24 of the measured fp32 FMA peak).
// RING: the rows are windows of the feature ring and the outputs go to the prediction ring (ape_mc_ff_ring); only the addressing
// of the input tile, the Philox counters (stream b, frame f instead of stream_id0 + row, frame0) and the store differ.
constexpr int FF_TR = 8, FF_KC = 32, FF_HB = 128;

template <int OP, bool RING>
__global__ void __launch_bounds__(FF_THREADS) mc_ff_kernel(FfArgs a, PhiloxRoundKeys rk) {
    extern __shared__ __align__(16) float sh[];
    const int KM = ((a.I > a.H ? a.I : a.H) + FF_KC - 1) / FF_KC * FF_KC;     // tile row: k-chunks never read past it
    float* act0 = sh;                                  // [FF_TR][KM]
    float* act1 = act0 + FF_TR * KM;                   // [FF_TR][KM]
    float* wch = act1 + FF_TR * KM;                    // [FF_KC][FF_HB]
    float* woT = wch + FF_KC * FF_HB;                  // [H][OP]
    const int tid = threadIdx.x, row0 = blockIdx.x * FF_TR;
    const int nr = min(FF_TR, a.rows - row0);
    for (int i = tid; i < FF_TR * KM; i += FF_THREADS) {
        const int r = i / KM, k = i - r * KM;
        float v = 0.0f;
        if (r < nr && k < a.I) {
            if constexpr (RING) {                      // frames before 0 read frame 0 (estimator.py:96-97, as ape_lstm_fma.cu)
                const int e = row0 + r, b = e / a.nF, t = k / a.Ifr;
                int fw = stream_frame0(a.stream_frames, (int)a.frame0, b) + e % a.nF - a.T + 1 + t;
                fw = fw < 0 ? 0 : fw;
                v = __ldg(a.x + ((size_t)b * a.feat_ring + fw % a.feat_ring) * a.Ifr + (k - t * a.Ifr));
            } else {
                v = a.x[(size_t)(row0 + r) * a.I + k];
            }
        }
        act0[i] = v;
    }
    const float* w = a.blob;
    int K = a.I;
    float* cur = act0;
    float* nxt = act1;
    const int r = tid >> 5, ug = tid & 31;             // this thread: row r of the tile, units hb + 4 ug .. + 3
    for (int l = 0; l <= a.Lh; ++l) {                  // input layer + Lh hidden layers, leaky_relu(0.01) after each
        const float* bias = w + (size_t)K * a.H;
        for (int hb = 0; hb < a.H; hb += FF_HB) {
            float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
            for (int kc0 = 0; kc0 < K; kc0 += FF_KC) {
                __syncthreads();                       // the previous chunk has been consumed (first pass: the input tile is complete)
#pragma unroll
                for (int i = 0; i < FF_KC * FF_HB / 4 / FF_THREADS; ++i) {
                    const int idx = tid + FF_THREADS * i, kk = idx >> 5, c4 = idx & 31;
                    float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                    if (kc0 + kk < K && hb + 4 * c4 < a.H) v = __ldg(reinterpret_cast<const float4*>(w + (size_t)(kc0 + kk) * a.H + hb + 4 * c4));
                    reinterpret_cast<float4*>(wch)[idx] = v;
                }
                __syncthreads();
                const float* xr = cur + r * KM + kc0;
#pragma unroll
                for (int kk = 0; kk < FF_KC; kk += 4) {
                    const float4 x4 = *reinterpret_cast<const float4*>(xr + kk);       // (zero beyond K: the tiles are zero-padded to KM)
                    const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float4 w4 = reinterpret_cast<const float4*>(wch + (kk + j) * FF_HB)[ug];
                        acc[0] = fmaf(w4.x, xs[j], acc[0]); acc[1] = fmaf(w4.y, xs[j], acc[1]);
                        acc[2] = fmaf(w4.z, xs[j], acc[2]); acc[3] = fmaf(w4.w, xs[j], acc[3]);
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int j = hb + 4 * ug + i;
                if (j < a.H) {
                    const float v = acc[i] + __ldg(bias + j);
                    nxt[r * KM + j] = v > 0.0f ? v : 0.01f * v;
                }
            }
        }
        for (int i = tid; i < FF_TR * (KM - a.H); i += FF_THREADS) {      // zero padding behind the H units (k-chunks read up to KM)
            const int rr = i / (KM - a.H), k = a.H + i - rr * (KM - a.H);
            nxt[rr * KM + k] = 0.0f;
        }
        float* t = cur; cur = nxt; nxt = t;
        w = bias + a.H;
        K = a.H;
    }
    // ---- output layer per (row, MC sample) -----------------------------------------------------------------------------------
    const float* wo = w;
    const float* bo = wo + (size_t)a.O * a.H;
    for (int i = tid; i < a.H * OP; i += FF_THREADS) {
        const int k = i / OP, o = i - k * OP;
        woT[i] = o < a.O ? __ldg(wo + (size_t)o * a.H + k) : 0.0f;
    }
    __syncthreads();                                   // the last layer's activations and W_o^T are in place
    for (int i = tid; i < FF_TR * a.H; i += FF_THREADS) {
        const int rr = i / a.H, k = i - rr * a.H;
        cur[rr * KM + k] *= a.keep_scale;              // 1 / (1 - p), applied to the kept units (nn.Dropout)
    }
    __syncthreads();
    for (int p = tid; p < nr * a.n; p += FF_THREADS) {
        const int rr = p / a.n, s = p - rr * a.n, row = row0 + rr;
        uint32_t sid = a.stream_id0 + (uint32_t)row, frm = a.frame0;
        int fb = 0;
        if constexpr (RING) {
            fb = stream_frame0(a.stream_frames, (int)a.frame0, row / a.nF);
            sid = a.stream_id0 + (uint32_t)(row / a.nF);
            frm = (uint32_t)(fb + row % a.nF);
        }
        const float* h = cur + rr * KM;
        float acc[OP];
#pragma unroll
        for (int o = 0; o < OP; ++o) acc[o] = 0.0f;
        for (int g = 0; g < a.H / 8; ++g) {
            uint32_t keep = 0xFFu;                     // bit j: unit 8 g + j is kept
            if (a.mask_mode == APE_MASK_INJECTED) {
                const uint2 mm = __ldg(reinterpret_cast<const uint2*>(a.masks + ((size_t)row * a.n + s) * a.H + 8 * g));
                keep = 0;
#pragma unroll
                for (int j = 0; j < 4; ++j) keep |= (((mm.x >> (8 * j)) & 0xFFu) ? 1u : 0u) << j | (((mm.y >> (8 * j)) & 0xFFu) ? 1u : 0u) << (4 + j);
            } else if (a.mask_mode == APE_MASK_PHILOX) {   // gap id 15 is reserved for the feed-forward output dropout
                const uint4 f = philox_keep_flags_rk(rk, sid, frm, (uint32_t)s, 15u, 0u, (uint32_t)g, a.keep_thr16);
                const uint32_t fw[4] = {f.x, f.y, f.z, f.w};
                keep = 0;
#pragma unroll
                for (int i = 0; i < 4; ++i) keep |= ((fw[i] >> 15) & 1u) << (2 * i) | ((fw[i] >> 31) & 1u) << (2 * i + 1);
            }
            const float4 ha = *reinterpret_cast<const float4*>(h + 8 * g), hb4 = *reinterpret_cast<const float4*>(h + 8 * g + 4);
            const float hv[8] = {ha.x, ha.y, ha.z, ha.w, hb4.x, hb4.y, hb4.z, hb4.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float v = (keep >> j) & 1u ? hv[j] : 0.0f;
                const float4* wr = reinterpret_cast<const float4*>(woT + (8 * g + j) * OP);
#pragma unroll
                for (int o4 = 0; o4 < OP / 4; ++o4) {
                    const float4 w4 = wr[o4];
                    acc[4 * o4] = fmaf(w4.x, v, acc[4 * o4]); acc[4 * o4 + 1] = fmaf(w4.y, v, acc[4 * o4 + 1]);
                    acc[4 * o4 + 2] = fmaf(w4.z, v, acc[4 * o4 + 2]); acc[4 * o4 + 3] = fmaf(w4.w, v, acc[4 * o4 + 3]);
                }
            }
        }
        float* dst = a.preds + ((size_t)row * a.n + s) * a.O;
        if constexpr (RING) {
            if (fb < 0) continue;                      // the stream sits this call out: its prediction ring stays untouched
            dst = a.preds + (((size_t)(row / a.nF) * a.pred_ring + frm % (uint32_t)a.pred_ring) * a.n + s) * a.O;
        }
#pragma unroll
        for (int o = 0; o < OP; ++o)
            if (o < a.O) dst[o] = acc[o] + __ldg(bo + o);
    }
}

static size_t ff_batched_smem(int I, int H, int OP) {
    const int KM = ((I > H ? I : H) + FF_KC - 1) / FF_KC * FF_KC;
    return sizeof(float) * ((size_t)2 * FF_TR * KM + (size_t)FF_KC * FF_HB + (size_t)H * OP);
}

// One dense layer  y = act(x W^T + b)  over many rows: the input layer of ImuPoseLSTM (nn_models.py:210-249: Linear(I, 256) + relu in
// front of a plain 2-layer LSTM).  W^T [K][H] pre-transposed like the feed-forward blob; a CTA stages DENSE_ROWS input rows in
// shared memory and its threads sweep the output units (coalesced weight reads, DENSE_ROWS accumulators per thread).
constexpr int DENSE_ROWS = 8;

__global__ void __launch_bounds__(FF_THREADS) dense_act_kernel(const float* __restrict__ wt, const float* __restrict__ bias,
                                                               const float* __restrict__ x, float* __restrict__ y,
                                                               int rows, int K, int H, int act) {
    extern __shared__ float sx[];                      // [DENSE_ROWS][K]
    const int row0 = blockIdx.x * DENSE_ROWS, tid = threadIdx.x;
    const int nr = min(DENSE_ROWS, rows - row0);
    for (int i = tid; i < DENSE_ROWS * K; i += FF_THREADS) sx[i] = i < nr * K ? x[(size_t)row0 * K + i] : 0.0f;
    __syncthreads();
    for (int j = tid; j < H; j += FF_THREADS) {
        float acc[DENSE_ROWS];
        const float b = bias[j];
#pragma unroll
        for (int r = 0; r < DENSE_ROWS; ++r) acc[r] = b;
        for (int k = 0; k < K; ++k) {
            const float w = __ldg(wt + (size_t)k * H + j);
#pragma unroll
            for (int r = 0; r < DENSE_ROWS; ++r) acc[r] = fmaf(w, sx[r * K + k], acc[r]);
        }
#pragma unroll
        for (int r = 0; r < DENSE_ROWS; ++r) {
            if (r < nr) {
                float v = acc[r];
                if (act == 1) v = v > 0.0f ? v : 0.0f;               // relu
                else if (act == 2) v = v > 0.0f ? v : 0.01f * v;     // leaky_relu(0.01)
                y[(size_t)(row0 + r) * H + j] = v;
            }
        }
    }
}

}  // namespace ape

extern "C" int ape_dense_act(const float* wt, const float* bias, const float* x, float* y, int rows, int K, int H, int act,
                             void* stream) {
    using namespace ape;
    if (!wt || !bias || !x || !y || rows < 0 || K < 1 || H < 1 || act < 0 || act > 2) return APE_ERR_BAD_ARG;
    if (rows == 0) return APE_OK;
    const size_t smem = sizeof(float) * (size_t)DENSE_ROWS * K;
    if (smem > 200 * 1024) return APE_ERR_UNSUPPORTED;
    if (smem > 48 * 1024)
        APE_CUDA_TRY(cudaFuncSetAttribute(dense_act_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dense_act_kernel<<<(rows + DENSE_ROWS - 1) / DENSE_ROWS, FF_THREADS, smem, (cudaStream_t)stream>>>(wt, bias, x, y, rows, K, H, act);
    return check_launch();
}

extern "C" int ape_ff_blob_floats(int I, int H, int Lh, int O, int64_t* floats) {
    if (!floats || I < 1 || H < 1 || Lh < 0 || O < 1) return APE_ERR_BAD_ARG;
    *floats = (int64_t)I * H + H + (int64_t)Lh * ((int64_t)H * H + H) + (int64_t)O * H + O;
    return APE_OK;
}

extern "C" int ape_mc_ff(const float* blob, int I, int H, int Lh, int O, float dropout_p, const float* x, int rows,
                         int n_samples, int mask_mode, const uint8_t* masks, uint64_t philox_seed, uint32_t stream_id0,
                         uint32_t frame0, float* preds, void* stream) {
    using namespace ape;
    if (!blob || !x || !preds || I < 1 || H < 1 || Lh < 0 || O < 1 || O > 20 || rows < 0 || n_samples < 1) return APE_ERR_BAD_ARG;
    if (mask_mode < APE_MASK_NONE || mask_mode > APE_MASK_PHILOX) return APE_ERR_BAD_ARG;
    if (mask_mode == APE_MASK_INJECTED && !masks) return APE_ERR_BAD_ARG;
    if (mask_mode != APE_MASK_NONE && !(dropout_p >= 0.0f && dropout_p < 1.0f)) return APE_ERR_BAD_ARG;
    // the Philox counter holds the sample in 20 bits (ape_common.cuh): samples s and s + 2^20 would draw the same mask
    if (mask_mode == APE_MASK_PHILOX && n_samples > (1 << 20)) return APE_ERR_UNSUPPORTED;
    if (rows == 0) return APE_OK;
    FfArgs a{blob, I, H, Lh, O, x, rows, n_samples, mask_mode, masks, philox_seed, stream_id0, frame0,
             keep_threshold16(dropout_p), mask_mode == APE_MASK_NONE ? 1.0f : 1.0f / (1.0f - dropout_p), preds,
             nullptr, I, 1, 1, 1, 1};
    // the batched kernel wants 16-byte rows of W^T / the masks (H % 8 == 0, aligned pointers) and its tiles in shared memory
    const int OP = O <= 16 ? 16 : 20;
    const size_t bsmem = ff_batched_smem(I, H, OP);
    const bool aligned = H % 8 == 0 && ((uintptr_t)blob & 15) == 0 && (mask_mode != APE_MASK_INJECTED || ((uintptr_t)masks & 7) == 0);
    if (aligned && bsmem <= 200 * 1024) {
        const PhiloxRoundKeys rk = philox_round_keys(philox_seed);
        const int grid = (rows + FF_TR - 1) / FF_TR;
        if (OP == 16) {
            if (bsmem > 48 * 1024) APE_CUDA_TRY(cudaFuncSetAttribute(mc_ff_kernel<16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem));
            mc_ff_kernel<16, false><<<grid, FF_THREADS, bsmem, (cudaStream_t)stream>>>(a, rk);
        } else {
            if (bsmem > 48 * 1024) APE_CUDA_TRY(cudaFuncSetAttribute(mc_ff_kernel<20, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem));
            mc_ff_kernel<20, false><<<grid, FF_THREADS, bsmem, (cudaStream_t)stream>>>(a, rk);
        }
        return check_launch();
    }
    const size_t smem = 2 * sizeof(float) * (size_t)(I > H ? I : H);      // any other shape: one CTA per row
    if (smem > 200 * 1024) return APE_ERR_UNSUPPORTED;
    if (smem > 48 * 1024)
        APE_CUDA_TRY(cudaFuncSetAttribute(mc_ff_row_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    mc_ff_row_kernel<<<rows, FF_THREADS, smem, (cudaStream_t)stream>>>(a);
    return check_launch();
}

extern "C" int ape_mc_ff_ring(const float* blob, int I, int T, int H, int Lh, int O, float dropout_p,
                              const float* feats, int feat_ring, int B, int nF, int frame0, const int32_t* stream_frames,
                              int n_samples, int mask_mode, const uint8_t* masks, uint64_t philox_seed, uint32_t stream_id0,
                              float* preds, int pred_ring, void* stream) {
    using namespace ape;
    if (!blob || !feats || !preds || I < 1 || T < 1 || H < 1 || Lh < 0 || O < 1 || O > 20 || B < 0 || nF < 1 || n_samples < 1)
        return APE_ERR_BAD_ARG;
    if (feat_ring < nF + T - 1 || frame0 < 0 || pred_ring < nF) return APE_ERR_BAD_ARG;
    if (mask_mode < APE_MASK_NONE || mask_mode > APE_MASK_PHILOX) return APE_ERR_BAD_ARG;
    if (mask_mode == APE_MASK_INJECTED && !masks) return APE_ERR_BAD_ARG;
    if (mask_mode != APE_MASK_NONE && !(dropout_p >= 0.0f && dropout_p < 1.0f)) return APE_ERR_BAD_ARG;
    if ((int64_t)I * T > (1 << 20) || (int64_t)B * nF > (1 << 30)) return APE_ERR_BAD_ARG;
    if (mask_mode == APE_MASK_PHILOX && n_samples > (1 << 20)) return APE_ERR_UNSUPPORTED;     // 20-bit sample field, as ape_mc_ff
    // the batched kernel only (no ring form of the one-CTA-per-row kernel): 16-byte rows of W^T / the masks, tiles in shared memory
    const int OP = O <= 16 ? 16 : 20;
    const size_t bsmem = ff_batched_smem(I * T, H, OP);
    const bool aligned = H % 8 == 0 && ((uintptr_t)blob & 15) == 0 && (mask_mode != APE_MASK_INJECTED || ((uintptr_t)masks & 7) == 0);
    if (!aligned || bsmem > 200 * 1024) return APE_ERR_UNSUPPORTED;
    const int rows = B * nF;
    if (rows == 0) return APE_OK;
    FfArgs a{blob, I * T, H, Lh, O, feats, rows, n_samples, mask_mode, masks, philox_seed, stream_id0, (uint32_t)frame0,
             keep_threshold16(dropout_p), mask_mode == APE_MASK_NONE ? 1.0f : 1.0f / (1.0f - dropout_p), preds,
             stream_frames, I, T, feat_ring, nF, pred_ring};
    const PhiloxRoundKeys rk = philox_round_keys(philox_seed);
    const int grid = (rows + FF_TR - 1) / FF_TR;
    if (OP == 16) {
        if (bsmem > 48 * 1024) APE_CUDA_TRY(cudaFuncSetAttribute(mc_ff_kernel<16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem));
        mc_ff_kernel<16, true><<<grid, FF_THREADS, bsmem, (cudaStream_t)stream>>>(a, rk);
    } else {
        if (bsmem > 48 * 1024) APE_CUDA_TRY(cudaFuncSetAttribute(mc_ff_kernel<20, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem));
        mc_ff_kernel<20, true><<<grid, FF_THREADS, bsmem, (cudaStream_t)stream>>>(a, rk);
    }
    return check_launch();
}
