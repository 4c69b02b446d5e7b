// Stage 2, fp32 FFMA variant: the MC-dropout LSTM regressor (nn_models.py:160-207) as one persistent kernel
// per layer.  A CTA owns a tile of R = 16*RT rows (layer 0: estimates; layers >= 1: (estimate, MC sample)
// pairs) for ALL T time steps: the cell state c and the hidden state h never leave shared memory, the packed
// gate weights stream from L2 through a 3-stage cp.async ring in K-slices of 16 rows x 128 gate columns, and
// every thread accumulates an RT x 8 register tile = RT rows x 2 hidden units x 4 gates, so the sigmoid/tanh
// cell update runs in registers right behind the contraction.  The inter-layer dropout mask (injected bytes or
// counter-based Philox) is applied when a layer READS its input, so layer 0 is evaluated once per estimate
// and only layers >= 1 are evaluated per MC sample (SURVEY.md §3.2).  Sequences between layers use the
// tile-local K-major layout [tile][T][H][R] so both sides move float4s with unit stride.
#include "ape_f32x2.cuh"
#ifndef APE_FMA_F32X2
#define APE_FMA_F32X2 1
#endif
#include "ape_common.cuh"
#include "ape_lstm_pack.h"
#include "ape_lstm_plan.cuh"

namespace ape {

constexpr int LSTM_THREADS = 256;
constexpr int CHUNK_UNITS = 32;            // hidden units per N-chunk
constexpr int CHUNK_COLS = 4 * CHUNK_UNITS;
constexpr int KS = APE_KSLICE;
constexpr int W_STAGES = 3;
constexpr int W_STAGE_FLOATS = KS * CHUNK_COLS;

enum { IN_WINDOW = 0, IN_DENSE = 1, IN_SHARED = 2, IN_TILED = 3 };

struct LayerArgs {
    const float* Wp;
    const float* bp;
    int Kin, Kin_pad, H, T;
    int in_mode;
    const float* in;
    int in_R;                 // IN_SHARED: tile rows of the producing layer
    int feat_ring, nF, frame0;
    const int32_t* stream_frames;   // per-stream frame counters (null: frame0 for all); < 0: the stream sits this call out
    int rows;                 // rows of this layer
    int n;                    // row -> estimate e = row / n, sample s = row % n
    int mask_mode;
    const uint8_t* masks;
    int gap, n_gaps;
    uint64_t seed;
    uint32_t stream_id0;
    float keep_scale;
    uint32_t keep_thr16;
    float* out_seq;           // [tiles][T][H][R] un-masked h_t, or null on the last layer
    const float* Wo;          // last layer: output_layer.weight (O, H) / bias (O)
    const float* bo;
    int O;
    float* preds;
    int pred_ring, all_steps, n_out;
    const float* h0;          // optional initial state of this layer, [rows][H] each (torch.nn.LSTM(x, (h_0, c_0))), or null
    const float* c0;
};

__device__ __forceinline__ float sigmoid_f(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float tanh_f(float x) { return 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * x)); }

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

template <int RT> __device__ __forceinline__ void ld_vec(const float* p, float* v) {
    if (RT == 4) { const float4 t = *reinterpret_cast<const float4*>(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
    else if (RT == 2) { const float2 t = *reinterpret_cast<const float2*>(p); v[0] = t.x; v[1] = t.y; }
    else v[0] = p[0];
}
template <int RT> __device__ __forceinline__ void st_vec(float* p, const float* v) {
    if (RT == 4) *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    else if (RT == 2) *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
    else p[0] = v[0];
}

// position of the weight-slice stream: (time step, N-chunk, K-slice)
struct SliceCursor {
    int t, chunk, ks;
    bool state0;                                               // a caller-supplied h_0: step 0 has a recurrent half too
    __device__ __forceinline__ void advance(int nsx, int nsh, int nchunks) {
        const int ns = nsx + ((t > 0 || state0) ? nsh : 0);     // h_{-1} = 0: step 0 skips the recurrent slices
        if (++ks == ns) { ks = 0; if (++chunk == nchunks) { chunk = 0; ++t; } }
    }
};

// NCH_REG = 0: cell state in shared memory, any H % 32 == 0.  NCH_REG = H / 32 > 0: the chunk loop is unrolled and the cell
// state lives in registers (RT x 2 values per chunk), which frees H*R floats of shared memory - H = 256 then fits 64-row
// tiles (twice the FFMA : LDS ratio of the 32-row tiles it would otherwise get).
template <int RT, int NCH_REG>
__global__ void __launch_bounds__(LSTM_THREADS, 1) lstm_layer_fma_kernel(LayerArgs a) {
    constexpr int R = 16 * RT;
    extern __shared__ __align__(16) float smem[];
    const int H = a.H, T = a.T;
    float* xt = smem;                               // [Kin_pad][R]  this step's (masked, scaled) input
    float* hbuf = xt + a.Kin_pad * R;               // [2][H][R]     h_{t-1} / h_t
    float* cbuf = hbuf + 2 * H * R;                 // [H][R]        cell state (NCH_REG == 0 only)
    float* ws = cbuf + (NCH_REG > 0 ? 0 : H * R);   // [W_STAGES][KS][CHUNK_COLS] weight ring
    float creg[NCH_REG > 0 ? NCH_REG : 1][2][RT];   // cell state in registers (NCH_REG > 0)

    const int tid = threadIdx.x, cg = tid & 15, rg = tid >> 4;
    const int tile = blockIdx.x, row0 = tile * R;
    const int nchunks = H / CHUNK_UNITS, nsx = a.Kin_pad / KS, nsh = H / KS;
    const int H4 = 4 * H;

    auto issue_slice = [&](const SliceCursor& c, int stage) {
        if (c.t < T) {
            const int krow = c.ks < nsx ? c.ks * KS : a.Kin_pad + (c.ks - nsx) * KS;
            const float* src = a.Wp + (size_t)krow * H4 + c.chunk * CHUNK_COLS;
            float* dst = ws + stage * W_STAGE_FLOATS;
#pragma unroll
            for (int j = 0; j < (KS * CHUNK_COLS / 4) / LSTM_THREADS; ++j) {
                const int idx = tid + j * LSTM_THREADS, kr = idx >> 5, c4 = idx & 31;
                cp_async16(dst + kr * CHUNK_COLS + c4 * 4, src + (size_t)kr * H4 + c4 * 4);
            }
        }
        cp_async_commit();
    };

    const bool state0 = a.h0 != nullptr;
    if (state0) {                                   // (h_0, c_0) of nn_models.py:180-189 instead of zeros
        for (int idx = tid; idx < H * R; idx += LSTM_THREADS) {
            const int r = idx % R, k = idx / R, row = row0 + r;
            hbuf[k * R + r] = row < a.rows ? __ldg(a.h0 + (size_t)row * H + k) : 0.0f;
            if (NCH_REG == 0) cbuf[k * R + r] = row < a.rows ? __ldg(a.c0 + (size_t)row * H + k) : 0.0f;
        }
        if (NCH_REG > 0) {
#pragma unroll
            for (int chunk = 0; chunk < (NCH_REG > 0 ? NCH_REG : 1); ++chunk)
#pragma unroll
                for (int half = 0; half < 2; ++half)
#pragma unroll
                    for (int r = 0; r < RT; ++r) {
                        const int row = row0 + rg * RT + r;
                        creg[chunk][half][r] = row < a.rows ? __ldg(a.c0 + (size_t)row * H + chunk * CHUNK_UNITS + cg + 16 * half) : 0.0f;
                    }
        }
        __syncthreads();
    }
    SliceCursor pf{0, 0, 0, state0};                // prefetch cursor runs W_STAGES-1 slices ahead
    for (int s = 0; s < W_STAGES - 1; ++s) { issue_slice(pf, s); pf.advance(nsx, nsh, nchunks); }
    int slice = 0, cur = 0;

    for (int t = 0; t < T; ++t) {
        // ---- this step's input rows -> xt[k][r] -------------------------------------------------------
        if (a.in_mode == IN_WINDOW || a.in_mode == IN_DENSE) {
            for (int idx = tid; idx < R * a.Kin_pad; idx += LSTM_THREADS) {
                const int r = idx % R, k = idx / R, row = row0 + r;
                float v = 0.0f;
                if (row < a.rows && k < a.Kin) {
                    if (a.in_mode == IN_DENSE) {
                        v = __ldg(a.in + ((size_t)row * T + t) * a.Kin + k);
                    } else {                                           // sliding window, clamped at frame 0 (estimator.py:96-97)
                        const int b = row / a.nF;
                        int fw = stream_frame0(a.stream_frames, a.frame0, b) + row % a.nF - T + 1 + t;
                        fw = fw < 0 ? 0 : fw;
                        v = __ldg(a.in + ((size_t)b * a.feat_ring + fw % a.feat_ring) * a.Kin + k);
                    }
                }
                xt[k * R + r] = v;
            }
        } else {
            for (int idx = tid; idx < R * (H / 8); idx += LSTM_THREADS) {
                const int r = idx % R, oct = idx / R, row = row0 + r;
                float v[8];
                uint32_t keep = 0xFFu;
                if (row < a.rows) {
                    const int e = row / a.n, s = row - e * a.n;
                    if (a.in_mode == IN_SHARED) {
                        const float* src = a.in + (((size_t)(e / a.in_R) * T + t) * H + oct * 8) * a.in_R + e % a.in_R;
#pragma unroll
                        for (int j = 0; j < 8; ++j) v[j] = __ldg(src + (size_t)j * a.in_R);
                    } else {
                        const float* src = a.in + (((size_t)tile * T + t) * H + oct * 8) * R + r;
#pragma unroll
                        for (int j = 0; j < 8; ++j) v[j] = __ldg(src + (size_t)j * R);
                    }
                    if (a.mask_mode == APE_MASK_INJECTED) {
                        const uint2 m = __ldg(reinterpret_cast<const uint2*>(
                            a.masks + ((((size_t)e * a.n_gaps + a.gap) * T + t) * a.n + s) * H + oct * 8));
                        keep = 0;
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            keep |= ((m.x >> (8 * j)) & 0xFFu ? 1u : 0u) << j;
                            keep |= ((m.y >> (8 * j)) & 0xFFu ? 1u : 0u) << (4 + j);
                        }
                    } else if (a.mask_mode == APE_MASK_PHILOX) {
                        const int b = e / a.nF, f = stream_frame0(a.stream_frames, a.frame0, b) + e % a.nF;
                        keep = philox_keep8(a.seed, a.stream_id0 + (uint32_t)b, (uint32_t)f, (uint32_t)s, (uint32_t)a.gap,
                                            (uint32_t)t, (uint32_t)oct, a.keep_thr16);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = 0.0f;
                }
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    xt[(oct * 8 + j) * R + r] = ((keep >> j) & 1u) ? v[j] * a.keep_scale : 0.0f;
            }
        }
        // (visibility of xt: the __syncthreads of the first slice below)

        const float* hcur = hbuf + cur * H * R;
        float* hnxt = hbuf + (cur ^ 1) * H * R;
        const int ns = nsx + ((t > 0 || state0) ? nsh : 0);

        auto chunk_body = [&](const int chunk, float (&cst)[2][RT]) {
            float acc[RT][8];
            {
                const float4 b0 = __ldg(reinterpret_cast<const float4*>(a.bp + chunk * CHUNK_COLS + cg * 4));
                const float4 b1 = __ldg(reinterpret_cast<const float4*>(a.bp + chunk * CHUNK_COLS + 64 + cg * 4));
#pragma unroll
                for (int r = 0; r < RT; ++r) {
                    acc[r][0] = b0.x; acc[r][1] = b0.y; acc[r][2] = b0.z; acc[r][3] = b0.w;
                    acc[r][4] = b1.x; acc[r][5] = b1.y; acc[r][6] = b1.z; acc[r][7] = b1.w;
                }
            }
            for (int ks = 0; ks < ns; ++ks, ++slice) {
                cp_async_wait<W_STAGES - 2>();
                __syncthreads();
                issue_slice(pf, (slice + W_STAGES - 1) % W_STAGES);
                pf.advance(nsx, nsh, nchunks);
                const float* As = (ks < nsx ? xt + ks * KS * R : hcur + (ks - nsx) * KS * R) + rg * RT;
                const float* Bs = ws + (slice % W_STAGES) * W_STAGE_FLOATS + cg * 4;
#pragma unroll
                for (int kk = 0; kk < KS; ++kk) {
                    float av[RT];
                    ld_vec<RT>(As + kk * R, av);
                    const float4 b0 = *reinterpret_cast<const float4*>(Bs + kk * CHUNK_COLS);
                    const float4 b1 = *reinterpret_cast<const float4*>(Bs + kk * CHUNK_COLS + 64);
#if APE_FMA_F32X2
                    // two gate columns per FFMA2 (packed fp32 pairs, ape_f32x2.cuh; the row value is a scalar-broadcast operand): the same
                    // fused multiply-adds in the same order, half the issue slots of the contraction
                    const F2 w01 = pk(b0.x, b0.y), w23 = pk(b0.z, b0.w), w45 = pk(b1.x, b1.y), w67 = pk(b1.z, b1.w);
#pragma unroll
                    for (int r = 0; r < RT; ++r) {
                        const F2 x = splat(av[r]);
                        F2 v;
                        v = fma2(w01, x, pk(acc[r][0], acc[r][1])); acc[r][0] = lo(v); acc[r][1] = hi(v);
                        v = fma2(w23, x, pk(acc[r][2], acc[r][3])); acc[r][2] = lo(v); acc[r][3] = hi(v);
                        v = fma2(w45, x, pk(acc[r][4], acc[r][5])); acc[r][4] = lo(v); acc[r][5] = hi(v);
                        v = fma2(w67, x, pk(acc[r][6], acc[r][7])); acc[r][6] = lo(v); acc[r][7] = hi(v);
                    }
#else
#pragma unroll
                    for (int r = 0; r < RT; ++r) {
                        acc[r][0] = fmaf(av[r], b0.x, acc[r][0]); acc[r][1] = fmaf(av[r], b0.y, acc[r][1]);
                        acc[r][2] = fmaf(av[r], b0.z, acc[r][2]); acc[r][3] = fmaf(av[r], b0.w, acc[r][3]);
                        acc[r][4] = fmaf(av[r], b1.x, acc[r][4]); acc[r][5] = fmaf(av[r], b1.y, acc[r][5]);
                        acc[r][6] = fmaf(av[r], b1.z, acc[r][6]); acc[r][7] = fmaf(av[r], b1.w, acc[r][7]);
                    }
#endif
                }
            }
            // ---- cell update for this thread's RT rows x 2 units (gate order i, f, g, o) ------------------
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int u = chunk * CHUNK_UNITS + cg + 16 * half;
                float cv[RT], hv[RT];
                if (NCH_REG > 0) {
#pragma unroll
                    for (int r = 0; r < RT; ++r) cv[r] = cst[half][r];
                } else if (t > 0 || state0) {
                    ld_vec<RT>(cbuf + u * R + rg * RT, cv);
                }
#pragma unroll
                for (int r = 0; r < RT; ++r) {
                    const float gi = sigmoid_f(acc[r][4 * half + 0]), gf = sigmoid_f(acc[r][4 * half + 1]);
                    const float gg = tanh_f(acc[r][4 * half + 2]), go = sigmoid_f(acc[r][4 * half + 3]);
                    const float c = (t > 0 || state0) ? fmaf(gf, cv[r], gi * gg) : gi * gg;
                    cv[r] = c;
                    hv[r] = go * tanh_f(c);
                }
                if (NCH_REG > 0) {
#pragma unroll
                    for (int r = 0; r < RT; ++r) cst[half][r] = cv[r];
                } else {
                    st_vec<RT>(cbuf + u * R + rg * RT, cv);
                }
                st_vec<RT>(hnxt + u * R + rg * RT, hv);
            }
        };
        if (NCH_REG > 0) {
#pragma unroll
            for (int chunk = 0; chunk < (NCH_REG > 0 ? NCH_REG : 1); ++chunk) chunk_body(chunk, creg[chunk]);
        } else {
            for (int chunk = 0; chunk < nchunks; ++chunk) chunk_body(chunk, creg[0]);
        }
        __syncthreads();                                               // h_t complete

        if (a.out_seq) {
            float4* dst = reinterpret_cast<float4*>(a.out_seq + ((size_t)tile * T + t) * H * R);
            const float4* src = reinterpret_cast<const float4*>(hnxt);
            for (int idx = tid; idx < H * R / 4; idx += LSTM_THREADS) dst[idx] = src[idx];
        }
        if (a.preds && (a.all_steps || t == T - 1)) {                  // output_layer (nn_models.py:189)
            for (int idx = tid; idx < R * a.O; idx += LSTM_THREADS) {
                const int r = idx % R, o = idx / R, row = row0 + r;
                if (row >= a.rows) continue;
                const float* w = a.Wo + (size_t)o * H;
                float sum = __ldg(a.bo + o);
                for (int k = 0; k < H; ++k) sum = fmaf(__ldg(w + k), hnxt[k * R + r], sum);
                if (a.all_steps) {
                    a.preds[((size_t)row * T + t) * a.O + o] = sum;
                } else {
                    const int e = row / a.n, s = row - e * a.n;
                    const int b = e / a.nF, fb = stream_frame0(a.stream_frames, a.frame0, b), f = fb + e % a.nF;
                    if (fb < 0) continue;                              // inactive stream: keep its prediction ring untouched
                    float* dst = a.preds + (((size_t)b * a.pred_ring + f % a.pred_ring) * a.n_out) * a.O + o;
                    if (a.n == 1 && a.n_out > 1) {                     // single-layer model: no dropout, samples identical
                        for (int s2 = 0; s2 < a.n_out; ++s2) dst[(size_t)s2 * a.O] = sum;
                    } else {
                        dst[(size_t)s * a.O] = sum;
                    }
                }
            }
        }
        cur ^= 1;
    }
    cp_async_wait<0>();
}

__global__ void philox_masks_kernel(uint64_t seed, uint32_t stream_id0, int nF, int frame0, int n_gaps, int T, int n,
                                    int H, uint32_t thr, uint8_t* masks, long long total_octets) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total_octets) return;
    const int H8 = H / 8;
    long long q = i;
    const int oct = (int)(q % H8); q /= H8;
    const int s = (int)(q % n); q /= n;
    const int t = (int)(q % T); q /= T;
    const int gap = (int)(q % n_gaps); q /= n_gaps;
    const int e = (int)q, b = e / nF, f = frame0 + e % nF;
    const uint32_t keep = philox_keep8(seed, stream_id0 + (uint32_t)b, (uint32_t)f, (uint32_t)s, (uint32_t)gap, (uint32_t)t,
                                       (uint32_t)oct, thr);
    uint2 out;
    out.x = (keep & 1u) | ((keep >> 1 & 1u) << 8) | ((keep >> 2 & 1u) << 16) | ((keep >> 3 & 1u) << 24);
    out.y = (keep >> 4 & 1u) | ((keep >> 5 & 1u) << 8) | ((keep >> 6 & 1u) << 16) | ((keep >> 7 & 1u) << 24);
    reinterpret_cast<uint2*>(masks)[i] = out;
}

// ---- host side -----------------------------------------------------------------------------------------

// rt >= 8 encodes "RT = 4 with the cell state in registers" (only instantiated for H = 256)
static size_t layer_smem_bytes(int rt, int H, int kin_pad) {
    const bool regc = rt >= 8;
    const int r = 16 * (regc ? 4 : rt);
    return sizeof(float) * ((size_t)r * (kin_pad + (regc ? 2 : 3) * H) + W_STAGES * W_STAGE_FLOATS);
}
static int max_rt_for(int H, int kin_pad_max) {
    if (layer_smem_bytes(4, H, kin_pad_max) <= 227 * 1024) return 4;
    if (H == 256 && layer_smem_bytes(8, H, kin_pad_max) <= 227 * 1024) return 8;
    for (int rt = 2; rt >= 1; rt >>= 1)
        if (layer_smem_bytes(rt, H, kin_pad_max) <= 227 * 1024) return rt;
    return 0;
}
static int rows_per_tile(int rt) { return 16 * (rt >= 8 ? 4 : rt); }
// rows per tile: the largest tile shared memory allows, shrunk while the grid would leave SMs idle
static int pick_rt(long long rows, int H, int kin_pad) {
    int rt = max_rt_for(H, kin_pad);
    while (rt > 1 && (rows + rows_per_tile(rt) - 1) / rows_per_tile(rt) < 148) rt = rt >= 8 ? 2 : rt >> 1;
    return rt;
}
static long long tiles_of(long long rows, int rt) { return (rows + rows_per_tile(rt) - 1) / rows_per_tile(rt); }
static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

int make_plan(int I, int H, int L, int T, long long E, int n, FmaPlan* p) {
    if (H % CHUNK_UNITS != 0 || H < CHUNK_UNITS) return APE_ERR_UNSUPPORTED;
    const int kp0 = ape_pack_kin_pad(0, I, H);
    if (max_rt_for(H, kp0 > H ? kp0 : H) == 0) return APE_ERR_UNSUPPORTED;
    p->rt0 = pick_rt(E, H, kp0);
    p->rt1 = pick_rt(E * n, H, H);
    p->tiles0 = tiles_of(E, p->rt0);
    p->tiles1 = tiles_of(E * n, p->rt1);
    p->seq0_bytes = L > 1 ? align256((size_t)p->tiles0 * T * H * rows_per_tile(p->rt0) * sizeof(float)) : 0;
    p->seq1_bytes = L > 2 ? align256((size_t)p->tiles1 * T * H * rows_per_tile(p->rt1) * sizeof(float)) : 0;
    p->total = p->seq0_bytes + (L > 3 ? 2 : 1) * p->seq1_bytes;
    return APE_OK;
}

template <int RT, int NCH_REG> static int launch_layer(int rt_code, const LayerArgs& a, long long tiles, cudaStream_t st) {
    const size_t smem = layer_smem_bytes(rt_code, a.H, a.Kin_pad);
    APE_CUDA_TRY(cudaFuncSetAttribute(lstm_layer_fma_kernel<RT, NCH_REG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    lstm_layer_fma_kernel<RT, NCH_REG><<<(unsigned)tiles, LSTM_THREADS, smem, st>>>(a);
    return check_launch();
}
static int launch_layer_rt(int rt, const LayerArgs& a, long long tiles, cudaStream_t st) {
    if (rt == 8) return launch_layer<4, 8>(rt, a, tiles, st);
    if (rt == 4) return launch_layer<4, 0>(rt, a, tiles, st);
    if (rt == 2) return launch_layer<2, 0>(rt, a, tiles, st);
    return launch_layer<1, 0>(rt, a, tiles, st);
}

int check_lstm_args(const ape_lstm_args* g) {
    if (!g || !g->weights || !g->preds) return APE_ERR_BAD_ARG;
    if (g->I < 1 || g->H < 1 || g->L < 1 || g->T < 1 || g->O < 1 || g->B < 0 || g->nF < 0 || g->n_samples < 1) return APE_ERR_BAD_ARG;
    if ((g->x_dense == nullptr) == (g->feat_ring_buf == nullptr)) return APE_ERR_BAD_ARG;
    if (g->feat_ring_buf && (g->feat_ring < g->nF + g->T - 1 || g->frame0 < 0)) return APE_ERR_BAD_ARG;
    if (!g->all_steps && (g->pred_ring < g->nF || g->pred_ring < 1)) return APE_ERR_BAD_ARG;
    if (g->all_steps && g->L == 1 && g->n_samples > 1) return APE_ERR_UNSUPPORTED;
    if (g->mask_mode < APE_MASK_NONE || g->mask_mode > APE_MASK_PHILOX) return APE_ERR_BAD_ARG;
    if (g->mask_mode == APE_MASK_INJECTED && g->L > 1 && !g->masks) return APE_ERR_BAD_ARG;
    if (g->mask_mode != APE_MASK_NONE && !(g->dropout_p >= 0.0f && g->dropout_p < 1.0f)) return APE_ERR_BAD_ARG;
    if ((long long)g->B * g->nF * g->n_samples > 0x7fffffffLL) return APE_ERR_BAD_ARG;
    // the Philox counter packs sample (20 bits), gap (4 bits) and step (8 bits) into one word (ape_common.cuh): beyond these
    // ranges masks of different steps / gaps / samples would alias
    if (g->mask_mode == APE_MASK_PHILOX && g->L > 1 && (g->T > 256 || g->L > 16 || g->n_samples > (1 << 20))) return APE_ERR_UNSUPPORTED;
    if ((g->h0 == nullptr) != (g->c0 == nullptr)) return APE_ERR_BAD_ARG;
    if (g->h0 && g->n_samples != 1) return APE_ERR_UNSUPPORTED;
    return APE_OK;
}

// one layer of the fp32 path; `seq_in` / `seq_out` are the inter-layer sequence buffers (null where unused)
int fma_launch_layer(const ape_lstm_args* g, int l, const FmaPlan& p, const float* seq_in, float* seq_out, cudaStream_t st) {
    const long long E = (long long)g->B * g->nF;
    const bool last = l == g->L - 1;
    LayerArgs a{};
    a.Wp = g->weights + ape_pack_layer_offset(l, g->I, g->H);
    a.bp = g->weights + ape_pack_bias_offset(l, g->I, g->H);
    a.Kin = l == 0 ? g->I : g->H;
    a.Kin_pad = ape_pack_kin_pad(l, g->I, g->H);
    a.H = g->H; a.T = g->T;
    a.feat_ring = g->feat_ring; a.nF = g->nF; a.frame0 = g->frame0; a.stream_frames = g->stream_frames;
    a.mask_mode = l == 0 ? APE_MASK_NONE : g->mask_mode;
    a.masks = g->masks; a.gap = l - 1; a.n_gaps = g->L - 1;
    a.seed = g->philox_seed; a.stream_id0 = g->stream_id0;
    a.keep_scale = g->mask_mode == APE_MASK_NONE ? 1.0f : 1.0f / (1.0f - g->dropout_p);
    a.keep_thr16 = keep_threshold16(g->dropout_p);
    a.Wo = g->weights + ape_pack_out_offset(g->I, g->H, g->L);
    a.bo = a.Wo + (size_t)g->O * g->H;
    a.O = g->O;
    a.pred_ring = g->pred_ring; a.all_steps = g->all_steps; a.n_out = g->n_samples;
    int rt; long long tiles;
    if (l == 0) {
        a.in_mode = g->x_dense ? IN_DENSE : IN_WINDOW;
        a.in = g->x_dense ? g->x_dense : g->feat_ring_buf;
        a.rows = (int)E; a.n = 1;
        rt = p.rt0; tiles = p.tiles0;
    } else {
        a.in_mode = l == 1 ? IN_SHARED : IN_TILED;
        a.in = seq_in;
        a.in_R = rows_per_tile(p.rt0);
        a.rows = (int)(E * g->n_samples); a.n = g->n_samples;
        rt = p.rt1; tiles = p.tiles1;
    }
    a.out_seq = last ? nullptr : seq_out;
    a.preds = last ? g->preds : nullptr;
    if (g->h0) {                                    // [L][E][H]; n_samples == 1, so every layer has E rows
        a.h0 = g->h0 + (size_t)l * E * g->H;
        a.c0 = g->c0 + (size_t)l * E * g->H;
    }
    return launch_layer_rt(rt, a, tiles, st);
}

}  // namespace ape

extern "C" int ape_mc_lstm_workspace_bytes(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes) {
    using namespace ape;
    if (!bytes || I < 1 || H < 1 || L < 1 || T < 1 || O < 1 || E < 0 || n_samples < 1) return APE_ERR_BAD_ARG;
    FmaPlan p;
    const int rc = make_plan(I, H, L, T, E, n_samples, &p);
    if (rc != APE_OK) return rc;
    *bytes = p.total + 256;
    return APE_OK;
}

extern "C" int ape_mc_lstm_fma(const ape_lstm_args* g, void* stream) {
    using namespace ape;
    int rc = check_lstm_args(g);
    if (rc != APE_OK) return rc;
    const long long E = (long long)g->B * g->nF;
    if (E == 0) return APE_OK;
    FmaPlan p;
    rc = make_plan(g->I, g->H, g->L, g->T, E, g->n_samples, &p);
    if (rc != APE_OK) return rc;
    if (p.total > 0 && !g->workspace) return APE_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;

    char* wsp = (char*)(((uintptr_t)g->workspace + 255) & ~(uintptr_t)255);
    float* seq0 = (float*)wsp;
    float* seq1[2] = {(float*)(wsp + p.seq0_bytes), (float*)(wsp + p.seq0_bytes + p.seq1_bytes)};

    LayerTimer timer(g->layer_ms, g->L, st);
    rc = timer.start();
    for (int l = 0; l < g->L && rc == APE_OK; ++l) {
        const float* seq_in = l == 0 ? nullptr : (l == 1 ? seq0 : seq1[(l - 2) & 1]);
        float* seq_out = l == 0 ? seq0 : seq1[(l - 1) & 1];
        rc = fma_launch_layer(g, l, p, seq_in, seq_out, st);
        if (rc == APE_OK) rc = timer.mark(l + 1);
    }
    return rc == APE_OK ? timer.finish() : rc;
}

extern "C" int ape_philox_masks(uint64_t philox_seed, uint32_t stream_id0, int B, int nF, int frame0, int L, int T,
                                int n_samples, int H, float dropout_p, uint8_t* masks, void* stream) {
    using namespace ape;
    if (B < 0 || nF < 0 || frame0 < 0 || L < 1 || T < 1 || n_samples < 1 || H < 8 || H % 8 != 0) return APE_ERR_BAD_ARG;
    const long long total = (long long)B * nF * (L - 1) * T * n_samples * (H / 8);
    if (total == 0) return APE_OK;
    if (!masks) return APE_ERR_BAD_ARG;
    const int threads = 256;
    const long long blocks = (total + threads - 1) / threads;
    if (blocks > 0x7fffffffLL) return APE_ERR_BAD_ARG;
    philox_masks_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(
        philox_seed, stream_id0, nF, frame0, L - 1, T, n_samples, H, keep_threshold16(dropout_p), masks, total);
    return check_launch();
}
