/*
 * ape_b200.h - C ABI of the B200-native per-frame arm-pose estimation path.
 *
 * The reference (wear_mocap_ape 1.2.3) has no FFI: its boundary is the Python class API
 * (SURVEY.md §8b).  This header is the C-ABI layer north_star prescribes underneath that API.
 * Every entry point takes raw DEVICE pointers + sizes + a cudaStream_t (passed as void*), allocates
 * nothing, keeps no global state, and returns an int status (APE_OK or an APE_ERR_* code; the Python
 * wrappers raise UserWarning on non-zero, the way the reference signals errors, nn_models.py:202).
 * All kernels are enqueued on `stream` and return without synchronising.
 *
 * Units.  One ESTIMATE = one frame of one stream (raw IMU row -> 25-float pose message).  A launch
 * covers E = B streams x nF consecutive frames; estimate e = b * nF + f_rel, absolute frame
 * f = frame0 + f_rel.  Frame-indexed device buffers are rings of `*_ring` frames per stream, slot
 * f % ring; frames before 0 clamp to frame 0, which reproduces the reference's "repeat the first
 * row / first prediction" warm-up (estimator.py:96-97, :114-115).
 *
 * Streams that do not advance in lock-step (many sockets feeding one GPU, each with the reference's
 * "drop the backlog" freshness policy, estimator.py:159-161): every stage takes an optional device array
 * `stream_frames[B]` of per-stream absolute frame numbers that replaces frame0; a NEGATIVE entry means
 * "no new frame for this stream in this call" - the stream's rings and outputs are left untouched.
 */
#ifndef APE_B200_H
#define APE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define APE_OK 0
#define APE_ERR_BAD_ARG 1        /* null pointer / size out of range */
#define APE_ERR_UNSUPPORTED 2    /* shape not supported by this kernel (e.g. H % 32 != 0) */
#define APE_ERR_CUDA 3           /* a CUDA runtime call failed; see ape_last_cuda_error() */
#define APE_ERR_NO_SM100 4       /* the current device is not compute capability 10.x */

/* estimator kinds: which parse_row_to_xx is followed */
#define APE_KIND_WATCH_ONLY 0    /* estimate/watch_only.py:46-82            -> 20 features */
#define APE_KIND_POCKET 1        /* estimate/watch_phone_pocket_nn.py:41-96  -> 22 features */
#define APE_KIND_UARM 2          /* estimate/watch_phone_uarm_nn.py:43-105   -> 38 features */

/* wire layouts of a raw row (data_types/messaging.py:20-68 and :96-187) */
#define APE_LAYOUT_WATCH_ONLY 0  /* 28 floats */
#define APE_LAYOUT_WATCH_PHONE 1 /* 55 floats */

/* network target sets (utility/names.py:4-29) */
#define APE_TARGET_ORI_CAL_LARM_UARM 0           /* O = 12 */
#define APE_TARGET_ORI_CAL_LARM_UARM_HIPS 1      /* O = 14 */
#define APE_TARGET_ORI_POS_CAL_LARM_UARM_HIPS 2  /* O = 20 */

/* dropout mask source of the MC-LSTM */
#define APE_MASK_NONE 0      /* eval mode: no dropout (DropoutLSTM.forward after .eval()) */
#define APE_MASK_INJECTED 1  /* caller supplies the Bernoulli masks (bit-comparable parity runs) */
#define APE_MASK_PHILOX 2    /* counter-based Philox4x32-10 keyed by (seed; stream, frame, sample, gap, t, unit) */

/* ---- library / device ------------------------------------------------------------------------ */

/* ABI version of this header (bumped on any signature change). */
int ape_abi_version(void);
/* cudaGetErrorString of the last failing CUDA call made by this library on the calling thread. */
const char* ape_last_cuda_error(void);
/* sm count / smem per block of the current device; returns APE_ERR_NO_SM100 off Blackwell. */
int ape_device_info(int* sm_count, int* smem_optin_bytes, int* cc_major, int* cc_minor);
/* number of floats of the packed weight blob (csrc/ape_lstm_pack.h) for a DropoutLSTM(I, H, L, O). */
int ape_lstm_blob_floats(int I, int H, int L, int O, int64_t* floats);

/* ---- stage 1: raw rows -> calibrated, normalised feature rows --------------------------------- */
/*
 * Replaces parse_row_to_xx (watch_only.py:46-82, watch_phone_pocket_nn.py:41-96,
 * watch_phone_uarm_nn.py:43-105) and the z-score of estimator.py:103-104 for B x nF rows at once.
 *   raw      [B][nF][ncols] float32, ncols = 28 (layout 0) or 55 (layout 1)
 *   xx_m/s   [I] float64 column means / stds (data_stats pickles)
 *   feats    [B][feat_ring][I] float32, row of absolute frame f written to slot f % feat_ring
 *   normalize 0: write raw features (what parse_row_to_xx returns), 1: (xx - m) / s
 * Arithmetic is float64 with the reference's float32 rounding point (watch_only.py:82) kept.
 */
int ape_features(const float* raw, int layout, int kind, const double* xx_m, const double* xx_s,
                 int normalize, float* feats, int B, int nF, int frame0, const int32_t* stream_frames,
                 int feat_ring, void* stream);

/*
 * The window update of add_xx_to_row_hist_and_make_prediction (estimator.py:93-104) for callers that use the reference's three
 * per-frame calls one by one: xx [B][I] float64 feature rows as parse_row_to_xx returned them -> z-score -> slot
 * frame % feat_ring of each stream's ring (frames before 0 are never written: readers clamp to frame 0, which is the
 * reference's "repeat the first row").
 */
int ape_features_push(const double* xx, int I, const double* xx_m, const double* xx_s, int normalize, float* feats,
                      int B, int frame0, const int32_t* stream_frames, int feat_ring, void* stream);

/* ---- stage 2: MC-dropout LSTM regressor -------------------------------------------------------- */
/*
 * Replaces DropoutLSTM.forward / .monte_carlo_predictions (nn_models.py:180-207) and the
 * "keep the last step" of make_prediction_from_row_hist (watch_only.py:84-97), batched over
 * (estimates x MC samples).  Layer 0 runs once per estimate (no dropout in front of it), layers >= 1
 * per (estimate, sample); the output layer is applied to the last step only unless all_steps != 0.
 */
typedef struct ape_lstm_args {
    /* model: packed by arm_pose_estimation_b200.estimate.nn_models.pack_lstm_weights() */
    const float* weights;      /* device blob, layout documented in csrc/ape_lstm_pack.h */
    int I, H, L, T, O;         /* input, hidden, layers, sequence length, outputs */
    float dropout_p;           /* Bernoulli drop probability of the inter-layer dropout */
    /* input: exactly one of x_dense / feat_ring_buf is non-null */
    const float* x_dense;      /* [E][T][I] normalised windows (DropoutLSTM.forward API) */
    const float* feat_ring_buf;/* [B][feat_ring][I] ring written by ape_features */
    int feat_ring;
    int B, nF, frame0;         /* E = B * nF estimates */
    int n_samples;             /* MC samples per estimate (rows of layers >= 1 = E * n_samples) */
    /* dropout masks */
    int mask_mode;             /* APE_MASK_* */
    const uint8_t* masks;      /* APE_MASK_INJECTED: [E][L-1][T][n_samples][H] of {0,1}, else null */
    uint64_t philox_seed;
    uint32_t stream_id0;       /* global id of stream 0 of this launch (shard offset) */
    /* workspace: ape_mc_lstm_workspace_bytes() bytes, 256-byte aligned */
    void* workspace;
    /* output */
    float* preds;              /* all_steps == 0: [B][pred_ring][n_samples][O], slot f % pred_ring
                                  all_steps != 0: [E][n_samples][T][O] */
    int pred_ring;
    int all_steps;
    /* tensor-core path only: fp16 gate weights of all layers packed by pack_lstm_weights_tc()
       (ape_lstm_tc_blob_bytes() bytes, layout in csrc/ape_lstm_tc.cu); ignored by ape_mc_lstm_fma */
    const void* weights_tc;
    /* profiling: null, or L floats on the HOST - the call then brackets every layer launch with CUDA events,
       synchronises the stream and writes each layer's device time in milliseconds (bench.py's roofline leg) */
    float* layer_ms;
    /* tensor-core path: run only layers [layer_begin, layer_end) (0, 0 = all) so a caller can put layer 0 of the next call
       on a second stream under the tail of this call; ws_parity (0 | 1) selects one of two copies of layer 0's output */
    int layer_begin, layer_end, ws_parity;
    /* debugging (tensor-core path): null, or a device buffer of 768 int64 that receives SM-clock stamps of the first
       tile of CTA 0 of layer `trace_layer` ([role: epilogue, loader, issuer][step < 16][event < 16]; needs a library built
       with -DAPE_TC_TRACE=1).  trace_layer < 0: instead the CTA timeline of every layer, a device buffer of [L][160 CTAs][4]
       int64 = {globaltimer ns at entry, after the set-up, at exit; SM id} (tools/lanes_timeline.py) */
    void* trace;
    int trace_layer;
    /* per-stream frame counters [B] on the device (null: every stream is at frame0); < 0: skip the stream */
    const int32_t* stream_frames;
    /* ---- ABI 5 ---- */
    /* tensor-core path: E = B * nF of the LARGEST call that uses this workspace (0: this call's own E).  The offsets of the
       buffers inside the workspace are computed from it, so calls of different sizes that are in flight on different streams
       (the cross-call pipeline, estimate/batched.py) agree on where the two copies of layer 0's output live. */
    int ws_E;
    /* tensor-core path, H = 128, L >= 3: how consecutive layers >= 1 are launched.  0 = automatic (a pair of layers runs as ONE
       two-layer wavefront launch, csrc/ape_lstm_tcw.cu, when the batch fills the GPU), 1 = one launch per layer always,
       2 = wavefront pairs always (no initial state), 3 = the SPLIT-PRECISION variant, initial state at H = 256 only (every operand an fp16 pair hi + lo, three tensor-core passes per
       product, ex2 / rcp cell update: fp32-grade results at ~0.4 of the single-pass throughput; needs weights_tcx; H = 128:
       csrc/ape_lstm_tcx.cu, H = 256: csrc/ape_lstm_tcxs.cu; all_steps != 0 needs the _all_steps workspace query),
       4 = the SMALL-BATCH kernel (csrc/ape_lstm_tcl.cu: B * nF * n_samples <= 8192 rows, L <= 4: all layers in one launch, one
       8-CTA cluster per 128 rows with the hidden units split across it - the real-time case of one to a few dozen streams; same
       arithmetic as 0..2; no initial state),
       5 = the SPLIT-PRECISION SMALL-BATCH kernel (csrc/ape_lstm_tcxl.cu: the arithmetic of 3 at H = 128 - bit-identical results - in
       the launch structure of 4: B * nF * n_samples <= 8192 rows, 2 <= L <= 4, T <= 40, O <= 16; needs weights_tcx and a workspace of
       ape_mc_lstm_tcxl_workspace_bytes(); no initial state, no all_steps, no layer range: APE_ERR_UNSUPPORTED; the same call of an
       H = 256 model goes to ape_mc_lstm_tcxsl, csrc/ape_lstm_tcxsl.cu) */
    int tc_flags;
    /* optional initial state (h_0, c_0) of torch.nn.LSTM(x, hs) (nn_models.py:180-189): [L][E][H] float32 each, both or neither
       (APE_ERR_BAD_ARG); needs n_samples == 1 (APE_ERR_UNSUPPORTED; a caller with per-sample states passes the samples as estimates).
       Taken by the fp32 path and by the tensor-core path with tc_flags 0 or 1 (the one-layer kernels; tc_flags 0 then never pairs
       layers) and with tc_flags 3 at H = 256 only (the split-precision kernel csrc/ape_lstm_tcxs.cu); both pointers 16-byte aligned,
       else APE_ERR_BAD_ARG.  tc_flags 2 and 4, and 3 at H = 128, refuse it with APE_ERR_UNSUPPORTED */
    const float* h0;
    const float* c0;
    /* ---- ABI 6 ---- */
    /* tensor-core path: SMs (rounded up to whole SM pairs) that the persistent launches of the layers >= 1 leave free, so that the
       few CTAs of stage 1 + layer 0 of the NEXT call (a high-priority side stream, ape_pipeline_submit) start at once instead of
       waiting for a persistent launch to retire CTAs; 0 = use every SM */
    int reserve_sms;
    /* split-precision tensor-core variant (tc_flags == 3; csrc/ape_lstm_tcx.cu, H = 128, or csrc/ape_lstm_tcxs.cu, H = 256): its
       weight blob, packed by pack_lstm_weights_tcx() (ape_lstm_tcx_blob_bytes() / ape_lstm_tcxs_blob_bytes() bytes); the workspace
       must then hold ape_mc_lstm_tcx_workspace_bytes() / ape_mc_lstm_tcxs_workspace_bytes() */
    const void* weights_tcx;
} ape_lstm_args;

int ape_mc_lstm_workspace_bytes(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes);
/* fp32 FFMA variant (parity anchor; H in {32, 64, 128, 256}). */
int ape_mc_lstm_fma(const ape_lstm_args* args, void* stream);
/*
 * Tensor-core variant (tcgen05, cta_group::2, TMEM accumulators): fp16 operands, fp32 accumulation and cell state.
 * H in {64, 128} (gate weights resident in shared memory; H = 128, L >= 3: pairs of layers >= 1 as one two-layer wavefront launch
 * with weights streamed from L2) or 256 (gate weights streamed from L2 through a cp.async.bulk ring), L >= 2; same arguments and
 * outputs as ape_mc_lstm_fma plus weights_tc, h0 / c0 included (tc_flags 0 and 1, and 3 at H = 256; see the h0 field).
 * Use when the streams x MC-samples batch is large (>= a few thousand rows); the fp32 variant is the exact path.
 */
int ape_mc_lstm_tc_supported(int I, int H, int L, int O);
int ape_lstm_tc_blob_bytes(int I, int H, int L, int64_t* bytes);
int ape_mc_lstm_tc_workspace_bytes(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes);
/* workspace of a call with all_steps != 0 (keeps the last layer's sequence for the per-step output layer) */
int ape_mc_lstm_tc_workspace_bytes_all_steps(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes);
int ape_mc_lstm_tc(const ape_lstm_args* args, void* stream);
/* split-precision variant (tc_flags == 3): supported shapes (H = 128, O <= 16, L >= 2), blob and workspace sizes */
int ape_mc_lstm_tcx_supported(int I, int H, int L, int O);
int ape_lstm_tcx_blob_bytes(int I, int H, int L, int64_t* bytes);
int ape_mc_lstm_tcx_workspace_bytes(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes);
/* workspace of a split-precision call with all_steps != 0 (keeps the last layer's sequence, hi and lo, for the per-step output layer) */
int ape_mc_lstm_tcx_workspace_bytes_all_steps(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes);
/* the same for the H = 256 split-precision kernel (csrc/ape_lstm_tcxs.cu; H = 256, I <= 256, O <= 32, L >= 2), which tc_flags == 3
   selects for an H = 256 model: its blob (packed by pack_lstm_weights_tcx() as well, the same layout at H = 256) also travels in
   weights_tcx, and the workspace must hold ape_mc_lstm_tcxs_workspace_bytes() */
int ape_mc_lstm_tcxs_supported(int I, int H, int L, int O);
int ape_lstm_tcxs_blob_bytes(int I, int H, int L, int64_t* bytes);
int ape_mc_lstm_tcxs_workspace_bytes(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes);
int ape_mc_lstm_tcxs_workspace_bytes_all_steps(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes);
/* workspace of a call on the split-precision small-batch kernel (tc_flags == 5: H = 128, 2 <= L <= 4, T <= 40, O <= 16,
   E * n_samples <= 8192): the h_t exchange buffer and the layer sequences, hi and lo, of one cluster per 128 rows */
int ape_mc_lstm_tcxl_workspace_bytes(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes);
/*
 * Split-precision small-batch kernel for H = 256 (csrc/ape_lstm_tcxsl.cu): the arithmetic and MMA order of tc_flags == 3 at H = 256 -
 * bit-identical results - with every layer of a call in ONE launch, one 16-CTA cluster per 128 rows (a non-portable cluster size).
 * Same arguments as ape_mc_lstm_tc with tc_flags == 5 (else APE_ERR_BAD_ARG) and the blob in weights_tcx.  APE_ERR_UNSUPPORTED for
 * an initial state, all_steps, a layer range, H != 256, L outside 2..4, O > 32, T > 40, I > 256 or B * nF * n_samples > 8192;
 * APE_ERR_BAD_ARG for a missing blob or workspace or ws_E < B * nF - all before any CUDA call; an empty call returns APE_OK.  Then
 * APE_ERR_UNSUPPORTED when the device cannot hold one cluster of the kernel (ape_mc_lstm_tcxsl_max_active_clusters() == 0).
 * layer_ms reports the one launch as layer 0.  The workspace must hold ape_mc_lstm_tcxsl_workspace_bytes() (the h_t exchange buffer
 * and the layer sequences, hi and lo, of one cluster per 128 rows).
 */
int ape_mc_lstm_tcxsl(const ape_lstm_args* args, void* stream);
int ape_mc_lstm_tcxsl_workspace_bytes(int I, int H, int L, int T, int O, int E, int n_samples, uint64_t* bytes);
/* 16-CTA clusters of ape_mc_lstm_tcxsl's launch the current device holds at once (cudaOccupancyMaxActiveClusters, cached per device);
   0 = the kernel cannot run there */
int ape_mc_lstm_tcxsl_max_active_clusters(int* clusters);
/* number of kernels ape_mc_lstm_tc launches for these arguments (layer pairs of an H = 128 model count once; tc_flags 4 and 5: 1) */
int ape_mc_lstm_tc_launch_count(const ape_lstm_args* args, int* launches);
/*
 * The Bernoulli keep-masks APE_MASK_PHILOX draws, written out as bytes in the APE_MASK_INJECTED layout
 * [E][L-1][T][n_samples][H] - lets a checker replay a Philox run through any injected-mask implementation.
 */
int ape_philox_masks(uint64_t philox_seed, uint32_t stream_id0, int B, int nF, int frame0, int L, int T,
                     int n_samples, int H, float dropout_p, uint8_t* masks, void* stream);

/*
 * MC-dropout feed-forward regressors (DropoutFF / DropoutFF2D, nn_models.py:252-370): Linear + leaky_relu stack evaluated once
 * per input row, dropout + output layer once per MC sample.
 *   blob   packed by pack_ff_weights(): layer 0 W^T [I][H], b [H]; Lh x (W^T [H][H], b [H]); output W [O][H], b [O]
 *   x      [rows][I] float32 (DropoutFF2D: the flattened [seq_len * input] window)
 *   masks  APE_MASK_INJECTED: [rows][n_samples][H] of {0,1}
 *   preds  [rows][n_samples][O] float32
 * APE_MASK_PHILOX with n_samples > 2^20 returns APE_ERR_UNSUPPORTED before any CUDA call (the counter's sample field has 20 bits).
 */
int ape_ff_blob_floats(int I, int H, int Lh, int O, int64_t* floats);
int ape_mc_ff(const float* blob, int I, int H, int Lh, int O, float dropout_p, const float* x, int rows,
              int n_samples, int mask_mode, const uint8_t* masks, uint64_t philox_seed, uint32_t stream_id0,
              uint32_t frame0, float* preds, void* stream);
/*
 * ape_mc_ff on the rings of the batched path: stage 2 of a feed-forward model between ape_features and ape_fk_reduce.
 * E = B * nF rows, row e = b * nF + j is frame f = (stream_frames ? stream_frames[b] : frame0) + j of stream b (a negative
 * stream_frames[b]: nothing of stream b is written).  Its input is the window of frames f - T + 1 .. f of the feature ring,
 * time-major (index t * I + k, DropoutFF2D._flatten of x [1, T, I]; T = 1: DropoutFF on the newest frame), frames before 0
 * read frame 0.  The hidden stack, FMA order and output layer are those of ape_mc_ff; the Philox counters are
 * (stream_id0 + b, f, sample, gap 15, 0, unit octet), so row e equals ape_mc_ff on its window with stream_id0 + b, frame0 = f.
 *   blob   pack_ff_weights() of a model with T * I inputs
 *   feats  [B][feat_ring][I] float32 (ape_features), feat_ring >= nF + T - 1
 *   masks  APE_MASK_INJECTED: [E][n_samples][H] of {0,1}
 *   preds  [B][pred_ring][n_samples][O] float32 (ape_fk_reduce's input), slot f % pred_ring, pred_ring >= nF
 * The batched kernel only: H % 8 != 0, a blob not 16-byte aligned, masks not 8-byte aligned or tiles over 200 KB of
 * shared memory return APE_ERR_UNSUPPORTED.  O <= 20.  APE_MASK_PHILOX with n_samples > 2^20: APE_ERR_UNSUPPORTED, as ape_mc_ff.
 * Every refusal comes before any CUDA call.
 */
int ape_mc_ff_ring(const float* blob, int I, int T, int H, int Lh, int O, float dropout_p,
                   const float* feats, int feat_ring, int B, int nF, int frame0, const int32_t* stream_frames,
                   int n_samples, int mask_mode, const uint8_t* masks, uint64_t philox_seed, uint32_t stream_id0,
                   float* preds, int pred_ring, void* stream);

/*
 * One dense layer over many rows, y = act(x W^T + b): the input layer of ImuPoseLSTM (nn_models.py:210-249: Linear + relu in front
 * of a plain LSTM; the LSTM itself runs through ape_mc_lstm_fma with x_dense).
 *   wt [K][H] float32 (the layer's weight transposed), bias [H], x [rows][K], y [rows][H]; act 0 none, 1 relu, 2 leaky_relu(0.01)
 */
int ape_dense_act(const float* wt, const float* bias, const float* x, float* y, int rows, int K, int H, int act, void* stream);

/* ---- stage 3: targets -> quaternions + forward kinematics + MC reduction ----------------------- */
/*
 * Replaces the de-normalisation of estimator.py:108-109, the smoothing stack of :112-118,
 * estimate_joints.arm_pose_from_nn_targets (estimate_joints.py:16-92) and
 * compose_msg.msg_from_nn_targets_est (compose_msg.py:13-108), plus the per-frame std over the
 * S = smooth * n_samples rows (SURVEY.md §8a "new").
 *   preds    [B][pred_ring][n_samples][O] float32 normalised network outputs
 *   yy_m/s   [O] float32 (null: preds are already de-normalised)
 *   body9    [9] float32: larm_vec, uarm_vec, uarm_orig_rh (estimator.py:57-68)
 *   msg      [E][25] float32: [larm_q, hand, larm_q, elbow, uarm_q, shoulder, hips_q]
 *   samples  [E][S][6] float32 or null: per-row hand xyz, elbow xyz (message tail of estimator.py:131-136)
 *   stdev    [E][6] float32 or null: population std of those rows
 *   est_rows [E][S][W] float32 or null: the full per-row output of arm_pose_from_nn_targets, W = 14 (target 0:
 *            hand3, elbow3, larm_q4, uarm_q4) or 21 (targets 1, 2: hand3, elbow3, shoulder3, larm_q4, uarm_q4, hips_q4)
 *   status   [E] int32 or null: 0 ok, 1 = a 6D pair was degenerate (the reference raises LinAlgError)
 */
int ape_fk_reduce(const float* preds, int pred_ring, const float* yy_m, const float* yy_s, const float* body9,
                  int target, int O, int B, int nF, int frame0, const int32_t* stream_frames, int n_samples, int smooth,
                  float* msg, float* samples, float* stdev, float* est_rows, int32_t* status, void* stream);
/*
 * ape_fk_reduce with one skeleton PER STREAM (the reference gives every estimator its own bonemap, estimator.py:57-68):
 *   bodies       [B][body_stride] float32, row b = the nine floats of body9 for stream b (the local index of this launch);
 *                body_stride 0: one row for every stream, which is ape_fk_reduce itself (the same kernel and arithmetic)
 * Every other argument and output is that of ape_fk_reduce.  A null bodies, a negative stride or a stride of 1 to 8 returns
 * APE_ERR_BAD_ARG before any CUDA call.  Rows of idle streams (stream_frames[b] < 0) are not used.
 */
int ape_fk_reduce_bodies(const float* preds, int pred_ring, const float* yy_m, const float* yy_s, const float* bodies,
                         int body_stride, int target, int O, int B, int nF, int frame0, const int32_t* stream_frames, int n_samples,
                         int smooth, float* msg, float* samples, float* stdev, float* est_rows, int32_t* status, void* stream);

/*
 * compose_msg.msg_from_nn_targets_est (compose_msg.py:13-108) on rows that already hold quaternions + origins:
 *   est [E][S][W] float32 rows as produced by arm_pose_from_nn_targets (W = 14 | 21, see est_rows above)
 *   msg [E][25], stdev [E][6] or null
 */
int ape_msg_from_est(const float* est, int W, const float* body9, int target, int E, int S, float* msg,
                     float* stdev, void* stream);

/* ---- the cross-call pipeline as one host call per batch (ABI 6) --------------------------------------------- */
/*
 * What the reference's loop body (estimator.py:174-176) becomes for B streams x nF frames when calls are queued back to back:
 * stage 1 + MC-LSTM layer 0 on a high-priority side stream (up to three calls ahead), the layers >= 1 + stage 3 on two alternating
 * lane streams (two calls in flight), the device-to-host copy of the results on a copy stream.  ape_pipeline_submit enqueues all
 * of it in ONE call (a few dozen CUDA API calls, no Python in between) and returns without waiting; ape_pipeline_wait blocks
 * until the results of a slot are in pinned host memory.  The tensor-core MC-LSTM only (ape_mc_lstm_tc), mask modes
 * APE_MASK_PHILOX / APE_MASK_NONE.  The object owns CUDA streams and events and nothing else: every buffer below is the
 * caller's and must outlive the pipeline.  One host thread per pipeline.
 *   result buffer layout (device and host, E_max = B * nF_max, S = smooth * n_samples):
 *     [msg E_max x 25 | std E_max x 6 | status E_max (int32) | samples E_max x S x 6 (if emit_samples)]
 *   a call of nF < nF_max frames packs its E = B * nF estimates at the front of each part.
 */
#define APE_PIPELINE_MAX_SLOTS 8
#define APE_PIPE_INPUT_PENDING 1  /* rows_dev is still being written on caller_stream: order stage 1 after it */
#define APE_PIPE_CALLER_WAITS 2   /* caller_stream waits for the call's results (device consumers of out_dev[slot]) */
#define APE_PIPE_D2H 4            /* copy the results to out_host[slot]; ape_pipeline_wait(slot) then blocks until they landed */
typedef struct ape_pipeline ape_pipeline;
typedef struct ape_pipeline_desc {
    /* stage 1 (ape_features) */
    int layout, kind, normalize, ncols;
    const double* xx_m;
    const double* xx_s;
    float* raw;                 /* device [B][nF_max][ncols]: where staged host rows are copied to */
    float* feats;               /* device [B][feat_ring][I] */
    int feat_ring;
    /* stage 2 (ape_mc_lstm_tc): model, dims, mask mode, seed, stream_id0, preds, pred_ring, weights_tc, ws_E, tc_flags, B, n_samples
       as for a direct call; nF, frame0, stream_frames, workspace, layer range and ws_parity are set per call by the pipeline */
    ape_lstm_args lstm;
    void* lane_workspace[2];    /* one ape_mc_lstm_tc workspace per lane */
    /* stage 3 (ape_fk_reduce) */
    const float* yy_m;
    const float* yy_s;
    const float* body9;
    int target, smooth, emit_samples;
    /* buffers */
    int B, nF_max, n_slots;     /* 2 <= n_slots <= APE_PIPELINE_MAX_SLOTS: calls in flight between submit and wait */
    float* out_dev[APE_PIPELINE_MAX_SLOTS];      /* device result buffers */
    float* raw_host[APE_PIPELINE_MAX_SLOTS];     /* pinned [B][nF_max][ncols] */
    float* out_host[APE_PIPELINE_MAX_SLOTS];     /* pinned result buffers */
    int32_t* frames_dev[4];                      /* optional (all null: not used): per-stream frame counters, device [B] x 4 */
    int32_t* frames_host[APE_PIPELINE_MAX_SLOTS];/* ... and their pinned staging [B] per slot */
} ape_pipeline_desc;
int ape_pipeline_create(const ape_pipeline_desc* desc, ape_pipeline** out);
int ape_pipeline_destroy(ape_pipeline* p);
/*
 * One call of B x nF estimates starting at absolute frame frame0 (or at stream_frames_host[b] per stream, host int32 [B], negative:
 * the stream sits this call out).  Exactly one of rows_host (any host memory, copied into the slot's pinned staging here) and
 * rows_dev (device rows, read in place) is non-null.  *slot = the result slot used (out_dev / out_host index); a slot is
 * reused after n_slots calls, after its previous results have landed.  A stream's counter may go back (a restarted stream, frame0
 * back to 0 after a reset) or jump while earlier calls are in flight: when this call would write a prediction-ring slot that the
 * previous call's smoothing window reads, its LSTM layers >= 1 wait for the previous call's stage 3.
 */
int ape_pipeline_submit(ape_pipeline* p, const float* rows_host, const float* rows_dev, int nF, int frame0,
                        const int32_t* stream_frames_host, int flags, void* caller_stream, int* slot);
int ape_pipeline_wait(ape_pipeline* p, int slot);              /* host-blocking: results of `slot` are in out_host[slot] */
int ape_pipeline_query(ape_pipeline* p, int slot, int* landed);/* non-blocking form */
int ape_pipeline_sync(ape_pipeline* p);                        /* host-blocking drain of all four streams */
int ape_pipeline_fence(ape_pipeline* p, void* stream);         /* later submits wait for what `stream` holds now */
/* The pipeline's CUDA streams (which: 0 side, 1 lane 0, 2 lane 1, 3 copy) as cudaStream_t, for a caller that orders its own work
   against one of them; the pipeline keeps owning them.  APE_ERR_BAD_ARG for a null pointer or another `which`. */
int ape_pipeline_stream(ape_pipeline* p, int which, void** stream);
/*
 * Per-stream skeletons for stage 3: every call submitted after this returns runs ape_fk_reduce_bodies on `bodies` ([B][body_stride]
 * float32 on the device, body_stride 0 or >= 9); a null `bodies` goes back to desc.body9.  The call does not synchronise and the
 * pipeline copies nothing: the caller must not overwrite a table that submitted calls may still read (ape_pipeline_sync first).
 * APE_ERR_BAD_ARG for a null p, a negative stride or a stride of 1 to 8.
 */
int ape_pipeline_set_bodies(ape_pipeline* p, const float* bodies, int body_stride);

/* ---- host self-check hooks (tests only; one row per call, never used by the product path) ------ */
/* The __host__ __device__ row math of the kernels, compiled for the host so a CPU-only box can pin it. */
int ape_selfcheck_philox(const uint32_t* ctr4, const uint32_t* key2, uint32_t* out4);
int ape_selfcheck_keep8(uint64_t seed, uint32_t stream, uint32_t frame, uint32_t sample, uint32_t gap,
                        uint32_t t, uint32_t group, float dropout_p, uint32_t* keep_bits);
/* The two-lane keep compare of the tensor-core and batched feed-forward kernels on n Philox output words: flags[i] has bit 15 set iff
 * the low 16-bit lane of words[i] is < keep_thr16 and bit 31 iff the high lane is (the other bits carry no meaning); keep_thr16 <= 65536
 * (65536: every lane kept). */
int ape_selfcheck_keep_flags(const uint32_t* words, int n, uint32_t keep_thr16, uint32_t* flags);
int ape_selfcheck_features(int kind, int layout, const float* row, double* xx, int* n_features);
int ape_selfcheck_row_pose(int target, const double* preds, const double* body9, int use_float, double* est, int* bad);
/* The per-step schedule of weight pieces of the H = 256 tensor-core kernel (csrc/ape_lstm_tcs.cu: walk_step) for an x-part of kgx
 * k-groups: entries [n][2] words; lets a CPU-only box check that every chunk's operands are covered exactly once, in an order
 * the ring can serve. */
int ape_selfcheck_tcs_schedule(int kgx, int first_step, uint32_t* entries, int max_entries, int* n_entries);
/* GPU self-test of the tcgen05 / TMEM plumbing: D[128*cta_group][N] (f32) = A * B^T with f16 operands packed in the
 * canonical K-major no-swizzle layout of csrc/ape_umma.cuh (a_packed: [cta][K/8][128][8], b_packed: [cta][K/8][N/cta][8]).
 * cta_group 1 | 2; + 16 routes the A operand through tensor memory (tcgen05.st, then the [a_tmem] form of tcgen05.mma). */
int ape_selftest_umma(const void* a_packed, const void* b_packed, float* d, int N, int K, int cta_group, void* stream);
/* Measured fp32 FMA peak (TFLOP/s) of the current device: best of `reps` launches of an unrolled register-only FFMA microkernel
 * (2 x sm_count CTAs x 1024 threads x iters x 128 FFMA).  scratch: >= 2 * sm_count floats on the device.  Synchronises `stream`.
 * bench.py's roofline denominator for the fp32 LSTM kernel (MEASURED_PEAKS.json has HBM and bf16 tensor figures only). */
int ape_selftest_ffma_peak(float* scratch, int iters, int reps, float* tflops, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* APE_B200_H */
