"""The batched per-frame estimation path: many streams x MC samples in one pass on one B200.

``BatchedEstimator`` is what the reference's per-stream loop (``estimator.py:155-178``: ``parse_row_to_xx`` ->
``add_xx_to_row_hist_and_make_prediction`` -> ``msg_from_pred``) becomes when B independent streams advance in
lockstep: one H2D copy of the raw rows ``[B, nF, 28|55]``, three kernel stages on one CUDA stream
(``ape_features`` -> ``ape_mc_lstm_*`` -> ``ape_fk_reduce``), one D2H copy of the 25-float messages (+ std, + per-sample
hand / elbow positions).  All history the reference keeps in Python lists (``_row_hist``, ``_smooth_hist``) lives in
device rings indexed by the absolute frame number; frames before 0 clamp to frame 0, which is the reference's
"repeat the first row / first prediction" warm-up.  Streams are independent, so a multi-GPU job is a static split
of the stream axis (``shard_streams``) with no collective.
"""
from dataclasses import dataclass

import ctypes
import os

import numpy as np
import torch

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200.data_types.bone_map import body_measurements_row
from arm_pose_estimation_b200.estimate import nn_models
from arm_pose_estimation_b200.utility.names import NNS_TARGETS

C_void = ctypes.c_void_p

TARGET_IDS = {
    NNS_TARGETS.ORI_CAL_LARM_UARM: N.TARGET_ORI_CAL_LARM_UARM,
    NNS_TARGETS.ORI_CAL_LARM_UARM_HIPS: N.TARGET_ORI_CAL_LARM_UARM_HIPS,
    NNS_TARGETS.ORI_POS_CAL_LARM_UARM_HIPS: N.TARGET_ORI_POS_CAL_LARM_UARM_HIPS,
}
EST_WIDTH = {N.TARGET_ORI_CAL_LARM_UARM: 14, N.TARGET_ORI_CAL_LARM_UARM_HIPS: 21, N.TARGET_ORI_POS_CAL_LARM_UARM_HIPS: 21}
KIND_FEATURES = {N.KIND_WATCH_ONLY: 20, N.KIND_POCKET: 22, N.KIND_UARM: 38}
LAYOUT_NCOLS = {N.LAYOUT_WATCH_ONLY: 28, N.LAYOUT_WATCH_PHONE: 55}


def shard_streams(n_streams, world_size, rank):
    """Static contiguous split of the stream axis: ``(first_stream, count)`` of ``rank`` (SURVEY.md §8e).
    The first ``n_streams % world_size`` ranks take one extra stream; no stream is shared, no exchange follows."""
    if world_size < 1 or not 0 <= rank < world_size or n_streams < 0:
        raise ValueError(f"bad shard request: n_streams={n_streams} world_size={world_size} rank={rank}")
    base, extra = divmod(n_streams, world_size)
    count = base + (1 if rank < extra else 0)
    first = rank * base + min(rank, extra)
    return first, count


def gather_host_results(local, first_stream, n_streams, group=None):
    """The only cross-rank step of a sharded job: rank 0 collects every rank's per-stream HOST results (a numpy array
    whose axis 0 is this rank's streams) into one array ordered by global stream id; other ranks get ``None``.
    Works on any ``torch.distributed`` backend (results are already on the host)."""
    import torch.distributed as dist
    local = np.ascontiguousarray(local)
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    parts = [None] * world if rank == 0 else None
    dist.gather_object((int(first_stream), local), parts, dst=0, group=group)
    if rank != 0:
        return None
    out = np.empty((n_streams,) + local.shape[1:], dtype=local.dtype)
    for first, arr in parts:
        out[first:first + len(arr)] = arr
    return out


def ring_slots(n_frames_per_call, history):
    """Slots a device ring needs so that one call of ``n_frames_per_call`` frames still finds the ``history - 1``
    frames before its first one (``history`` = sequence_len for features, smooth for predictions)."""
    return max(1, n_frames_per_call) + max(1, history) - 1


def pred_window_alias(f, nF, f1, nF1, smooth, ring):
    """Do frames ``f .. f + nF - 1`` of a stream share a slot of a prediction ring of ``ring`` frames with the smoothing windows of
    a call of ``nF1`` frames from frame ``f1`` (frames ``f1 - smooth + 1 .. f1 + nF1 - 1``, those before 0 read as frame 0)?
    Element-wise over arrays; the cross-call pipeline's ordering rule (csrc/ape_pipeline.cu has the same)."""
    f1 = np.asarray(f1, np.int64)
    lo = np.maximum(f1 - smooth + 1, 0)                   # oldest frame read
    o = (np.asarray(f, np.int64) - lo) % ring             # where the written frames start, counted from its slot
    return (o < f1 + nF1 - lo) | (o + nF > ring)


@dataclass
class EstimateBatch:
    """Results of one ``BatchedEstimator.step``; tensors live on the estimator's device until ``.host()``."""
    msg: torch.Tensor            # [B, nF, 25]   [larm_q, hand, larm_q, elbow, uarm_q, shoulder, hips_q] (compose_msg.py)
    std: torch.Tensor            # [B, nF, 6]    population std of the per-row hand / elbow positions
    samples: torch.Tensor        # [B, nF, S, 6] per-row hand xyz, elbow xyz (message tail of estimator.py:131-136) or None
    status: torch.Tensor         # [B, nF] int32, 1 = degenerate 6D output (the reference raises LinAlgError)
    frame0: int

    def host(self):
        f = lambda t: None if t is None else t.cpu().numpy()
        return EstimateBatch(f(self.msg), f(self.std), f(self.samples), f(self.status), self.frame0)


class PendingEstimate:
    """Handle of an enqueued ``BatchedEstimator.submit``: ``result()`` waits for its D2H copy and returns host arrays.
    ``event`` is the torch event of the copy, or ``None`` when the call went through the native pipeline (``ape_pipeline_wait``)."""

    def __init__(self, owner, slot, nF, frame0, event):
        self.owner, self.slot, self.nF, self.frame0, self.event = owner, slot, nF, frame0, event

    def done(self):
        if self.event is not None:
            return self.event.query()
        landed = ctypes.c_int(0)
        N.check(self.owner.lib.ape_pipeline_query(self.owner._pipe, self.slot, ctypes.byref(landed)), "ape_pipeline_query")
        return bool(landed.value)

    def result(self):
        if self.event is not None:
            self.event.synchronize()
        else:
            N.check(self.owner.lib.ape_pipeline_wait(self.owner._pipe, self.slot), "ape_pipeline_wait")
        msg, std, samples, status = self.owner._host_views(self.slot, self.nF)
        return EstimateBatch(msg, std, samples, status, self.frame0)


class _GraphCall:
    """State of the captured single-call graph (``BatchedEstimator.step_graph``): the graph, numpy views of its pinned staging
    block (frame counters + rows) and of its pinned result block."""


class BatchedEstimator:
    # largest call (streams x frames x MC samples) that runs on the cluster kernel (one 8-CTA cluster per 128 rows, csrc/ape_lstm_tcl.cu)
    SMALL_BATCH_ROWS = int(os.environ.get("APE_SMALL_BATCH_ROWS", "2048"))
    # largest call of an H = 256 model on the split-precision small-batch kernel (16-CTA clusters, csrc/ape_lstm_tcxsl.cu).  A B200 holds
    # 7 of its clusters at once, so calls above 896 rows run in waves; measured per single call (n = 128, B200 at 1000 W,
    # profiles/split_small256_bench.json) it still beats the split layer kernels at 3072 rows (pocket 0.334 / 0.349 ms, watch-only
    # 0.418 / 0.452) and loses at 4096 (0.408 / 0.352, 0.512 / 0.455): the crossover lies above SMALL_BATCH_ROWS, which stays the bound
    SPLIT256_SMALL_BATCH_ROWS = min(SMALL_BATCH_ROWS, 2048)
    N_SLOTS = int(os.environ.get("APE_N_SLOTS", "8"))      # staging / result buffer sets: up to N_SLOTS - 1 submitted calls may be outstanding while the next is staged
                     # (measured end to end, uarm 1024 x 100: 3 outstanding 0.413 ms/step, 5 outstanding 0.392, 7 outstanding 0.391)

    def __init__(self, kind, layout, state, seq_len, y_targets, stats, n_streams, mc_samples,
                 smooth=1, dropout=0.2, bonemap=None, frames_per_call=1, emit_samples=True, normalize=True,
                 mask_mode=N.MASK_PHILOX, philox_seed=0, first_stream=0, device=None,
                 lstm_variant="auto", tc_min_rows=1, tc_tolerance_m=5e-5, pipeline=True, lanes=True, tc_flags=None,
                 native_pipeline=None, small_batch_kernel=True, split_small_batch_kernel=False):
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedEstimator needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = N.load()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.kind, self.layout = int(kind), int(layout)
        self.I, self.H, self.L, self.O = nn_models.lstm_dims(state)
        if KIND_FEATURES[self.kind] != self.I:
            raise UserWarning(f"estimator kind {kind} produces {KIND_FEATURES[self.kind]} features, the model takes {self.I}")
        self.T, self.smooth, self.n = max(1, int(seq_len)), max(1, int(smooth)), int(mc_samples)
        self.S = self.smooth * self.n
        self.p = float(dropout)
        self.B, self.nF_max = int(n_streams), max(1, int(frames_per_call))
        self.target = TARGET_IDS[y_targets]
        if self.O != len(y_targets.value):
            raise UserWarning(f"model has {self.O} outputs, target set {y_targets.name} has {len(y_targets.value)}")
        self.mask_mode, self.philox_seed, self.first_stream = int(mask_mode), int(philox_seed), int(first_stream)
        self.emit_samples = bool(emit_samples)
        self.normalize = bool(normalize)
        # tensor-core path, H = 128, L >= 3: 0 = pairs of layers >= 1 as one wavefront launch when the batch fills the GPU,
        # 1 = always one launch per layer, 2 = always wavefront pairs (include/ape_b200.h: ape_lstm_args.tc_flags)
        self.tc_flags = int(os.environ.get("APE_TC_FLAGS", "0")) if tc_flags is None else int(tc_flags)     # (the variable: A/B runs of bench.py)
        self.reserve_sms = 0
        self.ncols = LAYOUT_NCOLS[self.layout]
        dev, f32 = self.device, torch.float32
        with torch.cuda.device(dev):
            self.weights = torch.from_numpy(nn_models.pack_lstm_weights(state)).to(dev)
            if normalize:
                self.xx_m = torch.as_tensor(np.asarray(stats["xx_m"], dtype=np.float64)).to(dev)
                self.xx_s = torch.as_tensor(np.asarray(stats["xx_s"], dtype=np.float64)).to(dev)
                self.yy_m = torch.as_tensor(np.asarray(stats["yy_m"], dtype=np.float32)).to(dev)
                self.yy_s = torch.as_tensor(np.asarray(stats["yy_s"], dtype=np.float32)).to(dev)
                self.yy_m_host, self.yy_s_host = np.asarray(stats["yy_m"], dtype=np.float64), np.asarray(stats["yy_s"], dtype=np.float64)
            else:
                self.xx_m = self.xx_s = self.yy_m = self.yy_s = None
            self.body = torch.as_tensor(body_measurements_row(bonemap).astype(np.float32).ravel()).to(dev)
            self.feat_ring = ring_slots(self.nF_max, self.T)
            # (two calls' worth of frames: with the two-lane pipeline the last layer of call k+1 may write its predictions
            # while stage 3 of call k still reads the smoothing window of call k)
            self.pred_ring = ring_slots(2 * self.nF_max, self.smooth)
            B, nF = self.B, self.nF_max
            self.raw = torch.zeros((B, nF, self.ncols), dtype=f32, device=dev)
            self.feats = torch.zeros((B, self.feat_ring, self.I), dtype=f32, device=dev)
            self.preds = torch.zeros((B, self.pred_ring, self.n, self.O), dtype=f32, device=dev)
            # results live in ONE device buffer [msg | std | status | samples] so a full call leaves in one D2H copy
            E = B * nF
            n_words = E * (25 + 6 + 1) + (E * self.S * 6 if emit_samples else 0)
            # (N_SLOTS of them: the D2H copy of call k runs on a side stream under the kernels of the calls after it)
            NS = self.N_SLOTS
            self.out_bufs = [torch.zeros(n_words, dtype=f32, device=dev) for _ in range(NS)]
            self.copy_stream = torch.cuda.Stream(device=dev)
            self.copy_done = [None] * NS
            self._use_out(0)
            # sized for the largest call; a shorter call re-tiles its rows, so leave one tile of slack per buffer
            ws_bytes = N.workspace_bytes(self.I, self.H, self.L, self.T, self.O, B * nF, self.n) + 3 * 64 * self.T * self.H * 4
            self.workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            # pinned staging for the host-facing calls: N_SLOTS slots, so the next calls can be staged and enqueued while the
            # results of call k are still on their way back (submit() / PendingEstimate.result())
            self.raw_host = [torch.zeros((B, nF, self.ncols), dtype=f32).pin_memory() for _ in range(NS)]
            self.out_host = [torch.zeros(n_words, dtype=f32).pin_memory() for _ in range(NS)]
            self.slot_event = [None] * NS
            self._g, self._g_stale = None, False           # captured single-call graph; stale: other calls were enqueued since its last replay
            self.frames_host = self.frames_dev = None      # per-stream frame counters (multi-stream front-end), made on first use
            self.submits = 0
            # ---- which LSTM kernel: fp32 FFMA (exact) or tcgen05 fp16-operand tensor cores ----------------------
            # Tensor cores when the fp16-operand result stays within tc_tolerance_m of the fp32 kernel on a probe batch of
            # THIS model's weights (and the batch has at least tc_min_rows rows: the measured crossover against the fp32
            # kernel is below one row - profiles/r1_crossover.md - so the default does not restrict).
            # "tcx" = the split-precision tensor-core kernels (csrc/ape_lstm_tcx.cu, H = 128; csrc/ape_lstm_tcxs.cu, H = 256): fp16 pairs
            # hi + lo, three passes per product, ex2 / rcp cell update - what "auto" takes when the single-pass probe fails, before it
            # falls back to the fp32 kernel.
            self.tc_weights = self.tcx_weights = None
            self.tc_probe_error_m = self.tcx_probe_error_m = None
            self.tc_split = False
            self.lstm_variant = "fp32"
            if lstm_variant not in ("auto", "fp32", "tc", "tcx"):
                raise UserWarning(f"lstm_variant must be 'auto', 'fp32', 'tc' or 'tcx', got {lstm_variant!r}")
            tc_ok = N.tc_supported(self.I, self.H, self.L, self.O) and self.T <= 40
            tcx_ok = N.split_supported(self.I, self.H, self.L, self.O) and self.T <= 40
            if lstm_variant == "tc" and not tc_ok:
                raise UserWarning(f"the tensor-core LSTM kernel does not support H={self.H}, L={self.L}")
            if lstm_variant == "tcx" and not tcx_ok:
                raise UserWarning(f"the split-precision tensor-core LSTM kernel does not support H={self.H}, L={self.L}, O={self.O}")
            if lstm_variant == "tc" or (lstm_variant == "auto" and tc_ok and B * nF * self.n >= tc_min_rows):
                self.tc_weights = torch.from_numpy(nn_models.pack_lstm_weights_tc(state)).to(dev)
                assert self.tc_weights.numel() == N.tc_blob_bytes(self.I, self.H, self.L)
                ws_tc = N.workspace_bytes(self.I, self.H, self.L, self.T, self.O, B * nF, self.n, tensor_core=True) + 3 * 256 * self.T * self.H * 4
                ws_tc += (2 + 2 * self.T) * (self.H // 8) * 2048 + 512          # (the small-batch kernel's exchange buffer and layer sequences)
                if ws_tc > self.workspace.numel():
                    self.workspace = torch.empty(ws_tc, dtype=torch.uint8, device=dev)
                self.tc_probe_error_m = self._probe_tc_error()
                if lstm_variant == "tc" or self.tc_probe_error_m <= tc_tolerance_m:
                    self.lstm_variant = "tc"
            if lstm_variant == "tcx" or (lstm_variant == "auto" and self.lstm_variant != "tc" and tcx_ok and B * nF * self.n >= tc_min_rows):
                self.tcx_weights = torch.from_numpy(nn_models.pack_lstm_weights_tcx(state)).to(dev)
                assert self.tcx_weights.numel() == N.split_blob_bytes(self.I, self.H, self.L)
                self.tcx_probe_error_m = self._probe_tc_error("tcx")
                if lstm_variant == "tcx" or self.tcx_probe_error_m <= tc_tolerance_m:
                    self.lstm_variant, self.tc_split, self.tc_flags = "tc", True, 3
                    ws_x = N.split_workspace_bytes(self.I, self.H, self.L, self.T, self.O, B * nF, self.n) + 1024
                    if ws_x > self.workspace.numel():
                        self.workspace = torch.empty(ws_x, dtype=torch.uint8, device=dev)
            # A call of <= 128 rows (one stream x 100 MC samples: the real-time case) can run ALL layers in one launch of one 8-CTA cluster
            # with the hidden units split across it (csrc/ape_lstm_tcl.cu) instead of one CTA pair walking every gate column of every
            # layer; a larger call takes one cluster per 128 rows in the same launch.  Up to 16 clusters (what a B200 holds at once: two per
            # GPC) the call costs what one cluster costs - measured per call, pocket model x 100 MC samples: 1 .. 16 streams 0.10 ms against
            # 0.19 ms on the layer kernels, 32 streams 0.16 against 0.19, 64 streams 0.27 against 0.19 (tools/tcl_crossover.py).  Same operand rounding, accumulation order and Philox keys as the layer kernels: results are bit-identical
            # (tests/test_gpu_tcl.py), so it is simply what such an estimator runs (small_batch_kernel=False: the layer kernels).
            self.small_batch = (bool(small_batch_kernel) and self.lstm_variant == "tc" and not self.tc_split and self.tc_flags == 0
                                and self.L <= 4 and self.H in (128, 256) and self.T <= 40 and B * nF * self.n <= self.SMALL_BATCH_ROWS)
            if self.small_batch:
                self.tc_flags = 4
            # The same for a model on the split-precision kernels (tc_flags = 5; H = 128: csrc/ape_lstm_tcxl.cu, H = 256:
            # csrc/ape_lstm_tcxsl.cu, its own entry point, on a device that holds one of its 16-CTA clusters): the layer kernels'
            # arithmetic and MMA order per accumulator, so the results are bit-identical to them (tests/test_gpu_tcxl.py,
            # tests/test_gpu_tcxsl.py).  Off by default; the single-stream estimator classes (estimator.py) turn it on.
            if (split_small_batch_kernel and self.tc_split and self.L <= 4 and self.T <= 40
                    and ((self.H == 128 and B * nF * self.n <= self.SMALL_BATCH_ROWS)
                         or (self.H == 256 and B * nF * self.n <= self.SPLIT256_SMALL_BATCH_ROWS and self._tcxsl_available()))):
                self.small_batch, self.tc_flags = True, 5
                ws_fn = N.tcxl_workspace_bytes if self.H == 128 else N.tcxsl_workspace_bytes
                ws_xl = ws_fn(self.I, self.H, self.L, self.T, self.O, B * nF, self.n)
                if ws_xl > self.workspace.numel():
                    self.workspace = torch.empty(ws_xl, dtype=torch.uint8, device=dev)
            # cross-call software pipeline (tensor-core path), two levels:
            #  * stage 1 + LSTM layer 0 of call k+1 (a few dozen CTAs) run on a side stream under call k's big layer kernels;
            #    layer 0's output is double-buffered by call parity;
            #  * the big layer kernels (persistent, one CTA pair per SM pair, a whole number of 256-row tiles per pair) and stage 3
            #    of consecutive calls go to two alternating "lane" streams with a workspace each: a layer's last round of tiles
            #    fills only part of the GPU (400 tiles over 74 pairs = 5.4 rounds), and the pairs that finish early pick up the
            #    next call's layer instead of idling until the launch drains.  At most two calls are in flight.
            self.pipeline = bool(pipeline) and self.lstm_variant == "tc" and not self.small_batch      # (one launch: nothing to overlap)
            # With the pipeline the persistent launches of the layers >= 1 leave ONE SM pair free for the side stream: stage 1 + layer 0
            # of the next calls (<= 8 CTAs) otherwise only get SMs in the ~50 us in which a big launch retires its CTAs, and a call
            # whose layer 0 misses that window stalls its lane.  Measured (uarm 1024 x 100, B200): 0 -> 2 reserved SMs: device-resident
            # 3.445M -> 3.498M est/s, end to end (H2D of the rows in front of stage 1) 3.206M -> 3.483M; 4 reserved SMs: the same.
            if self.pipeline:
                self.reserve_sms = int(os.environ.get("APE_RESERVE_SMS", "2"))
            # (high priority: its few dozen CTAs take the first SMs any big launch frees, so layer 0 is ready well before its call's turn)
            self.side_stream = torch.cuda.Stream(device=dev, priority=-1) if self.pipeline else None
            self.lanes = bool(lanes) and self.pipeline
            self.lane_streams = [torch.cuda.Stream(device=dev) for _ in range(2)] if self.lanes else None
            self.lane_ws = [self.workspace, torch.empty_like(self.workspace)] if self.lanes else None
            self.l1_done = [None] * 4             # completion of the last call that used buffer set (call & 3)
            self.lstm_done = None             # last LSTM layer of the previous call (its predictions feed this call's smoothing window)
            self._prev_call = None            # (stage-3 event, frames, nF) of the previous pipelined call: frame0, host counters or None
            # The same pipeline as ONE C call per batch (csrc/ape_pipeline.cu: ape_pipeline_submit): used for every call that needs
            # nothing call-specific from Python (no injected masks, no profiling / trace leg, no caller-owned frame counters).  The
            # Python-level pipeline below remains for those, and as the A/B switch (native_pipeline=False | APE_NATIVE_PIPELINE=0).
            if native_pipeline is None:
                native_pipeline = os.environ.get("APE_NATIVE_PIPELINE", "1") != "0"
            self._pipe = None
            self._pipe_busy = False
            self._py_dirty = False            # a Python-path call has run since the native pipeline last drained
            self._launch_cache = {}
            if native_pipeline and self.lanes and self.mask_mode != N.MASK_INJECTED and normalize:
                self._make_native_pipeline()
        self.calls = 0
        self.frame = 0
        self.launches = 0             # kernels launched so far (bench.py reports it)

    def _make_native_pipeline(self):
        d = N.PipelineDesc()
        d.layout, d.kind, d.normalize, d.ncols = self.layout, self.kind, 1 if self.normalize else 0, self.ncols
        d.xx_m, d.xx_s = self.xx_m.data_ptr(), self.xx_s.data_ptr()
        d.raw, d.feats, d.feat_ring = self.raw.data_ptr(), self.feats.data_ptr(), self.feat_ring
        d.lstm = self._lstm_args(self.nF_max, 0, None, None)[0]
        d.lane_workspace[0], d.lane_workspace[1] = self.lane_ws[0].data_ptr(), self.lane_ws[1].data_ptr()
        d.yy_m, d.yy_s, d.body9 = self.yy_m.data_ptr(), self.yy_s.data_ptr(), self.body.data_ptr()
        d.target, d.smooth, d.emit_samples = self.target, self.smooth, 1 if self.emit_samples else 0
        d.B, d.nF_max, d.n_slots = self.B, self.nF_max, self.N_SLOTS
        self.frames_host = [torch.zeros(self.B, dtype=torch.int32).pin_memory() for _ in range(self.N_SLOTS)]
        self.frames_dev = [torch.zeros(self.B, dtype=torch.int32, device=self.device) for _ in range(4)]
        for k in range(self.N_SLOTS):
            d.out_dev[k], d.raw_host[k], d.out_host[k] = self.out_bufs[k].data_ptr(), self.raw_host[k].data_ptr(), self.out_host[k].data_ptr()
            d.frames_host[k] = self.frames_host[k].data_ptr()
        for k in range(4):
            d.frames_dev[k] = self.frames_dev[k].data_ptr()
        handle = ctypes.c_void_p(None)
        N.check(self.lib.ape_pipeline_create(ctypes.byref(d), ctypes.byref(handle)), "ape_pipeline_create")
        self._pipe, self._pipe_desc = handle, d

    def __del__(self):
        pipe, self._pipe = getattr(self, "_pipe", None), None
        if pipe is not None:
            try:
                self.lib.ape_pipeline_destroy(pipe)
            except Exception:                        # interpreter shutdown: the library may already be gone
                pass

    def _native_call(self, rows_host, rows_dev, nF, sf_host, flags):
        """One ``ape_pipeline_submit``; returns (slot, frame0)."""
        if self._py_dirty:                           # buffers were last touched by the Python-level path: let it finish first
            torch.cuda.current_stream().synchronize()
            self.copy_stream.synchronize()
            self._py_dirty = False
        self._pipe_busy = True
        slot = ctypes.c_int(-1)
        N.check(self.lib.ape_pipeline_submit(self._pipe, rows_host, rows_dev, nF, self.frame, sf_host, flags,
                                             N.current_stream_ptr(), ctypes.byref(slot)), "ape_pipeline_submit")
        if nF not in self._launch_cache:
            self._launch_cache[nF] = 2 + self._lstm_launches(self._lstm_args(nF, 0, None, None)[0])
        self.launches += self._launch_cache[nF]
        frame0 = self.frame
        self.frame += nF
        self.calls += 1
        self.submits += 1
        return slot.value, frame0

    def _leave_native(self):
        """Before a Python-path call on an estimator that owns a native pipeline: drain the pipeline's streams."""
        if self._pipe is not None:
            if self._pipe_busy:
                N.check(self.lib.ape_pipeline_sync(self._pipe), "ape_pipeline_sync")
                self._pipe_busy = False
            self._py_dirty = True

    @staticmethod
    def _tcxsl_available():
        """Can the current device run the H = 256 split-precision small-batch kernel (at least one of its 16-CTA clusters at once)?
        A failed availability query counts as "no": the estimator then stays on the split layer kernels, which need no cluster of 16."""
        try:
            return N.tcxsl_max_active_clusters() >= 1
        except UserWarning:
            return False

    def _lstm_fn(self, variant=None):
        if variant is None and self.tc_flags == 5 and self.H == 256:
            return self.lib.ape_mc_lstm_tcxsl                  # the H = 256 split-precision small-batch kernel has its own entry point
        return self.lib.ape_mc_lstm_tc if (variant or self.lstm_variant) in ("tc", "tcx") else self.lib.ape_mc_lstm_fma

    def _lstm_launches(self, a):
        """Kernels the LSTM stage launches for the argument block ``a`` (pairs of layers of an H = 128 model count once)."""
        if self.lstm_variant != "tc":
            return self.L
        a.layer_begin = a.layer_end = 0
        n = ctypes.c_int(0)
        N.check(self.lib.ape_mc_lstm_tc_launch_count(a, ctypes.byref(n)), "ape_mc_lstm_tc_launch_count")
        return n.value

    def _probe_tc_error(self, which="tc", n_est=16, n_samples=64):
        """Max |position| difference (metres) between a tensor-core LSTM kernel (``which``: "tc" single pass | "tcx" split precision)
        and the fp32 kernel on a probe batch: N(0,1) normalised windows, the same Philox masks for both (the keying does not depend
        on the kernel)."""
        dev = self.device
        g = torch.Generator(device="cpu").manual_seed(1234)
        x = torch.randn((n_est, self.T, self.I), generator=g, dtype=torch.float32).to(dev)
        ws = torch.empty(max(N.workspace_bytes(self.I, self.H, self.L, self.T, self.O, n_est, n_samples),
                             N.split_workspace_bytes(self.I, self.H, self.L, self.T, self.O, n_est, n_samples) if which == "tcx" else
                             N.workspace_bytes(self.I, self.H, self.L, self.T, self.O, n_est, n_samples, tensor_core=True)),
                         dtype=torch.uint8, device=dev)
        outs = []
        for variant in ("fp32", which):
            preds = torch.zeros((n_est, 1, n_samples, self.O), dtype=torch.float32, device=dev)
            a = N.LstmArgs()
            a.weights = self.weights.data_ptr()
            a.weights_tc = None if self.tc_weights is None else self.tc_weights.data_ptr()
            if variant == "tcx":
                a.weights_tcx, a.tc_flags = self.tcx_weights.data_ptr(), 3
            a.I, a.H, a.L, a.T, a.O = self.I, self.H, self.L, self.T, self.O
            a.dropout_p = self.p
            a.x_dense, a.feat_ring_buf, a.feat_ring = x.data_ptr(), None, 0
            a.B, a.nF, a.frame0, a.n_samples = n_est, 1, 0, n_samples
            a.mask_mode, a.philox_seed, a.stream_id0 = N.MASK_PHILOX, 0x5EED, 0
            a.workspace = ws.data_ptr()
            a.preds, a.pred_ring, a.all_steps = preds.data_ptr(), 1, 0
            N.check(self._lstm_fn(variant)(a, N.current_stream_ptr()), f"ape_mc_lstm ({variant} probe)")
            est = torch.empty((n_est, n_samples, EST_WIDTH[self.target]), dtype=torch.float32, device=dev)
            msg = torch.empty((n_est, 25), dtype=torch.float32, device=dev)
            N.check(self.lib.ape_fk_reduce(N.ptr(preds), 1, N.ptr(self.yy_m), N.ptr(self.yy_s), N.ptr(self.body), self.target,
                                           self.O, n_est, 1, 0, None, n_samples, 1, N.ptr(msg), None, None, N.ptr(est), None,
                                           N.current_stream_ptr()), "ape_fk_reduce (probe)")
            outs.append(est[..., :9 if EST_WIDTH[self.target] == 21 else 6].clone())
        torch.cuda.current_stream().synchronize()
        return float((outs[0] - outs[1]).abs().max().item())

    def _use_out(self, k):
        """Point the result views at device output buffer ``k``."""
        B, nF, E = self.B, self.nF_max, self.B * self.nF_max
        self.out_slot, self.out_all = k, self.out_bufs[k]
        self.msg = self.out_all[: E * 25].view(B, nF, 25)
        self.std = self.out_all[E * 25: E * 31].view(B, nF, 6)
        self.status = self.out_all[E * 31: E * 32].view(torch.int32).view(B, nF)
        self.samples = self.out_all[E * 32:].view(B, nF, self.S, 6) if self.emit_samples else None

    def _use_out_mapped(self, host):
        """Point the result views at a PINNED HOST block of the same layout (zero-copy results of the CUDA-graph path: pinned memory
        is mapped into the device's address space under unified addressing, the kernels take its address like a device pointer)."""
        B, nF, E = self.B, self.nF_max, self.B * self.nF_max
        self.msg = host[: E * 25].view(B, nF, 25)
        self.std = host[E * 25: E * 31].view(B, nF, 6)
        self.status = host[E * 31: E * 32].view(torch.int32).view(B, nF)
        self.samples = host[E * 32:].view(B, nF, self.S, 6) if self.emit_samples else None

    def reset(self):
        """Forget all history, like ``Estimator.reset`` (estimator.py:88-91): the next row is frame 0 again."""
        self.frame = 0

    # ---- device path -----------------------------------------------------------------------------------
    def _lstm_args(self, nF, frame0, sf, masks):
        """The stage-2 argument block of one call over the feature ring (and the device copy of injected masks, kept alive
        by the caller until the launch is enqueued)."""
        B = self.B
        a = N.LstmArgs()
        a.weights = self.weights.data_ptr()
        a.I, a.H, a.L, a.T, a.O = self.I, self.H, self.L, self.T, self.O
        a.dropout_p = self.p
        a.x_dense, a.feat_ring_buf, a.feat_ring = None, self.feats.data_ptr(), self.feat_ring
        a.B, a.nF, a.frame0, a.n_samples = B, nF, frame0, self.n
        a.stream_frames = None if sf is None else sf.data_ptr()
        a.mask_mode = self.mask_mode if self.L > 1 else N.MASK_NONE
        md = None
        if a.mask_mode == N.MASK_INJECTED:
            if masks is None:
                raise UserWarning("mask_mode is MASK_INJECTED: pass masks [B, nF, L-1, T, n, H] uint8")
            md = torch.as_tensor(masks).to(device=self.device, dtype=torch.uint8).contiguous()
            if md.numel() != B * nF * (self.L - 1) * self.T * self.n * self.H:
                raise UserWarning("masks must be [B, nF, L-1, T, n, H]")
            a.masks = md.data_ptr()
        a.philox_seed, a.stream_id0 = self.philox_seed, self.first_stream
        a.workspace = self.workspace.data_ptr()
        a.preds, a.pred_ring, a.all_steps = self.preds.data_ptr(), self.pred_ring, 0
        a.weights_tc = None if self.tc_weights is None else self.tc_weights.data_ptr()
        # the workspace is laid out for the largest call, so short calls in flight beside full ones agree on every offset
        a.ws_E, a.tc_flags = B * self.nF_max, self.tc_flags
        a.reserve_sms = self.reserve_sms
        a.weights_tcx = None if self.tcx_weights is None else self.tcx_weights.data_ptr()
        return a, md

    # ---- the reference's three per-frame calls, one by one (estimator.py:174-176) ------------------------------------
    def step_features(self, xx, masks=None):
        """``add_xx_to_row_hist_and_make_prediction`` for all streams: ``xx [B, I]`` float64 rows as ``parse_row_to_xx`` returned
        them -> z-score -> feature ring -> MC-dropout LSTM -> prediction ring; returns the de-normalised predictions of the
        smoothing window ``[B, smooth * n, O]`` (oldest frame first, frames before 0 read as frame 0: the reference's
        ``_row_hist`` / ``_smooth_hist`` lists are the two device rings).  Advances the frame counter."""
        xx = np.ascontiguousarray(xx, dtype=np.float64).reshape(self.B, self.I)
        with torch.cuda.device(self.device):
            st = N.current_stream_ptr()
            xd = torch.from_numpy(xx).to(self.device)
            N.check(self.lib.ape_features_push(N.ptr(xd), self.I, N.ptr(self.xx_m), N.ptr(self.xx_s), 1 if self.normalize else 0,
                                               N.ptr(self.feats), self.B, self.frame, None, self.feat_ring, st), "ape_features_push")
            a, md = self._lstm_args(1, self.frame, None, masks)
            N.check(self._lstm_fn()(a, st), "ape_mc_lstm")
            slots = [max(0, k) % self.pred_ring for k in range(self.frame - self.smooth + 1, self.frame + 1)]
            window = self.preds[:, slots].cpu().numpy().astype(np.float64)          # [B, smooth, n, O]
        if self.normalize:
            window = window * self.yy_s_host + self.yy_m_host                       # estimator.py:108-109
        self.launches += 1 + self._lstm_launches(a)
        self.calls += 1
        self.frame += 1
        return window.reshape(self.B, self.S, self.O)

    def step_device(self, raw, *args, **kwargs):
        """See ``_step_device``; runs it with the estimator's device current (kernels, streams and events all belong to it)."""
        with torch.cuda.device(self.device):
            return self._step_device(raw, *args, **kwargs)

    def _step_device(self, raw, n_frames=None, masks=None, layer_ms=None, trace=None, trace_layer=1, raw_ready=False,
                     _h2d_from=None, stream_frames=None, _frames_from=None, _out_slot=None, timeline=None, _plain=False):
        """``raw``: device tensor ``[B, nF, ncols]`` float32 (nF <= frames_per_call).  Enqueues the three stages and returns an
        ``EstimateBatch`` of views into the estimator's device buffers (valid until the call after next).  ``raw_ready=True``
        promises that ``raw`` is already materialised (not pending on the current stream), which lets the pipelined path
        start stage 1 + layer 0 of this call under the previous call's kernels.  ``stream_frames``: optional device int32
        tensor ``[B]`` of per-stream absolute frame numbers for streams that do not advance in lock-step (a negative entry
        skips the stream in this call: its rings and outputs stay untouched); the shared frame counter is then not used.
        With the lanes, a call whose frames go back (a restarted stream, ``reset()`` with calls in flight) or jump orders its LSTM
        layers >= 1 behind the previous call's stage 3, which may still read the prediction slots this call writes; counters that
        exist only on the device (``stream_frames`` without a host copy) cannot be inspected without a sync, so such a call is
        always ordered so."""
        nF = int(raw.shape[1]) if n_frames is None else int(n_frames)
        self._g_stale = self._g_stale or not _plain
        if raw.shape[0] != self.B or nF > self.nF_max or raw.shape[2] != self.ncols or not raw.is_contiguous():
            raise UserWarning(f"raw rows must be a contiguous [B={self.B}, nF<={self.nF_max}, {self.ncols}] tensor, got {tuple(raw.shape)}")
        if raw.dtype != torch.float32:
            raise UserWarning("raw rows must be float32 (the wire format, messaging.py)")
        lib, B = self.lib, self.B
        if (self._pipe is not None and masks is None and layer_ms is None and trace is None and timeline is None and not _plain
                and _h2d_from is None and stream_frames is None):
            flags = N.PIPE_CALLER_WAITS | (0 if raw_ready else N.PIPE_INPUT_PENDING)
            slot, frame0 = self._native_call(None, C_void(raw.data_ptr()), nF, None, flags)
            self._use_out(slot)
            return EstimateBatch(self._view(self.msg, nF), self._view(self.std, nF), self._view(self.samples, nF),
                                 self._view(self.status, nF), frame0)
        self._leave_native()
        main = torch.cuda.current_stream()
        frame0, sf = (self.frame, None) if stream_frames is None else (0, stream_frames)
        if sf is not None and (sf.dtype != torch.int32 or sf.numel() != B or not sf.is_cuda):
            raise UserWarning("stream_frames must be a device int32 tensor of B entries")
        a, md = self._lstm_args(nF, frame0, sf, masks)
        if layer_ms is not None:                     # profiling leg: float32 host array of L entries, filled on return
            a.layer_ms = layer_ms.ctypes.data
        if trace is not None:                        # debugging: device int64[768] of SM-clock stamps (tensor-core path)
            a.trace, a.trace_layer = trace.data_ptr(), trace_layer
        if timeline is not None:                     # debugging: device int64[L, 160, 4] CTA timeline (does not leave the pipelined path)
            a.trace, a.trace_layer = timeline.data_ptr(), -1

        def features(stream_ptr):
            N.check(lib.ape_features(N.ptr(raw), self.layout, self.kind, N.ptr(self.xx_m), N.ptr(self.xx_s),
                                     1 if self.normalize else 0, N.ptr(self.feats), B, nF, frame0, N.ptr(sf), self.feat_ring, stream_ptr),
                    "ape_features")

        def stage3(stream_ptr):
            N.check(lib.ape_fk_reduce(N.ptr(self.preds), self.pred_ring, N.ptr(self.yy_m), N.ptr(self.yy_s), N.ptr(self.body),
                                      self.target, self.O, B, nF, frame0, N.ptr(sf), self.n, self.smooth,
                                      N.ptr(self.msg), N.ptr(self.samples), N.ptr(self.std), None, N.ptr(self.status), stream_ptr),
                    "ape_fk_reduce")

        if self.pipeline and self._pipe is None and layer_ms is None and trace is None and not _plain:
            # buffer set of this call: lane (stream + workspace) = call & 1; with lanes each workspace's two copies of layer 0's
            # output alternate as well, so stage 1 + layer 0 may run up to three calls ahead of the big kernels (whichever
            # launch's tail has room for their few dozen CTAs) and never gate the next call's first big layer
            side, parity = self.side_stream, self.calls & 1
            bufset = self.calls & 3 if self.lanes else parity
            lane = self.lane_streams[parity] if self.lanes else main      # (lanes off: the big kernels stay on the caller's stream)
            if self.lanes:
                a.workspace = self.lane_ws[parity].data_ptr()
            if _out_slot is None:
                self._use_out(self.calls % self.N_SLOTS)     # results of call k stay valid while the next calls are computed
            # inputs the caller may still have pending on its own stream (everything but the staged host-facing path)
            if (not raw_ready and _h2d_from is None) or md is not None or (sf is not None and _frames_from is None):
                ev_in = torch.cuda.Event()
                ev_in.record(main)
                side.wait_event(ev_in)
                if self.lanes:
                    lane.wait_event(ev_in)
                if md is not None and self.lanes:
                    md.record_stream(lane)           # (allocated on the caller's stream, read by the lane's kernels)
            if self.l1_done[bufset] is not None:
                side.wait_event(self.l1_done[bufset])    # the last call on this buffer set (layer 0's output, frames) has finished
            with torch.cuda.stream(side):
                if _h2d_from is not None:
                    raw.copy_(_h2d_from, non_blocking=True)
                if _frames_from is not None:
                    sf.copy_(_frames_from, non_blocking=True)
                sp = C_void(side.cuda_stream)
                features(sp)
                a.layer_begin, a.layer_end, a.ws_parity = 0, 1, (bufset >> 1) if self.lanes else parity
                N.check(lib.ape_mc_lstm_tc(a, sp), "ape_mc_lstm_tc (layer 0)")
                ev0 = torch.cuda.Event()
                ev0.record(side)
            lane.wait_event(ev0)
            if self.copy_done[self.out_slot] is not None:
                lane.wait_event(self.copy_done[self.out_slot])   # this output buffer has been read back (submit(), call k-2)
            frames = frame0 if sf is None else (None if _frames_from is None else _frames_from.numpy().copy())
            if self.lanes and self._prev_call is not None and self._writes_prev_window(frames, nF):
                lane.wait_event(self._prev_call[0])      # the previous call's stage 3 (the other lane) has read its window
            with torch.cuda.stream(lane):
                lp = C_void(lane.cuda_stream)
                a.layer_begin, a.layer_end = 1, self.L
                N.check(lib.ape_mc_lstm_tc(a, lp), "ape_mc_lstm_tc (layers >= 1)")
                if self.lstm_done is not None:
                    lane.wait_event(self.lstm_done)      # the smoothing window reaches into the previous call's predictions
                self.lstm_done = torch.cuda.Event()
                self.lstm_done.record(lane)
                stage3(lp)
                done = torch.cuda.Event()
                done.record(lane)
            self.l1_done[bufset] = done
            self._prev_call = (done, frames, nF)
            if self.lanes:
                main.wait_event(done)                    # the caller's stream sees the results, as without the lanes
        else:
            if _h2d_from is not None:
                raw.copy_(_h2d_from, non_blocking=True)
            if _frames_from is not None:
                sf.copy_(_frames_from, non_blocking=True)
            st = N.current_stream_ptr()
            features(st)
            N.check(self._lstm_fn()(a, st), "ape_mc_lstm")
            stage3(st)
        self.launches += 2 + self._lstm_launches(a)
        self.calls += 1
        out = EstimateBatch(self._view(self.msg, nF), self._view(self.std, nF), self._view(self.samples, nF),
                            self._view(self.status, nF), self.frame)
        self.frame += nF
        return out

    def _writes_prev_window(self, frames, nF):
        """Would a call of ``nF`` frames from ``frames`` (the shared frame0, host counters [B], or None: device counters only) write a
        prediction slot that the previous pipelined call's smoothing window reads?  A change of counter mode counts as yes."""
        _, prev, prev_nF = self._prev_call
        if frames is None or prev is None or isinstance(frames, int) != isinstance(prev, int):
            return True
        if isinstance(frames, int):
            return bool(pred_window_alias(frames, nF, prev, prev_nF, self.smooth, self.pred_ring))
        both = (frames >= 0) & (prev >= 0)                # a stream the previous call skipped has no window there
        return bool(pred_window_alias(frames[both], nF, prev[both], prev_nF, self.smooth, self.pred_ring).any())

    def _view(self, buf, nF):
        """The kernels pack a call's E = B * nF estimates densely: view the front of a [B, nF_max, ...] buffer."""
        if buf is None:
            return None
        tail = tuple(buf.shape[2:])
        return buf.reshape(-1)[: self.B * nF * int(np.prod(tail, dtype=np.int64))].view(self.B, nF, *tail)

    # ---- host-facing path: pinned H2D, the three stages, pinned D2H ------------------------------------------
    def submit(self, rows, masks=None, stream_frames=None):
        """Stage ``rows`` (host array ``[B, nF, ncols]`` or ``[B, ncols]`` of float32 wire rows) in pinned memory and
        enqueue H2D copy -> the three stages -> D2H copy on the current stream WITHOUT waiting.  Returns a
        ``PendingEstimate``; a slot is reused after ``N_SLOTS`` calls (the call then first waits for that slot's results to land).  ``stream_frames``: optional host int32
        array ``[B]`` of per-stream frame numbers (negative: the stream has no new row in this call), see ``step_device``."""
        rows = np.asarray(rows, dtype=np.float32)
        if rows.ndim == 2:
            rows = rows[:, None, :]
        nF = rows.shape[1]
        if rows.shape[0] != self.B or nF > self.nF_max or rows.shape[2] != self.ncols:
            raise UserWarning(f"rows must be [B={self.B}, nF<={self.nF_max}, {self.ncols}], got {rows.shape}")
        self._g_stale = True
        if self._pipe is not None and masks is None:
            rows = np.ascontiguousarray(rows)
            sf = None if stream_frames is None else np.ascontiguousarray(np.asarray(stream_frames, dtype=np.int32).reshape(self.B))
            with torch.cuda.device(self.device):
                slot, frame0 = self._native_call(C_void(rows.ctypes.data), None, nF, None if sf is None else C_void(sf.ctypes.data),
                                                 N.PIPE_D2H)
            return PendingEstimate(self, slot, nF, frame0, None)
        self._leave_native()
        slot = self.submits % self.N_SLOTS
        self.submits += 1
        if self.slot_event[slot] is not None:
            self.slot_event[slot].synchronize()           # the slot's previous results have landed; its staging is free
        with torch.cuda.device(self.device):
            E = self.B * nF
            stage = self.raw_host[slot].view(-1)[: E * self.ncols].view(self.B, nF, self.ncols)
            stage.numpy()[...] = rows
            raw = self.raw.view(-1)[: E * self.ncols].view(self.B, nF, self.ncols)
            main = torch.cuda.current_stream()
            self._use_out(slot)
            if self.copy_done[slot] is not None:
                main.wait_event(self.copy_done[slot])     # device buffer `slot` has been read back (call k-2)
            sf_dev = sf_host = None
            if stream_frames is not None:
                if self.frames_host is None:
                    self.frames_host = [torch.zeros(self.B, dtype=torch.int32).pin_memory() for _ in range(self.N_SLOTS)]
                    self.frames_dev = [torch.zeros(self.B, dtype=torch.int32, device=self.device) for _ in range(4)]
                sf_host, sf_dev = self.frames_host[slot], self.frames_dev[self.calls & 3]     # (device copies: one per buffer set)
                sf_host.numpy()[...] = np.asarray(stream_frames, dtype=np.int32).reshape(self.B)
            out = self.step_device(raw, nF, masks, _h2d_from=stage, stream_frames=sf_dev, _frames_from=sf_host, _out_slot=slot)
            computed = torch.cuda.Event()
            computed.record(main)
            host, dev_out = self.out_host[slot], self.out_all
            self.copy_stream.wait_event(computed)
            with torch.cuda.stream(self.copy_stream):
                if nF == self.nF_max:
                    host.copy_(dev_out, non_blocking=True)
                else:                                    # short call: the kernels packed E estimates at the front of each part
                    Em = self.B * self.nF_max
                    for off, width in ((0, 25), (Em * 25, 6), (Em * 31, 1)) + (((Em * 32, self.S * 6),) if self.emit_samples else ()):
                        host[off: off + E * width].copy_(dev_out[off: off + E * width], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self.copy_stream)
            self.slot_event[slot] = ev
            self.copy_done[slot] = ev
        return PendingEstimate(self, slot, nF, out.frame0, ev)

    # ---- single-call latency path: the whole call as one captured CUDA graph ------------------------------------
    def step_graph(self, rows, stream_frames=None):
        """``step`` for the latency-bound case (a few streams, one call at a time - BASELINE configs[1]): the whole call is captured
        ONCE as a CUDA graph and replayed with one launch per frame.  The graph has four nodes: ONE pinned H2D copy (the per-stream
        frame counters and the rows share a staging block, so the frame number reaches the kernels through device memory and the
        captured kernel arguments never change) and the three stages; stage 3 writes the messages, std and samples STRAIGHT into
        pinned host memory (mapped into the device's address space), so there is no D2H node.  Per frame the host does two small
        numpy copies, one ``cudaGraphLaunch`` and one stream synchronize.  Same kernels, same Philox keys: bit-equal to ``step``.
        ``stream_frames``: optional host int32 ``[B]`` of per-stream frame numbers (negative: no new row), as in ``submit``."""
        rows = np.asarray(rows, dtype=np.float32)
        if rows.ndim == 2:
            rows = rows[:, None, :]
        nF = rows.shape[1]
        g = self._g
        if g is None or g.nF != nF or self._g_stale or torch.cuda.current_device() != g.dev_index:
            g = self._graph_setup(rows, nF)                   # validates the shape, drains earlier pipelined calls, (re)captures
        g.frames_np[...] = self.frame if stream_frames is None else np.asarray(stream_frames, dtype=np.int32).reshape(self.B)
        g.rows_np[...] = rows
        g.graph.replay()
        torch.cuda.current_stream().synchronize()
        out = EstimateBatch(g.msg, g.std, g.samples, g.status, self.frame)
        self.frame += nF
        self.calls += 1
        self.launches += g.launches
        return out

    def _graph_setup(self, rows, nF):
        """Slow path of ``step_graph`` (first call, another call size, or pipelined calls were submitted in between)."""
        if rows.shape[0] != self.B or nF > self.nF_max or rows.shape[2] != self.ncols:
            raise UserWarning(f"rows must be [B={self.B}, nF<={self.nF_max}, {self.ncols}], got {rows.shape}")
        with torch.cuda.device(self.device):
            self._leave_native()
            for ev in self.slot_event:                       # nothing submitted earlier may still be using the rings / the workspace
                if ev is not None:
                    ev.synchronize()
            torch.cuda.current_stream().synchronize()
            self._g_stale = False
            g = self._g
            if g is None or g.nF != nF or torch.cuda.current_device() != g.dev_index:
                g = self._capture_graph(rows, nF)
        return g

    def _capture_graph(self, rows, nF):
        B, E, Em = self.B, self.B * nF, self.B * self.nF_max
        g = _GraphCall()
        g.nF, g.dev_index = nF, torch.cuda.current_device()
        fb = (B * 4 + 15) // 16 * 16                         # the frame counters first, the rows behind them (16-byte aligned)
        stage_host = torch.zeros(fb + E * self.ncols * 4, dtype=torch.uint8).pin_memory()
        stage_dev = torch.zeros(fb + E * self.ncols * 4, dtype=torch.uint8, device=self.device)
        g.frames_np = stage_host[: B * 4].view(torch.int32).numpy()
        g.rows_np = stage_host[fb:].view(torch.float32).view(B, nF, self.ncols).numpy()
        raw, sf = stage_dev[fb:].view(torch.float32).view(B, nF, self.ncols), stage_dev[: B * 4].view(torch.int32)
        # results: a pinned block of the device buffers' layout, written by the stage-3 kernel itself
        out_host = torch.zeros(self.out_bufs[0].numel(), dtype=torch.float32).pin_memory()
        host = out_host.numpy()
        g.msg = host[: E * 25].reshape(B, nF, 25)
        g.std = host[Em * 25: Em * 25 + E * 6].reshape(B, nF, 6)
        g.status = host[Em * 31: Em * 31 + E].view(np.int32).reshape(B, nF)
        g.samples = host[Em * 32: Em * 32 + E * self.S * 6].reshape(B, nF, self.S, 6) if self.emit_samples else None
        g.keep = (stage_host, stage_dev, out_host)
        # the first use stages THIS call before the eager pass below (the replay that follows repeats it with the same inputs and keys)
        g.frames_np[...] = self.frame
        g.rows_np[...] = rows
        saved = (self.frame, self.calls, self.launches)

        def enqueue():
            stage_dev.copy_(stage_host, non_blocking=True)
            self._use_out_mapped(out_host)
            try:
                self._step_device(raw, nF, stream_frames=sf, _plain=True)
            finally:
                self._use_out(0)

        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                        # one eager pass first (function attributes, lazy module loading)
            enqueue()
        side.synchronize()
        g.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g.graph, stream=side):
            enqueue()
        g.launches = (self.launches - saved[2]) // 2          # (the eager pass and the capture each counted one call)
        self.frame, self.calls, self.launches = saved
        self._g = g
        return g

    def _host_views(self, slot, nF):
        host, E, Em = self.out_host[slot].numpy(), self.B * nF, self.B * self.nF_max
        msg = host[: E * 25].reshape(self.B, nF, 25)
        std = host[Em * 25: Em * 25 + E * 6].reshape(self.B, nF, 6)
        status = host[Em * 31: Em * 31 + E].view(np.int32).reshape(self.B, nF)
        samples = host[Em * 32: Em * 32 + E * self.S * 6].reshape(self.B, nF, self.S, 6) if self.emit_samples else None
        return msg, std, samples, status

    def step(self, rows, masks=None, stream_frames=None):
        """``submit`` + wait.  Returns an ``EstimateBatch`` of HOST arrays (views of a pinned staging slot, valid until
        the slot is reused ``N_SLOTS`` calls later)."""
        return self.submit(rows, masks, stream_frames).result()

    @property
    def h2d_bytes_per_frame(self):
        return self.B * self.ncols * 4

    @property
    def d2h_bytes_per_frame(self):
        return self.B * ((25 + 6) * 4 + 4 + (self.S * 6 * 4 if self.emit_samples else 0))
