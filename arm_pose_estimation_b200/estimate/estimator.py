"""The per-stream estimation loop behind the reference's ``Estimator`` API (``estimate/estimator.py:17-218``).

Constructor arguments, method names, properties, the sensor-queue / message-queue contract and the error behaviour are the
reference's, so its socket listeners, UDP publishers and CSV recorders work unchanged around this class.  What sits behind
them is different: the reference keeps the input window and the smoothing stack in Python lists and runs the model on the
CPU; here both histories are device rings indexed by the absolute frame number (a frame before 0 reads as frame 0, which is
the reference's "repeat the first row / first prediction" start-up), owned by a one-stream ``BatchedEstimator``:

* ``processing_loop`` / ``estimate_row``: one CUDA-graph launch per frame (one H2D copy of frame counter + raw row, the three kernel stages,
  the message written by stage 3 into mapped pinned memory) - the fused form of the loop body ``parse_row_to_xx -> add_xx_to_row_hist_and_make_prediction ->
  msg_from_pred`` (estimator.py:174-176);
* the three calls one by one: each runs its own kernel stage (stage 1 with ``normalize=0``; ``ape_features_push`` + the
  MC-LSTM over the rings; stage 3 on the rows it is handed).

A subclass that brings its own ``make_prediction_from_row_hist`` (the reference's extension point, e.g. the direct-orientation
``WatchPhoneUarm``) or a model family without a fused kernel path (``DropoutFF``, ``ImuPoseLSTM``) still gets the same call
sequence; its window and smoothing stack then live in small host rings of the same "absolute frame, clamp at 0" design.
"""
import logging
import queue
import threading
import time

import numpy as np
import torch

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200.data_types.bone_map import BoneMap, body_measurements_row
from arm_pose_estimation_b200.estimate import estimate_joints
from arm_pose_estimation_b200.estimate.batched import BatchedEstimator
from arm_pose_estimation_b200.utility import data_stats
from arm_pose_estimation_b200.utility.names import NNS_INPUTS, NNS_TARGETS

BACKLOG_LIMIT = 5            # rows a sensor queue may hold before the loop sheds the oldest ones (estimator.py:160)
QUEUE_TIMEOUT_S = 2          # estimator.py:159
RATE_LOG_PERIOD_S = 5        # estimator.py:167-170


class _FrameRing:
    """The last ``depth`` per-frame arrays of one stream, by absolute frame number; frames before 0 read as frame 0."""

    def __init__(self, depth):
        self.depth = int(depth)
        self.clear()

    def clear(self):
        self.frames = 0
        self.slots = [None] * self.depth

    def push(self, item):
        self.slots[self.frames % self.depth] = item
        self.frames += 1

    def window(self):
        """The ``depth`` most recent items, oldest first."""
        newest = self.frames - 1
        return [self.slots[max(0, f) % self.depth] for f in range(newest - self.depth + 1, newest + 1)]


class Estimator:
    # set by the NN subclasses: which parse_row_to_xx the stage-1 kernel follows, and the wire layout of a raw row
    _kind = None
    _layout = None

    def __init__(self,
                 x_inputs: NNS_INPUTS,
                 y_targets: NNS_TARGETS,
                 normalize: bool = True,
                 smooth: int = 1,
                 seq_len: int = 1,
                 add_mc_samples: bool = True,
                 bonemap: BoneMap = None,
                 tag: str = "Estimator"):
        self.__tag = tag
        self._x_inputs, self._y_targets = x_inputs, y_targets
        self._sequence_len, self._smooth = max(1, seq_len), max(1, smooth)
        self._add_mc_samples = add_mc_samples
        self._bonemap = bonemap
        self._body_measurements = body_measurements_row(bonemap)                 # (1, 9): larm_vec, uarm_vec, uarm_orig
        self._larm_vec, self._uarm_vec, self._uarm_orig = np.split(self._body_measurements[0], 3)
        self._device = torch.device("cuda" if torch.cuda.is_available() else "cpu")
        self._normalize = normalize
        if normalize:
            self._take_stats(data_stats.get_norm_stats(x_inputs=x_inputs, y_targets=y_targets))
        self._active = False
        self._last_msg = self._last_std = None
        self._engines = {}                                  # one-stream BatchedEstimators by role: "graph" | "calls"
        self._xx_ring, self._pred_ring = _FrameRing(self._sequence_len), _FrameRing(self._smooth)

    # ---- state ---------------------------------------------------------------------------------------------------
    def _take_stats(self, stats):
        for key in ("xx_m", "xx_s", "yy_m", "yy_s"):
            setattr(self, "_" + key, stats[key])
        self._engines = {}                                  # device copies of the old statistics go with their engines

    def set_norm_stats(self, stats: dict):
        """overwrites the default norm stats loaded during the initialization"""
        self._take_stats(stats)
        logging.info("Replaced norm stats xx m+/-s and yy m+/-s")

    def reset(self):
        self._active = False
        self._xx_ring.clear()
        self._pred_ring.clear()
        for engine in self._engines.values():
            engine.reset()

    def terminate(self):
        self._active = False

    def is_active(self):
        return self._active

    def get_last_msg(self):
        return self._last_msg

    def get_last_std(self):
        """Population std of the per-row hand / elbow positions of the last fused estimate (new; SURVEY.md §8a)."""
        return self._last_std

    # ---- device engines ------------------------------------------------------------------------------------------
    def _has_device_path(self):
        """True when stage 2 of this estimator is the MC-LSTM kernel path over device rings."""
        return False

    def _make_fused(self, mask_mode=N.MASK_PHILOX):
        raise UserWarning("this estimator has no fused CUDA path")

    _mask_mode = N.MASK_PHILOX

    def _engine(self, role):
        if role not in self._engines:
            self._engines[role] = self._make_fused(mask_mode=self._mask_mode)
        return self._engines[role]

    def _fused_estimator(self):
        return self._engine("graph")

    # ---- the three per-frame calls, one by one (estimator.py:93-137) ---------------------------------------------------
    def add_xx_to_row_hist_and_make_prediction(self, xx, masks=None) -> np.array:
        """``masks`` (not in the reference): explicit dropout masks ``[L-1, T, n, H]`` for this frame instead of the Philox draw -
        needs ``_mask_mode = MASK_INJECTED`` before the first call; used by the parity tests."""
        if self._has_device_path():
            # window -> z-score -> MC forward passes -> de-normalise -> smoothing stack, all on the engine's device rings
            m = None if masks is None else np.asarray(masks)[None, None]
            return self._engine("calls").step_features(np.asarray(xx, dtype=np.float64)[None, :], masks=m)[0]
        self._xx_ring.push(np.asarray(xx))
        window = np.vstack(self._xx_ring.window())
        if self._normalize:
            window = (window - self._xx_m) / self._xx_s
        pred = self.make_prediction_from_row_hist(window) if masks is None else self.make_prediction_from_row_hist(window, masks=masks)
        if self._normalize:
            pred = pred * self._yy_s + self._yy_m
        if self._smooth == 1:
            return pred
        self._pred_ring.push(pred)
        return np.vstack(self._pred_ring.window())

    def msg_from_pred(self, pred: np.array, add_mc_samples: bool) -> np.array:
        est, msg, self._last_std = estimate_joints.fk_rows(pred, self._body_measurements, self._y_targets, want_msg=True)
        self._last_msg = msg.copy()
        if not add_mc_samples:
            return msg
        tail = est[:, :6].ravel().tolist() if len(est) > 1 else []      # hand xyz, elbow xyz of every row (estimator.py:131-136)
        return list(msg) + tail

    # ---- the same three stages as one launch sequence ---------------------------------------------------------------
    def estimate_row(self, row, add_mc_samples=None):
        """One frame of the loop body (estimator.py:174-176); returns the message."""
        with_samples = self._add_mc_samples if add_mc_samples is None else add_mc_samples
        if not self._has_device_path():
            return self.msg_from_pred(self.add_xx_to_row_hist_and_make_prediction(self.parse_row_to_xx(row)), with_samples)
        engine = self._engine("graph")
        out = engine.step_graph(np.asarray(row, dtype=np.float32).reshape(1, 1, -1))      # one CUDA-graph launch
        if out.status[0, 0] != 0:
            raise np.linalg.LinAlgError("degenerate 6D rotation (zero or collinear columns)")
        self._last_msg = out.msg[0, 0].astype(np.float64)
        self._last_std = out.std[0, 0].astype(np.float64)
        if not with_samples:
            return self._last_msg.copy()
        tail = out.samples[0, 0].astype(np.float64).ravel().tolist() if engine.S > 1 else []
        return list(self._last_msg) + tail

    # ---- queue in, queue out (estimator.py:139-178) -------------------------------------------------------------------
    def process_in_thread(self, sensor_q: queue):
        msg_q = queue.Queue()
        threading.Thread(target=self.processing_loop, args=(sensor_q, msg_q)).start()
        return msg_q

    def _freshest_row(self, sensor_q):
        """The next row to estimate: blocks up to the reference's 2 s, and sheds rows while more than five are waiting."""
        row = sensor_q.get(timeout=QUEUE_TIMEOUT_S)
        while sensor_q.qsize() > BACKLOG_LIMIT:
            row = sensor_q.get(timeout=QUEUE_TIMEOUT_S)
        return row

    def processing_loop(self, sensor_q: queue, msg_q: queue):
        logging.info(f"[{self.__tag}] wearable streaming loop")
        self.reset()
        self._active = True
        window_start, estimates = time.monotonic(), 0
        while self._active:
            try:
                row = self._freshest_row(sensor_q)
            except queue.Empty:
                logging.info(f"[{self.__tag}] no data")
                continue
            if time.monotonic() - window_start >= RATE_LOG_PERIOD_S:
                logging.info(f"[{self.__tag}] {estimates / RATE_LOG_PERIOD_S} Hz")
                window_start, estimates = time.monotonic(), 0
            msg_q.put(self.estimate_row(row, self._add_mc_samples))
            estimates += 1

    # ---- what a subclass provides ---------------------------------------------------------------------------------------
    def make_prediction_from_row_hist(self, xx_hist: np.array) -> np.array:
        raise NotImplementedError

    def parse_row_to_xx(self, row) -> np.array:
        raise NotImplementedError

    sequence_len = property(lambda self: self._sequence_len)
    body_measurements = property(lambda self: self._body_measurements)
    uarm_orig = property(lambda self: self._uarm_orig)
    uarm_vec = property(lambda self: self._uarm_vec)
    larm_vec = property(lambda self: self._larm_vec)
    device = property(lambda self: self._device)
    x_inputs = property(lambda self: self._x_inputs)
    y_targets = property(lambda self: self._y_targets)


def parsed_feature_row(row, layout, kind, n_features, dtype):
    """``parse_row_to_xx`` of the reference for one raw IMU row: the stage-1 kernel with ``normalize=0``."""
    if not torch.cuda.is_available():
        raise RuntimeError("arm_pose_estimation_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    ncols = 28 if layout == N.LAYOUT_WATCH_ONLY else 55
    flat = np.asarray(row, dtype=np.float32).ravel()
    if flat.size < ncols:
        raise UserWarning(f"a raw row of this estimator has {ncols} floats, got {flat.size}")
    raw = torch.from_numpy(np.ascontiguousarray(flat[:ncols])).cuda()
    out = torch.empty(n_features, dtype=torch.float32, device="cuda")
    N.check(N.load().ape_features(N.ptr(raw), layout, kind, None, None, 0, N.ptr(out), 1, 1, 0, None, 1,
                                  N.current_stream_ptr()), "ape_features")
    return out.cpu().numpy().astype(dtype)


class _NNEstimator(Estimator):
    """What the three NN estimators share: the deployed model, the stage-1 kernel per row, the MC forward passes."""
    _xx_dtype = np.float32

    def _init_nn(self, model_hash, smooth, add_mc_samples, monte_carlo_samples, bonemap, tag, philox_seed):
        from arm_pose_estimation_b200.estimate import nn_models
        self._mc_samples = monte_carlo_samples
        self._nn_model, params = nn_models.load_deployed_model_from_hash(hash_str=model_hash)
        self._params = params
        # the loader may hand back any of the three model families (nn_models.py:392-399); only DropoutLSTM has the fused kernels
        self._lstm_model = isinstance(self._nn_model, nn_models.DropoutLSTM)
        if philox_seed is not None:
            self._nn_model.philox_seed = int(philox_seed)
        self._philox_seed = int(getattr(self._nn_model, "philox_seed", 0))
        Estimator.__init__(
            self,
            x_inputs=NNS_INPUTS[params["x_inputs_n"]],
            y_targets=NNS_TARGETS[params["y_targets_n"]],
            smooth=smooth,
            normalize=params["normalize"],
            seq_len=params["sequence_len"],
            add_mc_samples=add_mc_samples,
            tag=tag,
            bonemap=bonemap,
        )

    def _has_device_path(self):
        # (a subclass that overrides make_prediction_from_row_hist goes through its override, like in the reference)
        return self._lstm_model and getattr(self.make_prediction_from_row_hist, "__func__", None) is _NNEstimator.make_prediction_from_row_hist

    def parse_row_to_xx(self, row):
        return parsed_feature_row(row, self._layout, self._kind, len(self._x_inputs.value), self._xx_dtype)

    def make_prediction_from_row_hist(self, xx_hist, masks=None):
        """``xx_hist [sequence_len, features]`` (z-scored) -> ``[mc_samples, outputs]``: the last step of the MC forward passes
        (watch_only.py:84-97)."""
        x = torch.tensor(np.asarray(xx_hist)[None, :, :], dtype=torch.float32)
        extra = {} if masks is None else {"masks": masks}
        return self._nn_model.monte_carlo_predictions(x=x, n_samples=self._mc_samples, **extra).numpy()[:, -1, :]

    def _make_fused(self, mask_mode=N.MASK_PHILOX):
        if not self._lstm_model:
            raise UserWarning(f"{type(self._nn_model).__name__} has no fused CUDA path: use the three per-frame calls")
        stats = dict(xx_m=self._xx_m, xx_s=self._xx_s, yy_m=self._yy_m, yy_s=self._yy_s) if self._normalize else None
        return BatchedEstimator(
            kind=self._kind, layout=self._layout, state=self._nn_model.state_dict(), seq_len=self._sequence_len,
            y_targets=self._y_targets, stats=stats, n_streams=1, mc_samples=self._mc_samples, smooth=self._smooth,
            dropout=self._nn_model.dropout, bonemap=self._bonemap, frames_per_call=1, emit_samples=True,
            normalize=self._normalize, mask_mode=mask_mode, philox_seed=self._philox_seed, split_small_batch_kernel=True)
