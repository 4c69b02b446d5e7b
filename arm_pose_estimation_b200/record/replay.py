"""Recorded-IMU CSV replay / offline relabelling front-end (SURVEY.md §8f.1).

File formats are the reference's own:
* raw IMU recording: header = the keys of ``WATCH_ONLY_IMU_LOOKUP`` (28 columns) in wire order, one row per frame written
  with ``",".join(map(str, row))`` (``record/arm_pose_to_csv.py:9-32``); the ``experimental_applications/watch_raw_record.py``
  variant with a leading ``timestamp`` column and 55-column watch+phone recordings are accepted too;
* pose estimates: ``time`` + the 24 named columns of ``EstOutputRecorder`` (``record/est_output.py:16-25``) = the 25-float
  message, one row per frame.

``relabel_recordings`` pushes whole recordings through ``BatchedEstimator`` - recordings are the stream axis, frames go
``frames_per_call`` at a time - so BASELINE config 4 (10k recordings x 3600 frames, sharded over GPUs by recording) is this
function called on each rank's shard.
"""
import datetime
from pathlib import Path

import numpy as np

from arm_pose_estimation_b200.data_types import messaging

EST_OUTPUT_HEADER = [
    "time",
    "hand_quat_w", "hand_quat_x", "hand_quat_y", "hand_quat_z",
    "hand_orig_rh_x", "hand_orig_rh_y", "hand_orig_rh_z",
    "larm_quat_rh_w", "larm_quat_rh_x", "larm_quat_rh_y", "larm_quat_rh_z",
    "larm_orig_rh_x", "larm_orig_rh_y", "larm_orig_rh_z",
    "uarm_quat_rh_w", "uarm_quat_rh_x", "uarm_quat_rh_y", "uarm_quat_rh_z",
    "uarm_orig_rh_x", "uarm_orig_rh_y", "uarm_orig_rh_z",
    "hips_quat_g_w", "hips_quat_g_x", "hips_quat_g_y", "hips_quat_g_z",
]
_LAYOUT_KEYS = {
    messaging.LAYOUT_WATCH_ONLY: list(messaging.WATCH_ONLY_IMU_LOOKUP.keys()),
    messaging.LAYOUT_WATCH_PHONE: list(messaging.WATCH_PHONE_IMU_LOOKUP.keys()),
}


def write_imu_csv(path, rows, layout=messaging.LAYOUT_WATCH_ONLY):
    """Write ``rows [frames, 28|55]`` in the reference recorder's format (``arm_pose_to_csv.py:11-24``)."""
    keys = _LAYOUT_KEYS[layout]
    rows = np.asarray(rows)
    if rows.ndim != 2 or rows.shape[1] != len(keys):
        raise UserWarning(f"a layout-{layout} recording has {len(keys)} columns, got {rows.shape}")
    with open(path, "w") as fd:
        fd.write(",".join(keys) + "\n")
        for row in rows:
            fd.write(",".join(map(str, row.tolist())) + "\n")


def read_imu_csv(path):
    """Read a raw IMU recording -> ``(rows [frames, ncols] float32, layout)``.  Columns are matched BY NAME against the
    wire layouts, so a leading ``timestamp`` column (watch_raw_record.py variant) or reordered columns are fine."""
    with open(path, "r") as fd:
        header = fd.readline().strip().split(",")
        body = fd.read().strip()
    for layout, keys in ((messaging.LAYOUT_WATCH_PHONE, _LAYOUT_KEYS[messaging.LAYOUT_WATCH_PHONE]),
                         (messaging.LAYOUT_WATCH_ONLY, _LAYOUT_KEYS[messaging.LAYOUT_WATCH_ONLY])):
        if all(k in header for k in keys):
            break
    else:
        raise UserWarning(f"{path}: header matches neither the 28-column watch layout nor the 55-column watch+phone layout")
    if not body:
        return np.zeros((0, len(keys)), np.float32), layout
    cols = [header.index(k) for k in keys]
    table = []
    for line in body.split("\n"):
        parts = line.split(",")
        if len(parts) != len(header):
            raise UserWarning(f"{path}: ragged line with {len(parts)} fields, header has {len(header)}")
        table.append([float(parts[c]) for c in cols])
    return np.asarray(table, dtype=np.float32), layout


def write_pose_csv(path, msgs, times=None):
    """Write ``msgs [frames, 25]`` as ``EstOutputRecorder`` does (``est_output.py:16-25, 53-57``)."""
    msgs = np.asarray(msgs)
    if msgs.ndim != 2 or msgs.shape[1] != 25:
        raise UserWarning(f"pose messages are [frames, 25], got {msgs.shape}")
    path = Path(path)
    if not path.parent.exists():
        raise UserWarning(f"Directory does not exist {path.parent}")
    with open(path, "w") as fd:
        fd.write(",".join(EST_OUTPUT_HEADER) + "\n")
        for i, m in enumerate(msgs):
            t = datetime.datetime.now() if times is None else times[i]
            fd.write(",".join([str(t)] + [str(x) for x in m.tolist()]) + "\n")


def read_pose_csv(path):
    """-> ``(times [frames] str, msgs [frames, 25] float64)``."""
    with open(path, "r") as fd:
        header = fd.readline().strip().split(",")
        if header != EST_OUTPUT_HEADER:
            raise UserWarning(f"{path}: not an EstOutputRecorder file")
        lines = [ln for ln in fd.read().split("\n") if ln]
    times = [ln.split(",", 1)[0] for ln in lines]
    msgs = np.asarray([[float(v) for v in ln.split(",")[1:]] for ln in lines], dtype=np.float64).reshape(len(lines), 25)
    return times, msgs


def pad_recordings(recordings):
    """List of ``[frames_i, ncols]`` -> ``([R, F_max, ncols] float32, lengths)``; short recordings repeat their last row
    (the padded frames are computed and discarded - frames of a stream only depend on earlier frames)."""
    lengths = np.asarray([len(r) for r in recordings], dtype=np.int64)
    if len(recordings) == 0 or lengths.max(initial=0) == 0:
        return np.zeros((len(recordings), 0, 0), np.float32), lengths
    ncols = recordings[int(np.argmax(lengths))].shape[1]
    out = np.zeros((len(recordings), int(lengths.max()), ncols), np.float32)
    for i, r in enumerate(recordings):
        if len(r):
            out[i, : len(r)] = r
            out[i, len(r):] = r[-1]
    return out, lengths


def relabel_recordings(recordings, make_estimator, frames_per_call=16, keep_samples=False, masks=None, bonemaps=None):
    """Offline relabelling: ``recordings`` = list of ``[frames_i, ncols]`` arrays (or one ``[R, F, ncols]`` array);
    ``make_estimator(n_streams, frames_per_call)`` returns a ``BatchedEstimator``.  Returns a list of dicts with
    ``msg [frames_i, 25]``, ``std [frames_i, 6]`` (and ``samples`` if asked).  The next calls are staged and enqueued while call k runs.
    ``masks``: explicit dropout masks ``[R, F, L-1, T, n, H]`` for an estimator built with ``MASK_INJECTED`` (parity runs); for a
    feed-forward model (``DropoutFF`` / ``DropoutFF2D``) its output-dropout masks ``[R, F, n, H]``.  ``bonemaps``: one skeleton per
    recording (R entries for ``body_measurements_rows``: recordings of different subjects), set on the estimator before its first
    call; ``None`` keeps the estimator's own."""
    if isinstance(recordings, np.ndarray) and recordings.ndim == 3:
        rows, lengths = np.asarray(recordings, dtype=np.float32), np.full(len(recordings), recordings.shape[1], np.int64)
    else:
        rows, lengths = pad_recordings(list(recordings))
    R, F = rows.shape[0], rows.shape[1]
    if R == 0 or F == 0:
        return [dict(msg=np.zeros((0, 25)), std=np.zeros((0, 6))) for _ in range(R)]
    be = make_estimator(R, min(frames_per_call, F))
    be.reset()
    if bonemaps is not None:
        be.set_bonemaps(bonemaps)
    msg = np.empty((R, F, 25), np.float32)
    std = np.empty((R, F, 6), np.float32)
    samples = np.empty((R, F, be.S, 6), np.float32) if keep_samples else None

    def collect(pending, f0, nf):
        out = pending.result()
        if (out.status != 0).any():
            raise np.linalg.LinAlgError("degenerate 6D rotation (zero or collinear columns) in a relabelled frame")
        msg[:, f0:f0 + nf], std[:, f0:f0 + nf] = out.msg, out.std
        if keep_samples:
            samples[:, f0:f0 + nf] = out.samples

    outstanding = []                                          # submitted, not yet collected (oldest first)
    for f0 in range(0, F, be.nF_max):
        nf = min(be.nF_max, F - f0)
        outstanding.append((be.submit(rows[:, f0:f0 + nf], masks=None if masks is None else masks[:, f0:f0 + nf]), f0, nf))
        if len(outstanding) >= be.N_SLOTS - 1:                # the next submit reuses the oldest one's staging slot
            collect(*outstanding.pop(0))
    for item in outstanding:
        collect(*item)
    msg64, std64 = msg.astype(np.float64), std.astype(np.float64)      # one conversion for all recordings; the per-recording results are views
    res = []
    for i in range(R):
        d = dict(msg=msg64[i, : lengths[i]], std=std64[i, : lengths[i]])
        if keep_samples:
            d["samples"] = samples[i, : lengths[i]]
        res.append(d)
    return res
