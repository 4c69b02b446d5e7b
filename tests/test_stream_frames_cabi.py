"""CPU: the C-ABI refusals around per-stream frame counters that return before any CUDA call, and the plain references of
tests/test_gpu_stream_frames.py pinned against the reference's own messages and window bookkeeping."""
import ctypes as C

import numpy as np
import pytest

from conftest import load_golden, unpack_masks
from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200 import synthetic as syn
from test_gpu_stream_frames import msg_errors, ref_features, ref_lstm, ref_stage3, window_frames, window_slots

P = C.c_void_p(256)                      # a non-null address that is never dereferenced: every call below refuses first


def test_features_refusals():
    lib = N.load()
    # a launch may not lap its own ring: nF > feat_ring
    assert lib.ape_features(P, 0, 0, None, None, 0, P, 4, 6, 0, None, 5, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_features(P, 0, 0, None, None, 0, P, 4, 6, 0, P, 5, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_features(P, 1, 2, None, None, 0, P, 4, 2, 0, P, 1, None) == N.APE_ERR_BAD_ARG
    # null rows / ring, normalize without statistics, no ring at all
    assert lib.ape_features(None, 0, 0, None, None, 0, P, 4, 1, 0, P, 5, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_features(P, 0, 0, None, None, 0, None, 4, 1, 0, P, 5, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_features(P, 0, 0, None, P, 1, P, 4, 1, 0, P, 5, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_features(P, 0, 0, None, None, 0, P, 4, 1, 0, P, 0, None) == N.APE_ERR_BAD_ARG


def test_features_push_refusals():
    lib = N.load()
    for ring in (0, -3):
        assert lib.ape_features_push(P, 20, None, None, 0, P, 4, 0, P, ring, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_features_push(None, 20, None, None, 0, P, 4, 0, P, 5, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_features_push(P, 20, None, None, 0, None, 4, 0, P, 5, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_features_push(P, 20, P, None, 1, P, 4, 0, P, 5, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_features_push(P, 0, None, None, 0, P, 4, 0, P, 5, None) == N.APE_ERR_BAD_ARG


def test_fk_reduce_refusals():
    lib = N.load()
    t, O = N.TARGET_ORI_CAL_LARM_UARM_HIPS, 14

    def fk(preds=P, ring=5, body=P, msg=P, nF=3, smooth=3, target=t, o=O, yy_m=None, yy_s=None):
        return lib.ape_fk_reduce(preds, ring, yy_m, yy_s, body, target, o, 4, nF, 0, P, 10, smooth, msg, None, None, None, None, None)

    # the smoothing window of the call's last frame must still be in the ring: nF + smooth - 1 <= pred_ring
    assert fk(ring=4, nF=3, smooth=3) == N.APE_ERR_BAD_ARG
    assert fk(ring=19, nF=1, smooth=20) == N.APE_ERR_BAD_ARG
    assert fk(ring=0, nF=1, smooth=1) == N.APE_ERR_BAD_ARG
    for kw in (dict(preds=None), dict(body=None), dict(msg=None), dict(yy_m=P), dict(yy_s=P), dict(o=12), dict(target=3),
               dict(smooth=0)):
        assert fk(**kw) == N.APE_ERR_BAD_ARG, kw


def test_msg_from_est_refusals():
    lib = N.load()
    assert lib.ape_msg_from_est(None, 14, P, 0, 3, 5, P, None, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_msg_from_est(P, 14, None, 0, 3, 5, P, None, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_msg_from_est(P, 14, P, 0, 3, 5, None, None, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_msg_from_est(P, 21, P, 0, 3, 5, P, None, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_msg_from_est(P, 14, P, 2, 3, 5, P, None, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_msg_from_est(P, 14, P, 0, 3, 0, P, None, None) == N.APE_ERR_BAD_ARG


def test_window_helper_matches_the_reference_history_and_the_estimator_slots():
    # the reference keeps its row / smoothing history as a list: append, pad to the window by repeating the newest entry (only
    # ever at the first frame), drop the oldest (estimator.py:93-118, restated by oracle.estimator)
    for length in (1, 2, 3, 6, 8, 20):
        hist = []
        for f in range(3 * length + 5):
            hist.append(f)
            while len(hist) < length:
                hist.append(f)
            while len(hist) > length:
                del hist[0]
            assert window_frames(f, length) == hist, (f, length)
            for ring in (1, length, length + 2, 7):
                # the slots BatchedEstimator.step_features reads (estimate/batched.py: max(0, k) % pred_ring over the window)
                assert window_slots(f, length, ring) == [max(0, k) % ring for k in range(f - length + 1, f + 1)]
    assert window_slots(1001, 3, 4) == [3, 0, 1]                     # across the ring wrap


@pytest.mark.parametrize("name", ["watch_only_s3", "pocket_s1", "uarm_s1", "uarm_s4"])
def test_windowed_references_reproduce_the_reference_messages(name, body9):
    # the three references of the GPU test chained on the CPU - features into a ring, the LSTM on the clamped window of the ring,
    # the normalised predictions into a second ring, stage 3 on the de-normalised smoothing window - reproduce the messages the
    # reference itself produced (tests/golden/make_golden.py) frame by frame
    g = load_golden(f"e2e_{name}.npz")
    kind = {"watch_only": syn.KIND_WATCH_ONLY, "pocket": syn.KIND_POCKET, "uarm": syn.KIND_UARM}[name.rsplit("_", 1)[0]]
    spec = syn.kind_spec(kind)
    state = syn.synth_state_dict(spec["I"], spec["H"], spec["L"], spec["O"], int(g["weight_seed"]))
    n, smooth, T = int(g["n"]), int(g["smooth"]), spec["T"]
    masks = unpack_masks(g)                                          # [F][L-1][T][n][H]
    rows, F = g["rows"], len(g["rows"])
    feat_ring, pred_ring = T + 1, smooth + 1                         # one slot more than a window: over 14 frames both rings wrap
    feats = np.full((feat_ring, spec["I"]), np.nan, np.float32)      # (a slot read before it was written would show as NaN)
    preds = np.full((pred_ring, n, spec["O"]), np.nan, np.float32)
    xx = ref_features(kind, rows, spec["stats"]["xx_m"], spec["stats"]["xx_s"])
    worst = 0.0
    for f in range(F):
        feats[f % feat_ring] = xx[f].astype(np.float32)
        preds[f % pred_ring] = ref_lstm(state, feats, f, T, masks[f], spec["p"])
        est, msg, _ = ref_stage3(preds, f, smooth, spec["stats"]["yy_m"], spec["stats"]["yy_s"], body9, spec["y_targets"].name)
        pos, q = msg_errors(msg, g["msgs"][f, :25])
        if n * smooth > 1:
            pos = max(pos, float(np.abs(est[:, :6].ravel() - g["msgs"][f, 25:]).max()))
        assert pos <= 1e-4 and q <= 2e-4, f"frame {f}: position {pos:.3g} m, quaternion {q:.3g}"
        worst = max(worst, pos)
    print(f"{name}: windowed CPU references vs the reference's messages over {F} frames: worst position error {worst:.3g} m")
