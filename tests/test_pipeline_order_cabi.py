"""CPU: the refusals of ape_pipeline_stream, the pipeline's ordering rule (``pred_window_alias``) against a brute-force slot count,
and the aliasing preconditions of the schedules tests/test_gpu_pipeline_order.py holds streams on - so an edit that makes those GPU
cases vacuous fails here, on a machine without a GPU."""
import ctypes as C
import itertools

import numpy as np

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200.estimate.batched import BatchedEstimator, pred_window_alias, ring_slots
from test_gpu_pipeline_order import (MATRIX_B, MATRIX_CALLS, SMOOTH, histories, matrix_schedule, overwritten_window_slots,
                                     reset_schedule, restart_schedule)
from test_gpu_stream_frames import window_slots

P = C.c_void_p(256)                      # a non-null address that is never dereferenced: every call below refuses first


def test_pipeline_stream_refusals():
    lib = N.load()
    s = C.c_void_p(None)
    assert lib.ape_pipeline_stream(None, 0, C.byref(s)) == N.APE_ERR_BAD_ARG
    assert lib.ape_pipeline_stream(P, 0, None) == N.APE_ERR_BAD_ARG
    for which in (-1, 4, 1 << 30):
        assert lib.ape_pipeline_stream(P, which, C.byref(s)) == N.APE_ERR_BAD_ARG
    assert s.value is None


def test_alias_rule_is_exact():
    """pred_window_alias(f, nF, f1, nF1) is true exactly when frames f .. f + nF - 1 share a ring slot with the smoothing windows of
    frames f1 .. f1 + nF1 - 1 (clamped to frame 0), over every ring the estimator builds for nF_max <= 3, smooth <= 3."""
    for nF_max, smooth in itertools.product((1, 2, 3), (1, 2, 3)):
        ring = ring_slots(2 * nF_max, smooth)
        for nF, nF1 in itertools.product(range(1, nF_max + 1), repeat=2):
            for f1 in range(0, 2 * ring + 2):
                read = {s for j in range(nF1) for s in window_slots(f1 + j, smooth, ring)}
                for f in range(0, f1 + 2 * ring + 2):
                    want = bool(read & {(f + j) % ring for j in range(nF)})
                    assert bool(pred_window_alias(f, nF, f1, nF1, smooth, ring)) == want, (nF_max, smooth, nF, nF1, f1, f)
                # a stream that moves on by exactly the previous call's frames never needs the fence
                assert not pred_window_alias(f1 + nF1, nF, f1, nF1, smooth, ring)


def test_restart_schedule_aliases():
    for B in (40, 64, 300, 1024):
        calls, K, b_own, b_prev = restart_schedule(B)
        ring = ring_slots(2, SMOOTH)
        f_own, f_prev = int(calls[K][1][b_own]), int(calls[K][1][b_prev])
        assert (f_own, f_prev) == (ring, ring + 1)
        assert calls[K + 1][1][b_own] == 0 and calls[K + 1][1][b_prev] == 0
        # call K + 1 overwrites the slot of call K's own frame (b_own) / of the frame before it, written by call K - 1 (b_prev)
        assert overwritten_window_slots(calls, K, b_own, ring) == {f_own % ring} == {0}
        assert overwritten_window_slots(calls, K, b_prev, ring) == {(f_prev - 1) % ring} == {0}
        # ... and nowhere else: every other stream and every other pair of calls moves forward without aliasing
        for k in range(len(calls) - 1):
            for b in range(B):
                hit = bool(overwritten_window_slots(calls, k, b, ring))
                assert hit == (k == K and b in (b_own, b_prev)), (B, k, b)
        hist = histories(calls, B)
        assert [len(hist[b]) for b in (b_own, b_prev)] == [2, 2] and all(len(h) == 1 for b, h in enumerate(hist) if b not in (b_own, b_prev))


def test_reset_schedule_aliases():
    calls, (K1, K2) = reset_schedule()
    ring = ring_slots(2, SMOOTH)
    assert [calls[K][2] for K in (K1, K2)] == [ring, ring + 1] and calls[K1 + 1][2] == calls[K2 + 1][2] == 0
    assert overwritten_window_slots(calls, K1, 0, ring) == {calls[K1][2] % ring}
    assert overwritten_window_slots(calls, K2, 0, ring) == {(calls[K2][2] - 1) % ring}
    assert [k for k in range(len(calls) - 1) if overwritten_window_slots(calls, k, 0, ring)] == [K1, K2]
    assert [len(seg) for seg in histories(calls, 3)[0]] == [ring + 1, ring + 2, 2]


def test_matrix_schedule_covers_what_it_claims():
    calls, late, restart = matrix_schedule(MATRIX_B, MATRIX_CALLS)
    assert len(calls) >= BatchedEstimator.N_SLOTS + 4                      # every result slot and all four buffer sets wrap
    assert {nF for nF, _, _ in calls} == {1, 2}                             # short calls among full ones
    sf = np.stack([c[1] for c in calls])
    assert (sf < 0).any(axis=1).all()                                       # skipped streams in every call
    assert (sf[:5, list(late)] < 0).all() and (sf[5:, list(late)] >= 0).mean() > 0.5
    hist = histories(calls, MATRIX_B)
    assert len(hist[restart]) == 2 and hist[late[0]]
    ring = ring_slots(2 * 2, SMOOTH)
    # the restart is the only call pair in which a stream goes back; forward moves never alias
    back = {(k, b) for k in range(len(calls) - 1) for b in range(MATRIX_B) if overwritten_window_slots(calls, k, b, ring)}
    assert {b for _, b in back} <= {restart}
