"""GPU (-m gpu): the cross-call pipeline's stream ordering, pinned with held streams instead of whatever interleaving the GPU picks.

The pipeline (csrc/ape_pipeline.cu, and its Python-level copy in estimate/batched.py) runs stage 1 + layer 0 on a side stream, the
LSTM layers >= 1 + stage 3 of consecutive calls on two alternating lane streams and the read-back on a copy stream, ordered by about
ten cross-stream edges.  A *hold* is a bounded clock spin (``torch.cuda._sleep``) enqueued on one of those streams before a chosen
``submit``: the work queued behind it waits ~10 ms, everything the ordering lets run ahead does, and a missing edge shows as a
wrong result every time rather than once in a while.  Every case feeds the same schedule to a ``pipeline=False`` estimator (serial)
and requires every call's ``msg``, ``std``, ``samples`` and ``status`` of the active streams bit for bit; the serial run's restarted
streams are checked against ``oracle.estimator.OracleEstimator`` with their own Philox masks (1e-4 m, 2e-4 in quaternions).

  a. a restarted stream: call K + 1 writes frame 0 into a prediction slot that call K's smoothing window reads (once the slot of
     call K's own frame, once the slot of the frame before it), with call K's lane held: on every pipelined kernel, native and
     Python-level pipeline;
  b. ``reset()`` of the shared frame counter with calls in flight, the same construction;
  c. a hold matrix: each of the four streams held before call 3 and before call N_SLOTS of a 12-call schedule (skipped streams, a
     late-joining block, a restart, short calls, smooth = 2) on the wavefront and the H = 256 kernels.

tests/test_pipeline_order_cabi.py checks on the CPU that the schedules below meet the aliasing preconditions they state."""
import ctypes

import numpy as np
import pytest
import torch

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200 import synthetic as syn
from arm_pose_estimation_b200.estimate.batched import BatchedEstimator, pred_window_alias, ring_slots
from test_gpu_stream_frames import SEED, _estimator, _model, msg_errors, philox_masks, window_slots

pytestmark = pytest.mark.gpu

POS_TOL, QUAT_TOL = 1e-4, 2e-4
SMOOTH = 2
HOLD_CYCLES = 20_000_000               # ~10 ms at the B200's ~2 GHz SM clock: > 20 calls of 1024 x 100 (~0.4 ms each)
STREAMS = ("side", "lane0", "lane1", "copy")     # ape_pipeline_stream's `which`: 0 .. 3


# ---- schedules (pure numpy: tests/test_pipeline_order_cabi.py checks their preconditions without a GPU) ----------------------------
# A call is (nF, per-stream counters int32 [B] or None, shared frame0); a negative counter skips the stream in that call.
def restart_schedule(B):
    """One-frame calls with per-stream counters in which two streams restart at frame 0 in call K + 1.  ``b_own`` reaches frame
    ``ring`` (slot 0: its own frame of call K) in call K, ``b_prev`` frame ``ring + 1`` (its window's older frame, written by
    call K - 1, is in slot 0); every other stream advances one frame per call.  Returns (calls, K, b_own, b_prev)."""
    ring = ring_slots(2, SMOOTH)
    K, b_own, b_prev = ring + 1, B // 3, B - 1
    frames = np.zeros(B, np.int64)
    calls = []
    for k in range(K + 3):
        active = np.ones(B, bool)
        active[b_own] = k > 0                                         # (joins one call late: frame ring, not ring + 1, in call K)
        if k == K + 1:
            frames[[b_own, b_prev]] = 0                               # MultiStreamEstimator.reset_stream
        sf = np.where(active, frames, -1).astype(np.int32)
        frames[active] += 1
        calls.append((1, sf, 0))
    return calls, K, b_own, b_prev


def reset_schedule():
    """One-frame calls on the shared counter: frames 0 .. ring, reset(), 0 .. ring + 1, reset(), 0 .. 1.  The last call before
    each reset has its own frame (first reset) / the frame before it (second reset) in slot 0.  Returns (calls, [K1, K2])."""
    ring = ring_slots(2, SMOOTH)
    f0s = list(range(ring + 1)) + list(range(ring + 2)) + [0, 1]
    return [(1, None, f) for f in f0s], [ring, 2 * ring + 2]


def matrix_schedule(B, n_calls, seed=5):
    """Two-frame calls with per-stream counters: a quarter of the streams idle per call at random, a block of 16 streams joins in
    call 5, one stream restarts in call 7, calls 5 and n_calls - 2 are short (one frame).  Returns (calls, late block, restart)."""
    rng = np.random.default_rng(seed)
    late, restart, restart_at = range(B // 4, B // 4 + 16), B // 2 + 3, 7
    frames = np.zeros(B, np.int64)
    calls = []
    for k in range(n_calls):
        nF = 1 if k in (5, n_calls - 2) else 2
        active = rng.random(B) >= 0.25
        active[list(late)] &= k >= 5
        if k == restart_at:
            frames[restart] = 0
        active[restart] |= k in (restart_at - 1, restart_at)
        sf = np.where(active, frames, -1).astype(np.int32)
        frames[active] += nF
        calls.append((nF, sf, 0))
    return calls, late, restart


def call_frames(call, B):
    """Per-stream frame of a call's first row (negative: skipped)."""
    nF, sf, f0 = call
    return np.full(B, f0, np.int64) if sf is None else sf.astype(np.int64)


def overwritten_window_slots(calls, k, b, ring):
    """Prediction slots of stream ``b`` that call k's smoothing windows read and call k + 1 writes."""
    f, f1 = (c[2] if c[1] is None else int(c[1][b]) for c in (calls[k], calls[k + 1]))
    if f < 0 or f1 < 0:
        return set()
    read = {s for j in range(calls[k][0]) for s in window_slots(f + j, SMOOTH, ring)}
    return read & {(f1 + j) % ring for j in range(calls[k + 1][0])}


def histories(calls, B):
    """Per stream: its segments (a restart or a reset opens one; each starts at frame 0) as lists of (call, row in call, column)."""
    hist, nxt, col = [[] for _ in range(B)], np.full(B, -1, np.int64), 0
    for k, call in enumerate(calls):
        nF, fr = call[0], call_frames(call, B)
        for b in np.flatnonzero(fr >= 0):
            if fr[b] != nxt[b]:
                assert fr[b] == 0, f"stream {b} starts a segment at frame {fr[b]}"
                hist[b].append([])
            hist[b][-1] += [(k, j, col + j) for j in range(nF)]
            nxt[b] = fr[b] + nF
        col += nF
    return hist


# ---- driving an estimator -------------------------------------------------------------------------------------------------------
def pipeline_streams(est):
    """The four streams of a pipelined estimator (side, lane 0, lane 1, copy) as torch streams."""
    if est._pipe is None:
        return [est.side_stream, est.lane_streams[0], est.lane_streams[1], est.copy_stream]
    out = []
    for which in range(4):
        s = ctypes.c_void_p(None)
        N.check(est.lib.ape_pipeline_stream(est._pipe, which, ctypes.byref(s)), "ape_pipeline_stream")
        out.append(torch.cuda.ExternalStream(s.value, device=est.device))
    return out


def run(est, rows, calls, holds=None):
    """Submit the schedule with at most N_SLOTS - 1 calls outstanding; ``holds`` {call: stream name or "lane" (the lane call k will
    take)}: hold that stream just before submitting call k.  A shared frame0 of 0 after call 0 is a reset().  Returns per call host
    copies of (msg, std, samples, status)."""
    holds = holds or {}
    streams = pipeline_streams(est) if holds else None
    got, pending, col = [], [], 0
    for k, (nF, sf, f0) in enumerate(calls):
        if len(pending) == est.N_SLOTS - 1:
            got.append(_copy(pending.pop(0).result()))
        if sf is None and f0 == 0 and k > 0:
            est.reset()
        if k in holds:
            which = 1 + (est.calls & 1) if holds[k] == "lane" else STREAMS.index(holds[k])
            with torch.cuda.stream(streams[which]):
                torch.cuda._sleep(HOLD_CYCLES)
        pending.append(est.submit(rows[:, col:col + nF], stream_frames=sf))
        assert sf is not None or pending[-1].frame0 == f0
        col += nF
    got += [_copy(p.result()) for p in pending]
    return got


def _copy(o):
    return o.msg.copy(), o.std.copy(), o.samples.copy(), o.status.copy()


def assert_bit_equal(got, want, calls, B, what):
    for k, (g, w) in enumerate(zip(got, want)):
        act = call_frames(calls[k], B) >= 0
        for name, x, y in zip(("msg", "std", "samples", "status"), g, w):
            x, y = x.view(np.int32)[act], y.view(np.int32)[act]
            if not np.array_equal(x, y):
                bad = np.flatnonzero(act)[(x != y).reshape(len(x), -1).any(axis=1)]
                raise AssertionError(f"{what}: call {k}: {name} differs from the serial estimator on {len(bad)} streams "
                                     f"(first {bad[:8].tolist()})")


def oracle_check(kind, state, n, rows, got, hist, streams):
    """The serial results of ``streams`` against OracleEstimator, segment by segment with each stream's own Philox masks."""
    from oracle import estimator as OE
    spec = syn.kind_spec(kind)
    L, T, H, p = spec["L"], spec["T"], spec["H"], spec["p"]
    worst, n_checked = 0.0, 0
    for b in streams:
        assert hist[b], f"stream {b} never ran"
        for seg in hist[b]:
            masks = philox_masks(SEED, b, len(seg), 0, L, T, n, H, p)
            orc = OE.OracleEstimator(syn.KIND_NAMES[kind], spec["lookup"], state, spec["stats"], spec["y_targets"].name, T, SMOOTH, n,
                                     None, p, mask_source=lambda f, m=masks: list(m[f]))
            for k, j, col in seg:
                want = np.asarray(orc.step(rows[b, col]), np.float64)
                pos, q = msg_errors(got[k][0][b, j], want[:25])
                pos = max(pos, float(np.abs(got[k][2][b, j].ravel() - want[25:]).max()))
                assert pos <= POS_TOL and q <= QUAT_TOL, f"stream {b}, call {k}: position {pos:.3g} m, quaternion {q:.3g} vs the oracle"
                worst = max(worst, pos)
                n_checked += 1
    return worst, n_checked


_SERIAL = {}


def serial_reference(key, kind, state, B, n, nF_max, calls, rows, check_streams, knobs):
    """Results of a ``pipeline=False`` estimator on the schedule (computed once per key), its ``check_streams`` vs the oracle."""
    if key not in _SERIAL:
        ref = _estimator(kind, state, B, n, nF_max, smooth=SMOOTH, pipeline=False, **knobs)
        assert not ref.pipeline and ref._pipe is None
        want = run(ref, rows, calls)
        worst, n_checked = oracle_check(kind, state, n, rows, want, histories(calls, B), check_streams)
        print(f"pipeline_order [serial {key}]: {n_checked} estimates of streams {list(check_streams)} vs the oracle, worst {worst:.3g} m")
        _SERIAL[key] = want
    return _SERIAL[key]


def pipelined(kind, state, B, n, nF_max, native, knobs):
    est = _estimator(kind, state, B, n, nF_max, smooth=SMOOTH, native_pipeline=native, **knobs)
    assert est.pipeline and est.lanes and not est.small_batch and est.tc_flags != 4       # the two-lane pipeline, no cluster kernel
    assert (est._pipe is not None) == native
    assert est.pred_ring == ring_slots(2 * nF_max, SMOOTH)
    return est


# ---- a / b. a stream that goes back while the previous call may still read its slot ------------------------------------------
# (name, kind, B, n, estimator knobs, tc_flags, H, launches per call)
KERNELS = [
    ("tc", syn.KIND_UARM, 64, 100, dict(lstm_variant="tc", tc_flags=1, small_batch_kernel=False), 1, 128, 2 + 3),
    ("tcw", syn.KIND_UARM, 1024, 100, dict(lstm_variant="tc", tc_flags=2), 2, 128, 2 + 2),
    ("tcs", syn.KIND_POCKET, 300, 7, dict(lstm_variant="tc", tc_flags=1, small_batch_kernel=False), 1, 256, 2 + 2),
    ("tcx", syn.KIND_UARM, 40, 100, dict(lstm_variant="tcx"), 3, 128, 2 + 3),
    ("tcxs", syn.KIND_POCKET, 300, 7, dict(lstm_variant="tcx"), 3, 256, 2 + 2),
]
KERNEL_IDS = [f"{c[0]}-{syn.KIND_NAMES[c[1]]}-{c[2]}x{c[3]}" for c in KERNELS]


def _check_kernel(est, name, tc_flags, H, launches, n_calls):
    assert est.tc_flags == tc_flags and est.H == H and est.tc_split == (name in ("tcx", "tcxs"))
    assert est.launches == n_calls * launches, f"launches {est.launches} != {n_calls} x {launches}"


@pytest.mark.parametrize("native", [True, False], ids=["native", "python"])
@pytest.mark.parametrize("name,kind,B,n,knobs,tc_flags,H,launches", KERNELS, ids=KERNEL_IDS)
def test_restarted_stream_waits_for_the_previous_window(name, kind, B, n, knobs, tc_flags, H, launches, native):
    spec, state = _model(kind, False)
    calls, K, b_own, b_prev = restart_schedule(B)
    ring = ring_slots(2, SMOOTH)
    # the aliasing the hold exposes: call K + 1 writes frame 0 into a slot call K's window reads
    assert overwritten_window_slots(calls, K, b_own, ring) == {int(calls[K][1][b_own]) % ring}
    assert overwritten_window_slots(calls, K, b_prev, ring) == {(int(calls[K][1][b_prev]) - 1) % ring}
    assert all(pred_window_alias(calls[K + 1][1][b], 1, calls[K][1][b], 1, SMOOTH, ring) for b in (b_own, b_prev))
    rows = syn.synth_rows(kind, B, len(calls), config_id=80 + kind)
    want = serial_reference(("restart", name, B, n), kind, state, B, n, 1, calls, rows, (b_own, b_prev), knobs)
    est = pipelined(kind, state, B, n, 1, native, knobs)
    got = run(est, rows, calls, holds={K: "lane"})
    _check_kernel(est, name, tc_flags, H, launches, len(calls))
    assert_bit_equal(got, want, calls, B, f"{name} {'native' if native else 'python'} restart")
    print(f"pipeline_order [restart] {name} {syn.KIND_NAMES[kind]} {B} x {n} {'native' if native else 'python'}: lane of call {K} "
          f"held, streams {b_own} / {b_prev} restart in call {K + 1}; {len(calls)} calls bit-equal to the serial estimator")


@pytest.mark.parametrize("native", [True, False], ids=["native", "python"])
@pytest.mark.parametrize("name,kind,B,n,knobs,tc_flags,H,launches", KERNELS, ids=KERNEL_IDS)
def test_reset_in_flight_waits_for_the_previous_window(name, kind, B, n, knobs, tc_flags, H, launches, native):
    spec, state = _model(kind, False)
    calls, Ks = reset_schedule()
    ring = ring_slots(2, SMOOTH)
    assert overwritten_window_slots(calls, Ks[0], 0, ring) == {calls[Ks[0]][2] % ring}
    assert overwritten_window_slots(calls, Ks[1], 0, ring) == {(calls[Ks[1]][2] - 1) % ring}
    rows = syn.synth_rows(kind, B, len(calls), config_id=90 + kind)
    want = serial_reference(("reset", name, B, n), kind, state, B, n, 1, calls, rows, (0, B - 1), knobs)
    est = pipelined(kind, state, B, n, 1, native, knobs)
    got = run(est, rows, calls, holds={k: "lane" for k in Ks})
    _check_kernel(est, name, tc_flags, H, launches, len(calls))
    assert_bit_equal(got, want, calls, B, f"{name} {'native' if native else 'python'} reset")
    print(f"pipeline_order [reset] {name} {syn.KIND_NAMES[kind]} {B} x {n} {'native' if native else 'python'}: lanes of calls {Ks} "
          f"held before the resets; {len(calls)} calls bit-equal to the serial estimator")


# ---- c. the hold matrix ------------------------------------------------------------------------------------------------------
MATRIX_MODELS = [("tcw", syn.KIND_UARM, dict(lstm_variant="tc", tc_flags=2), 2), ("tcs", syn.KIND_POCKET, dict(lstm_variant="tc"), 0)]
MATRIX_B, MATRIX_N, MATRIX_NF = 256, 20, 2
MATRIX_CALLS = BatchedEstimator.N_SLOTS + 4        # every result slot and all four buffer sets wrap


@pytest.mark.parametrize("at", [3, BatchedEstimator.N_SLOTS], ids=lambda a: f"call{a}")
@pytest.mark.parametrize("stream", STREAMS)
@pytest.mark.parametrize("native", [True, False], ids=["native", "python"])
@pytest.mark.parametrize("name,kind,knobs,tc_flags", MATRIX_MODELS, ids=[m[0] for m in MATRIX_MODELS])
def test_hold_matrix(name, kind, knobs, tc_flags, native, stream, at):
    spec, state = _model(kind, False)
    B, n = MATRIX_B, MATRIX_N
    calls, late, restart = matrix_schedule(B, MATRIX_CALLS)
    rows = syn.synth_rows(kind, B, sum(c[0] for c in calls), config_id=100 + kind)
    want = serial_reference(("matrix", name), kind, state, B, n, MATRIX_NF, calls, rows, (restart, late[0]), knobs)
    est = pipelined(kind, state, B, n, MATRIX_NF, native, knobs)
    got = run(est, rows, calls, holds={at: stream})
    assert est.tc_flags == tc_flags and est.launches == len(calls) * 4
    assert_bit_equal(got, want, calls, B, f"{name} {'native' if native else 'python'} {stream} held before call {at}")
    print(f"pipeline_order [matrix] {name} {B} x {n} {'native' if native else 'python'}: {stream} held before call {at}; "
          f"{len(calls)} calls bit-equal to the serial estimator")
