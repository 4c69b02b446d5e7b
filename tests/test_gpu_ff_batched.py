"""GPU: the MC-dropout feed-forward regressors (DropoutFF / DropoutFF2D) on the batched estimation path.

* ``ape_mc_ff_ring`` (the ring mode of csrc/ape_ff.cu) is bit-identical to ``ape_mc_ff`` on the same windows gathered on the host,
  called with stream id ``stream_id0 + b`` and frame ``f`` per row; streams that sit a call out keep every prediction slot.
* ``BatchedEstimator`` built from a feed-forward state dict matches a test-local oracle loop (oracle.features -> z-score ->
  oracle.ff on the flattened window -> oracle.fk) within 1e-4 m, and its entry points, shards and downstream users agree bit for bit.
"""
import queue

import numpy as np
import pytest
import torch

from arm_pose_estimation_b200 import _native as N, synthetic as syn
from arm_pose_estimation_b200.estimate import nn_models
from arm_pose_estimation_b200.estimate.batched import BatchedEstimator, shard_streams
from arm_pose_estimation_b200.estimate.multi_stream import MultiStreamEstimator
from arm_pose_estimation_b200.record import replay
from oracle import estimator as OE
from oracle import ff as OFF

pytestmark = pytest.mark.gpu
P = 0.2
SENTINEL = -7777.25


def _ring(blob, dims, feats, feat_ring, B, nF, frame0, sf, n, mode, masks, seed, sid0, preds, pred_ring):
    I, T, H, Lh, O = dims
    N.check(N.load().ape_mc_ff_ring(N.ptr(blob), I, T, H, Lh, O, P, N.ptr(feats), feat_ring, B, nF, frame0, N.ptr(sf), n, mode,
                                    N.ptr(masks), seed, sid0, N.ptr(preds), pred_ring, N.current_stream_ptr()), "ape_mc_ff_ring")


def _mc_ff(blob, dims, x, n, mode, masks, seed, sid0, frame0):
    I, T, H, Lh, O = dims
    xd = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).cuda()
    preds = torch.empty((x.shape[0], n, O), dtype=torch.float32, device="cuda")
    N.check(N.load().ape_mc_ff(N.ptr(blob), I * T, H, Lh, O, P, N.ptr(xd), x.shape[0], n, mode, N.ptr(masks), seed, sid0, frame0,
                               N.ptr(preds), N.current_stream_ptr()), "ape_mc_ff")
    return preds.cpu().numpy()


RING_CASES = [
    # name, I, T, H, Lh, O, B, nF, frame0, stream_frames, mask mode, stream_id0
    ("uarm-philox-warmup", 38, 6, 256, 2, 12, 13, 3, 1, None, N.MASK_PHILOX, 7),
    ("pocket-injected-idle", 22, 6, 256, 2, 14, 5, 4, 0, [0, -1, 9, 2, -5], N.MASK_INJECTED, 0),
    ("watch-none", 20, 8, 128, 1, 20, 9, 1, 0, None, N.MASK_NONE, 3),
    ("dropout-ff-T1-idle", 20, 1, 64, 0, 20, 3, 2, 0, [4, -1, 0], N.MASK_PHILOX, 100),
    ("uarm-philox-wrap-idle", 38, 6, 256, 2, 12, 11, 2, 0, [37, 0, -1, 5, 12, 1, -1, 3, 22, 8, 2], N.MASK_PHILOX, 1),
    ("pocket-injected-late", 22, 6, 256, 2, 14, 17, 1, 40, None, N.MASK_INJECTED, 0),
    ("O20-philox-frame0", 38, 6, 128, 2, 20, 6, 4, 0, None, N.MASK_PHILOX, 2),
]


@pytest.mark.parametrize("I,T,H,Lh,O,B,nF,frame0,sf,mode,sid0", [c[1:] for c in RING_CASES], ids=[c[0] for c in RING_CASES])
def test_ring_mode_is_bit_identical_to_mc_ff_on_gathered_windows(I, T, H, Lh, O, B, nF, frame0, sf, mode, sid0):
    rng = np.random.default_rng(I * 131 + B)
    dims, n, seed = (I, T, H, Lh, O), 24, 0xF00D
    blob = torch.from_numpy(nn_models.pack_ff_weights(syn.synth_ff_state_dict(T * I, H, Lh, O, seed=I + H))).cuda()
    feat_ring, pred_ring, E = nF + T - 1 + 2, nF + 2, B * nF
    feats_h = rng.normal(0, 1, (B, feat_ring, I)).astype(np.float32)
    feats = torch.from_numpy(feats_h).cuda()
    sf_d = None if sf is None else torch.tensor(sf, dtype=torch.int32, device="cuda")
    masks_h = (rng.random((E, n, H)) < 0.8).astype(np.uint8) if mode == N.MASK_INJECTED else None
    masks = None if masks_h is None else torch.from_numpy(masks_h).cuda()
    preds = torch.full((B, pred_ring, n, O), SENTINEL, dtype=torch.float32, device="cuda")
    _ring(blob, dims, feats, feat_ring, B, nF, frame0, sf_d, n, mode, masks, seed, sid0, preds, pred_ring)
    got = preds.cpu().numpy()
    # the windows on the host: frames f - T + 1 .. f of stream b, frames before 0 read frame 0
    fb = [frame0 if sf is None else sf[b] for b in range(B)]
    x = np.zeros((E, T * I), np.float32)
    for e in range(E):
        b, f = e // nF, fb[e // nF] + e % nF
        if fb[b] >= 0:
            x[e] = np.concatenate([feats_h[b, max(0, f - T + 1 + t) % feat_ring] for t in range(T)])
    if mode == N.MASK_PHILOX:                            # one call per row: its keys are (stream_id0 + b, f)
        ref = np.stack([_mc_ff(blob, dims, x[e:e + 1], n, mode, None, seed, sid0 + e // nF, max(0, fb[e // nF] + e % nF))[0]
                        for e in range(E)])
    else:
        ref = _mc_ff(blob, dims, x, n, mode, masks, seed, 0, 0)
    want = np.full_like(got, SENTINEL)
    for e in range(E):
        b, f = e // nF, fb[e // nF] + e % nF
        if fb[b] >= 0:
            want[b, f % pred_ring] = ref[e]
    assert np.isfinite(got).all()
    np.testing.assert_array_equal(got.view(np.int32), want.view(np.int32))
    if mode == N.MASK_PHILOX:
        assert np.abs(ref[:, 0] - ref[:, 1]).max() > 1e-4          # samples differ


def test_ring_philox_mean_is_the_eval_mode_output():
    """Dropout in front of the (linear) output layer is unbiased: the MC mean of the normalised outputs is the eval-mode output."""
    I, T, H, Lh, O, B, n = 38, 6, 256, 2, 12, 3, 4000
    dims = (I, T, H, Lh, O)
    blob = torch.from_numpy(nn_models.pack_ff_weights(syn.synth_ff_state_dict(T * I, H, Lh, O, seed=5))).cuda()
    feats = torch.from_numpy(np.random.default_rng(8).normal(0, 1, (B, T, I)).astype(np.float32)).cuda()
    out = {}
    for mode in (N.MASK_PHILOX, N.MASK_NONE):
        preds = torch.empty((B, 1, n, O), dtype=torch.float32, device="cuda")
        _ring(blob, dims, feats, T, B, 1, 9, None, n, mode, None, 77, 0, preds, 1)
        out[mode] = preds.cpu().numpy()[:, 0].astype(np.float64)
    y = out[N.MASK_PHILOX]
    y0 = out[N.MASK_NONE][:, 0]
    se = y.std(axis=1) / np.sqrt(n)
    assert (y.std(axis=1) > 0).all()
    assert (np.abs(y.mean(axis=1) - y0) < 5 * se + 1e-5).all()


# ---- BatchedEstimator on a feed-forward model ---------------------------------------------------------------------------------
def _ff_state(kind, model):
    spec = syn.kind_spec(kind)
    width = spec["I"] * (spec["T"] if model == "ff2d" else 1)
    return syn.synth_ff_state_dict(width, 256, 2, spec["O"], seed=99 + kind + (10 if model == "ff2d" else 0))


def _engine(kind, state, B, n, smooth=1, nF=1, mode=N.MASK_PHILOX, first_stream=0, **kw):
    spec = syn.kind_spec(kind)
    return BatchedEstimator(kind=kind, layout=spec["layout"], state=state, seq_len=spec["T"], y_targets=spec["y_targets"],
                            stats=spec["stats"], n_streams=B, mc_samples=n, smooth=smooth, dropout=spec["p"], frames_per_call=nF,
                            mask_mode=mode, philox_seed=21, first_stream=first_stream, **kw)


class FfOracle(OE.OracleEstimator):
    """The oracle's per-stream loop with the feed-forward model: the flattened window (DropoutFF2D) or the newest frame (DropoutFF)."""

    def __init__(self, *args, ff2d=True, **kw):
        super().__init__(*args, **kw)
        self.ff2d = ff2d

    def make_prediction_from_row_hist(self, xx_hist):
        x = np.asarray(xx_hist, dtype=np.float32)
        x = (x if self.ff2d else x[-1:]).reshape(1, -1)
        return OFF.forward_with_masks(self.state, np.repeat(x, self.n, 0), self.mask_source(self.frame), self.p)


def _oracle(kind, state, model, smooth, n, masks_b):
    spec = syn.kind_spec(kind)
    return FfOracle(syn.KIND_NAMES[kind], spec["lookup"], state, spec["stats"], spec["y_targets"].name, spec["T"], smooth, n, None,
                    spec["p"], mask_source=lambda f, m=masks_b: m[f], ff2d=model == "ff2d")


ORACLE_CASES = [(k, m, s) for k in (syn.KIND_WATCH_ONLY, syn.KIND_POCKET, syn.KIND_UARM) for m, s in (("ff2d", 1), ("ff2d", 3), ("ff", 3))]


@pytest.mark.parametrize("kind,model,smooth", ORACLE_CASES,
                         ids=[f"{syn.KIND_NAMES[k]}-{m}-smooth{s}" for k, m, s in ORACLE_CASES])
def test_batched_ff_matches_the_oracle_loop(kind, model, smooth):
    B, F, nF, n = 3, 7, 2, 16
    spec = syn.kind_spec(kind)
    state = _ff_state(kind, model)
    be = _engine(kind, state, B, n, smooth, nF=nF, mode=N.MASK_INJECTED)
    assert be.ff and be.T == (spec["T"] if model == "ff2d" else 1) and be.lstm_variant == "fp32" and be._pipe is None
    rows = syn.synth_rows(kind, B, F, config_id=3)
    masks = (np.random.default_rng(kind).random((B, F, n, be.H)) < 1 - spec["p"]).astype(np.uint8)
    msg, samples = [], []
    for f0 in range(0, F, nF):
        out = be.step(rows[:, f0:f0 + nF], masks=masks[:, f0:f0 + nF])
        assert (out.status == 0).all()
        msg.append(out.msg.copy())
        samples.append(out.samples.copy())
    msg, samples = np.concatenate(msg, 1), np.concatenate(samples, 1)
    worst = 0.0
    for b in range(B):
        orc = _oracle(kind, state, model, smooth, n, masks[b])
        for f in range(F):
            want = np.asarray(orc.step(rows[b, f]), dtype=np.float64)
            for a, c in ((4, 7), (11, 14), (18, 21)):                          # hand, elbow, shoulder positions
                worst = max(worst, float(np.abs(msg[b, f, a:c] - want[a:c]).max()))
            worst = max(worst, float(np.abs(samples[b, f].ravel() - want[25:]).max()))
    print(f"{syn.KIND_NAMES[kind]} {model} smooth {smooth}: worst position error vs the oracle {worst:.3g} m")
    assert worst <= 1e-4


def test_batched_ff_step_features_matches_the_oracle():
    kind, B, F, n, smooth = syn.KIND_POCKET, 2, 5, 8, 2
    spec = syn.kind_spec(kind)
    state = _ff_state(kind, "ff2d")
    be = _engine(kind, state, B, n, smooth, mode=N.MASK_INJECTED)
    rows = syn.synth_rows(kind, B, F, config_id=4)
    masks = (np.random.default_rng(1).random((B, F, n, be.H)) < 0.8).astype(np.uint8)
    orcs = [_oracle(kind, state, "ff2d", smooth, n, masks[b]) for b in range(B)]
    for f in range(F):
        xx = np.stack([orcs[b].parse_row_to_xx(rows[b, f]) for b in range(B)])
        got = be.step_features(xx, masks=masks[:, f:f + 1])
        for b in range(B):
            np.testing.assert_allclose(got[b], orcs[b].add_xx_to_row_hist_and_make_prediction(xx[b]), atol=5e-5, rtol=0)
    assert be.launches == 2 * F


def _same(a, b):
    for x, y in ((a.msg, b.msg), (a.std, b.std), (a.status, b.status), (a.samples, b.samples)):
        np.testing.assert_array_equal(np.asarray(x), np.asarray(y))


def test_batched_ff_entry_points_agree_bit_for_bit():
    kind, B, F, n, smooth = syn.KIND_UARM, 5, 6, 20, 2
    state = _ff_state(kind, "ff2d")
    rows = syn.synth_rows(kind, B, F, config_id=5)
    ref = _engine(kind, state, B, n, smooth)
    want = [ref.step(rows[:, f]) for f in range(F)]
    want = [type(w)(w.msg.copy(), w.std.copy(), w.samples.copy(), w.status.copy(), w.frame0) for w in want]
    assert ref.launches == 3 * F
    sub = _engine(kind, state, B, n, smooth)
    pend = [sub.submit(rows[:, f]) for f in range(F)]
    for w, p in zip(want, pend):
        _same(w, p.result())
    dev = _engine(kind, state, B, n, smooth)
    for f in range(F):
        _same(want[f], dev.step_device(torch.from_numpy(rows[:, f:f + 1].copy()).cuda()).host())
    gr = _engine(kind, state, B, n, smooth)
    for f in range(F):
        _same(want[f], gr.step_graph(rows[:, f]))
    assert gr.launches == 3 * F
    multi = _engine(kind, state, B, n, smooth, nF=3)             # one call of three frames = three single-frame calls
    for f0 in (0, 3):
        out = multi.step(rows[:, f0:f0 + 3])
        for j in range(3):
            for x, y in ((out.msg, want[f0 + j].msg), (out.std, want[f0 + j].std), (out.samples, want[f0 + j].samples)):
                np.testing.assert_array_equal(x[:, j:j + 1], y)
    lean = _engine(kind, state, B, n, smooth, emit_samples=False)
    for f in range(F):
        out = lean.step(rows[:, f])
        assert out.samples is None
        np.testing.assert_array_equal(out.msg, want[f].msg)
    for world in (2, 3):                                       # shards with first_stream = slices of the unsharded run
        for rank in range(world):
            first, count = shard_streams(B, world, rank)
            shard = _engine(kind, state, count, n, smooth, first_stream=first)
            for f in range(F):
                out = shard.step(rows[first:first + count, f])
                np.testing.assert_array_equal(out.msg, want[f].msg[first:first + count])
                np.testing.assert_array_equal(out.samples, want[f].samples[first:first + count])


def test_batched_ff_refuses_tensor_core_variants_and_bad_masks():
    state = _ff_state(syn.KIND_POCKET, "ff2d")
    for variant in ("tc", "tcx"):
        with pytest.raises(UserWarning):
            _engine(syn.KIND_POCKET, state, 2, 8, lstm_variant=variant)
    with pytest.raises(UserWarning):                             # a width that is neither the window nor one frame
        _engine(syn.KIND_POCKET, syn.synth_ff_state_dict(5 * 22, 64, 1, 14), 2, 8)
    be = _engine(syn.KIND_POCKET, state, 2, 8, mode=N.MASK_INJECTED)
    rows = syn.synth_rows(syn.KIND_POCKET, 2, 1)
    with pytest.raises(UserWarning):
        be.step(rows)
    with pytest.raises(UserWarning):
        be.step(rows, masks=np.ones((2, 1, 8, 255), np.uint8))


def test_multi_stream_over_a_ff_engine_matches_single_stream_engines():
    kind, B, n, smooth, F = syn.KIND_WATCH_ONLY, 4, 12, 3, 9
    state = _ff_state(kind, "ff2d")
    rows = syn.synth_rows(kind, B, F, config_id=17)
    rng = np.random.default_rng(5)
    ms = MultiStreamEstimator(_engine(kind, state, B, n, smooth), add_mc_samples=True)
    qs = [queue.Queue() for _ in range(B)]
    fed = [0] * B
    got = [[] for _ in range(B)]
    for tick in range(40):
        for b in range(B):
            arrives = rng.random() < (0.8, 0.4, 0.9, 0.6)[b] and not (b == 3 and tick < 6) and not (b == 1 and 10 <= tick < 20)
            if arrives and fed[b] < F:
                qs[b].put(rows[b, fed[b]])
                fed[b] += 1
        for b, m in ms.tick(ms.collect(qs)).items():
            got[b].append(np.asarray(m))
    assert [len(g) for g in got] == fed and min(fed) >= 5
    for b in range(B):
        solo = _engine(kind, state, 1, n, smooth, first_stream=b)
        for f in range(fed[b]):
            out = solo.step(rows[b:b + 1, f:f + 1])
            want = np.concatenate([out.msg[0, 0].astype(np.float64), out.samples[0, 0].astype(np.float64).ravel()])
            np.testing.assert_array_equal(got[b][f], want)


def test_relabel_recordings_with_a_ff_engine_equals_frame_by_frame_stepping():
    kind, R, F, n = syn.KIND_POCKET, 3, 11, 10
    state = _ff_state(kind, "ff")
    rows = syn.synth_rows(kind, R, F, config_id=9)
    masks = (np.random.default_rng(2).random((R, F, n, 256)) < 0.8).astype(np.uint8)
    res = replay.relabel_recordings(rows, lambda nS, fpc: _engine(kind, state, nS, n, 2, nF=fpc, mode=N.MASK_INJECTED),
                                    frames_per_call=4, keep_samples=True, masks=masks)
    one = _engine(kind, state, R, n, 2, mode=N.MASK_INJECTED)
    for f in range(F):
        out = one.step(rows[:, f], masks=masks[:, f:f + 1])
        for r in range(R):
            np.testing.assert_array_equal(res[r]["msg"][f], out.msg[r, 0].astype(np.float64))
            np.testing.assert_array_equal(res[r]["samples"][f], out.samples[r, 0])
