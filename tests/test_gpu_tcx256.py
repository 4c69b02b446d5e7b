"""GPU (-m gpu): the split-precision tensor-core kernel for H = 256 (csrc/ape_lstm_tcxs.cu: every operand an fp16 pair hi + lo, three
tcgen05 passes per product, ex2 / rcp cell update; h_t staged through L2 into single-buffered TMEM operands) - the tensor-core path
of the watch-only and pocket models when the single-pass kernel fails its probe.  Checked against the reference's own messages, against
the oracle with injected masks at weight scales 1x .. 8x, against the fp32 kernel on ragged / multi-tile shapes under Philox, on
L = 3 / T = 1 / odd T / O = 20 shapes, per stream against dedicated estimators, and through the pipeline."""
import queue

import numpy as np
import pytest
import torch

from conftest import load_golden, unpack_masks
from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200 import synthetic as syn
from arm_pose_estimation_b200.estimate import nn_models
from arm_pose_estimation_b200.estimate.batched import BatchedEstimator
from arm_pose_estimation_b200.estimate.multi_stream import MultiStreamEstimator
from oracle import estimator as OE
from oracle import lstm as OL
from test_gpu_parity import msg_close, POS_TOL
from test_gpu_tc import make, _scaled_state

pytestmark = pytest.mark.gpu
H256_KINDS = [syn.KIND_WATCH_ONLY, syn.KIND_POCKET]


@pytest.mark.parametrize("kind,name", [(syn.KIND_WATCH_ONLY, "watch_only_s3"), (syn.KIND_POCKET, "pocket_s1")])
def test_split256_whole_path_against_reference_messages(kind, name):
    g = load_golden(f"e2e_{name}.npz")
    n, smooth = int(g["n"]), int(g["smooth"])
    masks = unpack_masks(g)
    rows, F = g["rows"], len(g["rows"])
    be, spec, _ = make(kind, 1, n, "tcx", smooth=smooth, frames_per_call=F, mask_mode=N.MASK_INJECTED)
    assert be.lstm_variant == "tc" and be.tc_split and spec["H"] == 256
    out = be.step(rows[None], masks=masks[None])
    worst = msg_close(out.msg[0], g["msgs"][:, :25])
    err = np.abs(out.samples[0].reshape(F, -1) - g["msgs"][:, 25:]).max()
    print(f"{name} H = 256 split-precision path: worst position error vs the reference's messages {max(worst, err):.3g} m "
          f"(probe {be.tcx_probe_error_m:.3g} m)")
    assert err <= 1e-5


@pytest.mark.parametrize("kind", H256_KINDS)
@pytest.mark.parametrize("scale,forget_bias", [(1.0, 0.0), (1.0, 1.0), (2.0, 1.0), (4.0, 0.0), (8.0, 1.0)])
def test_split256_weight_scale_sweep_against_oracle(kind, scale, forget_bias):
    # the sweep of test_gpu_tc.py::test_weight_scale_sweep_against_oracle (same states, rows and masks): the split kernel holds 1e-4 m
    # at every scale, and "auto" ends on a tensor-core path - the split one whenever the single-pass probe exceeds its tolerance
    spec = syn.kind_spec(kind)
    B, nF, n = 2, 2, 48
    state = _scaled_state(kind, scale, forget_bias)
    rng = np.random.default_rng(int(scale * 10) + kind)
    rows = syn.synth_rows(kind, B, nF, config_id=44)
    masks = (rng.random(size=(B, nF, spec["L"] - 1, spec["T"], n, spec["H"])) < 0.8).astype(np.uint8)
    want = []
    for b in range(B):
        orc = OE.OracleEstimator(syn.KIND_NAMES[kind], spec["lookup"], state, spec["stats"], spec["y_targets"].name, spec["T"], 1, n,
                                 None, spec["p"], mask_source=lambda f, b=b: list(masks[b, f]))
        want.append([np.asarray(orc.step(rows[b, f])) for f in range(nF)])
    errs = {}
    for variant in ("tcx", "auto"):
        be, _, _ = make(kind, B, n, variant, state=state, frames_per_call=nF, mask_mode=N.MASK_INJECTED)
        out = be.step(rows, masks=masks)
        worst = 0.0
        for b in range(B):
            for f in range(nF):
                w = want[b][f]
                for a, c in ((4, 7), (11, 14), (18, 21)):
                    worst = max(worst, float(np.abs(out.msg[b, f, a:c] - w[a:c]).max()))
                worst = max(worst, float(np.abs(out.samples[b, f].ravel() - w[25:]).max()))
        errs[variant] = (worst, be.lstm_variant, be.tc_split, be.tc_probe_error_m, be.tcx_probe_error_m)
    print(f"{syn.KIND_NAMES[kind]} weights x{scale} forget bias +{forget_bias}: split precision {errs['tcx'][0]:.3g} m "
          f"(probe {errs['tcx'][4]:.3g} m); auto -> {'split' if errs['auto'][2] else 'single pass'} {errs['auto'][0]:.3g} m "
          f"(single-pass probe {errs['auto'][3]:.3g} m)")
    assert errs["tcx"][0] <= POS_TOL
    assert errs["auto"][1] == "tc" and errs["auto"][0] <= POS_TOL
    if errs["auto"][3] > 5e-5:
        assert errs["auto"][2]


@pytest.mark.parametrize("kind", H256_KINDS)
@pytest.mark.parametrize("B,n", [(1, 1), (3, 70), (5, 100), (200, 100)])
def test_split256_matches_fp32_kernel_with_philox(kind, B, n):
    # ragged row counts, one row, and 79 tiles > 74 CTA pairs (a pair runs on across tile boundaries)
    nF = 2
    rows = np.tile(syn.synth_rows(kind, min(B, 8), 3 * nF, config_id=7), ((B + 7) // 8, 1, 1))[:B]
    kw = dict(frames_per_call=nF, mask_mode=N.MASK_PHILOX, philox_seed=3, smooth=2)
    x, _, _ = make(kind, B, n, "tcx", **kw)
    r, _, _ = make(kind, B, n, "fp32", **kw)
    assert x.tc_split
    for c in range(3):
        a, b = x.step(rows[:, c * nF:(c + 1) * nF]), r.step(rows[:, c * nF:(c + 1) * nF])
        d = max(float(np.abs(a.samples - b.samples).max()), float(np.abs(a.msg - b.msg).max()), float(np.abs(a.std - b.std).max()))
        print(f"{syn.KIND_NAMES[kind]} split precision vs fp32 kernel, {B} x {nF} x {n}, call {c}: max |difference| {d:.3g} m")
        assert np.isfinite(a.msg).all() and d <= 5e-6


def _lstm_preds(state, x, masks, n, p, split):
    """Raw LSTM outputs of the last step through ape_mc_lstm_tc (tc_flags = 3) or ape_mc_lstm_fma: x (E, T, I), masks (E, L-1, T, n, H)."""
    I, H, L, O = OL.lstm_dims(state)
    E, T, _ = x.shape
    dev = torch.device("cuda")
    xd = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(dev)
    md = torch.from_numpy(np.ascontiguousarray(masks, dtype=np.uint8)).to(dev)
    w = torch.from_numpy(nn_models.pack_lstm_weights(state)).to(dev)
    wx = torch.from_numpy(nn_models.pack_lstm_weights_tcx(state)).to(dev) if split else None
    ws = torch.empty(N.tcxs_workspace_bytes(I, H, L, T, O, E, n) if split else N.workspace_bytes(I, H, L, T, O, E, n),
                     dtype=torch.uint8, device=dev)
    preds = torch.zeros((E, 1, n, O), dtype=torch.float32, device=dev)
    a = N.LstmArgs()
    a.weights = w.data_ptr()
    a.I, a.H, a.L, a.T, a.O = I, H, L, T, O
    a.dropout_p = p
    a.x_dense, a.feat_ring_buf, a.feat_ring = xd.data_ptr(), None, 0
    a.B, a.nF, a.frame0, a.n_samples = E, 1, 0, n
    a.mask_mode, a.masks = N.MASK_INJECTED, md.data_ptr()
    a.workspace = ws.data_ptr()
    a.preds, a.pred_ring, a.all_steps = preds.data_ptr(), 1, 0
    if split:
        a.weights_tcx, a.tc_flags = wx.data_ptr(), 3
    lib = N.load()
    fn = lib.ape_mc_lstm_tc if split else lib.ape_mc_lstm_fma
    N.check(fn(a, N.current_stream_ptr()), "ape_mc_lstm")
    torch.cuda.synchronize()
    return preds.cpu().numpy()[:, 0]


@pytest.mark.parametrize("I,L,T,O", [(20, 3, 8, 12), (22, 2, 1, 14), (20, 2, 7, 20), (38, 3, 5, 20)])
def test_split256_shapes_against_oracle(I, L, T, O):
    # L = 3: a middle layer that reads and writes hi / lo units through HBM; T = 1: no recurrent product at all; odd T; O = 20
    H, E, n, p = 256, 6, 50, 0.2
    state = syn.synth_state_dict(I, H, L, O, 100 + I + L + T + O)
    rng = np.random.default_rng(I * L * T)
    x = rng.standard_normal((E, T, I)).astype(np.float32)
    masks = (rng.random(size=(E, L - 1, T, n, H)) < 1 - p).astype(np.uint8)
    got = _lstm_preds(state, x, masks, n, p, split=True)
    ref = _lstm_preds(state, x, masks, n, p, split=False)
    om = [np.ascontiguousarray(masks[:, g].transpose(1, 0, 2, 3).reshape(T, E * n, H)) for g in range(L - 1)]
    want = OL.forward_with_masks(state, np.repeat(x, n, axis=0), om, p=p, last_only=True).reshape(E, n, O)
    d_or, d_fp = float(np.abs(got - want).max()), float(np.abs(got - ref).max())
    print(f"I{I} H256 L{L} T{T} O{O}: split kernel vs oracle {d_or:.3g}, vs fp32 kernel {d_fp:.3g} (raw outputs)")
    assert np.isfinite(got).all() and d_or <= 2e-5 and d_fp <= 2e-5


def test_split256_per_stream_frames_match_dedicated_estimators():
    # the multi-stream front-end drives per-stream frame counters (streams without a row sit a call out: -1); every stream's
    # estimates must be bit-equal to those of a dedicated single-stream estimator on the split kernel
    kind, B, n, smooth, F = syn.KIND_POCKET, 4, 20, 3, 7
    spec = syn.kind_spec(kind)
    state = syn.synth_state_dict(spec["I"], spec["H"], spec["L"], spec["O"], 1234 + kind)

    def engine(n_streams, first_stream):
        return BatchedEstimator(kind=kind, layout=spec["layout"], state=state, seq_len=spec["T"], y_targets=spec["y_targets"],
                                stats=spec["stats"], n_streams=n_streams, mc_samples=n, smooth=smooth, dropout=spec["p"],
                                frames_per_call=1, mask_mode=N.MASK_PHILOX, philox_seed=11, first_stream=first_stream,
                                lstm_variant="tcx")

    rows = syn.synth_rows(kind, B, F, config_id=17)
    rng = np.random.default_rng(5)
    eng = engine(B, 0)
    assert eng.tc_split
    ms = MultiStreamEstimator(eng, add_mc_samples=True)
    qs = [queue.Queue() for _ in range(B)]
    fed, got, idle = [0] * B, [[] for _ in range(B)], 0
    for tick in range(30):
        for b in range(B):
            arrives = rng.random() < (0.8, 0.4, 0.9, 0.6)[b] and not (b == 3 and tick < 4) and not (b == 1 and 6 <= tick < 12)
            if arrives and fed[b] < F:
                qs[b].put(rows[b, fed[b]])
                fed[b] += 1
        active = ms.collect(qs)
        idle += int(active.any() and not active.all())
        for b, m in ms.tick(active).items():
            got[b].append(np.asarray(m))
    assert [len(g) for g in got] == fed and min(fed) >= 4 and idle > 0
    for b in range(B):
        solo = engine(1, b)
        for f in range(fed[b]):
            out = solo.step(rows[b:b + 1, f:f + 1])
            want = np.concatenate([out.msg[0, 0].astype(np.float64), out.samples[0, 0].astype(np.float64).ravel()])
            np.testing.assert_array_equal(got[b][f], want)


def test_split256_pipeline_is_bitwise_invisible_and_repeats():
    # submitted back to back through the native pipeline vs one call at a time; then the full 1024 x 100 batch twice, bit for bit
    kind, B, n, calls = syn.KIND_WATCH_ONLY, 300, 100, 4
    rows = np.tile(syn.synth_rows(kind, 8, calls, config_id=9), (38, 1, 1))[:B]
    kw = dict(frames_per_call=1, mask_mode=N.MASK_PHILOX, philox_seed=8, smooth=3)
    piped, _, _ = make(kind, B, n, "tcx", **kw)
    plain, _, _ = make(kind, B, n, "tcx", pipeline=False, **kw)
    assert piped._pipe is not None and plain._pipe is None and piped.tc_split
    pend = [piped.submit(rows[:, k:k + 1]) for k in range(calls)]
    for k, p in enumerate(pend):
        got, want = p.result(), plain.step(rows[:, k:k + 1])
        np.testing.assert_array_equal(got.msg, want.msg, err_msg=f"call {k}")
        np.testing.assert_array_equal(got.samples, want.samples, err_msg=f"call {k}")
        np.testing.assert_array_equal(got.std, want.std, err_msg=f"call {k}")
    big_rows = np.tile(syn.synth_rows(kind, 8, 1, config_id=3), (128, 1, 1))
    outs = []
    for _ in range(2):
        be, _, _ = make(kind, 1024, 100, "tcx", frames_per_call=1, mask_mode=N.MASK_PHILOX, philox_seed=21, pipeline=False)
        outs.append(be.step(big_rows))
    np.testing.assert_array_equal(outs[0].msg, outs[1].msg)
    np.testing.assert_array_equal(outs[0].samples, outs[1].samples)
    assert np.isfinite(outs[0].msg).all()
