"""GPU (-m gpu): the H = 256 split-precision small-batch kernel (ape_mc_lstm_tcxsl, csrc/ape_lstm_tcxsl.cu: all layers of a call in one
launch, one 16-CTA cluster per 128 rows, the arithmetic of the H = 256 split layer kernels) - what a single-stream watch-only or pocket
estimator whose model fails the single-pass probe runs per frame.
It keeps the split layer kernels' operand splits, MMA order per accumulator, cell update and Philox keys, so it must be BIT-identical to
them; like them it is held against the oracle, the reference's own messages and a float64 restatement of the LSTM."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import load_golden, unpack_masks
from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200 import synthetic as syn
from arm_pose_estimation_b200.estimate import estimator as estimator_module, nn_models
from arm_pose_estimation_b200.estimate.batched import BatchedEstimator
from oracle import estimator as OE
from oracle import lstm as OL
from test_gpu_parity import deploy, msg_close, POS_TOL  # noqa: F401  (deploy: the synthetic deployed models, a fixture)
from test_gpu_tc import make, _scaled_state
import test_gpu_stream_frames as SF
from test_gpu_lstm_envelope import EXACT_TOL, GUARD, PATTERN, inputs, last_step_error, pick, reference, run_lstm, saturating_state

pytestmark = pytest.mark.gpu
KINDS = {"watch_only": syn.KIND_WATCH_ONLY, "pocket": syn.KIND_POCKET}
WEIGHTS = {"1x": (1.0, 0.0), "4x+fb": (4.0, 1.0)}
BOUND = BatchedEstimator.SPLIT256_SMALL_BATCH_ROWS


def test_the_device_holds_a_16_cta_cluster():
    n = N.tcxsl_max_active_clusters()
    print(f"ape_mc_lstm_tcxsl: {n} 16-CTA clusters active at once on {torch.cuda.get_device_name()}")
    assert n >= 1


def _pair(kind, B, n, weights, **kw):
    """The same split-precision estimator on the new kernel and on the split layer kernels."""
    state = _scaled_state(kind, *WEIGHTS[weights])
    small, spec, _ = make(kind, B, n, "tcx", state=state, split_small_batch_kernel=True, **kw)
    layers, _, _ = make(kind, B, n, "tcx", state=state, **kw)
    assert spec["H"] == 256
    assert small.tc_split and small.small_batch and small.tc_flags == 5 and small._pipe is None and not small.pipeline
    assert small._lstm_fn() == small.lib.ape_mc_lstm_tcxsl
    assert layers.tc_split and not layers.small_batch and layers.tc_flags == 3
    return small, layers, spec


def _equal(a, b, what=""):
    assert np.isfinite(a.msg).all()
    np.testing.assert_array_equal(a.samples, b.samples, err_msg=what)
    np.testing.assert_array_equal(a.msg, b.msg, err_msg=what)
    np.testing.assert_array_equal(a.std, b.std, err_msg=what)


@pytest.mark.parametrize("kind", list(KINDS))
@pytest.mark.parametrize("weights", list(WEIGHTS))
@pytest.mark.parametrize("mode", [N.MASK_PHILOX, N.MASK_INJECTED])
@pytest.mark.parametrize("B,n,nF", [(1, 100, 1), (1, 1, 1), (1, 128, 1),
                                    # several clusters: an estimate straddling two, more estimates than a cluster has rows, two frames
                                    # per call, the largest call the estimator gives the kernel
                                    (3, 100, 1), (130, 1, 1), (20, 7, 2), (BOUND // 128, 128, 1)])
def test_split256_small_batch_kernel_is_bit_identical_to_the_split_layer_kernels(kind, B, n, nF, mode, weights):
    k = KINDS[kind]
    rows = syn.synth_rows(k, B, 3 * nF, config_id=6)
    small, layers, spec = _pair(k, B, n, weights, frames_per_call=nF, mask_mode=mode, philox_seed=11, smooth=2)
    rng = np.random.default_rng(2)
    for c in range(3):
        masks = None
        if mode == N.MASK_INJECTED:
            masks = (rng.random(size=(B, nF, spec["L"] - 1, spec["T"], n, spec["H"])) < 0.8).astype(np.uint8)
        _equal(small.step(rows[:, c * nF:(c + 1) * nF], masks=masks), layers.step(rows[:, c * nF:(c + 1) * nF], masks=masks), f"call {c}")
    assert small.launches == 3 * 3                                            # stage 1, ONE LSTM launch, stage 3 per call


# ---- direct C ABI on dense windows ----------------------------------------------------------------------------------------

def run_tcxsl(state, x, masks, n):
    """ape_mc_lstm_tcxsl on dense windows (E, T, I), guard regions behind the workspace and the predictions, NaN-filled predictions;
    checks the launch count and the per-layer times.  Returns the predictions (E, n, O)."""
    I, H, L, O = OL.lstm_dims(state)
    E, T, _ = x.shape
    dev = torch.device("cuda")
    a = N.LstmArgs()
    w = torch.from_numpy(nn_models.pack_lstm_weights(state)).to(dev)
    wx = torch.from_numpy(nn_models.pack_lstm_weights_tcx(state)).to(dev)
    a.weights, a.weights_tcx = w.data_ptr(), wx.data_ptr()
    ws_bytes = N.tcxsl_workspace_bytes(I, H, L, T, O, E, n)
    ws = torch.empty(ws_bytes + GUARD, dtype=torch.uint8, device=dev)
    ws[ws_bytes:] = PATTERN
    n_pred = E * n * O
    pbuf = torch.empty(4 * n_pred + GUARD, dtype=torch.uint8, device=dev)
    pbuf[4 * n_pred:] = PATTERN
    preds = pbuf[:4 * n_pred].view(torch.float32)
    preds.fill_(float("nan"))
    xd = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(dev)
    a.I, a.H, a.L, a.T, a.O = I, H, L, T, O
    a.dropout_p = 0.2
    a.x_dense, a.feat_ring_buf, a.feat_ring = xd.data_ptr(), None, 0
    a.B, a.nF, a.frame0, a.n_samples = E, 1, 0, n
    md = None
    if masks is None:
        a.mask_mode = N.MASK_NONE
    else:
        md = torch.from_numpy(np.ascontiguousarray(masks, dtype=np.uint8)).to(dev)
        a.mask_mode, a.masks = N.MASK_INJECTED, md.data_ptr()
    a.workspace = ws.data_ptr()
    a.preds, a.pred_ring, a.all_steps = preds.data_ptr(), 1, 0
    a.tc_flags = 5
    lib = N.load()
    count = C.c_int(0)
    N.check(lib.ape_mc_lstm_tc_launch_count(a, C.byref(count)), "ape_mc_lstm_tc_launch_count")
    assert count.value == 1
    ms = (C.c_float * L)(*([-1.0] * L))
    a.layer_ms = C.addressof(ms)
    N.check(lib.ape_mc_lstm_tcxsl(a, N.current_stream_ptr()), "ape_mc_lstm_tcxsl")
    assert ms[0] > 0.0 and all(ms[l] == 0.0 for l in range(1, L)), list(ms)     # the one launch is layer 0's time
    torch.cuda.synchronize()
    assert bool((ws[ws_bytes:] == PATTERN).all()), f"bytes behind the workspace ({ws_bytes} B) were written"
    assert bool((pbuf[4 * n_pred:] == PATTERN).all()), "bytes behind the predictions were written"
    out = preds.cpu().numpy()
    assert not np.isnan(out).any(), f"{int(np.isnan(out).sum())} predictions were never written"
    return out.reshape(E, n, O)


@pytest.mark.parametrize("L,T,I,E,n,saturate", [
    (2, 1, 9, 1, 100, False),        # one step, the narrowest layer 0
    (3, 1, 256, 3, 100, False),      # the widest layer 0 (two 16-k-group pieces), an estimate straddling two clusters
    (4, 40, 256, 3, 100, False),
    (3, 40, 22, 2, 64, False),
    (2, 6, 22, 64, 128, False),      # 8192 rows: 64 clusters
    (4, 40, 256, 3, 100, True),      # saturating gates, cells that grow towards |c| = T
])
def test_direct_abi_against_float64(L, T, I, E, n, saturate):
    H, O = 256, 32
    state = (saturating_state if saturate else syn.synth_state_dict)(I, H, L, O, 600 + L + T + I)
    x, masks = inputs(I, H, L, T, E, n, seed=L * 1000 + T + I)
    sel = pick(E, n)
    want, c_max = reference(state, x, masks, n, sel)
    got = run_tcxsl(state, x, masks, n)
    err = last_step_error(got, want, sel, n)
    layers = run_lstm(state, x, masks, n, "split")
    label = f"tcxsl I{I} H{H} L{L} T{T} O{O} E{E} n{n}{' saturating' if saturate else ''}"
    print(f"{label}: vs float64 {err:.3g} (bound {EXACT_TOL:g}), max |c_T| {c_max:.3g}")
    if saturate:
        assert c_max > 30.0
    assert err <= EXACT_TOL
    np.testing.assert_array_equal(got, layers)                                # bit for bit the split layer kernels


# ---- accuracy through the estimator ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", list(KINDS))
@pytest.mark.parametrize("scale,forget_bias", [(1.0, 0.0), (4.0, 1.0), (8.0, 1.0)])
def test_weight_scale_sweep_against_oracle(kind, scale, forget_bias):
    k = KINDS[kind]
    B, nF, n = 2, 2, 48
    state = _scaled_state(k, scale, forget_bias)
    spec = syn.kind_spec(k)
    rng = np.random.default_rng(int(scale * 10) + k)
    rows = syn.synth_rows(k, B, nF, config_id=44)
    masks = (rng.random(size=(B, nF, spec["L"] - 1, spec["T"], n, spec["H"])) < 0.8).astype(np.uint8)
    be, _, _ = make(k, B, n, "tcx", state=state, frames_per_call=nF, mask_mode=N.MASK_INJECTED, split_small_batch_kernel=True)
    assert be.tc_flags == 5 and be.H == 256
    out = be.step(rows, masks=masks)
    worst = 0.0
    for b in range(B):
        orc = OE.OracleEstimator(syn.KIND_NAMES[k], spec["lookup"], state, spec["stats"], spec["y_targets"].name, spec["T"], 1, n,
                                 None, spec["p"], mask_source=lambda f, b=b: list(masks[b, f]))
        for f in range(nF):
            w = np.asarray(orc.step(rows[b, f]))
            for a, c in ((4, 7), (11, 14), (18, 21)):
                worst = max(worst, float(np.abs(out.msg[b, f, a:c] - w[a:c]).max()))
            worst = max(worst, float(np.abs(out.samples[b, f].ravel() - w[25:]).max()))
    print(f"{kind} weights x{scale} forget bias +{forget_bias}: H = 256 split small-batch kernel {worst:.3g} m vs oracle")
    assert worst <= POS_TOL


@pytest.mark.parametrize("kind,name", [("watch_only", "watch_only_s3"), ("pocket", "pocket_s1")])
def test_whole_path_against_reference_messages(kind, name):
    g = load_golden(f"e2e_{name}.npz")
    n, smooth = int(g["n"]), int(g["smooth"])
    masks = unpack_masks(g)
    rows, F = g["rows"], len(g["rows"])
    be, _, _ = make(KINDS[kind], 1, n, "tcx", smooth=smooth, frames_per_call=1, mask_mode=N.MASK_INJECTED, split_small_batch_kernel=True)
    assert be.tc_flags == 5 and be.H == 256
    worst = 0.0
    for f in range(F):                                                        # frame by frame: the streaming call pattern
        out = be.step(rows[None, f:f + 1], masks=masks[None, f:f + 1])
        worst = max(worst, msg_close(out.msg[0, 0], g["msgs"][f, :25]))
        err = float(np.abs(out.samples[0, 0] - g["msgs"][f, 25:].reshape(n * smooth, 6)).max())
        assert err <= 1e-5
        worst = max(worst, err)
    print(f"{name} H = 256 split small-batch kernel: worst position error vs the reference's messages over {F} frames: {worst:.3g} m")


# ---- graph and multi-stream paths -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", list(KINDS))
def test_graph_path_equals_eager_and_the_layer_kernels(kind):
    k = KINDS[kind]
    B, n = 1, 100
    rows = syn.synth_rows(k, B, 5, config_id=12)
    small, layers, _ = _pair(k, B, n, "4x+fb", mask_mode=N.MASK_PHILOX, philox_seed=4)
    graph, _, _ = make(k, B, n, "tcx", state=_scaled_state(k, *WEIGHTS["4x+fb"]), mask_mode=N.MASK_PHILOX, philox_seed=4,
                       split_small_batch_kernel=True)
    assert graph.tc_flags == 5
    for f in range(5):
        a, b, c = graph.step_graph(rows[:, f:f + 1]), small.step(rows[:, f:f + 1]), layers.step(rows[:, f:f + 1])
        for other in (b, c):
            np.testing.assert_array_equal(a.msg, other.msg, err_msg=f"frame {f}")
            np.testing.assert_array_equal(a.samples, other.samples, err_msg=f"frame {f}")
            np.testing.assert_array_equal(a.std, other.std, err_msg=f"frame {f}")


@pytest.mark.parametrize("kind", list(KINDS))
def test_ticks_with_idle_streams_match_the_layer_kernels(kind):
    k = KINDS[kind]
    B, n, ticks = 6, 100, 6
    rows = syn.synth_rows(k, B, ticks, config_id=21)
    small, layers, _ = _pair(k, B, n, "4x+fb", mask_mode=N.MASK_PHILOX, philox_seed=5, smooth=2)
    graph, _, _ = make(k, B, n, "tcx", state=_scaled_state(k, *WEIGHTS["4x+fb"]), mask_mode=N.MASK_PHILOX, philox_seed=5, smooth=2,
                       split_small_batch_kernel=True)
    rng = np.random.default_rng(3)
    frames = np.zeros(B, np.int32)
    for t in range(ticks):
        active = rng.random(B) < 0.6
        active[t % B] = True
        sf = np.where(active, frames, -1).astype(np.int32)                    # idle streams sit the tick out
        before = small.preds.clone()
        a = small.step(rows[:, t:t + 1], stream_frames=sf)
        idle = torch.from_numpy(~active).to(small.preds.device)
        assert torch.equal(small.preds[idle], before[idle]), f"tick {t}: an idle stream's prediction ring was written"
        b = layers.step(rows[:, t:t + 1], stream_frames=sf)
        c = graph.step_graph(rows[:, t:t + 1], stream_frames=sf)
        for got in (a, c):
            np.testing.assert_array_equal(got.msg[active], b.msg[active], err_msg=f"tick {t}")
            np.testing.assert_array_equal(got.samples[active], b.samples[active], err_msg=f"tick {t}")
            np.testing.assert_array_equal(got.std[active], b.std[active], err_msg=f"tick {t}")
        frames += active


@pytest.mark.parametrize("kind,B,n", [("watch_only", 6, 100), ("pocket", 27, 25)])   # 1800 / 2025 rows at 3 frames per call
def test_idle_streams_leave_their_rings_and_outputs_untouched(kind, B, n):
    # the per-stream frame counter schedule of test_gpu_stream_frames.py (idle streams, streams far ahead, 1- and 3-frame calls, runs
    # across the 128-row cluster boundaries): every feature slot, prediction slot and result word of an idle stream keeps its bits,
    # every one of an active stream is written, its predictions match the oracle - and all of it bit for bit the split layer kernels
    k = KINDS[kind]
    spec, state = SF._model(k, False)
    nF_max = max(SF.NF_PER_CALL)
    be = SF._estimator(k, state, B, n, nF_max, pipeline=False, lstm_variant="tcx", split_small_batch_kernel=True)
    assert be.tc_flags == 5 and be.small_batch and be._lstm_fn() == be.lib.ape_mc_lstm_tcxsl and B * nF_max * n <= BOUND
    calls, _, _ = SF.lstm_schedule(B, n, SF.NF_PER_CALL, seed=B + n)
    rows = syn.synth_rows(k, B, sum(SF.NF_PER_CALL), config_id=50 + k)
    worst_f, worst_p, kept = SF.run_lstm_schedule(be, k, state, calls, list(range(B)), SF.PRED_TOL, rows, keep=True)
    assert be.launches == len(calls) * (2 + 1)
    print(f"stream_frames [tcxsl] {kind} {B} x {n}: worst feature error {worst_f:.3g}, worst normalised-output error {worst_p:.3g}")
    layers = SF._estimator(k, state, B, n, nF_max, pipeline=False, lstm_variant="tcx")
    assert layers.tc_flags == 3
    _, _, kept1 = SF.run_lstm_schedule(layers, k, state, calls, [], SF.PRED_TOL, rows, keep=True)
    for c, ((pa, oa), (pb, ob)) in enumerate(zip(kept, kept1)):
        np.testing.assert_array_equal(pa, pb, err_msg=f"call {c}: prediction ring, new kernel vs layer kernels")
        np.testing.assert_array_equal(oa, ob, err_msg=f"call {c}: results, new kernel vs layer kernels")


# ---- routing ----------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", list(KINDS))
def test_single_stream_estimator_routes_a_split_model_to_the_new_kernel(kind, monkeypatch, deploy):
    from arm_pose_estimation_b200.data_deploy.nn import deploy_models
    from arm_pose_estimation_b200.estimate.watch_only import WatchOnlyNN
    from arm_pose_estimation_b200.estimate.watch_phone_pocket_nn import WatchPhonePocketNN

    def new_estimator():
        if kind == "watch_only":
            est = WatchOnlyNN(monte_carlo_samples=100, philox_seed=1)
        else:
            est = WatchPhonePocketNN(model_hash=deploy_models.LSTM.WATCH_PHONE_POCKET.value, monte_carlo_samples=100, philox_seed=1)
        st = {k: np.asarray(v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else v, dtype=np.float32).copy()
              for k, v in est._nn_model.state_dict().items()}
        H = st["lstm.weight_hh_l0"].shape[1]
        for k in st:
            if k.startswith("lstm.weight_"):
                st[k] = (st[k] * np.float32(4.0)).astype(np.float32)
            if k.startswith("lstm.bias_ih_l"):
                st[k][H:2 * H] += np.float32(1.0)
        est._nn_model.load_state_dict({k: torch.from_numpy(v) for k, v in st.items()})
        return est

    new, old = new_estimator(), new_estimator()
    rows = syn.synth_rows(KINDS[kind], 1, 6, config_id=3)[0]
    got = [np.asarray(new.estimate_row(r)) for r in rows]
    engine = new._engine("graph")
    assert engine.tc_split and engine.tc_flags == 5 and engine.small_batch and engine.H == 256
    # the same class on the split layer kernels
    base = estimator_module.BatchedEstimator
    monkeypatch.setattr(estimator_module, "BatchedEstimator", lambda **kw: base(**{**kw, "split_small_batch_kernel": False}))
    want = [np.asarray(old.estimate_row(r)) for r in rows]
    assert old._engine("graph").tc_flags == 3
    for f in range(len(rows)):
        np.testing.assert_array_equal(got[f], want[f], err_msg=f"frame {f}")


@pytest.mark.parametrize("answer", ["zero", "error"])
def test_a_device_without_a_cluster_keeps_the_layer_kernels(answer, monkeypatch):
    # the availability query answering 0, or failing, leaves the estimator on the split layer kernels
    def query():
        if answer == "error":
            raise UserWarning("ape_mc_lstm_tcxsl_max_active_clusters: CUDA error")
        return 0
    monkeypatch.setattr(N, "tcxsl_max_active_clusters", query)
    be, _, _ = make(syn.KIND_POCKET, 1, 100, "tcx", state=_scaled_state(syn.KIND_POCKET, *WEIGHTS["4x+fb"]), split_small_batch_kernel=True)
    assert be.tc_split and be.tc_flags == 3 and not be.small_batch
    rows = syn.synth_rows(syn.KIND_POCKET, 1, 1, config_id=8)
    assert np.isfinite(be.step(rows).msg).all()


def test_above_the_row_bound_the_estimator_stays_on_the_layer_kernels():
    be, _, _ = make(syn.KIND_POCKET, BOUND // 128 + 1, 128, "tcx", state=_scaled_state(syn.KIND_POCKET, *WEIGHTS["4x+fb"]),
                    split_small_batch_kernel=True)
    assert be.tc_split and be.tc_flags == 3 and not be.small_batch
