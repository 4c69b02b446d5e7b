"""GPU (-m gpu): every LSTM kernel across the shapes its ``supported`` predicate accepts, not only the three deployed models - against a
float64 restatement of oracle.lstm.forward_with_masks.  The corners: layer-0 inputs up to I = H (at H = 128 the one-layer kernel's
dynamic shared memory is then 231 680 of the 232 448 bytes a block may have), the widest output layer of each kernel, T = 1 / odd / 40,
L = 2 .. 5 (the wavefront kernel beside and below another pair, the split kernels' layer walk past L = 3, the cluster kernel's layer 3),
row counts with a ragged last tile and with more 256-row tiles than CTA pairs, cells that grow towards |c| = T, per-step outputs at
T = 40 and an estimator whose 40-frame feature window is clamped at frame 0 and then wraps its ring.

Every call is pinned to one kernel (``tc_flags``), checks the routing (``ape_mc_lstm_tc_launch_count`` and the per-layer times) and
runs with a guard region behind the workspace and behind the predictions, and NaN in the predictions: a workspace query that is too
small at a corner shape, or a store past the last row, changes guard bytes or leaves a NaN.

Bounds (raw LSTM outputs against float64): fp32 and split-precision kernels 2e-5; single-pass fp16-operand kernels 2e-4 at T <= 8 and
5e-4 at T = 40 (h_t is rounded to fp16 on every step; test_gpu_split_model_api.py::test_large_cell_state measured ~2.7e-4 for that
accumulation at T = 40 on a B200).  Every worst error is printed."""
import ctypes as C

import numpy as np
import pytest
import torch

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200 import synthetic as syn
from arm_pose_estimation_b200.estimate import nn_models
from arm_pose_estimation_b200.estimate.batched import BatchedEstimator
from oracle import estimator as OE
from oracle import lstm as OL
from test_gpu_parity import msg_close, POS_TOL

pytestmark = pytest.mark.gpu

EXACT_TOL = 2e-5                     # fp32 FFMA kernel and split-precision kernels
SINGLE_TOL = 2e-4                    # single-pass fp16 operands, T <= 8
SINGLE_TOL_LONG = 5e-4               # single-pass fp16 operands, T = 40: fp16 rounding of h_t accumulates over the steps
TCW_VS_TC = 5e-5                     # wavefront vs one-layer launches (bias inside the accumulator, see test_gpu_tcw.py)
FLAGS = {"tc": 1, "tcw": 2, "split": 3, "tcl": 4, "tcxl": 5, "tcxsl": 5}
GUARD, PATTERN = 4096, 0xA5
P = 0.2


def single_tol(T):
    return SINGLE_TOL if T <= 8 else SINGLE_TOL_LONG


# ---- float64 reference ------------------------------------------------------------------------------------------------------

def lstm64(state, x, masks=None, p=P):
    """oracle.lstm.forward_with_masks with every array in float64: x (R, T, I), masks a list of L-1 {0,1} arrays (T, R, H) or None.
    Returns the outputs of every step (R, T, O) and the largest |c_T| over the layers."""
    st = {k: np.asarray(v, dtype=np.float64) for k, v in state.items()}
    I, H, L, O = OL.lstm_dims(state)
    seq = np.asarray(x, dtype=np.float64)
    R, T, _ = seq.shape
    c_max = 0.0
    for l in range(L):
        w_ih, w_hh = st[f"lstm.weight_ih_l{l}"], st[f"lstm.weight_hh_l{l}"]
        bias = st[f"lstm.bias_ih_l{l}"] + st[f"lstm.bias_hh_l{l}"]
        h, c = np.zeros((R, H)), np.zeros((R, H))
        out = np.empty((R, T, H))
        for t in range(T):
            g = seq[:, t, :] @ w_ih.T + h @ w_hh.T + bias
            gi, gf = 1.0 / (1.0 + np.exp(-g[:, :H])), 1.0 / (1.0 + np.exp(-g[:, H:2 * H]))
            gg, go = np.tanh(g[:, 2 * H:3 * H]), 1.0 / (1.0 + np.exp(-g[:, 3 * H:]))
            c = gf * c + gi * gg
            h = go * np.tanh(c)
            out[:, t, :] = h
        c_max = max(c_max, float(np.abs(c).max()))
        if l < L - 1 and masks is not None:
            out = out * np.asarray(masks[l], dtype=np.float64).transpose(1, 0, 2) / (1.0 - p)
        seq = out
    return seq @ st["output_layer.weight"].T + st["output_layer.bias"], c_max


def pick(E, n):
    """Estimates the reference recomputes: the first and the last ones (the first tile and the ragged last tile), ~256 rows."""
    k = max(1, 128 // n)
    return np.unique(np.r_[0:min(k, E), max(0, E - k):E])


def reference(state, x, masks, n, sel, p=P):
    """float64 outputs of every step for the rows of estimates ``sel``: (len(sel) * n, T, O), and the largest |c_T|."""
    T = x.shape[1]
    xs = np.repeat(x[sel], n, axis=0)
    ms = None
    if masks is not None:
        H = masks.shape[-1]
        ms = [np.ascontiguousarray(masks[sel, g].transpose(1, 0, 2, 3).reshape(T, len(sel) * n, H)) for g in range(masks.shape[1])]
    return lstm64(state, xs, ms, p)


# ---- driver -----------------------------------------------------------------------------------------------------------------

def expected_launches(kernel, L, T, all_steps):
    """(launches, layers that start a launch) of ape_mc_lstm_tc pinned to ``kernel``."""
    if kernel in ("tcl", "tcxl", "tcxsl"):                 # every layer in one launch
        return 1, [0]
    if kernel == "tcw" and T >= 2:                       # layer 0 alone, then pairs (1, 2), (3, 4) .. and a lone last layer
        starts = [0] + list(range(1, L, 2))
    else:
        starts = list(range(L))
    return len(starts) + (1 if all_steps else 0), starts


def run_lstm(state, x, masks, n, kernel, all_steps=False, p=P, philox=None, nF=1, frame0=0, stream_frames=None):
    """One LSTM call on dense windows x (E, T, I) with injected masks (E, L-1, T, n, H) (None: no dropout), pinned to one kernel:
    "fp32" (ape_mc_lstm_fma), "tc" / "tcw" / "split" / "tcl" / "tcxl" (ape_mc_lstm_tc with tc_flags 1 / 2 / 3 / 4 / 5) or "tcxsl"
    (ape_mc_lstm_tcxsl).  ``philox`` = (seed, stream_id0): APE_MASK_PHILOX instead (masks None).  The E = B * nF estimates are
    nF frames of each of B streams, from frame0 or from the host counters ``stream_frames`` [B]; the predictions go through a ring
    of nF slots.  Returns the predictions (E, n, O), or with ``all_steps`` those of every step (E * n, T, O).  Checks the routing
    and the guard bytes."""
    I, H, L, O = OL.lstm_dims(state)
    E, T, _ = x.shape
    assert E % nF == 0 and (masks is None or philox is None) and (nF == 1 or not all_steps)
    B = E // nF
    dev = torch.device("cuda")
    keep = []
    a = N.LstmArgs()
    w = torch.from_numpy(nn_models.pack_lstm_weights(state)).to(dev)
    keep.append(w)
    a.weights = w.data_ptr()
    if kernel == "fp32":
        ws_bytes = N.workspace_bytes(I, H, L, T, O, E, n)
    elif kernel in ("split", "tcxl", "tcxsl"):
        wx = torch.from_numpy(nn_models.pack_lstm_weights_tcx(state)).to(dev)
        keep.append(wx)
        a.weights_tcx = wx.data_ptr()
        if kernel == "split":
            ws_bytes = (N.tcx_workspace_bytes if H == 128 else N.tcxs_workspace_bytes)(I, H, L, T, O, E, n, all_steps=all_steps)
        else:
            ws_bytes = (N.tcxl_workspace_bytes if kernel == "tcxl" else N.tcxsl_workspace_bytes)(I, H, L, T, O, E, n)
    else:
        wt = torch.from_numpy(nn_models.pack_lstm_weights_tc(state)).to(dev)
        keep.append(wt)
        a.weights_tc = wt.data_ptr()
        ws_bytes = N.workspace_bytes(I, H, L, T, O, E, n, tensor_core=True, all_steps=all_steps)
    ws = torch.empty(ws_bytes + GUARD, dtype=torch.uint8, device=dev)
    ws[ws_bytes:] = PATTERN
    n_pred = E * n * (T if all_steps else 1) * O
    pbuf = torch.empty(4 * n_pred + GUARD, dtype=torch.uint8, device=dev)
    pbuf[4 * n_pred:] = PATTERN
    preds = pbuf[:4 * n_pred].view(torch.float32)
    preds.fill_(float("nan"))
    xd = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(dev)
    a.I, a.H, a.L, a.T, a.O = I, H, L, T, O
    a.dropout_p = p
    a.x_dense, a.feat_ring_buf, a.feat_ring = xd.data_ptr(), None, 0
    a.B, a.nF, a.frame0, a.n_samples = B, nF, frame0, n
    if stream_frames is not None:
        sfd = torch.tensor(stream_frames, dtype=torch.int32, device=dev)
        keep.append(sfd)
        a.stream_frames = sfd.data_ptr()
    if philox is not None:
        a.mask_mode, (a.philox_seed, a.stream_id0) = N.MASK_PHILOX, philox
    elif masks is None:
        a.mask_mode = N.MASK_NONE
    else:
        md = torch.from_numpy(np.ascontiguousarray(masks, dtype=np.uint8)).to(dev)
        keep.append(md)
        a.mask_mode, a.masks = N.MASK_INJECTED, md.data_ptr()
    a.workspace = ws.data_ptr()
    a.preds, a.pred_ring, a.all_steps = preds.data_ptr(), nF, int(all_steps)
    lib = N.load()
    if kernel == "fp32":
        N.check(lib.ape_mc_lstm_fma(a, N.current_stream_ptr()), "ape_mc_lstm_fma")
    else:
        a.tc_flags = FLAGS[kernel]
        want_launches, starts = expected_launches(kernel, L, T, all_steps)
        count = C.c_int(0)
        N.check(lib.ape_mc_lstm_tc_launch_count(a, C.byref(count)), "ape_mc_lstm_tc_launch_count")
        assert count.value == want_launches, f"{kernel}: {count.value} launches, expected {want_launches}"
        ms = (C.c_float * L)(*([-1.0] * L))
        a.layer_ms = C.addressof(ms)
        call = lib.ape_mc_lstm_tcxsl if kernel == "tcxsl" else lib.ape_mc_lstm_tc
        N.check(call(a, N.current_stream_ptr()), f"ape_mc_lstm_tc ({kernel})")
        for l in range(L):                               # a launch's time goes to its first layer; the second of a pair reads 0
            if l in starts:
                assert ms[l] > 0.0, f"{kernel}: layer {l} has no launch of its own (time {ms[l]})"
            else:
                assert ms[l] == 0.0, f"{kernel}: layer {l} ran in a launch of its own (time {ms[l]})"
    torch.cuda.synchronize()
    assert bool((ws[ws_bytes:] == PATTERN).all()), f"{kernel}: bytes behind the workspace ({ws_bytes} B) were written"
    assert bool((pbuf[4 * n_pred:] == PATTERN).all()), f"{kernel}: bytes behind the predictions were written"
    out = preds.cpu().numpy()
    assert not np.isnan(out).any(), f"{kernel}: {int(np.isnan(out).sum())} predictions were never written"
    if all_steps:
        return out.reshape(E * n, T, O)
    ring = out.reshape(B, nF, n, O)                      # slot f % nF of each stream: back to estimate order
    fb = np.full(B, frame0) if stream_frames is None else np.asarray(stream_frames)
    return np.stack([ring[e // nF, (int(fb[e // nF]) + e % nF) % nF] for e in range(E)])


def inputs(I, H, L, T, E, n, seed, masked=True):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((E, T, I)).astype(np.float32)
    masks = (rng.random(size=(E, L - 1, T, n, H)) < 1 - P).astype(np.uint8) if masked else None
    return x, masks


def last_step_error(got, want, sel, n):
    """max |kernel - float64| over the last step of the reference rows."""
    O = got.shape[-1]
    return float(np.abs(got[sel].reshape(-1, O).astype(np.float64) - want[:, -1, :]).max())


def check_kernel(state, x, masks, n, kernel, tol, label, want=None, sel=None):
    """Run ``kernel`` and the fp32 kernel on the same call and hold both against the float64 reference; returns the kernel's outputs."""
    E = x.shape[0]
    if want is None:
        sel = pick(E, n)
        want, _ = reference(state, x, masks, n, sel)
    got = run_lstm(state, x, masks, n, kernel)
    ref32 = run_lstm(state, x, masks, n, "fp32")
    e_k, e_32 = last_step_error(got, want, sel, n), last_step_error(ref32, want, sel, n)
    print(f"{label}: {kernel} vs float64 {e_k:.3g} (bound {tol:g}), fp32 kernel vs float64 {e_32:.3g}")
    assert e_32 <= EXACT_TOL
    assert e_k <= tol
    return got


# ---- one-layer kernel, H = 64 / 128 (tc_flags = 1) ------------------------------------------------------------------------------

@pytest.mark.parametrize("H,I,L,T,E,n", [
    (64, 64, 2, 1, 600, 1),          # I = H; one step; 600 estimates: layer 0 on 128-row CTAs
    (64, 49, 5, 7, 5, 60),           # I = H - 15 (the same k-groups); odd T; layer 0 on 32-row CTAs
    (64, 64, 5, 40, 5, 60),
    (64, 49, 2, 40, 600, 1),
    (128, 128, 2, 1, 5, 60),
    (128, 113, 5, 7, 600, 1),
    (128, 128, 2, 7, 600, 1),        # the widest layer 0 on 128-row CTAs: 231 680 B of dynamic shared memory
    (128, 128, 5, 40, 600, 1),
    (128, 113, 2, 40, 5, 60),
])
def test_one_layer_kernel_corners(H, I, L, T, E, n):
    O = 16
    state = syn.synth_state_dict(I, H, L, O, 10 + H + I + L + T)
    x, masks = inputs(I, H, L, T, E, n, seed=H * T + I)
    check_kernel(state, x, masks, n, "tc", single_tol(T), f"one-layer I{I} H{H} L{L} T{T} O{O} E{E} n{n}")


def test_streamed_weights_kernel_corner():
    I, H, L, T, O, E, n = 256, 256, 4, 40, 20, 3, 100
    state = syn.synth_state_dict(I, H, L, O, 77)
    x, masks = inputs(I, H, L, T, E, n, seed=7)
    check_kernel(state, x, masks, n, "tc", single_tol(T), f"streamed-weights I{I} H{H} L{L} T{T} O{O} E{E} n{n}")


# ---- wavefront kernel (tc_flags = 2) ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("L,T,E,n", [
    (4, 1, 3, 100),                  # T = 1: no pair launch at all (L one-layer launches)
    (4, 2, 3, 100), (4, 7, 3, 100), (4, 40, 3, 100),     # pair (1, 2) writes units for layer 3; layer 3 alone
    (5, 2, 3, 100), (5, 7, 3, 100), (5, 40, 3, 100),     # pair (3, 4) reads the units pair (1, 2) wrote
    (5, 7, 200, 100),                # 20 000 rows = 79 pair tiles > 74 CTA pairs
])
def test_wavefront_kernel_below_and_beside_another_pair(L, T, E, n):
    I, H, O = 38, 128, 16
    state = syn.synth_state_dict(I, H, L, O, 200 + L + T)
    x, masks = inputs(I, H, L, T, E, n, seed=L * 100 + T)
    sel = pick(E, n)
    want, _ = reference(state, x, masks, n, sel)
    label = f"wavefront I{I} H{H} L{L} T{T} O{O} E{E} n{n}"
    pair = check_kernel(state, x, masks, n, "tcw", single_tol(T), label, want, sel)
    single = run_lstm(state, x, masks, n, "tc")
    d = float(np.abs(pair - single).max())
    print(f"{label}: wavefront vs one-layer launches over all {E * n} rows {d:.3g}, one-layer vs float64 {last_step_error(single, want, sel, n):.3g}")
    assert d <= TCW_VS_TC


# ---- cluster kernel (tc_flags = 4) --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("H,L", [(128, 2), (128, 4), (256, 2), (256, 4)])
@pytest.mark.parametrize("E,n", [(1, 100), (3, 100)])   # one cluster; three clusters, estimate 1 straddles clusters 0 and 1
def test_cluster_kernel_corners(H, L, E, n):
    I, T = H, 40
    O = 16 if H == 128 else 20
    state = syn.synth_state_dict(I, H, L, O, 300 + H + L)
    x, masks = inputs(I, H, L, T, E, n, seed=H + L + E)
    label = f"cluster I{I} H{H} L{L} T{T} O{O} E{E} n{n}"
    got = check_kernel(state, x, masks, n, "tcl", single_tol(T), label)
    np.testing.assert_array_equal(got, run_lstm(state, x, masks, n, "tc"))       # bit-identical to the layer kernels


def test_cluster_kernel_refuses_five_layers():
    I, H, L, T, O, E, n = 38, 128, 5, 6, 12, 1, 10
    state = syn.synth_state_dict(I, H, L, O, 5)
    x, _ = inputs(I, H, L, T, E, n, seed=1, masked=False)
    with pytest.raises(UserWarning, match="not supported"):
        run_lstm(state, x, None, n, "tcl")


# ---- split-precision kernels (tc_flags = 3) -----------------------------------------------------------------------------------

@pytest.mark.parametrize("L", [2, 4, 5])
@pytest.mark.parametrize("T", [1, 7, 40])
def test_split128_corners(L, T):
    I, H, O, E, n = 128, 128, 16, 3, 100
    state = syn.synth_state_dict(I, H, L, O, 400 + L + T)
    x, masks = inputs(I, H, L, T, E, n, seed=L * 10 + T)
    check_kernel(state, x, masks, n, "split", EXACT_TOL, f"split I{I} H{H} L{L} T{T} O{O} E{E} n{n}")


@pytest.mark.parametrize("L", [4, 5])
def test_split256_corners(L):
    I, H, T, O, E, n = 256, 256, 40, 32, 3, 100
    state = syn.synth_state_dict(I, H, L, O, 500 + L)
    x, masks = inputs(I, H, L, T, E, n, seed=L)
    check_kernel(state, x, masks, n, "split", EXACT_TOL, f"split I{I} H{H} L{L} T{T} O{O} E{E} n{n}")


# ---- cells that grow towards |c| = T ------------------------------------------------------------------------------------------

def saturating_state(I, H, L, O, seed):
    """Two runs of units (the first and the last 16 of every layer) whose input and forget gates sit near 1 and whose g sits near
    +1 / -1 on every step: their cells add ~0.97 per step and keep ~0.998 of it, so |c_T| approaches T."""
    state = {k: v.copy() for k, v in syn.synth_state_dict(I, H, L, O, seed).items()}
    units = np.r_[0:16, H - 16:H]
    sign = np.where(np.arange(units.size) % 2 == 0, 1.0, -1.0).astype(np.float32)
    for l in range(L):
        b = state[f"lstm.bias_ih_l{l}"]
        b[units] += np.float32(4.0)              # i
        b[H + units] += np.float32(6.0)          # f
        b[2 * H + units] += np.float32(3.0) * sign   # g
    return state


@pytest.mark.parametrize("kernel,H,L", [("fp32", 128, 4), ("tc", 128, 4), ("tc", 256, 2), ("tcw", 128, 5), ("tcl", 256, 2),
                                        ("split", 128, 4), ("split", 256, 4)])
def test_saturating_cells_at_T40(kernel, H, L):
    I, T, E, n = H, 40, 3, 100
    O = 16 if H == 128 else 20
    state = saturating_state(I, H, L, O, 600 + H + L)
    x, masks = inputs(I, H, L, T, E, n, seed=H + L)
    sel = pick(E, n)
    want, c_max = reference(state, x, masks, n, sel)
    got = run_lstm(state, x, masks, n, kernel)
    err = last_step_error(got, want, sel, n)
    tol = EXACT_TOL if kernel in ("fp32", "split") else SINGLE_TOL_LONG
    print(f"saturating cells, {kernel} I{I} H{H} L{L} T{T} O{O} E{E} n{n}: largest |c_T| {c_max:.3g}, vs float64 {err:.3g} (bound {tol:g})")
    assert c_max > 30.0
    assert np.isfinite(got).all() and err <= tol


# ---- per-step outputs (the model API: all_steps = 1) at T = 40 ----------------------------------------------------------------

@pytest.mark.parametrize("kernel,H", [("tc", 128), ("tc", 256), ("split", 128), ("split", 256)])
def test_per_step_outputs_at_T40(kernel, H):
    I, L, T, E, n = 20, 4, 40, 300, 1
    O = 16 if H == 128 else 20
    state = syn.synth_state_dict(I, H, L, O, 700 + H)
    x, masks = inputs(I, H, L, T, E, n, seed=H)
    sel = np.r_[0:64, E - 64:E]
    want, _ = reference(state, x, masks, n, sel)
    got = run_lstm(state, x, masks, n, kernel, all_steps=True)
    err = float(np.abs(got[sel].astype(np.float64) - want).max())
    worst_step = int(np.abs(got[sel].astype(np.float64) - want).max(axis=(0, 2)).argmax())
    tol = EXACT_TOL if kernel == "split" else SINGLE_TOL_LONG
    print(f"per-step outputs, {kernel} I{I} H{H} L{L} T{T} O{O}, {E} rows: vs float64 over every step {err:.3g} (at step {worst_step}; bound {tol:g})")
    assert err <= tol


# ---- an estimator with a 40-frame window --------------------------------------------------------------------------------------

def _long_window_estimator(state, B, n, variant, **kw):
    spec = syn.kind_spec(syn.KIND_UARM)
    return BatchedEstimator(kind=syn.KIND_UARM, layout=spec["layout"], state=state, seq_len=40, y_targets=spec["y_targets"],
                            stats=spec["stats"], n_streams=B, mc_samples=n, dropout=spec["p"], lstm_variant=variant, **kw)


@pytest.mark.parametrize("variant", ["tc", "tcx"])
def test_estimator_with_a_40_frame_window_against_oracle(variant):
    # frames 0 .. 39 read a window clamped at frame 0; from frame 40 on the feature ring wraps
    kind, B, n, F, T = syn.KIND_UARM, 2, 20, 45, 40
    spec = syn.kind_spec(kind)
    state = syn.synth_state_dict(spec["I"], spec["H"], spec["L"], spec["O"], 1234 + kind)
    be = _long_window_estimator(state, B, n, variant, frames_per_call=1, mask_mode=N.MASK_INJECTED)
    if variant == "tc":                                  # 40 rows per call: the cluster kernel
        assert be.lstm_variant == "tc" and be.small_batch and be.tc_flags == 4
    else:
        assert be.lstm_variant == "tc" and be.tc_split and be.tc_flags == 3
    rows = syn.synth_rows(kind, B, F, config_id=45)
    rng = np.random.default_rng(40)
    masks = (rng.random(size=(B, F, spec["L"] - 1, T, n, spec["H"])) < 1 - spec["p"]).astype(np.uint8)
    checked = (0, 1, 38, 39, 40, 44)
    outs = {}
    for f in range(F):
        out = be.step(rows[:, f:f + 1], masks=masks[:, f:f + 1])
        if f in checked:                                 # (the result views are reused by later calls)
            outs[f] = (np.array(out.msg), np.array(out.samples))
    worst = 0.0
    for b in range(B):
        orc = OE.OracleEstimator(syn.KIND_NAMES[kind], spec["lookup"], state, spec["stats"], spec["y_targets"].name, T, 1, n, None,
                                 spec["p"], mask_source=lambda f, b=b: list(masks[b, f]))
        for f in range(F):
            want = np.asarray(orc.step(rows[b, f]))
            if f in checked:
                worst = max(worst, msg_close(outs[f][0][b, 0], want[:25]))
                err = float(np.abs(outs[f][1][b, 0].ravel() - want[25:]).max())
                assert err <= POS_TOL, f"stream {b} frame {f}: {err:.3g} m"
                worst = max(worst, err)
    print(f"uarm, seq_len 40, lstm_variant {variant} (tc_flags {be.tc_flags}): worst position error vs oracle on frames {checked}: {worst:.3g} m")


def test_estimator_with_a_40_frame_window_pipeline_is_bitwise_invisible():
    kind, B, n, F = syn.KIND_UARM, 4, 50, 45
    spec = syn.kind_spec(kind)
    state = syn.synth_state_dict(spec["I"], spec["H"], spec["L"], spec["O"], 1234 + kind)
    kw = dict(frames_per_call=1, mask_mode=N.MASK_PHILOX, philox_seed=40, smooth=3, small_batch_kernel=False)
    piped = _long_window_estimator(state, B, n, "tc", **kw)
    plain = _long_window_estimator(state, B, n, "tc", pipeline=False, **kw)
    assert piped._pipe is not None and plain._pipe is None and not piped.small_batch
    rows = syn.synth_rows(kind, B, F, config_id=46)
    ahead = 4                                            # calls in flight (fewer than the estimator's result slots)
    pend = {f: piped.submit(rows[:, f:f + 1]) for f in range(ahead)}
    for f in range(F):
        got = pend.pop(f).result()
        if f + ahead < F:
            pend[f + ahead] = piped.submit(rows[:, f + ahead:f + ahead + 1])
        want = plain.step(rows[:, f:f + 1])
        assert np.isfinite(got.msg).all()
        np.testing.assert_array_equal(got.msg, want.msg, err_msg=f"frame {f}")
        np.testing.assert_array_equal(got.samples, want.samples, err_msg=f"frame {f}")
        np.testing.assert_array_equal(got.std, want.std, err_msg=f"frame {f}")
