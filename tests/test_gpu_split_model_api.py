"""GPU (-m gpu): DropoutLSTM's model API on the split-precision tensor-core kernels (lstm_variant / hs_variant "tcx":
csrc/ape_lstm_tcx.cu for H = 128, csrc/ape_lstm_tcxs.cu for H = 256) - per-step outputs and an initial state (h_0, c_0) at H = 256
against torch, the output product behind a state at tile boundaries, a zero state bit-equal to none, large cell states, weights
that defeat the single-pass kernels, and the refusals."""
import ctypes as C

import numpy as np
import pytest
import torch

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200 import synthetic as syn
from arm_pose_estimation_b200.estimate import nn_models
from oracle import lstm as OL

pytestmark = pytest.mark.gpu
TOL = 2e-5                                     # normalised outputs: the raw-output bound of the split kernels (test_gpu_tcx256.py)
P = 0.3
BIG = 148 * 256 + 1000                         # > one 256-row tile per CTA pair: pairs run on across tile boundaries
DEPLOYED = [(38, 128, 3, 6, 12), (20, 256, 2, 8, 12), (22, 256, 2, 6, 14)]     # upper-arm, watch-only, pocket
SHAPES = DEPLOYED + [(20, 256, 3, 5, 12), (20, 256, 2, 1, 12), (38, 128, 3, 1, 12), (22, 256, 2, 7, 14), (20, 256, 2, 4, 20)]


def _model(I, H, L, O, seed=31, state=None, **kw):
    state = syn.synth_state_dict(I, H, L, O, seed) if state is None else state
    kw.setdefault("lstm_variant", "tcx")
    kw.setdefault("hs_variant", "tcx")
    return nn_models.DropoutLSTM(I, H, L, O, P, philox_seed=77, **kw).load_state_dict(state).eval(), state


def _hs(rng, L, rows, H, scale=0.5, c=None):
    h = torch.from_numpy((scale * rng.normal(size=(L, rows, H))).astype(np.float32))
    c = torch.from_numpy((scale * rng.normal(size=(L, rows, H))).astype(np.float32)) if c is None else c
    return h, c


def _mc_against_torch(m, tm, x1, n, T, H, L, hs=None):
    masks = OL.replay_torch_masks(5, T, n, H, L, P)
    torch.manual_seed(5)
    with torch.no_grad():
        want = tm.monte_carlo_predictions(n, x1, hs).numpy()
    tm.eval()
    got = m.monte_carlo_predictions(n, x1, hs=hs, masks=np.stack(masks)).numpy()
    m.eval()
    assert got.shape == want.shape
    return float(np.abs(got - want).max())


def _rows_cases(shape):
    return [37, 600] + ([BIG] if shape in DEPLOYED else [])


@pytest.mark.parametrize("I,H,L,T,O,rows", [s + (r,) for s in SHAPES for r in _rows_cases(s)])
def test_per_step_outputs_against_torch(I, H, L, T, O, rows):
    # forward(x) and monte_carlo_predictions(n, x, masks=...) with lstm_variant = "tcx": every step's output (all_steps = 1)
    m, state = _model(I, H, L, O)
    tm = OL.TorchDropoutLSTM.from_state(state, P)
    rng = np.random.default_rng(I + H + L + T + O + rows)
    x = torch.from_numpy(rng.normal(size=(rows, T, I)).astype(np.float32))
    with torch.no_grad():
        want = tm(x).numpy()
    got = m(x).numpy()
    assert got.shape == want.shape and np.isfinite(got).all()
    e1 = float(np.abs(got - want).max())
    e2 = _mc_against_torch(m, tm, x[:1], min(rows, 600), T, H, L)
    print(f"(I,H,L,T,O)={(I, H, L, T, O)} rows {rows} split precision, per-step outputs: forward |d|={e1:.3g}  mc |d|={e2:.3g}")
    assert e1 <= TOL and e2 <= TOL


@pytest.mark.parametrize("I,H,L,T,O", [(20, 256, 2, 8, 12), (22, 256, 2, 6, 14), (20, 256, 3, 5, 12), (20, 256, 2, 1, 12)])
@pytest.mark.parametrize("rows", [37, 600, BIG])
def test_initial_state_against_torch(I, H, L, T, O, rows):
    # forward(x, hs) and monte_carlo_predictions(n, x, hs, masks=...) with hs_variant = "tcx" (ape_lstm_tcxs.cu)
    m, state = _model(I, H, L, O)
    tm = OL.TorchDropoutLSTM.from_state(state, P)
    rng = np.random.default_rng(H + L + T + rows)
    x = torch.from_numpy(rng.normal(size=(rows, T, I)).astype(np.float32))
    hs = _hs(rng, L, rows, H)
    with torch.no_grad():
        want = tm(x, hs).numpy()
    got = m(x, hs).numpy()
    assert got.shape == want.shape and np.isfinite(got).all()
    e1 = float(np.abs(got - want).max())
    n = min(rows, 600)
    e2 = _mc_against_torch(m, tm, x[:1], n, T, H, L, _hs(rng, L, n, H))
    print(f"(I,H,L,T,O)={(I, H, L, T, O)} rows {rows} split precision with (h_0, c_0): forward |d|={e1:.3g}  mc |d|={e2:.3g}")
    assert e1 <= TOL and e2 <= TOL


def _direct(m, x, hs, kernel, all_steps=0, mask_mode=N.MASK_PHILOX):
    """One ape_mc_lstm_tc (tc_flags = 3) / ape_mc_lstm_fma call, one row per estimate: all_steps = 0 -> the last step's outputs
    [E, O] (on the split kernel the output product inside the last layer's kernel); all_steps = 1 -> [E, T, O]."""
    I, H, L, O = m._dims()
    E, T, _ = x.shape
    split = kernel == "tcx"
    preds = torch.full((E, T if all_steps else 1, O), float("nan"), dtype=torch.float32, device="cuda")
    a = N.LstmArgs()
    a.weights = m.packed_weights().data_ptr()
    a.I, a.H, a.L, a.T, a.O = I, H, L, T, O
    a.dropout_p = P
    a.x_dense, a.B, a.nF, a.frame0, a.n_samples = x.data_ptr(), E, 1, 3, 1
    a.mask_mode, a.philox_seed = mask_mode, 99
    if hs is not None:
        a.h0, a.c0 = hs[0].data_ptr(), hs[1].data_ptr()
    if split:
        a.weights_tcx, a.tc_flags = m.packed_weights_tcx().data_ptr(), 3
        need = N.split_workspace_bytes(I, H, L, T, O, E, 1, all_steps=bool(all_steps))
    else:
        need = N.workspace_bytes(I, H, L, T, O, E, 1)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    a.workspace = ws.data_ptr()
    a.preds, a.pred_ring, a.all_steps = preds.data_ptr(), 1, all_steps
    fn = N.load().ape_mc_lstm_tc if split else N.load().ape_mc_lstm_fma
    N.check(fn(C.byref(a), N.current_stream_ptr()), "ape_mc_lstm_tc" if split else "ape_mc_lstm_fma")
    torch.cuda.synchronize()
    return preds.cpu().numpy() if all_steps else preds.reshape(E, O).cpu().numpy()


@pytest.mark.parametrize("I,H,L,T,O", [(20, 256, 2, 8, 12), (20, 256, 3, 5, 12), (22, 256, 2, 1, 14)])
def test_output_product_with_state_across_tiles(I, H, L, T, O):
    # all_steps = 0 with a state: the last layer's kernel multiplies h_T by W_o on tensor cores, and the epilogue writes the next tile's
    # h_0 into the same TMEM columns only after that product has been read.  Two or three tiles per CTA pair; T = 1: step 0 is also
    # the last step.  Against the fp32 kernel under the same Philox masks, and run to run.
    m, _ = _model(I, H, L, O)
    rng = np.random.default_rng(T + L)
    x = torch.from_numpy(rng.normal(size=(BIG, T, I)).astype(np.float32)).cuda()
    hs = tuple(v.cuda() for v in _hs(rng, L, BIG, H))
    got = _direct(m, x, hs, "tcx")
    want = _direct(m, x, hs, "fp32")
    d = float(np.abs(got - want).max())
    print(f"(I,H,L,T,O)={(I, H, L, T, O)} {BIG} rows, all_steps = 0 with (h_0, c_0): |split - fp32| = {d:.3g}")
    assert np.isfinite(got).all() and d <= TOL
    np.testing.assert_array_equal(_direct(m, x, hs, "tcx"), got)


@pytest.mark.parametrize("I,H,L,T,O", [(20, 256, 2, 8, 12), (20, 256, 3, 5, 12), (22, 256, 2, 1, 14)])
def test_zero_state_equals_no_state(I, H, L, T, O):
    m, _ = _model(I, H, L, O)
    rng = np.random.default_rng(3)
    rows = 600
    x = torch.from_numpy(rng.normal(size=(rows, T, I)).astype(np.float32)).cuda()
    zeros = (torch.zeros(L, rows, H), torch.zeros(L, rows, H))
    m.train()                                  # Philox masks: the same keys with and without a state (one sample per row)
    m._calls = 9
    want = m(x).cpu().numpy()
    m._calls = 9
    got = m(x, zeros).cpu().numpy()
    np.testing.assert_array_equal(got, want)
    m.eval()
    n = 40
    masks = (rng.random(size=(L - 1, T, n, H)) < 0.7).astype(np.uint8)
    want = m.monte_carlo_predictions(n, x[:1], masks=masks).cpu().numpy()
    got = m.monte_carlo_predictions(n, x[:1], hs=(torch.zeros(L, n, H), torch.zeros(L, n, H)), masks=masks).cpu().numpy()
    np.testing.assert_array_equal(got, want)
    # the in-kernel output product (all_steps = 0) as well, and a nonzero state changes the outputs
    m.eval()
    zd = tuple(v.cuda() for v in zeros)
    np.testing.assert_array_equal(_direct(m, x, zd, "tcx"), _direct(m, x, None, "tcx"))
    moved = m(x, _hs(rng, L, rows, H)).cpu().numpy()
    assert np.abs(moved - m(x).cpu().numpy()).max() > 1e-3


def test_large_cell_state():
    # |c_0| up to 60 over T = 40 steps: |c_t| reaches ~100, far beyond the stateless |c_t| <= t bound; every ex2 argument of the
    # cell update is clamped (tc::lstm_cell2), so the outputs stay finite and fp32-grade
    I, H, L, O, T = 20, 256, 2, 12, 40
    m, state = _model(I, H, L, O)
    tm = OL.TorchDropoutLSTM.from_state(state, P)
    rng = np.random.default_rng(11)
    rows = 64
    x = torch.from_numpy(rng.normal(size=(rows, T, I)).astype(np.float32))
    hs = _hs(rng, L, rows, H, c=torch.from_numpy(rng.uniform(-60.0, 60.0, size=(L, rows, H)).astype(np.float32)))
    with torch.no_grad():
        want = tm(x, hs).numpy()
    got = m(x, hs).numpy()
    d = float(np.abs(got - want).max())
    print(f"H {H}: |c_0| <= 60, T = 40, split precision: |d| = {d:.3g}")
    assert np.isfinite(got).all() and d <= TOL


def _scaled(I, H, L, O, scale):
    state = syn.synth_state_dict(I, H, L, O, 31)
    return {k: (v * np.float32(scale)).astype(np.float32) if k.startswith("lstm.weight_") else v for k, v in state.items()}


@pytest.mark.parametrize("I,H,L,T,O", [(38, 128, 3, 6, 12), (20, 256, 2, 3, 12)])
def test_scaled_weights_stay_fp32_grade(I, H, L, T, O):
    # weights x 8: the single-pass kernels leave the 2e-4 tolerance (hs_variant = "auto" then picks fp32); the split kernels hold 2e-5
    state = _scaled(I, H, L, O, 8.0)
    tm = OL.TorchDropoutLSTM.from_state(state, P)
    rng = np.random.default_rng(1)
    x = torch.from_numpy(rng.normal(size=(64, T, I)).astype(np.float32))
    hs = _hs(rng, L, 64, H)
    split, _ = _model(I, H, L, O, state=state)
    single, _ = _model(I, H, L, O, state=state, lstm_variant="tc", hs_variant="tc")
    with torch.no_grad():
        want, want_hs = tm(x).numpy(), tm(x, hs).numpy()
    e_single, e_single_hs = float(np.abs(single(x).numpy() - want).max()), float(np.abs(single(x, hs).numpy() - want_hs).max())
    e_split = float(np.abs(split(x).numpy() - want).max())
    msg = f"H {H} weights x8 vs torch: forward(x) single pass {e_single:.3g}, split {e_split:.3g}"
    if H == 256:
        e_split_hs = float(np.abs(split(x, hs).numpy() - want_hs).max())
        msg += f"; forward(x, hs) single pass {e_single_hs:.3g}, split {e_split_hs:.3g}"
        assert e_split_hs <= TOL
    print(msg)
    assert e_split <= TOL


@pytest.mark.parametrize("I,H,L,T,O", [(38, 128, 3, 6, 12), (20, 256, 2, 8, 12), (20, 256, 3, 5, 12)])
def test_per_step_output_matches_in_kernel_product(I, H, L, T, O):
    # the per-step output layer (fp32 FMA chain over h = hi + lo) at t = T - 1 against the last layer's in-kernel tensor-core product
    # (all_steps = 0); and ape_mc_lstm_tc_launch_count reports the L layer launches + the output layer
    m, _ = _model(I, H, L, O)
    rng = np.random.default_rng(L * T)
    rows = 1000
    x = torch.from_numpy(rng.normal(size=(rows, T, I)).astype(np.float32)).cuda()
    every = _direct(m, x, None, "tcx", all_steps=1, mask_mode=N.MASK_NONE)
    last = _direct(m, x, None, "tcx", all_steps=0, mask_mode=N.MASK_NONE)
    np.testing.assert_array_equal(every, m(x).cpu().numpy())
    d = float(np.abs(every[:, T - 1] - last).max())
    print(f"(I,H,L,T,O)={(I, H, L, T, O)}: per-step output at T-1 vs in-kernel product |d| = {d:.3g}")
    assert d <= TOL
    a = N.LstmArgs()
    a.I, a.H, a.L, a.T, a.O = I, H, L, T, O
    a.B, a.nF, a.n_samples, a.all_steps, a.tc_flags = rows, 1, 1, 1, 3
    out = C.c_int(0)
    N.check(N.load().ape_mc_lstm_tc_launch_count(C.byref(a), C.byref(out)), "ape_mc_lstm_tc_launch_count")
    assert out.value == L + 1


def test_tcx_refuses_unsupported_shapes():
    rng = np.random.default_rng(0)
    m128, _ = _model(38, 128, 3, 12)
    with pytest.raises(UserWarning):           # no initial state on the H = 128 split kernel
        m128(torch.zeros(2, 6, 38), _hs(rng, 3, 2, 128))
    m256, _ = _model(20, 256, 2, 12)
    with pytest.raises(UserWarning):           # T > 40
        m256(torch.zeros(2, 41, 20))
    with pytest.raises(UserWarning):
        m256(torch.zeros(2, 41, 20), _hs(rng, 2, 2, 256))
    for shape in ((38, 128, 3, 17), (20, 256, 2, 33), (20, 256, 1, 12)):    # outside split_supported: O > 16 / O > 32, L = 1
        assert not N.split_supported(*shape)
        other, _ = _model(*shape)
        with pytest.raises(UserWarning):
            other(torch.zeros(2, 4, shape[0]))
