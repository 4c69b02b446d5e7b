"""GPU (-m gpu): DropoutLSTM's model API with a caller-supplied initial state (h_0, c_0) on the one-layer tensor-core kernels
(hs_variant="tc": csrc/ape_lstm_tc.cu for H = 64 / 128, csrc/ape_lstm_tcs.cu for H = 256) - against torch.nn.LSTM, bit-equal to
the stateless kernel for a zero state, with large cell states, on ragged / both layer-0 row modes / multi-tile shapes, never on the
wavefront kernel, the hs_variant="auto" probe, and run-to-run."""
import ctypes as C

import numpy as np
import pytest
import torch

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200 import synthetic as syn
from arm_pose_estimation_b200.estimate import nn_models
from oracle import lstm as OL

pytestmark = pytest.mark.gpu
TC_TOL = 2e-4                                  # normalised outputs: the single-pass fp16-operand bound of the tensor-core path
SHAPES = [(9, 64, 2, 5, 14), (38, 128, 3, 6, 12), (20, 256, 2, 3, 12)]
P = 0.3


def _model(I, H, L, O, seed=31, hs_variant="tc", state=None):
    state = syn.synth_state_dict(I, H, L, O, seed) if state is None else state
    return nn_models.DropoutLSTM(I, H, L, O, P, philox_seed=77, hs_variant=hs_variant).load_state_dict(state).eval(), state


def _hs(rng, L, rows, H, scale=0.5, c_scale=None):
    h = (scale * rng.normal(size=(L, rows, H))).astype(np.float32)
    c = ((scale if c_scale is None else c_scale) * rng.normal(size=(L, rows, H))).astype(np.float32)
    return torch.from_numpy(h), torch.from_numpy(c)


@pytest.mark.parametrize("I,H,L,T,O", SHAPES)
@pytest.mark.parametrize("rows", [37, 600])   # ragged; layer 0 on 32-row CTAs (< 512 estimates) and on 128-row CTAs
def test_initial_state_against_torch(I, H, L, T, O, rows):
    m, state = _model(I, H, L, O)
    tm = OL.TorchDropoutLSTM.from_state(state, P)
    rng = np.random.default_rng(H + L + rows)
    x = torch.from_numpy(rng.normal(size=(rows, T, I)).astype(np.float32))
    hs = _hs(rng, L, rows, H)
    with torch.no_grad():
        want = tm(x, hs).numpy()
    got = m(x.cuda(), hs).cpu().numpy()
    e1 = np.abs(got - want).max()
    n = 6
    hs_n = _hs(rng, L, n, H)
    masks = OL.replay_torch_masks(5, T, n, H, L, P)
    torch.manual_seed(5)
    with torch.no_grad():
        want_mc = tm.monte_carlo_predictions(n, x[:1], hs_n).numpy()
    tm.eval()
    got_mc = m.monte_carlo_predictions(n, x[:1], hs=hs_n, masks=np.stack(masks)).numpy()
    e2 = np.abs(got_mc - want_mc).max()
    print(f"(I,H,L,T,O)={(I, H, L, T, O)} rows {rows} with (h_0, c_0) on tensor cores: forward |d|={e1:.3g}  mc |d|={e2:.3g}")
    assert got.shape == want.shape and got_mc.shape == want_mc.shape
    assert e1 <= TC_TOL and e2 <= TC_TOL


@pytest.mark.parametrize("I,H,L,T,O", SHAPES)
def test_zero_state_equals_no_state(I, H, L, T, O):
    m, _ = _model(I, H, L, O)
    m.lstm_variant = "tc"
    rng = np.random.default_rng(3)
    rows = 300
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
    # ... and a nonzero state changes the outputs
    m.eval()
    moved = m(x, _hs(rng, L, rows, H)).cpu().numpy()
    assert np.abs(moved - m(x).cpu().numpy()).max() > 1e-3


@pytest.mark.parametrize("I,H,L,T,O", SHAPES)
def test_large_cell_state(I, H, L, T, O):
    # |c_0| up to 60 over T = 40 steps: |c_t| reaches ~100, beyond the stateless kernels' |c_t| <= t bound.  The bound is wider than
    # TC_TOL, which holds for the deployed sequence lengths (<= 8): over 40 steps the fp16 rounding of h_t adds up to ~2.7e-4 (B200)
    T = 40
    m, state = _model(I, H, L, O)
    tm = OL.TorchDropoutLSTM.from_state(state, P)
    rng = np.random.default_rng(11)
    rows = 64
    x = torch.from_numpy(rng.normal(size=(rows, T, I)).astype(np.float32))
    h = torch.from_numpy((0.5 * rng.normal(size=(L, rows, H))).astype(np.float32))
    c = torch.from_numpy(rng.uniform(-60.0, 60.0, size=(L, rows, H)).astype(np.float32))
    with torch.no_grad():
        want = tm(x, (h, c)).numpy()
    got = m(x, (h, c)).numpy()
    print(f"H {H}: |c_0| <= 60, T = 40: |d| = {np.abs(got - want).max():.3g}")
    assert np.isfinite(got).all()
    np.testing.assert_allclose(got, want, rtol=0, atol=5e-4)


def _launch_count(I, H, L, T, O, rows, with_state):
    a = N.LstmArgs()
    a.I, a.H, a.L, a.T, a.O = I, H, L, T, O
    a.B, a.nF, a.n_samples, a.all_steps = rows, 1, 1, 1
    if with_state:
        a.h0 = a.c0 = 256
    out = C.c_int(0)
    N.check(N.load().ape_mc_lstm_tc_launch_count(C.byref(a), C.byref(out)), "ape_mc_lstm_tc_launch_count")
    return out.value


@pytest.mark.parametrize("I,H,L,T,O", [(38, 128, 3, 4, 12), (20, 256, 2, 3, 12)])
def test_multi_tile_against_fp32(I, H, L, T, O):
    # more than 148 x 256 rows in layers >= 1: CTA pairs take several tiles, so h_0 / c_0 are reloaded at tile boundaries (behind the
    # previous tile's output product).  At this size tc_flags 0 would pair the H = 128 layers into the wavefront kernel; with a
    # state it must not.
    rows = 148 * 256 + 1000
    if H == 128:
        assert _launch_count(I, H, L, T, O, rows, False) == L
        assert _launch_count(I, H, L, T, O, rows, True) == L + 1
    m, state = _model(I, H, L, O)
    ref = nn_models.DropoutLSTM(I, H, L, O, P, hs_variant="fp32").load_state_dict(state).eval()
    rng = np.random.default_rng(rows)
    x = torch.from_numpy(rng.normal(size=(rows, T, I)).astype(np.float32)).cuda()
    hs = tuple(v.cuda() for v in _hs(rng, L, rows, H))
    got, want = m(x, hs), ref(x, hs)
    d = (got - want).abs().max().item()
    print(f"H {H} L {L}: {rows} rows with (h_0, c_0): |tc - fp32| = {d:.3g}")
    assert d <= TC_TOL
    np.testing.assert_array_equal(m(x, hs).cpu().numpy(), got.cpu().numpy())     # run to run


def _last_step(m, x, hs, tc, tc_flags=0):
    """ape_mc_lstm_tc / ape_mc_lstm_fma as the estimators call them: all_steps = 0, the output layer of the last step only (on the
    tensor-core path the output product inside the last layer's kernel, issued at tile boundaries), Philox masks, one row per estimate."""
    I, H, L, O = m._dims()
    E, T, _ = x.shape
    preds = torch.full((E, 1, 1, O), float("nan"), dtype=torch.float32, device="cuda")
    a = N.LstmArgs()
    a.weights = m.packed_weights().data_ptr()
    a.weights_tc = m.packed_weights_tc().data_ptr() if tc else None
    a.I, a.H, a.L, a.T, a.O = I, H, L, T, O
    a.dropout_p = P
    a.x_dense, a.B, a.nF, a.frame0, a.n_samples = x.data_ptr(), E, 1, 3, 1
    a.mask_mode, a.philox_seed, a.tc_flags = N.MASK_PHILOX, 99, tc_flags
    if hs is not None:
        a.h0, a.c0 = hs[0].data_ptr(), hs[1].data_ptr()
    ws = torch.empty(N.workspace_bytes(I, H, L, T, O, E, 1, tensor_core=tc), dtype=torch.uint8, device="cuda")
    a.workspace = ws.data_ptr()
    a.preds, a.pred_ring, a.all_steps = preds.data_ptr(), 1, 0
    fn = N.load().ape_mc_lstm_tc if tc else N.load().ape_mc_lstm_fma
    N.check(fn(C.byref(a), N.current_stream_ptr()), "ape_mc_lstm_tc" if tc else "ape_mc_lstm_fma")
    torch.cuda.synchronize()
    return preds.reshape(E, O).cpu().numpy()


@pytest.mark.parametrize("I,H,L,T,O", SHAPES)
def test_last_step_output_product_multi_tile(I, H, L, T, O):
    # all_steps = 0 with a state: the last layer's kernel runs its output product, which with a state goes ahead of step 0 of the next
    # tile; 153 tiles per layer >= 1 give every CTA pair two or three tiles.  Against the fp32 kernel, and bit for bit against the
    # stateless one-layer kernels for h_0 = c_0 = 0.  tc_flags = 0 with a state must not pair the H = 128 layers.
    rows = 148 * 256 + 1000
    m, _ = _model(I, H, L, O)
    rng = np.random.default_rng(rows + H)
    x = torch.from_numpy(rng.normal(size=(rows, T, I)).astype(np.float32)).cuda()
    hs = tuple(v.cuda().contiguous() for v in _hs(rng, L, rows, H))
    got = _last_step(m, x, hs, True)
    want = _last_step(m, x, hs, False)
    assert np.isfinite(got).all()
    d = np.abs(got - want).max()
    print(f"H {H} L {L}: {rows} rows, all_steps = 0 with (h_0, c_0): |tc - fp32| = {d:.3g}")
    assert d <= TC_TOL
    np.testing.assert_array_equal(_last_step(m, x, hs, True), got)                  # run to run
    zeros = tuple(torch.zeros_like(v) for v in hs)                                  # (tc_flags = 1: the same one-layer kernels)
    np.testing.assert_array_equal(_last_step(m, x, zeros, True), _last_step(m, x, None, True, tc_flags=1))


def _scaled(I, H, L, O, scale):
    state = syn.synth_state_dict(I, H, L, O, 31)
    return {k: (v * np.float32(scale)).astype(np.float32) if k.startswith("lstm.weight_") else v for k, v in state.items()}


@pytest.mark.parametrize("I,H,L,T,O", [(38, 128, 3, 6, 12), (20, 256, 2, 3, 12)])
def test_hs_variant_auto(I, H, L, T, O):
    rng = np.random.default_rng(1)
    x = torch.from_numpy(rng.normal(size=(8, T, I)).astype(np.float32))
    hs = _hs(rng, L, 8, H)
    m, state = _model(I, H, L, O, hs_variant="auto")
    got = m(x, hs).numpy()
    print(f"H {H} seeded weights: hs probe {m.hs_probe_error:.3g} -> {m.hs_choice}")
    assert m.hs_choice == "tc" and m.hs_probe_error <= TC_TOL
    with torch.no_grad():
        np.testing.assert_allclose(got, OL.TorchDropoutLSTM.from_state(state, P)(x, hs).numpy(), rtol=0, atol=TC_TOL)
    big, state8 = _model(I, H, L, O, hs_variant="auto", state=_scaled(I, H, L, O, 8.0))
    got8 = big(x, hs).numpy()
    print(f"H {H} weights x8: hs probe {big.hs_probe_error:.3g} -> {big.hs_choice}")
    assert big.hs_choice == "fp32" and big.hs_probe_error > TC_TOL
    exact, _ = _model(I, H, L, O, hs_variant="fp32", state=state8)
    np.testing.assert_array_equal(got8, exact(x, hs).numpy())


def test_hs_variant_tc_refuses_unsupported_shapes():
    m, _ = _model(20, 64, 2, 12)
    rng = np.random.default_rng(0)
    with pytest.raises(UserWarning):           # T > 40
        m(torch.zeros(2, 41, 20), _hs(rng, 2, 2, 64))
    one, _ = _model(20, 64, 1, 12)             # L = 1: no tensor-core kernel
    with pytest.raises(UserWarning):
        one(torch.zeros(2, 4, 20), _hs(rng, 1, 2, 64))
