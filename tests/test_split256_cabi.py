"""CPU: the H = 256 split-precision kernel's C-ABI queries and its weight blob (csrc/ape_lstm_tcxs.cu; no compute calls)."""
import numpy as np

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200 import synthetic as syn
from arm_pose_estimation_b200.estimate import nn_models


def test_split256_symbols_are_bound():
    lib = N.load()
    for name in ("ape_mc_lstm_tcxs_supported", "ape_lstm_tcxs_blob_bytes", "ape_mc_lstm_tcxs_workspace_bytes"):
        assert name in N.SYMBOLS and getattr(lib, name) is not None


def test_split256_supported_shapes():
    # the deployed watch-only (I20 H256 L2 O12) and pocket (I22 H256 L2 O14) models, and an L = 3 / O = 20 model
    for shape in [(20, 256, 2, 12), (22, 256, 2, 14), (38, 256, 3, 20), (20, 256, 2, 32)]:
        assert N.tcxs_supported(*shape) and N.split_supported(*shape), shape
    for shape in [(20, 128, 2, 12), (38, 128, 3, 12), (20, 64, 2, 12), (20, 256, 1, 12), (20, 256, 2, 33), (300, 256, 2, 12)]:
        assert not N.tcxs_supported(*shape), shape
    # the H = 128 query keeps answering for its own kernel only
    assert not N.tcx_supported(20, 256, 2, 12) and N.tcx_supported(38, 128, 3, 12)
    assert N.split_supported(38, 128, 3, 12)
    assert N.tcxs_workspace_bytes(20, 256, 2, 8, 12, 1024, 100) > 0
    lib = N.load()
    assert lib.ape_mc_lstm_tcxs_workspace_bytes(20, 128, 2, 8, 12, 16, 4, None) == N.APE_ERR_BAD_ARG


def test_split256_blob_layout():
    # pack_lstm_weights_tcx at H = 256: per layer 2 CTAs x 8 chunks x [Wx_hi + bias K step | Wx_lo | Wh_hi | Wh_lo], then the output
    # layer (32 columns, rounding and remainder); hi + lo reproduce the halved weights to ~2^-20 and the size is the library's
    I, H, L, O = 20, 256, 3, 20
    state = syn.synth_state_dict(I, H, L, O, 7)
    blob = nn_models.pack_lstm_weights_tcx(state)
    assert blob.size == N.tcxs_blob_bytes(I, H, L) == N.split_blob_bytes(I, H, L)
    halfs = blob.view(np.float16)
    kin_pad = 32
    p0, p1, ph = (kin_pad + 16) * 64, kin_pad * 64, H * 64
    chunk0 = p0 + p1 + 2 * ph
    layer0 = 2 * (H // 32) * chunk0
    n = np.arange(64)
    scale = np.where(n % 4 != 2, 0.5, 1.0)

    def tile(at, k):
        return halfs[at:at + k * 64].reshape(k // 8, 64, 8).transpose(1, 0, 2).reshape(64, k).astype(np.float64)

    for r, c in ((0, 0), (1, 5)):                                          # CTA r of the pair, 32-unit chunk c
        rows = (n % 4) * H + 32 * c + (64 * r + n) // 4
        at = (r * (H // 32) + c) * chunk0
        hi, lo = tile(at, kin_pad + 16), tile(at + p0, kin_pad)
        w = state["lstm.weight_ih_l0"][rows].astype(np.float64) * scale[:, None]
        assert np.abs(hi[:, :I] + lo[:, :I] - w).max() <= 2.0 ** -20 * np.abs(w).max() and not hi[:, I:kin_pad].any()
        b = (state["lstm.bias_ih_l0"] + state["lstm.bias_hh_l0"])[rows].astype(np.float64) * scale
        assert np.abs(hi[:, kin_pad] + hi[:, kin_pad + 1] - b).max() <= 2.0 ** -20 * np.abs(b).max() and not hi[:, kin_pad + 2:].any()
        wh = state["lstm.weight_hh_l0"][rows].astype(np.float64) * scale[:, None]
        assert np.abs(tile(at + p0 + p1, H) + tile(at + p0 + p1 + ph, H) - wh).max() <= 2.0 ** -20 * np.abs(wh).max()
    # layer 1 (x-part of H K-values), CTA 0, chunk 7
    p0, p1 = (H + 16) * 64, H * 64
    rows = (n % 4) * H + 32 * 7 + n // 4
    at = layer0 + 7 * (p0 + p1 + 2 * ph)
    w = state["lstm.weight_ih_l1"][rows].astype(np.float64) * scale[:, None]
    assert np.abs(tile(at, H + 16)[:, :H] + tile(at + p0, H) - w).max() <= 2.0 ** -20 * np.abs(w).max()
    # output layer: 2 x [H/8][32][8] halfs at the end, rows >= O zero
    wo = halfs[-2 * H * 32:].reshape(2, H // 8, 32, 8).transpose(0, 2, 1, 3).reshape(2, 32, H).astype(np.float64)
    want = state["output_layer.weight"].astype(np.float64)
    assert np.abs(wo[0, :O] + wo[1, :O] - want).max() <= 2.0 ** -20 * np.abs(want).max() and not wo[:, O:].any()
