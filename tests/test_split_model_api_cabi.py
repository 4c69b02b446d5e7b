"""CPU: DropoutLSTM's model API on the split-precision tensor-core kernels (tc_flags = 3) - the all-steps workspace queries, the
C ABI's refusals of an initial state and of per-step outputs with a layer range, which all come before the first CUDA call, and the
"tcx" variant arguments."""
import ctypes as C

import pytest

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200.estimate import nn_models


def _args(H=256, h0=True, c0=True, n_samples=1, all_steps=1, layer_range=(0, 0)):
    a = N.LstmArgs()
    a.weights = a.weights_tcx = a.preds = a.x_dense = a.workspace = 256    # never dereferenced: every case is refused first
    a.I, a.H, a.L, a.T, a.O = 20, H, 3, 8, 12
    a.B, a.nF, a.n_samples = 64, 1, n_samples
    a.mask_mode, a.pred_ring, a.all_steps = N.MASK_NONE, 1, all_steps
    a.tc_flags = 3
    a.h0 = 512 if h0 else None
    a.c0 = 768 if c0 else None
    a.layer_begin, a.layer_end = layer_range
    return a


def test_split_all_steps_symbols_are_bound():
    lib = N.load()
    for name in ("ape_mc_lstm_tcx_workspace_bytes_all_steps", "ape_mc_lstm_tcxs_workspace_bytes_all_steps"):
        assert name in N.SYMBOLS and getattr(lib, name) is not None


def _u1(T, H, E, n):                          # one (hi or lo) buffer of a layer >= 1's sequence, 256-byte rounded
    tiles1 = -(-E * n // 256)
    return (tiles1 * 256 * T * H * 2 + 255) & ~255


@pytest.mark.parametrize("I,H,O", [(38, 128, 12), (20, 256, 12), (22, 256, 14)])
@pytest.mark.parametrize("T,E,n", [(8, 1, 100), (20, 600, 1), (40, 4096, 3)])
def test_split_all_steps_workspace(I, H, O, T, E, n):
    for L in (2, 3, 4):
        plain = N.split_workspace_bytes(I, H, L, T, O, E, n)
        every = N.split_workspace_bytes(I, H, L, T, O, E, n, all_steps=True)
        assert every >= plain
        if L == 2:                            # the kept last-layer sequence: one more (hi, lo) pair of layers >= 1
            assert every - plain == 2 * _u1(T, H, E, n)
        if L == 4:                            # two pairs already alternate between layers 1..3
            assert every == plain
    # the existing queries keep their values, and the dispatching helper matches the per-kernel ones
    assert N.split_workspace_bytes(I, H, 2, T, O, E, n) == (N.tcxs_workspace_bytes if H == 256 else N.tcx_workspace_bytes)(I, H, 2, T, O, E, n)
    lib = N.load()
    other = lib.ape_mc_lstm_tcxs_workspace_bytes_all_steps if H == 128 else lib.ape_mc_lstm_tcx_workspace_bytes_all_steps
    assert other(I, H, 2, T, O, E, n, C.byref(C.c_uint64(0))) == N.APE_ERR_UNSUPPORTED
    assert lib.ape_mc_lstm_tcxs_workspace_bytes_all_steps(I, H, 2, T, O, E, n, None) == N.APE_ERR_BAD_ARG


def test_split256_refuses_bad_initial_state_before_the_device():
    lib = N.load()
    assert lib.ape_mc_lstm_tc(_args(c0=False), None) == N.APE_ERR_BAD_ARG
    assert lib.ape_mc_lstm_tc(_args(h0=False), None) == N.APE_ERR_BAD_ARG
    for h0, c0 in ((516, 768), (512, 776)):   # the kernel reads float4 rows: 16-byte aligned pointers only
        a = _args()
        a.h0, a.c0 = h0, c0
        assert lib.ape_mc_lstm_tc(a, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_mc_lstm_tc(_args(n_samples=2), None) == N.APE_ERR_UNSUPPORTED
    # the H = 128 split kernel still takes no state
    assert lib.ape_mc_lstm_tc(_args(H=128), None) == N.APE_ERR_UNSUPPORTED


@pytest.mark.parametrize("H", [128, 256])
def test_split_all_steps_refuses_a_layer_range(H):
    lib = N.load()
    for rng in ((0, 1), (1, 3)):
        assert lib.ape_mc_lstm_tc(_args(H=H, h0=False, c0=False, layer_range=rng), None) == N.APE_ERR_UNSUPPORTED, rng
    if H == 256:
        assert lib.ape_mc_lstm_tc(_args(H=H, layer_range=(0, 1)), None) == N.APE_ERR_UNSUPPORTED


def test_dropout_lstm_tcx_variant_arguments():
    for H in (128, 256):
        m = nn_models.DropoutLSTM(20, H, 2, 12, lstm_variant="tcx", hs_variant="tcx")
        assert m.lstm_variant == "tcx" and m.hs_variant == "tcx"
    with pytest.raises(UserWarning):
        nn_models.DropoutLSTM(20, 256, 2, 12, lstm_variant="tcxs")
    with pytest.raises(UserWarning):
        nn_models.DropoutLSTM(20, 256, 2, 12, hs_variant="split")
    # "auto" keeps its two choices: single pass, else fp32
    m = nn_models.DropoutLSTM(20, 256, 2, 12)
    assert m.lstm_variant == "auto" and m.hs_variant == "fp32"
