"""CPU: the corner shapes of every tensor-core LSTM kernel (tests/test_gpu_lstm_envelope.py runs them on the GPU) through the C-ABI
queries alone - the packers write exactly the bytes the library will read, the ``supported`` predicates take each shape and refuse
the next step past each limit (I = H + 1, O one past the kernel's output width).  T = 41 is pinned in test_tc_driver_cabi.py; the
cluster kernel's L <= 4 is checked after the device query, so its refusal of L = 5 is a GPU test."""
import ctypes as C

import pytest

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200 import synthetic as syn
from arm_pose_estimation_b200.estimate import nn_models

# (I, H, L, O) of the single-pass kernels (tc_flags 1, 2, 4): the one-layer kernel at H = 64 / 128 (I = H and I = H - 15, which pads
# to the same k-groups), the streamed-weights kernel at H = 256, the wavefront kernel at L = 4 / 5, the cluster kernel at L = 2 / 4
SINGLE_PASS = [(64, 64, 2, 16), (49, 64, 5, 16), (128, 128, 2, 16), (113, 128, 5, 16), (256, 256, 4, 20),
               (38, 128, 4, 16), (38, 128, 5, 16), (128, 128, 4, 16), (256, 256, 2, 20)]
# the split-precision kernels (tc_flags 3): H = 128 up to O = 16, H = 256 up to O = 32
SPLIT = [(128, 128, 2, 16), (128, 128, 4, 16), (128, 128, 5, 16), (256, 256, 4, 32), (256, 256, 5, 32)]
O_MAX_SINGLE = {64: 16, 128: 16, 256: 20}
O_MAX_SPLIT = {128: 16, 256: 32}


@pytest.mark.parametrize("I,H,L,O", SINGLE_PASS)
def test_single_pass_corner_shapes(I, H, L, O):
    state = syn.synth_state_dict(I, H, L, O, 3 + I + L)
    assert nn_models.pack_lstm_weights_tc(state).size == N.tc_blob_bytes(I, H, L)
    assert N.tc_supported(I, H, L, O)
    assert not N.tc_supported(H + 1, H, L, O)                        # layer 0's input k-groups past H
    assert not N.tc_supported(I, H, L, O_MAX_SINGLE[H] + 1)          # one output past the output product
    assert N.tc_supported(I, H, L, O_MAX_SINGLE[H])
    for all_steps in (False, True):
        assert N.workspace_bytes(I, H, L, 40, O, 600, 1, tensor_core=True, all_steps=all_steps) > 0


@pytest.mark.parametrize("I,H,L,O", SPLIT)
def test_split_corner_shapes(I, H, L, O):
    state = syn.synth_state_dict(I, H, L, O, 5 + I + L)
    assert nn_models.pack_lstm_weights_tcx(state).size == N.split_blob_bytes(I, H, L)
    assert N.split_supported(I, H, L, O)
    assert (N.tcx_supported if H == 128 else N.tcxs_supported)(I, H, L, O)
    assert not N.split_supported(H + 1, H, L, O)
    assert not N.split_supported(I, H, L, O_MAX_SPLIT[H] + 1)
    assert N.split_supported(I, H, L, O_MAX_SPLIT[H])
    for all_steps in (False, True):
        assert N.split_workspace_bytes(I, H, L, 40, O, 300, 1, all_steps=all_steps) > 0
    # a query that belongs to the other width refuses the shape
    other = N.load().ape_mc_lstm_tcxs_workspace_bytes if H == 128 else N.load().ape_mc_lstm_tcx_workspace_bytes
    out = C.c_uint64(0)
    assert other(I, H, L, 40, O, 300, 1, C.byref(out)) == N.APE_ERR_UNSUPPORTED


def test_wide_output_is_split_only():
    # O = 21 .. 32 at H = 256 runs on the split kernel only; the single-pass kernels refuse it
    for O in (21, 32):
        assert N.split_supported(256, 256, 4, O) and not N.tc_supported(256, 256, 4, O)
