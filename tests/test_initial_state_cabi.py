"""CPU: the initial-state (h_0, c_0) surface of the tensor-core LSTM path - the C ABI's refusals, which all come before the first
CUDA call, the step schedule of the H = 256 kernel for the first step of a tile with a state, and DropoutLSTM's hs_variant."""
import ctypes as C

import pytest

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200.estimate import nn_models

NCH, KG, SLICE_KG = 8, 32, 4                   # H = 256: 8 chunks of 32 units, 32 k-groups, K-slices of 4 k-groups


def _args(h0=True, c0=True, n_samples=1, tc_flags=0):
    a = N.LstmArgs()
    a.weights = a.weights_tc = a.preds = a.x_dense = a.workspace = 256      # never dereferenced: every case is refused first
    a.I, a.H, a.L, a.T, a.O = 20, 128, 3, 8, 12
    a.B, a.nF, a.n_samples = 64, 1, n_samples
    a.mask_mode, a.pred_ring, a.all_steps = N.MASK_NONE, 1, 1
    a.tc_flags = tc_flags
    a.h0 = 512 if h0 else None
    a.c0 = 768 if c0 else None
    return a


def test_tc_refuses_bad_initial_state_before_the_device():
    lib = N.load()
    assert lib.ape_mc_lstm_tc(_args(c0=False), None) == N.APE_ERR_BAD_ARG
    assert lib.ape_mc_lstm_tc(_args(h0=False), None) == N.APE_ERR_BAD_ARG
    assert lib.ape_mc_lstm_tc(_args(n_samples=2), None) == N.APE_ERR_UNSUPPORTED
    for flags in (2, 3, 4):                    # wavefront, split-precision and small-batch kernels take no state
        assert lib.ape_mc_lstm_tc(_args(tc_flags=flags), None) == N.APE_ERR_UNSUPPORTED, flags
    for h0, c0 in ((516, 768), (512, 776)):    # the state kernels read float4 rows: 16-byte aligned pointers only
        a = _args()
        a.h0, a.c0 = h0, c0
        assert lib.ape_mc_lstm_tc(a, None) == N.APE_ERR_BAD_ARG


def _schedule(kgx, first_step):
    lib = N.load()
    buf = (C.c_uint32 * (2 * 64))()
    n = C.c_int(0)
    assert lib.ape_selfcheck_tcs_schedule(kgx, first_step, buf, 64, C.byref(n)) == N.APE_OK
    return [(buf[2 * i], buf[2 * i + 1]) for i in range(n.value)]


def _piece(x):
    slot, is_h, nmma, src = x & 1, bool(x & 2), (x >> 8) & 0x1F, x >> 17
    return slot, is_h, nmma, src


@pytest.mark.parametrize("kgx", [4, 12, 32])
def test_tcs_first_step_with_state_schedule(kgx):
    ent = _schedule(kgx, 2)
    cover_x = {c: [] for c in range(NCH)}
    cover_h = {c: [] for c in range(NCH)}
    begun, done, x_done, out_at = [], [], [], []
    seen_h = False
    for i, (x, y) in enumerate(ent):
        slot, is_h, nmma, src = _piece(x)
        chunk, off = divmod(src, kgx + KG)
        assert chunk % 2 == slot and 1 <= nmma <= 16
        if x & 8:
            begun.append(chunk)
        if x & 64:
            out_at.append(i)
            assert not seen_h                  # the previous tile's output piece goes ahead of every recurrent piece
        if is_h:
            seen_h = True
            kg0 = off - kgx
            assert y == kg0 * 4 and ((x >> 13) & 0xF) == -(-(kg0 + 2 * nmma) // SLICE_KG)
            cover_h[chunk] += list(range(kg0, kg0 + 2 * nmma))
        else:
            assert off + 2 * nmma <= kgx and y == off * 128 and not (x >> 13) & 0xF
            cover_x[chunk] += list(range(off, off + 2 * nmma))
        if x & 16:
            done.append(chunk)
        if x & 32:
            x_done.append(chunk)
    for c in range(NCH):                       # every operand exactly once
        assert cover_x[c] == list(range(kgx)) and sorted(cover_h[c]) == list(range(KG)), c
    assert begun == list(range(NCH)) and sorted(done) == list(range(NCH)) and x_done == [NCH - 2, NCH - 1]
    assert len(out_at) == 1 and _piece(ent[out_at[0]][0])[:2] == (1, False)      # on chunk 1's x-part, as without a state
    for c in range(NCH):                       # the recurrent part of a chunk starts after its x-part
        xs = [i for i, (x, _) in enumerate(ent) if not x & 2 and _piece(x)[3] // (kgx + KG) == c]
        hs = [i for i, (x, _) in enumerate(ent) if x & 2 and _piece(x)[3] // (kgx + KG) == c]
        assert max(xs) < min(hs)
    # the x-part MMAs of every chunk are those of the stateless first step, in the same order and with the same overwrite flag:
    # with h_0 = c_0 = 0 the accumulators then hold the same bits
    x_of = lambda e: [(x & 0x7, (x >> 8) & 0x1F, x >> 17, y) for x, y in e if not x & 2]
    assert x_of(ent) == x_of(_schedule(kgx, 1))
    assert N.load().ape_selfcheck_tcs_schedule(kgx, 3, (C.c_uint32 * 128)(), 64, C.byref(C.c_int(0))) == N.APE_ERR_BAD_ARG


def test_dropout_lstm_hs_variant_argument():
    with pytest.raises(UserWarning):
        nn_models.DropoutLSTM(20, 64, 2, 12, hs_variant="bogus")
    m = nn_models.DropoutLSTM(20, 64, 2, 12)
    assert m.hs_variant == "fp32" and m.hs_choice is None and m.hs_probe_error is None
    for v in ("auto", "fp32", "tc"):
        assert nn_models.DropoutLSTM(20, 256, 2, 12, hs_variant=v).hs_variant == v
