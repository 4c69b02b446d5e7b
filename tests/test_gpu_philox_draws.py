"""GPU (-m gpu): every kernel's in-kernel Philox dropout draw, bit for bit, against the numpy reference ``oracle/philox.py``.

A kernel in APE_MASK_PHILOX mode and the same kernel in APE_MASK_INJECTED mode with the reference's masks build the same keep decisions and
apply them the same way (the same AND mask or select, the same 1 / (1 - p) scale), so their predictions must be equal to the bit.  A
single keep bit drawn differently - a lane on the threshold, the other half of the branch-free two-lane compare (p > 0.5), a lost seed
word, a counter field cut short - changes some prediction, which no tolerance comparison at p = 0.2 would see.

Every case runs at keep thresholds THR (both ends, both sides of bit 15, p = 0.2) and at p = 0.2 itself, with a seed whose high word is
not zero, stream ids that wrap at 2^32, frames near 2^31 and two frames per stream; the LSTM kernels also with per-stream frame counters.
At p = 0 Philox mode must equal APE_MASK_NONE.  ``ape_philox_masks`` (the export a checker replays) is held to the reference directly.
The shapes are small: the point is the counters, not the rows."""
import ctypes as C

import numpy as np
import pytest
import torch

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200 import synthetic as syn
from arm_pose_estimation_b200.estimate import nn_models
from oracle import philox as OP
import test_gpu_stream_frames as SF
from test_gpu_lstm_envelope import inputs, run_lstm

pytestmark = pytest.mark.gpu

THR = [65536, 65535, 52429, 32769, 32768, 32767, 16384, 1, 0]


def p_of(thr):
    """The float32 drop probability of keep threshold ``thr`` (exact: 1 - thr / 65536); thr 0: p = 1 - 2^-18, as p = 1 is refused."""
    return float(np.float32(1.0 - 2.0 ** -18)) if thr == 0 else float(np.float32(1.0 - thr / 65536.0))


P_SWEEP = [p_of(t) for t in THR] + [0.2]
SEED = 0x9E37_79B9_7F4A_7C15                   # both key words non-zero
SEED_HI = 1 << 32                              # low key word zero: only the high word tells it from seed 0
SID0 = 2 ** 32 - 3                             # stream ids 2^32 - 3 .. wrap to 0, 1, ... from the fourth stream on


def test_thresholds_of_the_sweep():
    assert [OP.keep_threshold16(p) for p in P_SWEEP] == THR + [52429]


def sweep(run, lanes, label):
    """``run(mask_mode, p, masks)`` -> predictions; Philox mode against injected mode with the reference's masks at every p of the sweep,
    and Philox mode at p = 0 against APE_MASK_NONE.  Asserts the case is not vacuous."""
    outs = {}
    for p in P_SWEEP:
        thr = OP.keep_threshold16(p)
        masks = OP.masks_from_lanes(lanes, p)
        kept = int(masks.sum())
        if thr == 65536:
            assert kept == masks.size
        elif thr == 0:
            assert kept == 0
        else:
            assert 0 < kept < masks.size, f"{label}: keep_thr16 {thr}: {kept} of {masks.size} units kept - a vacuous case"
        got = run(N.MASK_PHILOX, p, None)
        want = run(N.MASK_INJECTED, p, masks)
        if p == 0.2:                                            # (at p near 1 the scale 1 / (1 - p) may overflow fp16 operands)
            assert np.isfinite(got).all(), f"{label}: non-finite predictions at p = 0.2"
        np.testing.assert_array_equal(got.view(np.int32), want.view(np.int32),
                                      err_msg=f"{label}: Philox vs injected reference masks, keep_thr16 {thr} (p = {p!r})")
        outs[p] = got
    assert not np.array_equal(outs[p_of(52429)], outs[p_of(32767)]), f"{label}: the predictions do not depend on the masks"
    np.testing.assert_array_equal(outs[0.0].view(np.int32), run(N.MASK_NONE, 0.0, None).view(np.int32),
                                  err_msg=f"{label}: Philox at p = 0 vs no dropout")
    print(f"{label}: Philox = injected reference masks bit for bit at keep_thr16 {THR} and p = 0.2; p = 0 = no dropout "
          f"({lanes.size} units per call)")


# ---- a. the export ----------------------------------------------------------------------------------------------------------------
# (B, nF, L, T, n, H): three streams across the 2^32 wrap; gap 14 with t 255; samples >= 256 with t 255
EXPORT = [(3, 2, 3, 5, 7, 16), (1, 2, 16, 256, 2, 8), (1, 1, 2, 256, 300, 8)]


@pytest.mark.parametrize("B,nF,L,T,n,H", EXPORT)
def test_exported_masks_equal_the_reference(B, nF, L, T, n, H):
    sid0, f0 = 2 ** 32 - 2, 2 ** 31 - nF
    lanes = OP.lstm_lanes(SEED, sid0, B, nF, f0, L, T, n, H)
    m = torch.empty((B * nF, L - 1, T, n, H), dtype=torch.uint8, device="cuda")
    for p in P_SWEEP:
        m.fill_(7)
        N.check(N.load().ape_philox_masks(SEED, sid0, B, nF, f0, L, T, n, H, p, N.ptr(m), N.current_stream_ptr()), "ape_philox_masks")
        np.testing.assert_array_equal(m.cpu().numpy(), OP.masks_from_lanes(lanes, p), err_msg=f"keep_thr16 {OP.keep_threshold16(p)}")


# ---- b / c. every LSTM kernel -------------------------------------------------------------------------------------------------
# (kernel of run_lstm, H, I, L, T, O, B, nF, n)
LSTM_CASES = [
    ("fp32", 32, 20, 16, 256, 12, 4, 1, 3),        # gap 14, t 255
    ("fp32", 128, 38, 4, 40, 16, 1, 2, 300),
    ("tc", 64, 38, 3, 3, 16, 4, 2, 300),
    ("tc", 128, 38, 3, 3, 16, 4, 2, 300),
    ("tc", 256, 38, 2, 3, 20, 4, 2, 300),          # tcs
    ("tcw", 128, 38, 5, 3, 16, 4, 2, 300),
    ("split", 128, 38, 3, 3, 16, 4, 2, 300),       # tcx
    ("split", 256, 38, 2, 3, 20, 4, 2, 300),       # tcxs
    ("tcl", 128, 38, 3, 3, 16, 4, 2, 300),
    ("tcl", 256, 38, 2, 3, 20, 4, 2, 300),
    ("tcxl", 128, 38, 3, 3, 16, 4, 2, 300),
    ("tcxsl", 256, 38, 2, 3, 20, 4, 2, 300),
]
LSTM_IDS = [f"{k}-H{H}-L{L}-T{T}-{B}x{nF}x{n}" for k, H, I, L, T, O, B, nF, n in LSTM_CASES]


def _lstm_case(H, I, L, T, O, B, nF, n):
    state = syn.synth_state_dict(I, H, L, O, 900 + H + L + T)
    x, _ = inputs(I, H, L, T, B * nF, n, seed=H * L + T, masked=False)
    return state, x


@pytest.mark.parametrize("kernel,H,I,L,T,O,B,nF,n", LSTM_CASES, ids=LSTM_IDS)
def test_lstm_philox_equals_injected_reference_masks(kernel, H, I, L, T, O, B, nF, n):
    state, x = _lstm_case(H, I, L, T, O, B, nF, n)
    f0 = 2 ** 31 - 8
    lanes = OP.lstm_lanes(SEED, SID0, B, nF, f0, L, T, n, H)

    def run(mode, p, masks):
        return run_lstm(state, x, masks, n, kernel, p=p, philox=(SEED, SID0) if mode == N.MASK_PHILOX else None, nF=nF, frame0=f0)

    sweep(run, lanes, f"{kernel} H{H} L{L} T{T} {B} streams x {nF} frames x {n} samples")


@pytest.mark.parametrize("kernel,H,I,L,T,O,B,nF,n", LSTM_CASES, ids=LSTM_IDS)
def test_lstm_philox_with_per_stream_frames(kernel, H, I, L, T, O, B, nF, n):
    state, x = _lstm_case(H, I, L, T, O, B, nF, n)
    sf = [2 ** 31 - 9, 5, 0, 1000][:B]                         # one stream far ahead
    lanes = OP.lstm_lanes(SEED_HI, SID0, B, nF, 0, L, T, n, H, stream_frames=sf)
    for b in range(B):                                          # the export, per stream at its own frame, agrees
        for p in (0.2, p_of(32767)):
            np.testing.assert_array_equal(SF.philox_masks(SEED_HI, (SID0 + b) & 0xFFFFFFFF, nF, sf[b], L, T, n, H, p),
                                          OP.masks_from_lanes(lanes[b * nF:(b + 1) * nF], p))
    outs = {}
    for p in (0.2, p_of(32767)):
        masks = OP.masks_from_lanes(lanes, p)
        assert 0 < masks.sum() < masks.size
        got = run_lstm(state, x, None, n, kernel, p=p, philox=(SEED_HI, SID0), nF=nF, stream_frames=sf)
        want = run_lstm(state, x, masks, n, kernel, p=p, nF=nF, stream_frames=sf)
        np.testing.assert_array_equal(got.view(np.int32), want.view(np.int32), err_msg=f"{kernel}: stream_frames {sf}, p = {p!r}")
        outs[p] = got
    assert not np.array_equal(*outs.values())


# ---- b / c. the feed-forward kernels ----------------------------------------------------------------------------------------------
def _ff_blob(I, H, Lh, O, seed, offset_floats):
    """The packed blob on the device, ``offset_floats`` floats past a 256-byte aligned allocation; (pointer, owner)."""
    blob = nn_models.pack_ff_weights(syn.synth_ff_state_dict(I, H, Lh, O, seed=seed))
    buf = torch.zeros(blob.size + offset_floats, dtype=torch.float32, device="cuda")
    buf[offset_floats:] = torch.from_numpy(blob).cuda()
    return C.c_void_p(buf.data_ptr() + 4 * offset_floats), buf


# (label, I, H, Lh, O, rows, n, blob offset in floats): the batched kernel; the one-CTA-per-row kernel for H % 8 != 0 and for a blob
# that is not 16-byte aligned (ape_mc_ff's routing rule)
FF_CASES = [("batched", 38, 256, 2, 20, 5, 300, 0), ("row-H100", 38, 100, 1, 12, 8, 400, 0), ("row-unaligned-blob", 38, 256, 2, 20, 5, 300, 1)]


@pytest.mark.parametrize("label,I,H,Lh,O,rows,n,off", FF_CASES, ids=[c[0] for c in FF_CASES])
def test_ff_philox_equals_injected_reference_masks(label, I, H, Lh, O, rows, n, off):
    blob, keep = _ff_blob(I, H, Lh, O, 31 + H, off)
    x = torch.from_numpy(np.random.default_rng(H).normal(0, 1, (rows, I)).astype(np.float32)).cuda()
    frame0 = 0xFFFFFFF0                                         # ape_mc_ff takes any uint32 frame
    lanes = OP.ff_lanes(SEED, SID0, rows, frame0, n, H)

    def run(mode, p, masks):
        md = None if masks is None else torch.from_numpy(masks).cuda()
        preds = torch.full((rows, n, O), float("nan"), dtype=torch.float32, device="cuda")
        N.check(N.load().ape_mc_ff(blob, I, H, Lh, O, p, N.ptr(x), rows, n, mode, N.ptr(md), SEED, SID0, frame0, N.ptr(preds),
                                   N.current_stream_ptr()), "ape_mc_ff")
        return preds.cpu().numpy()

    sweep(run, lanes, f"ape_mc_ff {label} H{H} {rows} rows x {n} samples")


def test_ff_ring_philox_equals_injected_reference_masks():
    I, T, H, Lh, O, B, nF, n = 38, 6, 256, 2, 20, 5, 2, 300
    sf = [2 ** 31 - 9, -1, 0, 7, 1000]                          # stream 1 sits the call out
    feat_ring, pred_ring = nF + T, nF
    blob, keep = _ff_blob(I * T, H, Lh, O, 5, 0)
    feats = torch.from_numpy(np.random.default_rng(9).normal(0, 1, (B, feat_ring, I)).astype(np.float32)).cuda()
    sfd = torch.tensor(sf, dtype=torch.int32, device="cuda")
    lanes = OP.ff_ring_lanes(SEED, SID0, B, nF, 0, n, H, stream_frames=sf)
    written = np.repeat(np.array(sf) >= 0, pred_ring)           # [B * pred_ring] slots: all of an active stream, none of stream 1

    def run(mode, p, masks):
        md = None if masks is None else torch.from_numpy(masks).cuda()
        preds = torch.empty((B, pred_ring, n, O), dtype=torch.float32, device="cuda")
        SF._fill_sentinel(preds)
        N.check(N.load().ape_mc_ff_ring(blob, I, T, H, Lh, O, p, N.ptr(feats), feat_ring, B, nF, 0, N.ptr(sfd), n, mode, N.ptr(md), SEED,
                                        SID0, N.ptr(preds), pred_ring, N.current_stream_ptr()), "ape_mc_ff_ring")
        bits = SF._bits(preds).reshape(B * pred_ring, -1)
        assert (bits[~written] == SF.SENT).all() and (bits[written] != SF.SENT).all()
        out = preds.cpu().numpy().reshape(B * pred_ring, n, O)
        out[~written] = 0.0                                     # (the sentinel is a NaN)
        return out

    sweep(run, lanes, f"ape_mc_ff_ring {B} streams x {nF} frames x {n} samples, stream_frames {sf}")
