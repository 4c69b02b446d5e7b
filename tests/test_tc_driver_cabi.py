"""CPU: the refusals of ape_mc_lstm_tc that come before the first CUDA call, for each layer-kernel family behind it (tc_flags 0 / 1:
one launch per layer or automatic pairing, 2: wavefront pairs, 3: split precision at H = 128 and 256, 4: the small-batch kernel).
The pointers are placeholders that are never dereferenced: every case stops at an argument check, with or without a GPU."""
import pytest

from arm_pose_estimation_b200 import _native as N

OK, BAD, UNSUP = N.APE_OK, N.APE_ERR_BAD_ARG, N.APE_ERR_UNSUPPORTED


def _args(H=128, tc_flags=0, **kw):
    a = N.LstmArgs()
    a.weights = a.preds = a.x_dense = a.weights_tc = a.weights_tcx = 256
    a.I, a.H, a.L, a.T, a.O = 20, H, 3, 8, 12
    a.B, a.nF, a.n_samples = 64, 1, 1
    a.mask_mode, a.pred_ring = N.MASK_NONE, 1
    a.tc_flags = tc_flags
    a.workspace = None                     # with E > 0 the call stops here at the latest
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def _cases():
    for H in (128, 256):
        for f in (0, 1, 2, 3):
            blob, other = ("weights_tcx", "weights_tc") if f == 3 else ("weights_tc", "weights_tcx")
            # E = 0: the single-pass path returns before it looks at the workspace, the split path checks the workspace first
            yield f"H{H}-f{f}-empty-no-workspace", dict(H=H, tc_flags=f, B=0), BAD if f == 3 else OK
            yield f"H{H}-f{f}-empty", dict(H=H, tc_flags=f, B=0, workspace=512), OK
            # each variant reads its own blob, and checks it before the E = 0 return
            yield f"H{H}-f{f}-empty-no-blob", dict(H=H, tc_flags=f, B=0, workspace=512, **{blob: None}), BAD
            yield f"H{H}-f{f}-no-blob", dict(H=H, tc_flags=f, workspace=512, **{blob: None}), BAD
            yield f"H{H}-f{f}-empty-no-other-blob", dict(H=H, tc_flags=f, B=0, workspace=512, **{other: None}), OK
            yield f"H{H}-f{f}-no-workspace", dict(H=H, tc_flags=f), BAD
            yield f"H{H}-f{f}-layer-range-all-steps", dict(H=H, tc_flags=f, all_steps=1, layer_begin=0, layer_end=2), UNSUP
            yield f"H{H}-f{f}-T41", dict(H=H, tc_flags=f, T=41), UNSUP
            # an initial state: refused by the wavefront and the H = 128 split kernel, else the call goes on to the workspace check
            yield f"H{H}-f{f}-state", dict(H=H, tc_flags=f, h0=512, c0=768), UNSUP if f == 2 or (f == 3 and H == 128) else BAD
        yield f"H{H}-f4-state", dict(H=H, tc_flags=4, h0=512, c0=768), UNSUP
        yield f"H{H}-f4-empty-no-workspace", dict(H=H, tc_flags=4, B=0), OK
    # shapes: the single-pass path takes H = 64 / 128 with O <= 16 and H = 256 with O <= 20, the split path H = 128 with O <= 16 and
    # H = 256 with O <= 32; an accepted shape goes on to the workspace check
    want = {(64, 12): (BAD, UNSUP), (128, 16): (BAD, BAD), (128, 17): (UNSUP, UNSUP), (256, 20): (BAD, BAD), (256, 21): (UNSUP, BAD),
            (256, 32): (UNSUP, BAD), (256, 33): (UNSUP, UNSUP)}
    for (H, O), codes in want.items():
        for f, code in zip((0, 3), codes):
            yield f"H{H}-f{f}-O{O}", dict(H=H, tc_flags=f, O=O), code
    for f in (0, 3):
        yield f"H128-f{f}-L1", dict(tc_flags=f, L=1), UNSUP
        yield f"H256-f{f}-I300", dict(H=256, tc_flags=f, I=300), UNSUP


CASES = list(_cases())


@pytest.mark.parametrize("kw,want", [c[1:] for c in CASES], ids=[c[0] for c in CASES])
def test_tc_refusals_before_the_device(kw, want):
    assert N.load().ape_mc_lstm_tc(_args(**kw), None) == want
