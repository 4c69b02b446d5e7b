"""CPU: the ring mode of the feed-forward kernel (ape_mc_ff_ring, csrc/ape_ff.cu) - its binding and its refusals, which all come before
the first CUDA call - and the window rule of a feed-forward model on the batched path (batched.ff_window).  The pointers are
placeholders that are never dereferenced."""
import pytest

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200.estimate.batched import KIND_FEATURES, ff_window

OK, BAD, UNSUP = N.APE_OK, N.APE_ERR_BAD_ARG, N.APE_ERR_UNSUPPORTED


def _call(**kw):
    """ape_mc_ff_ring with the uarm DropoutFF2D of tools/ff_batched_bench.py (6 x 38 inputs, H = 256, Lh = 2, O = 12), 4 streams x 2 frames."""
    a = dict(blob=256, I=38, T=6, H=256, Lh=2, O=12, p=0.2, feats=512, feat_ring=7, B=4, nF=2, frame0=0, stream_frames=None,
             n=100, mask_mode=N.MASK_PHILOX, masks=None, seed=1, stream_id0=0, preds=768, pred_ring=2)
    a.update(kw)
    return N.load().ape_mc_ff_ring(a["blob"], a["I"], a["T"], a["H"], a["Lh"], a["O"], a["p"], a["feats"], a["feat_ring"], a["B"],
                                   a["nF"], a["frame0"], a["stream_frames"], a["n"], a["mask_mode"], a["masks"], a["seed"],
                                   a["stream_id0"], a["preds"], a["pred_ring"], None)


def test_ff_ring_symbol_is_bound():
    assert "ape_mc_ff_ring" in N.SYMBOLS
    assert N.load().ape_mc_ff_ring.restype is not None and len(N.load().ape_mc_ff_ring.argtypes) == 21


CASES = [
    # null pointers
    ("no-blob", dict(blob=None), BAD),
    ("no-feats", dict(feats=None), BAD),
    ("no-preds", dict(preds=None), BAD),
    ("injected-no-masks", dict(mask_mode=N.MASK_INJECTED), BAD),
    # the rings
    ("feat-ring-short", dict(feat_ring=6), BAD),                  # nF + T - 1 = 7
    ("feat-ring-short-T1", dict(T=1, feat_ring=1), BAD),
    ("frame0-negative", dict(frame0=-1), BAD),
    ("pred-ring-short", dict(pred_ring=1), BAD),
    # outputs, mask mode, dropout
    ("O21", dict(O=21), BAD),
    ("O0", dict(O=0), BAD),
    ("mask-mode-3", dict(mask_mode=3), BAD),
    ("mask-mode-neg", dict(mask_mode=-1), BAD),
    ("p1", dict(p=1.0), BAD),
    ("p-neg", dict(p=-0.1), BAD),
    ("p-nan", dict(p=float("nan")), BAD),
    # other sizes
    ("I0", dict(I=0), BAD),
    ("T0", dict(T=0), BAD),
    ("H0", dict(H=0), BAD),
    ("Lh-neg", dict(Lh=-1), BAD),
    ("B-neg", dict(B=-1), BAD),
    ("nF0", dict(nF=0), BAD),
    ("n0", dict(n=0), BAD),
    # shapes the batched kernel does not take (there is no ring form of the one-CTA-per-row kernel)
    ("H100", dict(H=100), UNSUP),
    ("blob-unaligned", dict(blob=260), UNSUP),
    ("masks-unaligned", dict(mask_mode=N.MASK_INJECTED, masks=1028), UNSUP),
    ("smem-over-200KB", dict(T=40, I=160, feat_ring=41), UNSUP),   # 6400 inputs: 2 x 8 x 6400 floats of tiles alone
    # accepted; an empty call is done before the device
    ("empty", dict(B=0), OK),
    ("empty-T1", dict(B=0, T=1, feat_ring=2), OK),
    ("empty-O20-injected", dict(B=0, O=20, mask_mode=N.MASK_INJECTED, masks=1024), OK),
    ("empty-none-p1", dict(B=0, mask_mode=N.MASK_NONE, p=1.0), OK),      # (eval mode: p is not used)
    ("empty-stream-frames", dict(B=0, stream_frames=2048), OK),
]


@pytest.mark.parametrize("kw,want", [c[1:] for c in CASES], ids=[c[0] for c in CASES])
def test_ff_ring_refusals_before_the_device(kw, want):
    assert _call(**kw) == want


@pytest.mark.parametrize("kind", sorted(KIND_FEATURES))
def test_ff_window_rule(kind):
    I = KIND_FEATURES[kind]
    assert ff_window(6 * I, I, 6) == 6                  # DropoutFF2D: the flattened window
    assert ff_window(I, I, 6) == 1                      # DropoutFF: the newest frame
    assert ff_window(I, I, 1) == 1 and ff_window(I, I, 0) == 1
    assert ff_window(8 * I, I, 8) == 8
    for width in (5 * I, 6 * I + 1, I - 1, 2 * I):
        with pytest.raises(UserWarning, match=str(width)):
            ff_window(width, I, 6)
