"""GPU (-m gpu): per-stream frame counters (``stream_frames[B]``, include/ape_b200.h) on every kernel that re-derives a stream's frame.

A stream with a negative counter has no new row in the call: its rows still sit in the tiles, but nothing of it may be written.  An
active stream writes exactly its slots ``f_b .. f_b + nF - 1`` (mod ring) of the feature and prediction rings, keys its Philox draws
by (its global id, its own frame) and reads a window clamped to frame 0.  Checked here:

  * every LSTM kernel (fp32, tc at H = 64 / 128, tcs, tcw, tcl, tcx, tcxs), pinned one at a time: ring slots and outputs against
    NaN sentinels and the previous contents (bit for bit), predictions against ``oracle.lstm`` on the stream's own window;
  * stage 1 (``ape_features``, ``ape_features_push``) and stage 3 (``ape_fk_reduce``, ``ape_msg_from_est``) through the C ABI
    against float64 references, with skipped streams, ring wraps, windows reaching back past frame 0 and degenerate rows;
  * the estimator entry points at serving scale (1024 streams x 100 samples, ragged arrivals, a late-joining block, a restarted
    stream): the native pipeline's ``submit``, ``step`` and ``step_graph`` bit for bit, and sampled streams against a dedicated
    single-stream estimator and the oracle.

Tolerances are the suite's (tests/test_gpu_parity.py): features 2e-6, normalised LSTM outputs 2e-5 (fp32 and split kernels) /
2e-4 (single-pass tensor-core kernels), positions 1e-4 m, quaternions 2e-4 up to sign.  The references below are also pinned on
the CPU by tests/test_stream_frames_cabi.py."""
import numpy as np
import pytest
import torch

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200 import synthetic as syn
from oracle import features as OF, fk as OFK, lstm as OL, quat as OQ

pytestmark = pytest.mark.gpu

FEAT_TOL, PRED_TOL, PRED_TOL_TC, POS_TOL, QUAT_TOL = 2e-6, 2e-5, 2e-4, 1e-4, 2e-4
SENT = 0x7FC0DEAD                      # a quiet-NaN bit pattern no kernel produces: "nothing was written here"
TARGET_NAMES = {N.TARGET_ORI_CAL_LARM_UARM: "ORI_CAL_LARM_UARM", N.TARGET_ORI_CAL_LARM_UARM_HIPS: "ORI_CAL_LARM_UARM_HIPS",
                N.TARGET_ORI_POS_CAL_LARM_UARM_HIPS: "ORI_POS_CAL_LARM_UARM_HIPS"}
TARGET_O = {N.TARGET_ORI_CAL_LARM_UARM: 12, N.TARGET_ORI_CAL_LARM_UARM_HIPS: 14, N.TARGET_ORI_POS_CAL_LARM_UARM_HIPS: 20}


# ---- plain references (float64 / the oracle's float32 LSTM), usable without a GPU ------------------------------------------------
def window_frames(f, length):
    """Absolute frames of the window of ``length`` frames that ends at frame ``f``, oldest first; frames before 0 clamp to frame 0
    (the reference pads its row and smoothing histories by repeating the first entry, estimator.py:96-97, :114-115)."""
    return [max(0, k) for k in range(f - length + 1, f + 1)]


def window_slots(f, length, ring):
    """Ring slots of that window in a ring of ``ring`` frames per stream."""
    return [k % ring for k in window_frames(f, length)]


def ref_features(kind, rows, xx_m=None, xx_s=None):
    """Stage 1 in float64: ``oracle.features.parse_row`` of each raw row (keeping the reference's float32 rounding point), then
    the z-score when ``xx_m`` / ``xx_s`` are given.  ``rows [..., ncols]`` -> ``[..., I]`` float64."""
    rows = np.asarray(rows)
    lk = syn.kind_spec(kind)["lookup"]
    flat = rows.reshape(-1, rows.shape[-1])
    xx = np.stack([OF.parse_row(syn.KIND_NAMES[kind], r, lk).astype(np.float64) for r in flat])
    if xx_m is not None:
        xx = (xx - np.asarray(xx_m, np.float64)) / np.asarray(xx_s, np.float64)
    return xx.reshape(rows.shape[:-1] + (xx.shape[-1],))


def ref_lstm(state, feat_ring, f, T, masks, p):
    """Stage 2 of one estimate: the MC-dropout LSTM (``oracle.lstm.forward_with_masks``) on the window of ``T`` frames ending at
    frame ``f`` of one stream's feature ring ``[ring][I]``; ``masks [L-1][T][n][H]`` (the injected-mask layout of one estimate).
    Returns the last step's normalised outputs ``[n][O]``."""
    x = np.asarray(feat_ring, np.float32)[window_slots(f, T, len(feat_ring))]
    n = masks.shape[2]
    return OL.forward_with_masks(state, np.repeat(x[None], n, axis=0), list(masks) if len(masks) else None, p, last_only=True)


def ref_stage3(pred_ring, f, smooth, yy_m, yy_s, body9, target):
    """Stage 3 of one estimate: the de-normalised smoothing window of ``smooth`` frames ending at frame ``f`` of one stream's
    prediction ring ``[ring][n][O]``, through ``oracle.fk``.  Returns (est rows [S][W], message [25], std [6])."""
    win = np.asarray(pred_ring, np.float64)[window_slots(f, smooth, len(pred_ring))]
    rows = win.reshape(-1, win.shape[-1])
    if yy_m is not None:
        rows = rows * np.asarray(yy_s, np.float64) + np.asarray(yy_m, np.float64)
    est = OFK.arm_pose_from_nn_targets(rows, body9, target)
    return est, OFK.msg_from_est(est, body9, target), OFK.sample_std(est)


def quat_err(a, b):
    """Largest distance between quaternions of the last axis of ``a`` and ``b`` (of 4 columns each), up to sign."""
    a, b = np.asarray(a, np.float64).reshape(-1, 4), np.asarray(b, np.float64).reshape(-1, 4)
    return float(np.minimum(np.abs(a - b).max(axis=-1), np.abs(a + b).max(axis=-1)).max())


def msg_errors(mine, want):
    """(worst position error, worst quaternion error) between two 25-float messages."""
    mine, want = np.asarray(mine, np.float64), np.asarray(want, np.float64)
    pos = max(float(np.abs(mine[a:b] - want[a:b]).max()) for a, b in ((4, 7), (11, 14), (18, 21)))
    return pos, max(quat_err(mine[a:b], want[a:b]) for a, b in ((0, 4), (7, 11), (14, 18), (21, 25)))


# ---- device helpers ---------------------------------------------------------------------------------------------------------------
def _fill_sentinel(t):
    t.view(-1).view(torch.int32).fill_(SENT)


def _bits(t):
    """The 32-bit words of a device tensor, as int32 on the host."""
    return t.detach().contiguous().view(-1).view(torch.int32).cpu().numpy().reshape(t.shape)


def philox_masks(seed, stream, nF, f0, L, T, n, H, p):
    """The keep-masks APE_MASK_PHILOX draws for ONE stream at its own frames f0 .. f0 + nF - 1: [nF][L-1][T][n][H]."""
    if L < 2:
        return np.zeros((nF, 0, T, n, H), np.uint8)
    m = torch.empty((1, nF, L - 1, T, n, H), dtype=torch.uint8, device="cuda")
    N.check(N.load().ape_philox_masks(seed, stream, 1, nF, f0, L, T, n, H, p, N.ptr(m), N.current_stream_ptr()), "ape_philox_masks")
    return m.cpu().numpy()[0]


def _written_slots(sf, nF, ring):
    """[B][ring] bool: the slots a call with counters ``sf`` and ``nF`` frames writes."""
    w = np.zeros((len(sf), ring), bool)
    for b in np.flatnonzero(sf >= 0):
        w[b, [(int(sf[b]) + j) % ring for j in range(nF)]] = True
    return w


def _out_written(be, sf, nF):
    """Bool mask over the whole int32 view of an estimator's result buffer: the words a call writes ([msg | std | status | samples],
    the call's E = B x nF estimates packed at the front of each part)."""
    B, Em, E, S = be.B, be.B * be.nF_max, be.B * nF, be.S
    w = np.zeros(be.out_bufs[0].numel(), bool)
    act = np.repeat(sf >= 0, nF)
    for off, width in ((0, 25), (Em * 25, 6), (Em * 31, 1)) + (((Em * 32, S * 6),) if be.emit_samples else ()):
        w[off: off + E * width] = np.repeat(act, width)
    return w


# ---- a. every LSTM kernel, one at a time --------------------------------------------------------------------------------------
# (name, kind, B, n, estimator knobs, H = 64 synthetic model, launches per call, normalised-output tolerance)
LSTM_CASES = [
    ("fma", syn.KIND_UARM, 300, 7, dict(lstm_variant="fp32"), False, 2 + 3, PRED_TOL),
    ("fma", syn.KIND_POCKET, 260, 1, dict(lstm_variant="fp32"), False, 2 + 2, PRED_TOL),
    ("tc", syn.KIND_WATCH_ONLY, 300, 7, dict(lstm_variant="tc", tc_flags=1, small_batch_kernel=False), True, 2 + 2, PRED_TOL_TC),
    ("tc", syn.KIND_UARM, 260, 1, dict(lstm_variant="tc", tc_flags=1, small_batch_kernel=False), False, 2 + 3, PRED_TOL_TC),
    ("tc", syn.KIND_UARM, 64, 100, dict(lstm_variant="tc", tc_flags=1, small_batch_kernel=False), False, 2 + 3, PRED_TOL_TC),
    ("tcs", syn.KIND_POCKET, 300, 7, dict(lstm_variant="tc", tc_flags=1, small_batch_kernel=False), False, 2 + 2, PRED_TOL_TC),
    ("tcs", syn.KIND_WATCH_ONLY, 1024, 100, dict(lstm_variant="tc", tc_flags=1, small_batch_kernel=False), False, 2 + 2, PRED_TOL_TC),
    ("tcw", syn.KIND_UARM, 300, 7, dict(lstm_variant="tc", tc_flags=2), False, 2 + 2, PRED_TOL_TC),
    ("tcw", syn.KIND_UARM, 1024, 100, dict(lstm_variant="tc", tc_flags=2), False, 2 + 2, PRED_TOL_TC),
    ("tcl", syn.KIND_UARM, 260, 1, dict(lstm_variant="tc", tc_flags=4, small_batch_kernel=False), False, 2 + 1, PRED_TOL_TC),
    ("tcl", syn.KIND_POCKET, 27, 100, dict(lstm_variant="tc", tc_flags=4, small_batch_kernel=False), False, 2 + 1, PRED_TOL_TC),
    ("tcx", syn.KIND_UARM, 300, 7, dict(lstm_variant="tcx"), False, 2 + 3, PRED_TOL),
    ("tcx", syn.KIND_UARM, 40, 100, dict(lstm_variant="tcx"), False, 2 + 3, PRED_TOL),
    ("tcxs", syn.KIND_POCKET, 300, 7, dict(lstm_variant="tcx"), False, 2 + 2, PRED_TOL),
    ("tcxs", syn.KIND_WATCH_ONLY, 1024, 100, dict(lstm_variant="tcx"), False, 2 + 2, PRED_TOL),
]
NF_PER_CALL = [1, 3, 3, 1, 3]
SEED = 29


def _model(kind, h64):
    spec = syn.kind_spec(kind)
    if h64:                                         # a synthetic H = 64, L = 2 model on this kind's features
        return spec, syn.synth_state_dict(spec["I"], 64, 2, spec["O"], 64)
    return spec, syn.synth_state_dict(spec["I"], spec["H"], spec["L"], spec["O"], 1234 + kind)


def _estimator(kind, state, B, n, nF_max, first_stream=0, smooth=1, **kw):
    from arm_pose_estimation_b200.estimate.batched import BatchedEstimator
    spec = syn.kind_spec(kind)
    return BatchedEstimator(kind=kind, layout=spec["layout"], state=state, seq_len=spec["T"], y_targets=spec["y_targets"],
                            stats=spec["stats"], n_streams=B, mc_samples=n, smooth=smooth, dropout=spec["p"], frames_per_call=nF_max,
                            mask_mode=N.MASK_PHILOX, philox_seed=SEED, first_stream=first_stream, **kw)


def boundary_streams(B, n, nFs):
    """Streams whose estimates hold rows 127 / 128 and 255 / 256 of a call (the 128-row cluster tiles and the 256-row pair tiles:
    of the per-estimate layer 0 and of the per-sample layers >= 1), with their neighbours: a run across every tile boundary."""
    out = set()
    for nF in nFs:
        E = B * nF
        for r in (127, 128, 255, 256):
            for e in (r, r // n):
                if e < E:
                    out.update(b for b in (e // nF - 1, e // nF, e // nF + 1) if 0 <= b < B)
    return sorted(out)


def lstm_schedule(B, n, nFs, seed):
    """Counters of consecutive calls: 30 % of the streams idle per call at random; stream 0 idle in calls 0 and 2, the last stream
    in calls 1 and 3, the tile-boundary run in calls 0 and 2 (so each comes back once or twice); an eighth of the streams far
    ahead (frame ~1000: both rings wrap, and their windows read slots never written in this run); the others start at frame 0 and
    stay in their warm-up (f < T - 1) for the first calls.  Returns ([(nF, counters)], boundary run, far streams)."""
    rng = np.random.default_rng(seed)
    frames = np.zeros(B, np.int64)
    far = rng.choice(np.arange(1, B - 1), size=max(1, B // 8), replace=False)
    frames[far] = 1000 + rng.integers(0, 97, size=far.size)
    bnd = boundary_streams(B, n, set(nFs))
    calls = []
    for k, nF in enumerate(nFs):
        active = rng.random(B) >= 0.3
        active[bnd] = k not in (0, 2)
        active[0] = k not in (0, 2)
        active[-1] = k not in (1, 3)
        sf = np.where(active, frames, -1).astype(np.int32)
        frames[active] += nF
        calls.append((nF, sf))
    return calls, bnd, far


def run_lstm_schedule(be, kind, state, calls, sample, tol, rows, keep=False):
    """Drive ``be`` (pipeline=False) through ``calls``; check the rings and the result buffer after every call.  Returns
    (worst feature error, worst normalised-output error, [per call: prediction ring bits, result buffer bits] if ``keep``)."""
    spec = syn.kind_spec(kind)
    L, T, H, n, p = be.L, be.T, be.H, be.n, be.p
    ring_f, ring_p = be.feat_ring, be.pred_ring
    g = torch.Generator(device="cpu").manual_seed(7)
    be.feats.copy_(torch.randn(be.feats.shape, generator=g))          # "previous contents" of slots no call of this run writes
    feats_model = be.feats.cpu().numpy().copy()                       # what the feature ring must hold: the reference's features
    xm, xs = spec["stats"]["xx_m"], spec["stats"]["xx_s"]
    worst_f = worst_p = 0.0
    kept = []
    col = 0
    for k, (nF, sf) in enumerate(calls):
        r = np.ascontiguousarray(rows[:, col:col + nF])
        col += nF
        feats_before = _bits(be.feats)
        _fill_sentinel(be.preds)                                      # smooth = 1: nothing reads an older prediction
        _fill_sentinel(be.out_bufs[0])
        raw = torch.from_numpy(r).cuda()
        sfd = torch.from_numpy(sf).cuda()
        be.step_device(raw, n_frames=nF, stream_frames=sfd)
        torch.cuda.synchronize()
        # stage 1: active streams write exactly their nF slots (to the reference's values), every other slot keeps its bits
        wf = _written_slots(sf, nF, ring_f)
        feats_after = _bits(be.feats)
        assert (feats_after[~wf] == feats_before[~wf]).all(), f"call {k}: a feature slot outside f_b .. f_b + nF - 1 changed"
        want = ref_features(kind, r, xm, xs)                          # [B, nF, I]
        for b in np.flatnonzero(sf >= 0):
            for j in range(nF):
                feats_model[b, (int(sf[b]) + j) % ring_f] = want[b, j].astype(np.float32)
        got_f = be.feats.cpu().numpy()
        err = np.abs(got_f[wf] - feats_model[wf]) / (1 + np.abs(feats_model[wf]))
        worst_f = max(worst_f, float(err.max()) if err.size else 0.0)
        assert worst_f <= FEAT_TOL, f"call {k}: features off by {worst_f:.3g}"
        # stage 2: the prediction ring - written exactly in the active streams' slots
        wp = _written_slots(sf, nF, ring_p)
        pb = _bits(be.preds)                                          # [B, ring, n, O]
        untouched = (pb == SENT).reshape(be.B, ring_p, -1).all(axis=-1)
        fresh = (pb != SENT).reshape(be.B, ring_p, -1).all(axis=-1)
        assert (untouched == ~wp).all() and (fresh == wp).all(), \
            f"call {k}: prediction slots written {np.argwhere(~untouched & ~wp)[:5].tolist()} / missed {np.argwhere(~fresh & wp)[:5].tolist()}"
        preds = be.preds.cpu().numpy()
        assert np.isfinite(preds[wp]).all()
        for b in sample:
            if sf[b] < 0:
                continue
            masks = philox_masks(SEED, be.first_stream + int(b), nF, int(sf[b]), L, T, n, H, p)
            for j in range(nF):
                f = int(sf[b]) + j
                want_p = ref_lstm(state, feats_model[b], f, T, masks[j], p)
                e = float(np.abs(preds[b, f % ring_p] - want_p).max())
                assert e <= tol, f"call {k}, stream {b}, frame {f}: normalised outputs off by {e:.3g}"
                worst_p = max(worst_p, e)
        # stage 3 outputs: exactly the active streams' estimates, nothing past E
        ob = _bits(be.out_bufs[0])
        wo = _out_written(be, sf, nF)
        assert (ob[~wo] == SENT).all(), f"call {k}: a result word of a skipped stream (or past E) was written"
        assert (ob[wo] != SENT).all(), f"call {k}: a result word of an active stream was not written"
        if keep:
            kept.append((pb, ob))
    return worst_f, worst_p, kept


@pytest.mark.parametrize("name,kind,B,n,knobs,h64,launches,tol", LSTM_CASES,
                         ids=[f"{c[0]}-{syn.KIND_NAMES[c[1]]}{'-h64' if c[5] else ''}-{c[2]}x{c[3]}" for c in LSTM_CASES])
def test_lstm_kernel_honours_stream_frames(name, kind, B, n, knobs, h64, launches, tol):
    spec, state = _model(kind, h64)
    be = _estimator(kind, state, B, n, max(NF_PER_CALL), pipeline=False, **knobs)
    # the kernel this case pins
    assert not be.pipeline and be._pipe is None
    if name == "fma":
        assert be.lstm_variant == "fp32"
    else:
        assert be.lstm_variant == "tc" and be.tc_split == (name in ("tcx", "tcxs")) and not be.small_batch
        assert be.tc_flags == {"tc": 1, "tcs": 1, "tcw": 2, "tcl": 4, "tcx": 3, "tcxs": 3}[name]
        assert be.H == {"tc": 64 if h64 else 128, "tcs": 256, "tcw": 128, "tcl": be.H, "tcx": 128, "tcxs": 256}[name]
    if name == "tcl":
        assert B * max(NF_PER_CALL) * n <= 8192 and be.L <= 4
    calls, bnd, far = lstm_schedule(B, n, NF_PER_CALL, seed=B + n)
    rows = syn.synth_rows(kind, B, sum(NF_PER_CALL), config_id=50 + kind)
    if B <= 64:
        sample = list(range(B))
    else:
        rng = np.random.default_rng(n)
        sample = sorted(set(bnd) | {0, 1, B - 2, B - 1} | set(far[:6].tolist()) | set(rng.choice(B, 8, replace=False).tolist()))
    worst_f, worst_p, kept = run_lstm_schedule(be, kind, state, calls, sample, tol, rows, keep=name == "tcl")
    assert be.launches == len(calls) * launches, f"launches {be.launches} != {len(calls)} x {launches}"
    print(f"stream_frames [{name}] {syn.KIND_NAMES[kind]}{' H=64' if h64 else ''} {B} x {n}: tc_flags {be.tc_flags}, split {be.tc_split}, "
          f"{be.launches // len(calls)} launches/call; worst feature error {worst_f:.3g}, worst normalised-output error {worst_p:.3g} "
          f"over {len(sample)} sampled streams (bound {tol:g})")
    if name == "tcl":
        # the cluster kernel keeps the layer kernels' arithmetic: the same per-stream run must match them bit for bit
        layers = _estimator(kind, state, B, n, max(NF_PER_CALL), pipeline=False, lstm_variant="tc", tc_flags=1, small_batch_kernel=False)
        _, _, kept1 = run_lstm_schedule(layers, kind, state, calls, [], tol, rows, keep=True)
        for k, ((pa, oa), (pb, ob)) in enumerate(zip(kept, kept1)):
            np.testing.assert_array_equal(pa, pb, err_msg=f"call {k}: prediction ring, cluster vs layer kernels")
            np.testing.assert_array_equal(oa, ob, err_msg=f"call {k}: results, cluster vs layer kernels")


# ---- b. stage 1 and stage 3 through the C ABI ------------------------------------------------------------------------------------
@pytest.mark.parametrize("normalize", [0, 1])
@pytest.mark.parametrize("kind", [syn.KIND_WATCH_ONLY, syn.KIND_POCKET, syn.KIND_UARM])
def test_features_kernels_honour_stream_frames(kind, normalize):
    spec = syn.kind_spec(kind)
    B, ring, I = 37, 5, spec["I"]
    lib = N.load()
    xm_h, xs_h = spec["stats"]["xx_m"], spec["stats"]["xx_s"]
    xm, xs = (torch.as_tensor(np.asarray(xm_h, np.float64)).cuda(), torch.as_tensor(np.asarray(xs_h, np.float64)).cuda()) if normalize else (None, None)
    feats = torch.empty((B, ring, I), dtype=torch.float32, device="cuda")
    _fill_sentinel(feats)
    model = _bits(feats).view(np.float32).copy()
    rng = np.random.default_rng(kind * 2 + normalize)
    # counters: skips (first, last, a run), f_b beyond the ring, nF > 1 wrapping the ring; one call without counters at frame0 > ring
    far = 1000 + np.arange(B)
    calls = [(3, np.where(rng.random(B) < 0.3, -1, far)), (1, np.where(np.arange(B) % 4 == 1, -1, np.arange(B) % 7)),
             (3, np.where((np.arange(B) >= 10) & (np.arange(B) < 20), -1, far + 3)), (2, None)]
    calls[0][1][[0, B - 1]] = -1
    worst = 0.0
    for k, (nF, sf) in enumerate(calls):
        rows = syn.synth_rows(kind, B, nF, config_id=60 + k)
        before = _bits(feats)
        sfd = None if sf is None else torch.from_numpy(sf.astype(np.int32)).cuda()
        frame0 = 2 * ring + 3
        raw = torch.from_numpy(rows).cuda()                           # (every device argument is bound to a name for the whole call)
        N.check(lib.ape_features(N.ptr(raw), spec["layout"], kind, N.ptr(xm), N.ptr(xs), normalize, N.ptr(feats),
                                 B, nF, frame0, N.ptr(sfd), ring, N.current_stream_ptr()), "ape_features")
        fb = np.full(B, frame0) if sf is None else sf
        want = ref_features(kind, rows, xm_h if normalize else None, xs_h if normalize else None)
        for b in np.flatnonzero(fb >= 0):
            for j in range(nF):
                model[b, (int(fb[b]) + j) % ring] = want[b, j]
        w = _written_slots(fb, nF, ring)
        after = _bits(feats)
        assert (after[~w] == before[~w]).all(), f"call {k}: a slot outside f_b .. f_b + nF - 1 changed"
        got = after.view(np.float32)
        np.testing.assert_allclose(got[w], model[w], rtol=FEAT_TOL, atol=FEAT_TOL, err_msg=f"call {k}")
        worst = max(worst, float((np.abs(got[w] - model[w]) / (1 + np.abs(model[w]))).max()))
    # the one-row-per-stream push (ape_features_push): float64 rows as parse_row_to_xx returned them
    for k, sf in enumerate([np.where(np.arange(B) % 3 == 0, -1, 2000 + 5 * np.arange(B)), np.where(np.arange(B) < 4, -1, np.arange(B))]):
        xx = rng.normal(size=(B, I))
        before = _bits(feats)
        xxd, sfd = torch.from_numpy(xx).cuda(), torch.from_numpy(sf.astype(np.int32)).cuda()
        N.check(lib.ape_features_push(N.ptr(xxd), I, N.ptr(xm), N.ptr(xs), normalize, N.ptr(feats), B, 0, N.ptr(sfd), ring,
                                      N.current_stream_ptr()), "ape_features_push")
        want = (xx - xm_h) / xs_h if normalize else xx
        w = _written_slots(sf, 1, ring)
        for b in np.flatnonzero(sf >= 0):
            model[b, int(sf[b]) % ring] = want[b]
        after = _bits(feats)
        assert (after[~w] == before[~w]).all(), f"push {k}: a slot of a skipped stream or another frame changed"
        np.testing.assert_allclose(after.view(np.float32)[w], model[w], rtol=FEAT_TOL, atol=FEAT_TOL, err_msg=f"push {k}")
    print(f"stream_frames [features] {syn.KIND_NAMES[kind]} normalize={normalize}: worst feature error {worst:.3g}")


def _stage3_preds(target, B, ring, n, rng):
    """De-normalised network outputs of a stream: one pose per stream plus 3 % noise per row (so the sign-aligned averages are far
    from their decision boundaries), [B][ring][n][O] float64."""
    O = TARGET_O[target]
    base = np.zeros((B, O))
    for b in range(B):
        ql, qu = [q / np.linalg.norm(q) for q in rng.normal(size=(2, 4))]
        sl, su = OQ.quat_to_six(ql), OQ.quat_to_six(qu)
        yaw = rng.uniform(-np.pi, np.pi)
        if target == N.TARGET_ORI_CAL_LARM_UARM:
            base[b] = np.r_[sl, su]
        elif target == N.TARGET_ORI_CAL_LARM_UARM_HIPS:
            base[b] = np.r_[sl, su, np.sin(yaw), np.cos(yaw)]
        else:
            base[b] = np.r_[rng.normal(size=3) * 0.3, sl, rng.normal(size=3) * 0.3, su, np.sin(yaw), np.cos(yaw)]
    return base[:, None, None, :] + 0.03 * rng.normal(size=(B, ring, n, O))


# (target, n, smooth, nF, de-normalise with yy_m / yy_s) - without yy_m / yy_s a zero 6D row stays zero: the degenerate cases
FK_CASES = [(0, 1, 20, 3, True), (0, 5, 3, 1, False), (0, 16, 1, 3, True), (1, 33, 3, 1, True), (1, 100, 1, 1, False),
            (1, 5, 20, 1, True), (2, 16, 3, 3, False), (2, 100, 1, 3, True), (2, 1, 3, 1, True), (2, 5, 20, 1, False)]


@pytest.mark.parametrize("target,n,smooth,nF,yy", FK_CASES)
def test_fk_reduce_honours_stream_frames(target, n, smooth, nF, yy, body9):
    O, W, tname = TARGET_O[target], 14 if target == 0 else 21, TARGET_NAMES[target]
    B, S = 11, smooth * n                                             # E = 11 or 33: the last warp's second half-warp has no estimate
    ring = nF + smooth                                                # one slot more than the window needs
    rng = np.random.default_rng(target * 1000 + n * 10 + smooth + nF)
    # counters: 0 / 1 / 2 (windows reaching back past frame 0), ~1000 (across the ring wrap), skipped streams next to active ones
    # in the same warp (estimates 2k and 2k + 1 share a warp)
    sf = np.array([0, -1, 1, 5, -1, 1000, 1001, 17, -1, 2, 1003], np.int32)
    dn = _stage3_preds(target, B, ring, n, rng)
    yy_m, yy_s = (rng.normal(size=O) * 0.3).astype(np.float32), rng.uniform(0.5, 1.5, size=O).astype(np.float32)
    preds_h = ((dn - yy_m) / yy_s if yy else dn).astype(np.float32)
    bad = np.zeros((B, ring, n), bool)                                # rows whose lower-arm 6D is zero: degenerate
    if not yy:
        ol = 3 if target == N.TARGET_ORI_POS_CAL_LARM_UARM_HIPS else 0
        for b in (2, 4):                                              # an active stream (its neighbour 3 is active) and a skipped one
            slot = (max(int(sf[b]), 0)) % ring
            preds_h[b, slot, 0, ol:ol + 6] = 0.0
            bad[b, slot, 0] = True
    preds = torch.from_numpy(preds_h).cuda()
    E = B * nF
    outs = {k: torch.empty(shape, dtype=torch.float32, device="cuda") for k, shape in
            (("msg", (E, 25)), ("samples", (E, S, 6)), ("stdev", (E, 6)), ("est", (E, S, W)))}
    status = torch.empty(E, dtype=torch.int32, device="cuda")
    for t in list(outs.values()) + [status]:
        _fill_sentinel(t)
    preds_before = _bits(preds)
    ym, ys = (torch.from_numpy(yy_m).cuda(), torch.from_numpy(yy_s).cuda()) if yy else (None, None)
    body = torch.from_numpy(np.asarray(body9, np.float32).ravel()).cuda()
    sfd = torch.from_numpy(sf).cuda()
    N.check(N.load().ape_fk_reduce(N.ptr(preds), ring, N.ptr(ym), N.ptr(ys), N.ptr(body), target, O, B, nF, 0,
                                   N.ptr(sfd), n, smooth, N.ptr(outs["msg"]), N.ptr(outs["samples"]),
                                   N.ptr(outs["stdev"]), N.ptr(outs["est"]), N.ptr(status), N.current_stream_ptr()), "ape_fk_reduce")
    torch.cuda.synchronize()
    assert (_bits(preds) == preds_before).all()
    got = {k: v.cpu().numpy() for k, v in outs.items()}
    bits = {k: _bits(v) for k, v in outs.items()}
    st = status.cpu().numpy()
    worst_pos = worst_q = worst_sd = 0.0
    n_bad = 0
    for b in range(B):
        for j in range(nF):
            e = b * nF + j
            if sf[b] < 0:                                             # the kernel writes nothing for a skipped stream
                assert st[e] == SENT, f"estimate {e} (skipped stream {b}): status written"
                for k in bits:
                    assert (bits[k][e] == SENT).all(), f"estimate {e} (skipped stream {b}): {k} written"
                continue
            f = int(sf[b]) + j
            for k in bits:
                assert (bits[k][e] != SENT).all(), f"estimate {e}: {k} not written"
            if bad[b][window_slots(f, smooth, ring)].any():
                assert st[e] == 1, f"estimate {e}: a degenerate 6D row, status {st[e]}"
                n_bad += 1
                continue
            assert st[e] == 0, f"estimate {e}: status {st[e]}"
            est, msg, sd = ref_stage3(preds_h[b], f, smooth, yy_m if yy else None, yy_s if yy else None, body9, tname)
            pos, q = msg_errors(got["msg"][e], msg)
            q0 = 6 if W == 14 else 9
            pos = max(pos, float(np.abs(got["samples"][e] - est[:, :6]).max()), float(np.abs(got["est"][e][:, :q0] - est[:, :q0]).max()))
            q = max(q, *(quat_err(got["est"][e][:, c:c + 4], est[:, c:c + 4]) for c in range(q0, W, 4)))
            np.testing.assert_allclose(got["stdev"][e], sd, rtol=5e-3, atol=2e-6, err_msg=f"estimate {e}")
            assert pos <= POS_TOL and q <= QUAT_TOL, f"estimate {e} (stream {b}, frame {f}): position {pos:.3g} m, quaternion {q:.3g}"
            worst_pos, worst_q = max(worst_pos, pos), max(worst_q, q)
            worst_sd = max(worst_sd, float(np.abs(got["stdev"][e] - sd).max()))
    assert n_bad == (0 if yy else sum(1 for j in range(nF) if bad[2][window_slots(int(sf[2]) + j, smooth, ring)].any()))
    if not yy:
        assert n_bad >= 1
    print(f"stream_frames [fk_reduce] {tname} n={n} smooth={smooth} nF={nF} yy={yy}: worst position error {worst_pos:.3g} m, "
          f"quaternion {worst_q:.3g}, std {worst_sd:.3g} m; {n_bad} degenerate estimates flagged")


@pytest.mark.parametrize("target", [0, 1, 2])
def test_msg_from_est_many_estimates_ragged_rows(target, body9):
    tname, W = TARGET_NAMES[target], 14 if target == 0 else 21
    E, S = 7, 37                                                      # S not a multiple of the 16 lanes of an estimate
    rng = np.random.default_rng(target + 3)
    dn = _stage3_preds(target, E, 1, S, rng)[:, 0]                    # [E][S][O]
    est = np.stack([OFK.arm_pose_from_nn_targets(dn[e], body9, tname) for e in range(E)]).astype(np.float32)
    msg = torch.empty((E, 25), dtype=torch.float32, device="cuda")
    sd = torch.empty((E, 6), dtype=torch.float32, device="cuda")
    est_d, body = torch.from_numpy(est).cuda(), torch.from_numpy(np.asarray(body9, np.float32).ravel()).cuda()
    N.check(N.load().ape_msg_from_est(N.ptr(est_d), W, N.ptr(body), target, E, S, N.ptr(msg), N.ptr(sd), N.current_stream_ptr()),
            "ape_msg_from_est")
    got_m, got_s = msg.cpu().numpy(), sd.cpu().numpy()
    worst = 0.0
    for e in range(E):
        pos, q = msg_errors(got_m[e], OFK.msg_from_est(est[e].astype(np.float64), body9, tname))
        assert pos <= POS_TOL and q <= QUAT_TOL, f"estimate {e}: position {pos:.3g} m, quaternion {q:.3g}"
        np.testing.assert_allclose(got_s[e], OFK.sample_std(est[e]), rtol=5e-3, atol=2e-6)
        worst = max(worst, pos)
    print(f"stream_frames [msg_from_est] {tname} E={E} S={S}: worst position error {worst:.3g} m")


# ---- c. the estimator entry points at serving scale -------------------------------------------------------------------------
@pytest.mark.parametrize("kind", [syn.KIND_UARM, syn.KIND_WATCH_ONLY, syn.KIND_POCKET])
def test_serving_scale_entry_points_agree_per_stream(kind):
    from oracle import estimator as OE
    spec, state = _model(kind, False)
    B, n, smooth, n_calls = 1024, 100, 2, 11
    late, restart, restart_at = range(300, 364), 517, 6
    rows = syn.synth_rows(kind, B, n_calls, config_id=70 + kind)
    rng = np.random.default_rng(kind + 40)
    frames = np.zeros(B, np.int64)
    schedule, history = [], [[[]] for _ in range(B)]                  # per stream: segments (a restart opens one) of call indices
    for k in range(n_calls):
        active = rng.random(B) >= 0.3
        active[list(late)] &= k >= 4                                  # a block of streams joins late
        if k == restart_at:                                           # MultiStreamEstimator.reset_stream: the next row is frame 0 again
            frames[restart] = 0
            active[restart] = True
            history[restart].append([])
        if k == restart_at - 1:
            active[restart] = True                                    # (so the restart cuts a non-empty history)
        sf = np.where(active, frames, -1).astype(np.int32)
        frames[active] += 1
        for b in np.flatnonzero(active):
            history[b][-1].append(k)
        schedule.append(sf)
    mk = lambda **kw: _estimator(kind, state, B, n, 1, smooth=smooth, lstm_variant="tc", **kw)
    piped, plain, graph = mk(), mk(pipeline=False), mk()
    assert piped._pipe is not None and piped.lanes and plain._pipe is None
    assert piped.tc_flags == 0 and not piped.small_batch and not piped.tc_split
    want_kernel = "tcw" if spec["H"] == 128 else "tcs"
    # the native pipeline: N_SLOTS - 1 calls in flight (the device copies of the counters, frames_dev[call & 3], are reused)
    got_p, pending = [], []
    for k in range(n_calls):
        if len(pending) == piped.N_SLOTS - 1:
            o = pending.pop(0).result()
            got_p.append((o.msg.copy(), o.std.copy(), o.samples.copy(), o.status.copy()))
        pending.append(piped.submit(rows[:, k:k + 1], stream_frames=schedule[k]))
    for p in pending:
        o = p.result()
        got_p.append((o.msg.copy(), o.std.copy(), o.samples.copy(), o.status.copy()))
    assert piped.submits == n_calls
    for k in range(n_calls):
        o = plain.step(rows[:, k:k + 1], stream_frames=schedule[k])
        a = (o.msg.copy(), o.std.copy(), o.samples.copy(), o.status.copy())
        o = graph.step_graph(rows[:, k:k + 1], stream_frames=schedule[k])
        g = (o.msg.copy(), o.std.copy(), o.samples.copy(), o.status.copy())
        act = schedule[k] >= 0
        for name, x, y, z in zip(("msg", "std", "samples", "status"), got_p[k], a, g):
            np.testing.assert_array_equal(x[act], y[act], err_msg=f"call {k}: {name}, submit vs step")
            np.testing.assert_array_equal(z[act], y[act], err_msg=f"call {k}: {name}, step_graph vs step")
        assert (a[3][act] == 0).all() and np.isfinite(a[0][act]).all()
        got_p[k] = a
    assert plain.launches == n_calls * 4, f"{plain.launches} launches"   # features, layer 0, ONE launch for layers >= 1 (wavefront pair / L = 2), stage 3
    # sampled streams against a dedicated single-stream estimator on the same kernel (bit for bit) and the oracle (1e-4 m)
    pin = dict(tc_flags=2, small_batch_kernel=False) if want_kernel == "tcw" else dict(small_batch_kernel=False)
    sample = [0, B - 1, late[0], late[-1], restart] + rng.choice(B, 4, replace=False).tolist()
    L, T, H, p = spec["L"], spec["T"], spec["H"], spec["p"]
    worst, n_checked = 0.0, 0
    for b in sample:
        for seg in history[b]:
            if not seg:
                continue
            solo = _estimator(kind, state, 1, n, 1, first_stream=b, smooth=smooth, lstm_variant="tc", pipeline=False, **pin)
            masks = philox_masks(SEED, b, len(seg), 0, L, T, n, H, p)
            orc = OE.OracleEstimator(syn.KIND_NAMES[kind], spec["lookup"], state, spec["stats"], spec["y_targets"].name, T, smooth, n,
                                     None, p, mask_source=lambda f, m=masks: list(m[f]))
            for f, k in enumerate(seg):
                assert schedule[k][b] == f
                o = solo.step(rows[b:b + 1, k:k + 1])
                np.testing.assert_array_equal(got_p[k][0][b], o.msg[0], err_msg=f"stream {b}, call {k}: msg vs a dedicated estimator")
                np.testing.assert_array_equal(got_p[k][2][b], o.samples[0], err_msg=f"stream {b}, call {k}: samples vs a dedicated estimator")
                want = np.asarray(orc.step(rows[b, k]), np.float64)
                pos, q = msg_errors(got_p[k][0][b, 0], want[:25])
                pos = max(pos, float(np.abs(got_p[k][2][b, 0].ravel() - want[25:]).max()))
                assert pos <= POS_TOL and q <= QUAT_TOL, f"stream {b}, call {k}: position {pos:.3g} m, quaternion {q:.3g} vs the oracle"
                worst = max(worst, pos)
                n_checked += 1
    assert len(history[restart]) == 2 and history[restart][0] and history[restart][1]
    print(f"stream_frames [serving] {syn.KIND_NAMES[kind]} {B} x {n}, {n_calls} calls ({want_kernel}): submit / step / step_graph bit-equal; "
          f"{n_checked} estimates of {len(sample)} streams bit-equal to dedicated estimators, worst position error vs the oracle {worst:.3g} m")
