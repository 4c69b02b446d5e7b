"""GPU: one skeleton per stream on the batched path (the reference's per-instance ``bonemap``, estimator.py:57-68).

* ``ape_fk_reduce_bodies`` with stride 0, or with a table of equal rows, is bit-identical to ``ape_fk_reduce``; with distinct rows every
  estimate is bit-identical to ``ape_fk_reduce`` called with its stream's row alone - also when the two estimates of a warp pair an
  x-axis skeleton with one off the axis - and within 1e-5 m of the float64 host FK (oracle.fk) with that row.
* ``BatchedEstimator(bonemaps=...)``: its entry points agree bit for bit, every stream equals the estimator built with ``bonemap=`` its
  skeleton, and a few streams match the oracle loop with their own body; ``set_bonemap`` orders against calls in flight and against a
  captured ``step_graph``; ``MultiStreamEstimator``, ``relabel_recordings`` and shards carry the skeletons through.
"""
import queue

import numpy as np
import pytest
import torch

from arm_pose_estimation_b200 import _native as N, synthetic as syn
from arm_pose_estimation_b200.data_types.bone_map import BoneMap, body_measurements_row, body_measurements_rows
from arm_pose_estimation_b200.estimate.batched import BatchedEstimator, EST_WIDTH, shard_streams
from arm_pose_estimation_b200.estimate.multi_stream import MultiStreamEstimator
from arm_pose_estimation_b200.record import replay
from oracle import estimator as OE
from oracle import fk as OFK

pytestmark = pytest.mark.gpu
SENTINEL = -7777.25
SEED = 0x5EED5
TNAMES = {0: "ORI_CAL_LARM_UARM", 1: "ORI_CAL_LARM_UARM_HIPS", 2: "ORI_POS_CAL_LARM_UARM_HIPS"}
O_OF = {0: 12, 1: 14, 2: 20}
OFF_A = [-0.21, 0.04, -0.03, -0.27, -0.05, 0.02, -0.16, 0.44, 0.01]       # bone vectors off the x axis: the general rotation
OFF_B = [-0.18, -0.06, 0.05, -0.30, 0.03, -0.04, -0.19, 0.41, -0.02]
# neighbouring streams alternate between the x-axis rotation and the general one
SKELETONS = [BoneMap(0.25, 0.31, [-0.18, 0.45, 0.0]), OFF_A, None, OFF_B, BoneMap(0.19, 0.23, [-0.15, 0.40, -0.02])]


def _bits(a):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    return np.ascontiguousarray(a).view(np.int32)


# ---- the kernel ---------------------------------------------------------------------------------------------------------------
def _stage3(fn, preds, ring, yy, table, stride, target, B, nF, frame0, sf, n, smooth):
    """One stage-3 launch into sentinel-filled outputs; ``fn``: "bodies" (table, stride) or "one" (ape_fk_reduce, table = one row)."""
    E, S, W = B * nF, smooth * n, EST_WIDTH[target]
    out = dict(msg=torch.full((E, 25), SENTINEL, device="cuda"), samples=torch.full((E, S, 6), SENTINEL, device="cuda"),
               stdev=torch.full((E, 6), SENTINEL, device="cuda"), est=torch.full((E, S, W), SENTINEL, device="cuda"),
               status=torch.full((E,), -3, dtype=torch.int32, device="cuda"))
    ym, ys = (None, None) if yy is None else yy
    lib, common = N.load(), (target, O_OF[target], B, nF, frame0, N.ptr(sf), n, smooth, N.ptr(out["msg"]), N.ptr(out["samples"]),
                             N.ptr(out["stdev"]), N.ptr(out["est"]), N.ptr(out["status"]), N.current_stream_ptr())
    if fn == "bodies":
        N.check(lib.ape_fk_reduce_bodies(N.ptr(preds), ring, N.ptr(ym), N.ptr(ys), N.ptr(table), stride, *common), "ape_fk_reduce_bodies")
    else:
        N.check(lib.ape_fk_reduce(N.ptr(preds), ring, N.ptr(ym), N.ptr(ys), N.ptr(table), *common), "ape_fk_reduce")
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def _same_outputs(a, b, rows=None):
    for k in a:
        x, y = (a[k], b[k]) if rows is None else (a[k][rows], b[k][rows])
        np.testing.assert_array_equal(_bits(x), _bits(y), err_msg=k)


KERNEL_CASES = [
    # target, B, nF, smooth, frame0, stream_frames, normalised
    (0, 7, 1, 1, 0, None, True),
    (0, 5, 2, 3, 4, [3, -1, 0, 7, 1], True),
    (1, 9, 3, 3, 0, None, False),
    (1, 5, 4, 1, 9, [9, 2, -1, 0, 5], True),
    (2, 7, 1, 3, 2, None, True),
    (2, 3, 2, 1, 0, [6, -1, 1], False),
]


def _kernel_inputs(target, B, nF, smooth, normalised, seed):
    rng = np.random.default_rng(seed)
    n, O = 12, O_OF[target]
    ring = nF + smooth - 1 + 1
    preds_h = rng.normal(0, 1, (B, ring, n, O)).astype(np.float32)
    yy = None
    if normalised:
        yy = (torch.from_numpy(rng.uniform(-0.1, 0.1, O).astype(np.float32)).cuda(),
              torch.from_numpy(rng.uniform(0.5, 1.5, O).astype(np.float32)).cuda())
    return preds_h, ring, n, yy


@pytest.mark.parametrize("target,B,nF,smooth,frame0,sf,normalised", KERNEL_CASES,
                         ids=[f"{TNAMES[c[0]]}-B{c[1]}-nF{c[2]}-s{c[3]}{'-idle' if c[5] else ''}" for c in KERNEL_CASES])
def test_kernel_table_is_bit_identical_to_one_row_calls(target, B, nF, smooth, frame0, sf, normalised):
    preds_h, ring, n, yy = _kernel_inputs(target, B, nF, smooth, normalised, 100 * target + B)
    if not normalised:                    # a degenerate 6D row in the last stream's first frame: status 1 for the estimates that read it
        off, fb = 3 if target == 2 else 0, frame0 if sf is None else sf[-1]
        preds_h[B - 1, fb % ring, 0, off:off + 6] = 0.0
    preds = torch.from_numpy(preds_h).cuda()
    sf_d = None if sf is None else torch.tensor(sf, dtype=torch.int32, device="cuda")
    rows = body_measurements_rows([SKELETONS[b % len(SKELETONS)] for b in range(B)], B).astype(np.float32)
    default = torch.from_numpy(body_measurements_row().astype(np.float32).ravel()).cuda()
    args = (target, B, nF, frame0, sf_d, n, smooth)
    one = _stage3("one", preds, ring, yy, default, 0, *args)
    # stride 0 and tables of equal rows (strides 9 and 12) are the one-row call
    _same_outputs(_stage3("bodies", preds, ring, yy, default, 0, *args), one)
    for stride in (9, 12):
        tab = np.zeros((B, stride), np.float32)
        tab[:, :9] = body_measurements_row().astype(np.float32)
        tab[:, 9:] = np.nan                              # (padding the kernel must not read)
        _same_outputs(_stage3("bodies", preds, ring, yy, torch.from_numpy(tab).cuda(), stride, *args), one)
    # distinct rows: each estimate is the one-row call with its stream's row
    for stride in (9, 16):
        tab = np.full((B, stride), np.nan, np.float32)
        tab[:, :9] = rows
        got = _stage3("bodies", preds, ring, yy, torch.from_numpy(tab).cuda(), stride, *args)
        for b in range(B):
            want = _stage3("one", preds, ring, yy, torch.from_numpy(rows[b].copy()).cuda(), 0, *args)
            _same_outputs(got, want, slice(b * nF, (b + 1) * nF))
    # idle streams keep their outputs; the skeletons change the positions
    for b in range(B):
        live = sf is None or sf[b] >= 0
        e = slice(b * nF, (b + 1) * nF)
        assert (got["msg"][e] != SENTINEL).all() == live and (got["msg"][e] == SENTINEL).all() == (not live)
        assert (got["status"][e] >= 0).all() == live
    assert np.abs(got["msg"][0, 18:21] - one["msg"][0, 18:21]).max() > 1e-3          # (stream 0 is live in every case)
    assert got["status"].max() == (0 if normalised else 1)


@pytest.mark.parametrize("target", [0, 1, 2], ids=[TNAMES[t] for t in (0, 1, 2)])
@pytest.mark.parametrize("smooth", [1, 3])
def test_kernel_table_against_float64_fk(target, smooth):
    B, nF, frame0 = 5, 2, 3
    preds_h, ring, n, yy = _kernel_inputs(target, B, nF, smooth, True, 7 + target + smooth)
    preds = torch.from_numpy(preds_h).cuda()
    rows = body_measurements_rows(SKELETONS, B)
    got = _stage3("bodies", preds, ring, yy, torch.from_numpy(rows.astype(np.float32)).cuda(), 9, target, B, nF, frame0, None, n, smooth)
    ym, ys = (t.cpu().numpy().astype(np.float64) for t in yy)
    worst = 0.0
    for b in range(B):
        body = rows[b:b + 1].astype(np.float32).astype(np.float64)
        for j in range(nF):
            f, e = frame0 + j, b * nF + j
            slots = [max(0, w) % ring for w in range(f - smooth + 1, f + 1)]
            win = preds_h[b, slots].astype(np.float64).reshape(-1, O_OF[target]) * ys + ym
            est = OFK.arm_pose_from_nn_targets(win, body, TNAMES[target])
            msg = OFK.msg_from_est(est, body, TNAMES[target])
            for a, c in ((4, 7), (11, 14), (18, 21)):
                worst = max(worst, float(np.abs(got["msg"][e, a:c] - msg[a:c]).max()))
            worst = max(worst, float(np.abs(got["est"][e][:, :6] - est[:, :6]).max()))
            np.testing.assert_allclose(got["stdev"][e], OFK.sample_std(est), rtol=0, atol=1e-5)
    print(f"{TNAMES[target]} smooth {smooth}: worst position error vs float64 FK {worst:.3g} m")
    assert worst <= 1e-5


# ---- the estimator ------------------------------------------------------------------------------------------------------------
def _state(kind, model):
    spec = syn.kind_spec(kind)
    if model == "ff2d":
        return syn.synth_ff_state_dict(spec["I"] * spec["T"], 256, 2, spec["O"], seed=40 + kind)
    return syn.synth_state_dict(spec["I"], spec["H"], spec["L"], spec["O"], 1234 + kind)


def _engine(kind, state, B, n, smooth=1, nF=1, first_stream=0, **kw):
    spec = syn.kind_spec(kind)
    return BatchedEstimator(kind=kind, layout=spec["layout"], state=state, seq_len=spec["T"], y_targets=spec["y_targets"],
                            stats=spec["stats"], n_streams=B, mc_samples=n, smooth=smooth, dropout=spec["p"], frames_per_call=nF,
                            mask_mode=N.MASK_PHILOX, philox_seed=SEED, first_stream=first_stream, **kw)


def _keep(out):
    c = lambda a: None if a is None else np.array(a, copy=True)
    return type(out)(c(out.msg), c(out.std), c(out.samples), c(out.status), out.frame0)


def _same(a, b, streams=slice(None)):
    for x, y in ((a.msg, b.msg), (a.std, b.std), (a.status, b.status), (a.samples, b.samples)):
        np.testing.assert_array_equal(np.asarray(x)[streams], np.asarray(y)[streams])


ENGINE_CASES = [
    # name, kind, model, engine keywords
    ("uarm-native-pipeline", syn.KIND_UARM, "lstm", dict(lstm_variant="tc", small_batch_kernel=False)),
    ("uarm-python-pipeline", syn.KIND_UARM, "lstm", dict(lstm_variant="tc", small_batch_kernel=False, native_pipeline=False)),
    ("pocket", syn.KIND_POCKET, "lstm", dict(lstm_variant="tc")),
    ("watch-only", syn.KIND_WATCH_ONLY, "lstm", dict(lstm_variant="tc")),
    ("uarm-ff2d", syn.KIND_UARM, "ff2d", dict()),
]


@pytest.mark.parametrize("kind,model,kw", [c[1:] for c in ENGINE_CASES], ids=[c[0] for c in ENGINE_CASES])
def test_estimator_entry_points_and_single_skeleton_estimators_agree(kind, model, kw):
    B, F, n, smooth = 5, 5, 16, 2
    state = _state(kind, model)
    rows = syn.synth_rows(kind, B, F, config_id=31)
    ref = _engine(kind, state, B, n, smooth, bonemaps=SKELETONS, **kw)
    if kw.get("native_pipeline", True) and kw.get("small_batch_kernel", True) is False:
        assert ref._pipe is not None
    np.testing.assert_array_equal(ref.body_rows, body_measurements_rows(SKELETONS, B).astype(np.float32))
    want = [_keep(ref.step(rows[:, f])) for f in range(F)]
    sub = _engine(kind, state, B, n, smooth, bonemaps=SKELETONS, **kw)
    pend = [sub.submit(rows[:, f]) for f in range(F)]
    for w, p in zip(want, pend):
        _same(w, p.result())
    dev = _engine(kind, state, B, n, smooth, bonemaps=SKELETONS, **kw)
    for f in range(F):
        _same(want[f], dev.step_device(torch.from_numpy(rows[:, f:f + 1].copy()).cuda()).host())
    gr = _engine(kind, state, B, n, smooth, bonemaps=np.asarray(body_measurements_rows(SKELETONS, B)), **kw)
    for f in range(F):
        _same(want[f], gr.step_graph(rows[:, f]))
    multi = _engine(kind, state, B, n, smooth, nF=F, bonemaps=SKELETONS, **kw)
    out = multi.step(rows)
    for f in range(F):
        _same(want[f], type(out)(out.msg[:, f:f + 1], out.std[:, f:f + 1], out.samples[:, f:f + 1], out.status[:, f:f + 1], 0))
    # every stream is what the estimator with that one skeleton for all streams computes for it
    for b in range(B):
        one = _engine(kind, state, B, n, smooth, bonemap=SKELETONS[b], **kw)
        for f in range(F):
            _same(want[f], one.step(rows[:, f]), slice(b, b + 1))
    # the skeletons move the joints
    default = _engine(kind, state, B, n, smooth, **kw)
    for f in range(F):
        out = default.step(rows[:, f])
        _same(want[f], out, slice(2, 3))
        assert np.abs(want[f].msg[0, 0, 11:14] - out.msg[0, 0, 11:14]).max() > 1e-3


def test_estimator_refuses_both_forms_and_bad_tables():
    kind = syn.KIND_UARM
    state = _state(kind, "ff2d")
    with pytest.raises(UserWarning, match="not both"):
        _engine(kind, state, 2, 8, bonemap=BoneMap(), bonemaps=[None, None])
    with pytest.raises(UserWarning, match="3 skeletons for 2 streams"):
        _engine(kind, state, 2, 8, bonemaps=[None] * 3)
    be = _engine(kind, state, 2, 8)
    with pytest.raises(UserWarning):
        be.set_bonemap(2, None)
    with pytest.raises(UserWarning, match="not finite"):
        be.set_bonemap(0, [np.nan] * 9)
    np.testing.assert_array_equal(be.body_rows, np.repeat(body_measurements_row().astype(np.float32), 2, axis=0))


def test_estimator_against_the_oracle_with_own_bodies():
    kind, B, F, n, smooth = syn.KIND_UARM, 3, 4, 16, 2
    spec = syn.kind_spec(kind)
    state = _state(kind, "lstm")
    L, T, H, p = spec["L"], spec["T"], spec["H"], spec["p"]
    be = _engine(kind, state, B, n, smooth, first_stream=4, bonemaps=SKELETONS[:B], lstm_variant="fp32")
    rows = syn.synth_rows(kind, B, F, config_id=12)
    outs = [_keep(be.step(rows[:, f])) for f in range(F)]
    masks = torch.empty((B, F, L - 1, T, n, H), dtype=torch.uint8, device="cuda")
    N.check(N.load().ape_philox_masks(SEED, 4, B, F, 0, L, T, n, H, p, N.ptr(masks), N.current_stream_ptr()), "ape_philox_masks")
    masks = masks.cpu().numpy()
    table = body_measurements_rows(SKELETONS[:B], B)
    worst = 0.0
    for b in range(B):
        orc = OE.OracleEstimator(syn.KIND_NAMES[kind], spec["lookup"], state, spec["stats"], spec["y_targets"].name, T, smooth, n,
                                 table[b:b + 1], p, mask_source=lambda f, b=b: list(masks[b, f]))
        for f in range(F):
            want = np.asarray(orc.step(rows[b, f]), dtype=np.float64)
            for a, c in ((4, 7), (11, 14), (18, 21)):
                worst = max(worst, float(np.abs(outs[f].msg[b, 0, a:c] - want[a:c]).max()))
            worst = max(worst, float(np.abs(outs[f].samples[b, 0].ravel() - want[25:]).max()))
    print(f"worst position error vs the oracle with per-stream bodies {worst:.3g} m")
    assert worst <= 1e-4


NEW = [OFF_B, BoneMap(0.28, 0.33), OFF_A, None]
OLD = [None, OFF_A, BoneMap(0.21, 0.27), OFF_B]


def test_set_bonemap_with_calls_in_flight_on_the_native_pipeline():
    kind, B, F, n, smooth, k = syn.KIND_UARM, 4, 8, 16, 3, 4
    state = _state(kind, "lstm")
    kw = dict(lstm_variant="tc", small_batch_kernel=False)
    rows = syn.synth_rows(kind, B, F, config_id=8)
    refs = {name: _engine(kind, state, B, n, smooth, bonemaps=bm, **kw) for name, bm in (("old", OLD), ("new", NEW))}
    want = {name: [_keep(r.step(rows[:, f])) for f in range(F)] for name, r in refs.items()}
    be = _engine(kind, state, B, n, smooth, bonemaps=OLD, **kw)
    assert be._pipe is not None
    pend = [be.submit(rows[:, f]) for f in range(k)]                # in flight while the skeletons change
    for b in range(B):
        be.set_bonemap(b, NEW[b])
    pend += [be.submit(rows[:, f]) for f in range(k, F)]
    for f, pe in enumerate(pend):
        _same(want["old" if f < k else "new"][f], pe.result())
    np.testing.assert_array_equal(be.body_rows, body_measurements_rows(NEW, B).astype(np.float32))
    # step_device on the native pipeline, then set_bonemaps for all streams at once
    be2 = _engine(kind, state, B, n, smooth, bonemaps=OLD, **kw)
    got = [be2.step_device(torch.from_numpy(rows[:, f:f + 1].copy()).cuda()) for f in range(2)]
    be2.set_bonemaps(NEW)
    for f in range(2):
        _same(want["old"][f], got[f].host())
    for f in range(2, F):
        _same(want["new"][f], be2.step_device(torch.from_numpy(rows[:, f:f + 1].copy()).cuda()).host())


def test_set_bonemap_between_graph_ticks_without_recapture():
    kind, B, F, n, smooth = syn.KIND_POCKET, 4, 6, 12, 2
    state = _state(kind, "lstm")
    rows = syn.synth_rows(kind, B, F, config_id=6)
    want = {name: [_keep(_e.step(rows[:, f])) for f in range(F)] for name, _e in
            (("old", _engine(kind, state, B, n, smooth, bonemaps=OLD, lstm_variant="tc")),
             ("new", _engine(kind, state, B, n, smooth, bonemaps=NEW, lstm_variant="tc")))}
    be = _engine(kind, state, B, n, smooth, bonemaps=OLD, lstm_variant="tc")
    for f in range(3):
        _same(want["old"][f], be.step_graph(rows[:, f]))
    g = be._g
    be.set_bonemaps(NEW)
    for f in range(3, F):
        _same(want["new"][f], be.step_graph(rows[:, f]))
    assert be._g is g


# ---- the front-ends -----------------------------------------------------------------------------------------------------------
def test_multi_stream_with_per_stream_skeletons_and_a_new_user():
    kind, B, n, smooth, F = syn.KIND_WATCH_ONLY, 4, 12, 3, 16
    state = _state(kind, "ff2d")
    rows = syn.synth_rows(kind, B, F, config_id=23)
    bms = [OFF_A, None, BoneMap(0.24, 0.29), OFF_B]
    newcomer = BoneMap(0.18, 0.22, [-0.14, 0.39, 0.02])
    rng = np.random.default_rng(11)
    ms = MultiStreamEstimator(_engine(kind, state, B, n, smooth, bonemaps=bms), add_mc_samples=True)
    qs = [queue.Queue() for _ in range(B)]
    fed, got, switch = [0] * B, [[] for _ in range(B)], None
    for tick in range(60):
        if tick == 10:                                         # a new user takes over stream 2
            ms.reset_stream(2)
            ms.set_bonemap(2, newcomer)
            switch = len(got[2])
        for b in range(B):
            if rng.random() < (0.8, 0.5, 0.9, 0.6)[b] and fed[b] < F and not (b == 3 and tick < 5):
                qs[b].put(rows[b, fed[b]])
                fed[b] += 1
        for b, m in ms.tick(ms.collect(qs)).items():
            got[b].append(np.asarray(m))
    assert [len(g) for g in got] == fed and 0 < switch < fed[2]

    def solo(b, bm, segment):
        one = _engine(kind, state, 1, n, smooth, first_stream=b, bonemap=bm)
        res = []
        for r in segment:
            out = one.step(r[None, None])
            res.append(np.concatenate([out.msg[0, 0].astype(np.float64), out.samples[0, 0].astype(np.float64).ravel()]))
        return res

    for b in range(B):
        segments = [(bms[b], 0, fed[b])] if b != 2 else [(bms[2], 0, switch), (newcomer, switch, fed[2])]
        for bm, lo, hi in segments:
            for g, w in zip(got[b][lo:hi], solo(b, bm, rows[b, lo:hi])):
                np.testing.assert_array_equal(g, w)


def test_relabel_recordings_with_one_skeleton_per_recording():
    kind, R, F, n = syn.KIND_POCKET, 3, 9, 10
    state = _state(kind, "ff2d")
    rows = syn.synth_rows(kind, R, F, config_id=9)
    bms = [OFF_A, BoneMap(0.26, 0.32), None]
    res = replay.relabel_recordings(rows, lambda nS, fpc: _engine(kind, state, nS, n, 2, nF=fpc), frames_per_call=4,
                                    keep_samples=True, bonemaps=bms)
    for r in range(R):
        alone = replay.relabel_recordings(rows[r:r + 1], lambda nS, fpc, r=r: _engine(kind, state, nS, n, 2, nF=fpc, first_stream=r),
                                          frames_per_call=4, keep_samples=True, bonemaps=[bms[r]])[0]
        np.testing.assert_array_equal(res[r]["msg"], alone["msg"])
        np.testing.assert_array_equal(res[r]["samples"], alone["samples"])
    plain = replay.relabel_recordings(rows, lambda nS, fpc: _engine(kind, state, nS, n, 2, nF=fpc), frames_per_call=4)
    np.testing.assert_array_equal(res[2]["msg"], plain[2]["msg"])
    assert np.abs(res[0]["msg"][:, 4:7] - plain[0]["msg"][:, 4:7]).max() > 1e-3


def test_shards_with_their_slices_equal_the_unsharded_estimator():
    kind, B, F, n, smooth = syn.KIND_UARM, 5, 4, 16, 2
    state = _state(kind, "lstm")
    rows = syn.synth_rows(kind, B, F, config_id=4)
    full = _engine(kind, state, B, n, smooth, bonemaps=SKELETONS, lstm_variant="tc")
    want = [_keep(full.step(rows[:, f])) for f in range(F)]
    for rank in range(2):
        first, count = shard_streams(B, 2, rank)
        shard = _engine(kind, state, count, n, smooth, first_stream=first, bonemaps=SKELETONS[first:first + count], lstm_variant="tc")
        for f in range(F):
            out = shard.step(rows[first:first + count, f])
            np.testing.assert_array_equal(out.msg, want[f].msg[first:first + count])
            np.testing.assert_array_equal(out.samples, want[f].samples[first:first + count])
