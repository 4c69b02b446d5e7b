"""CPU: the dropout draw of APE_MASK_PHILOX, bit for bit.

``oracle/philox.py`` restates Philox4x32-10 and the counter layout of ``philox_keep8`` (csrc/ape_common.cuh) in numpy.  Here it is
pinned to the Random123 known answers and to the library's host twins: ``ape_selfcheck_keep8`` (the plain compare of the fp32 LSTM and
feed-forward row kernels) at every counter field's edges and at every keep threshold class, and ``ape_selfcheck_keep_flags`` (the
branch-free two-lane compare of the tensor-core and batched feed-forward kernels) at every 16-bit lane value.  The reference draw's
statistics show that every counter field and both seed words reach the output.  The 20-bit sample field aliases samples s and
s + 2^20, so the feed-forward entry points refuse more than 2^20 samples in Philox mode, like the LSTM entry points.
tests/test_gpu_philox_draws.py holds every kernel's draw to this reference on the device."""
import ctypes as C

import numpy as np
import pytest

from arm_pose_estimation_b200 import _native as N
from oracle import philox as OP

U32 = 0xFFFFFFFF
# thresholds where a compare goes wrong: both ends, the bit-15 boundary from both sides, p = 0.2 (52429)
EDGE_THR = [0, 1, 2, 0x7FFE, 0x7FFF, 0x8000, 0x8001, 52429, 0xFFFE, 0xFFFF, 65536]
SEEDS = [0, 1 << 32, (1 << 64) - 1, 0x9C3E_57A1_D402_B86F]


def p_of(thr):
    """A float32 drop probability whose keep_threshold16 is ``thr``: 1 - thr / 65536 is exact in float32; thr 0 needs p < 1."""
    return float(np.float32(1.0 - 2.0 ** -18)) if thr == 0 else float(np.float32(1.0 - thr / 65536.0))


def lib_keep8(seed, stream, frame, sample, gap, t, group, p):
    out = C.c_uint32(0)
    assert N.load().ape_selfcheck_keep8(seed, stream, frame, sample, gap, t, group, p, C.byref(out)) == N.APE_OK
    return out.value


def lib_keep_flags(words, thr):
    w = np.ascontiguousarray(words, dtype=np.uint32)
    out = np.empty_like(w)
    P = C.POINTER(C.c_uint32)
    assert N.load().ape_selfcheck_keep_flags(w.ctypes.data_as(P), w.size, thr, out.ctypes.data_as(P)) == N.APE_OK
    return out


def test_reference_reproduces_the_random123_known_answers():
    for ctr, key, want in [([0, 0, 0, 0], [0, 0], [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
                           ([U32] * 4, [U32] * 2, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
                           ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0],   # both key words non-zero
                            [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1])]:
        assert [int(v) for v in OP.philox4x32_10(*ctr, *key)] == want


@pytest.mark.parametrize("thr", EDGE_THR)
def test_threshold_of_each_probability_is_exact(thr):
    p = p_of(thr)
    assert OP.keep_threshold16(p) == thr
    assert abs(thr / 65536 - (1.0 - p)) <= 2.0 ** -17


@pytest.mark.parametrize("p", [0.0, 0.1, 0.2, 0.25, 0.5, 0.9, float(np.float32(1.0 - 2.0 ** -18))])
def test_threshold_is_within_half_a_step_of_one_minus_p(p):
    thr = OP.keep_threshold16(p)
    assert 0 <= thr <= 65536 and abs(thr / 65536 - (1.0 - float(np.float32(p)))) <= 2.0 ** -17


def _counters(rng):
    """Counters (stream, frame, sample, gap, t, group): every field at 0 and at its maximum in all combinations, then random ones."""
    edges = [(0, U32), (0, U32), (0, (1 << 20) - 1), (0, 15), (0, 255), (0, 31)]
    corner = np.array(np.meshgrid(*edges, indexing="ij"), dtype=np.uint64).reshape(6, -1).T
    highs = [1 << 32, 1 << 32, 1 << 20, 16, 256, 1 << 32]
    rand = np.stack([rng.integers(0, h, size=700, dtype=np.uint64) for h in highs], axis=1)
    return np.concatenate([corner, rand])


@pytest.mark.parametrize("seed", SEEDS, ids=["0", "2^32", "2^64-1", "random"])
def test_reference_equals_the_library_draw(seed):
    ctr = _counters(np.random.default_rng(seed & 0xFFFF))
    words = OP.draw_words(seed, *ctr.T)
    lanes = OP.words_to_lanes(words)
    for thr in EDGE_THR:
        p = p_of(thr)
        want = OP.keep8(seed, *ctr.T, thr)
        np.testing.assert_array_equal((lanes < np.uint64(thr)).astype(np.uint64) @ (1 << np.arange(8, dtype=np.uint64)), want)
        got = np.array([lib_keep8(seed, *(int(v) for v in c), p) for c in ctr], dtype=np.uint64)
        np.testing.assert_array_equal(got, want, err_msg=f"seed {seed:#x}, keep_thr16 {thr}")
    if seed == SEEDS[-1]:                       # the kept fraction of these counters is not degenerate at p = 0.2
        kept = np.unpackbits(OP.keep8(seed, *ctr.T, 52429).astype(np.uint8)).mean()
        assert 0.75 < kept < 0.85


def _words_with_every_lane_value():
    """Every 16-bit value once in the low lane and once in the high lane, the other lane always a different value."""
    v = np.arange(65536, dtype=np.uint32)
    return np.concatenate([v | ((v ^ 0xA5A5) << 16), (v << 16) | (v ^ 0x5A5A), (v << 16) | (0xFFFF - v)])


@pytest.mark.parametrize("which", ["edges", "random"])
def test_two_lane_compare_equals_lane_less_than_threshold(which):
    words = _words_with_every_lane_value()
    thrs = EDGE_THR if which == "edges" else sorted(np.random.default_rng(17).integers(0, 65537, size=200).tolist())
    for thr in thrs:
        want = OP.keep_flags(words, thr).astype(np.uint32)
        got = lib_keep_flags(words, thr) & np.uint32(0x80008000)          # the other bits are by-products no kernel reads
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, f"keep_thr16 {thr}: {bad.size} words differ, first {words[bad[0]]:#010x}: {got[bad[0]]:#010x} != {want[bad[0]]:#010x}"
    assert (lib_keep_flags(words, 65536) == 0x80008000).all()
    assert (lib_keep_flags(words, 0) & 0x80008000 == 0).all()


def test_keep_flags_hook_refusals():
    w = (C.c_uint32 * 2)(1, 2)
    out = (C.c_uint32 * 2)()
    lib = N.load()
    assert lib.ape_selfcheck_keep_flags(None, 2, 5, out) == N.APE_ERR_BAD_ARG
    assert lib.ape_selfcheck_keep_flags(w, 2, 5, None) == N.APE_ERR_BAD_ARG
    assert lib.ape_selfcheck_keep_flags(w, -1, 5, out) == N.APE_ERR_BAD_ARG
    assert lib.ape_selfcheck_keep_flags(w, 2, 65537, out) == N.APE_ERR_BAD_ARG
    assert lib.ape_selfcheck_keep_flags(w, 0, 5, out) == N.APE_OK


# ---- statistics of the reference draw -------------------------------------------------------------------------------------------
N_DRAWS = 1 << 17                              # x 8 lanes = 1 048 576 lanes per sample


def _random_counters(rng, n=N_DRAWS):
    return [rng.integers(0, h, size=n, dtype=np.uint64) for h in (1 << 32, 1 << 32, 1 << 20, 16, 256, 1 << 32)]


def _five_sigma(q, n):
    return 5.0 * np.sqrt(q * (1.0 - q) / n) + 1.0 / n


def test_keep_rate_is_the_threshold():
    rng = np.random.default_rng(3)
    lanes = OP.words_to_lanes(OP.draw_words(0x0123_4567_89AB_CDEF, *_random_counters(rng))).ravel()
    for thr in EDGE_THR + [16384, 32767, 32768, 32769]:
        q = thr / 65536
        rate = float((lanes < np.uint64(thr)).mean())
        assert abs(rate - q) <= _five_sigma(q, lanes.size), f"keep_thr16 {thr}: kept {rate:.6f}, expected {q:.6f}"


FIELDS = ["stream", "frame", "sample", "gap", "t", "group"]
# (field, bit flipped): the lowest and the highest bit of every field, both words of the seed
CHANGES = [(f, b) for f, top in zip(FIELDS, (31, 31, 19, 3, 7, 31)) for b in (0, top)] + \
          [("seed", b) for b in (0, 31, 32, 63)]


@pytest.mark.parametrize("field,bit", CHANGES, ids=[f"{f}-bit{b}" for f, b in CHANGES])
def test_every_counter_field_and_seed_word_reaches_the_draw(field, bit):
    rng = np.random.default_rng(CHANGES.index((field, bit)))
    ctr = _random_counters(rng)
    seed = 0x5EED_0000_FACE_0001
    a = OP.words_to_lanes(OP.draw_words(seed, *ctr))
    if field == "seed":
        b = OP.words_to_lanes(OP.draw_words(seed ^ (1 << bit), *ctr))
    else:
        i = FIELDS.index(field)
        ctr2 = list(ctr)
        ctr2[i] = ctr[i] ^ np.uint64(1 << bit)
        b = OP.words_to_lanes(OP.draw_words(seed, *ctr2))
    for thr in (52429, 32768):
        q = thr / 65536
        agree = float(((a < np.uint64(thr)) == (b < np.uint64(thr))).mean())
        want = q * q + (1 - q) ** 2
        assert abs(agree - want) <= _five_sigma(want, a.size), f"{field} bit {bit}: agreement {agree:.5f}, independent draws {want:.5f}"


@pytest.mark.parametrize("j,k", [(0, 1), (0, 2), (1, 7), (3, 4), (6, 7)])
def test_units_within_an_octet_are_independent(j, k):
    lanes = OP.words_to_lanes(OP.draw_words(77, *_random_counters(np.random.default_rng(j * 8 + k), 1 << 20)))
    for thr in (52429, 32768):
        q = thr / 65536
        agree = float(((lanes[:, j] < np.uint64(thr)) == (lanes[:, k] < np.uint64(thr))).mean())
        want = q * q + (1 - q) ** 2
        assert abs(agree - want) <= _five_sigma(want, lanes.shape[0])


# ---- the 20-bit sample field: demonstrated, and refused where it would bite ------------------------------------------------------
def test_samples_two_to_the_twenty_apart_share_their_mask():
    rng = np.random.default_rng(20)
    seed, s = 0xABCD_EF01_2345_6789, rng.integers(0, 1 << 20, size=64, dtype=np.uint64)
    for g in (0, 15):
        a = OP.keep8(seed, 5, 9, s, g, 3, 2, 52429)
        np.testing.assert_array_equal(OP.keep8(seed, 5, 9, s + np.uint64(1 << 20), g, 3, 2, 52429), a)
        assert [lib_keep8(seed, 5, 9, int(v) + (1 << 20), g, 3, 2, 0.2) for v in s] == [int(v) for v in a]
    # ... and the samples of an n > 2^20 call would be exactly that: rows 0 and 2^20 of ff_lanes' counters
    np.testing.assert_array_equal(OP.ff_lanes(seed, 0, 1, 4, 2, 16)[0, 0], OP.unit_lanes(seed, 0, 4, 1 << 20, 15, 0, 16))


def _ff(**kw):
    """ape_mc_ff, DropoutFF of 38 inputs, H = 256, two hidden layers, O = 12 on 4 rows; the pointers are placeholders."""
    a = dict(blob=256, I=38, H=256, Lh=2, O=12, p=0.2, x=512, rows=4, n=(1 << 20) + 1, mask_mode=N.MASK_PHILOX, masks=None, seed=1,
             stream_id0=0, frame0=0, preds=768)
    a.update(kw)
    return N.load().ape_mc_ff(a["blob"], a["I"], a["H"], a["Lh"], a["O"], a["p"], a["x"], a["rows"], a["n"], a["mask_mode"],
                              a["masks"], a["seed"], a["stream_id0"], a["frame0"], a["preds"], None)


def _ff_ring(**kw):
    """ape_mc_ff_ring, the uarm DropoutFF2D (6 x 38 inputs, H = 256, Lh = 2, O = 12), 4 streams x 2 frames; placeholder pointers."""
    a = dict(blob=256, I=38, T=6, H=256, Lh=2, O=12, p=0.2, feats=512, feat_ring=7, B=4, nF=2, frame0=0, stream_frames=None,
             n=(1 << 20) + 1, mask_mode=N.MASK_PHILOX, masks=None, seed=1, stream_id0=0, preds=768, pred_ring=2)
    a.update(kw)
    return N.load().ape_mc_ff_ring(a["blob"], a["I"], a["T"], a["H"], a["Lh"], a["O"], a["p"], a["feats"], a["feat_ring"], a["B"],
                                   a["nF"], a["frame0"], a["stream_frames"], a["n"], a["mask_mode"], a["masks"], a["seed"],
                                   a["stream_id0"], a["preds"], a["pred_ring"], None)


@pytest.mark.parametrize("call", [_ff, _ff_ring], ids=["ape_mc_ff", "ape_mc_ff_ring"])
def test_feed_forward_refuses_more_philox_samples_than_the_counter_holds(call):
    empty = dict(rows=0) if call is _ff else dict(B=0)
    assert call() == N.APE_ERR_UNSUPPORTED                                        # before the first CUDA call
    assert call(n=1 << 30) == N.APE_ERR_UNSUPPORTED
    assert call(**empty) == N.APE_ERR_UNSUPPORTED                                 # before the empty-call shortcut, as the LSTM rule
    assert call(n=1 << 20, **empty) == N.APE_OK                                   # 2^20 samples fit the field
    assert call(mask_mode=N.MASK_INJECTED, masks=1024, **empty) == N.APE_OK       # other mask modes draw nothing
    assert call(mask_mode=N.MASK_NONE, **empty) == N.APE_OK
