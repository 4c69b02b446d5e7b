"""The dropout draw of ``APE_MASK_PHILOX`` in numpy: Philox4x32-10 (Salmon et al. 2011) and the counter layout of
``philox_keep8`` (csrc/ape_common.cuh), written out independently of the library.

Counter (stream id, absolute frame, sample | gap << 20 | t << 24, unit octet), key = the 64-bit seed.  Output word i of a draw
holds two 16-bit lanes, unit 2i in the low half and unit 2i + 1 in the high half; a unit is kept iff its lane < keep_thr16.  The
LSTM kernels use gap = the layer gap (0 .. L-2) and t = the step; the feed-forward kernels gap 15 and t 0.

Every array is uint64 with the 32-bit values in its low half, so the 32 x 32 -> 64-bit products of the rounds are exact.  The
draw does not depend on p: the ``*_lanes`` builders return the lanes (uint32), ``lanes < keep_threshold16(p)`` are the keep-masks.
Test infrastructure only.
"""
import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57          # round multipliers
W0, W1 = 0x9E3779B9, 0xBB67AE85          # Weyl key increments
MASK32 = np.uint64(0xFFFFFFFF)
SAMPLE_BITS, GAP_BITS, T_BITS = 20, 4, 8
FF_GAP = 15                              # the feed-forward output dropout's gap id


def _u32(v):
    return np.asarray(v, dtype=np.uint64) & MASK32


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of broadcastable counter words c0..c3 and key words k0, k1 -> the four output words (uint64 arrays)."""
    c0, c1, c2, c3, k0, k1 = np.broadcast_arrays(*(_u32(v) for v in (c0, c1, c2, c3, k0, k1)))
    m0, m1, s32 = np.uint64(M0), np.uint64(M1), np.uint64(32)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2
        c0, c1, c2, c3 = ((p1 >> s32) ^ c1 ^ k0), p1 & MASK32, ((p0 >> s32) ^ c3 ^ k1), p0 & MASK32
        k0, k1 = (k0 + np.uint64(W0)) & MASK32, (k1 + np.uint64(W1)) & MASK32
    return c0, c1, c2, c3


def keep_threshold16(p):
    """``keep_threshold16`` in float32 arithmetic: (1 - p) * 65536 + 0.5, truncated, clamped to [0, 65536]."""
    k = (np.float32(1.0) - np.float32(p)) * np.float32(65536.0) + np.float32(0.5)
    return 65536 if k >= np.float32(65536.0) else (0 if k <= np.float32(0.0) else int(k))


def counter_word2(sample, gap, t):
    """Third counter word: sample (20 bits) | gap (4 bits) << 20 | t (8 bits) << 24.  Wider values wrap into their field."""
    s, g, tt = (np.asarray(v, dtype=np.uint64) for v in (sample, gap, t))
    return (s & np.uint64((1 << SAMPLE_BITS) - 1)) | ((g & np.uint64((1 << GAP_BITS) - 1)) << np.uint64(20)) | \
        ((tt & np.uint64((1 << T_BITS) - 1)) << np.uint64(24))


def draw_words(seed, stream, frame, sample, gap, t, group):
    """The four output words of the draw of unit octet ``group``: (..., 4) uint64."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    w = philox4x32_10(stream, frame, counter_word2(sample, gap, t), group, seed & 0xFFFFFFFF, seed >> 32)
    return np.stack(w, axis=-1)


def words_to_lanes(words):
    """(..., 4) output words -> (..., 8) 16-bit lanes, unit 2i = low half of word i, unit 2i + 1 = high half."""
    lo, hi = words & np.uint64(0xFFFF), words >> np.uint64(16)
    return np.stack([lo, hi], axis=-1).reshape(words.shape[:-1] + (8,))


def keep8(seed, stream, frame, sample, gap, t, group, keep_thr16):
    """``philox_keep8``: bit j of the result is set iff unit 8 group + j is kept."""
    kept = words_to_lanes(draw_words(seed, stream, frame, sample, gap, t, group)) < np.uint64(keep_thr16)
    return (kept.astype(np.uint64) << np.arange(8, dtype=np.uint64)).sum(axis=-1)


def keep_flags(words, keep_thr16):
    """The plain compare the kernels' two-lane keep flags stand for: bit 15 iff the low lane < thr, bit 31 iff the high lane < thr."""
    w = _u32(words)
    lo = (w & np.uint64(0xFFFF)) < np.uint64(keep_thr16)
    hi = (w >> np.uint64(16)) < np.uint64(keep_thr16)
    return (lo.astype(np.uint64) << np.uint64(15)) | (hi.astype(np.uint64) << np.uint64(31))


def unit_lanes(seed, stream, frame, sample, gap, t, H):
    """Lanes of units 0 .. H-1 of broadcastable (stream, frame, sample, gap, t): (..., H) uint32.  A last octet that H does not fill
    is drawn whole and cut (the one-CTA-per-row feed-forward kernel takes any H)."""
    groups = np.arange((H + 7) // 8, dtype=np.uint64)
    ex = lambda v: np.asarray(v, dtype=np.uint64)[..., None]
    words = draw_words(seed, ex(stream), ex(frame), ex(sample), ex(gap), ex(t), groups)
    return words_to_lanes(words).reshape(words.shape[:-2] + (groups.size * 8,))[..., :H].astype(np.uint32)


def stream_frame_list(B, nF, frame0, stream_frames=None):
    """Absolute frame of each of the E = B * nF estimates (row e = b * nF + j): (stream_frames[b] or frame0) + j."""
    fb = np.full(B, frame0, np.int64) if stream_frames is None else np.asarray(stream_frames, np.int64)
    return (fb[:, None] + np.arange(nF)[None, :]).reshape(-1)


def lstm_lanes(seed, stream_id0, B, nF, frame0, L, T, n, H, stream_frames=None):
    """Lanes in the injected-mask layout of the LSTM kernels, [E][L-1][T][n][H]: estimate e = b * nF + j draws with stream
    stream_id0 + b (mod 2^32) at its frame, sample s, gap l, step t."""
    E = B * nF
    stream = (np.uint64(stream_id0) + (np.arange(E, dtype=np.uint64) // np.uint64(nF))) & MASK32
    frame = stream_frame_list(B, nF, frame0, stream_frames).astype(np.uint64) & MASK32
    sh = (E, L - 1, T, n)
    st = np.broadcast_to(stream[:, None, None, None], sh)
    fr = np.broadcast_to(frame[:, None, None, None], sh)
    gap = np.broadcast_to(np.arange(L - 1)[None, :, None, None], sh)
    t = np.broadcast_to(np.arange(T)[None, None, :, None], sh)
    s = np.broadcast_to(np.arange(n)[None, None, None, :], sh)
    return unit_lanes(seed, st, fr, s, gap, t, H)


def ff_lanes(seed, stream_id0, rows, frame0, n, H):
    """Lanes of ``ape_mc_ff``, [rows][n][H]: row r draws with stream stream_id0 + r (mod 2^32), frame frame0, gap 15, t 0."""
    stream = (np.uint64(stream_id0) + np.arange(rows, dtype=np.uint64)) & MASK32
    sh = (rows, n)
    return unit_lanes(seed, np.broadcast_to(stream[:, None], sh), frame0, np.broadcast_to(np.arange(n)[None, :], sh), FF_GAP, 0, H)


def ff_ring_lanes(seed, stream_id0, B, nF, frame0, n, H, stream_frames=None):
    """Lanes of ``ape_mc_ff_ring``, [E][n][H]: row e = b * nF + j draws with stream stream_id0 + b (mod 2^32) at its frame f."""
    E = B * nF
    stream = (np.uint64(stream_id0) + (np.arange(E, dtype=np.uint64) // np.uint64(nF))) & MASK32
    frame = stream_frame_list(B, nF, frame0, stream_frames).astype(np.uint64) & MASK32
    sh = (E, n)
    return unit_lanes(seed, np.broadcast_to(stream[:, None], sh), np.broadcast_to(frame[:, None], sh),
                      np.broadcast_to(np.arange(n)[None, :], sh), FF_GAP, 0, H)


def masks_from_lanes(lanes, p):
    """{0,1} uint8 keep-masks of the lanes at drop probability p."""
    return (lanes < keep_threshold16(p)).astype(np.uint8)
