"""Body measurements that enter the hot path as nine floats (``estimator.py:57-68`` of the reference).

Only the defaults (``data_types/bone_map.py:42-45``) and the three attributes the estimator reads are
provided; parsing Motive skeleton XML is outside the hot path (SURVEY.md §2 row 10) - any object with the
same three attributes (e.g. the reference's own ``BoneMap``) can be passed as ``bonemap``.
"""
import numpy as np


class BoneMap:
    DEFAULT_LARM_LEN = 0.22
    DEFAULT_UARM_LEN = 0.26
    DEFAULT_UARM_ORIG_RH = np.array([-0.1704612, 0.4309841, -0.00670862])

    def __init__(self, left_lower_arm_length=None, left_upper_arm_length=None, left_upper_arm_origin_rh=None):
        self.left_lower_arm_length = self.DEFAULT_LARM_LEN if left_lower_arm_length is None else float(left_lower_arm_length)
        self.left_upper_arm_length = self.DEFAULT_UARM_LEN if left_upper_arm_length is None else float(left_upper_arm_length)
        self.left_upper_arm_origin_rh = (
            self.DEFAULT_UARM_ORIG_RH.copy() if left_upper_arm_origin_rh is None
            else np.asarray(left_upper_arm_origin_rh, dtype=np.float64)
        )


def body_measurements_row(bonemap=None):
    """``[larm_vec(-len,0,0), uarm_vec(-len,0,0), uarm_orig_rh]`` as a ``(1, 9)`` float64 array."""
    bm = BoneMap() if bonemap is None else bonemap
    larm = np.array([-bm.left_lower_arm_length, 0.0, 0.0])
    uarm = np.array([-bm.left_upper_arm_length, 0.0, 0.0])
    return np.r_[larm, uarm, np.asarray(bm.left_upper_arm_origin_rh, dtype=np.float64)][np.newaxis, :]


def body_measurements_rows(bonemaps, n):
    """One skeleton per stream: the ``(n, 9)`` float64 table whose row ``b`` is ``body_measurements_row`` of stream ``b``.

    ``bonemaps``: ``None`` (every stream has the default skeleton), an ``(n, 9)`` array, or a sequence of ``n`` entries, each a
    BoneMap-like object, ``None`` (the default skeleton) or nine floats ``[larm_vec, uarm_vec, uarm_orig_rh]`` as they are (bone
    vectors off the x axis included).  A wrong count or length, or a non-finite value, raises ``UserWarning``."""
    n = int(n)
    if bonemaps is None:
        return np.repeat(body_measurements_row(), n, axis=0)
    entries = list(bonemaps)
    if len(entries) != n:
        raise UserWarning(f"{len(entries)} skeletons for {n} streams")
    rows = np.empty((n, 9), dtype=np.float64)
    for b, bm in enumerate(entries):
        if bm is None or hasattr(bm, "left_lower_arm_length"):
            rows[b] = body_measurements_row(bm)[0]
        else:
            v = np.asarray(bm, dtype=np.float64).ravel()
            if v.size != 9:
                raise UserWarning(f"skeleton of stream {b}: 9 floats (larm_vec, uarm_vec, uarm_orig_rh) expected, got {v.size}")
            rows[b] = v
    if not np.isfinite(rows).all():
        bad = int(np.flatnonzero(~np.isfinite(rows).all(axis=1))[0])
        raise UserWarning(f"skeleton of stream {bad} is not finite: {rows[bad]}")
    return rows
