"""CPU: per-stream skeletons on the batched path - the two entry points (ape_fk_reduce_bodies, ape_pipeline_set_bodies), their
bindings and their refusals, which all come before the first CUDA call, and the host-side table (bone_map.body_measurements_rows).
The pointers are placeholders that are never dereferenced."""
import numpy as np
import pytest

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200.data_types.bone_map import BoneMap, body_measurements_row, body_measurements_rows

OK, BAD = N.APE_OK, N.APE_ERR_BAD_ARG


def _call(**kw):
    """ape_fk_reduce_bodies of a uarm-shaped stage 3 (O = 12), 4 streams x 2 frames, 10 samples, smooth 3."""
    a = dict(preds=1024, ring=6, yy_m=None, yy_s=None, bodies=2048, stride=9, target=N.TARGET_ORI_CAL_LARM_UARM, O=12, B=4, nF=2,
             frame0=0, sf=None, n=10, smooth=3, msg=4096)
    a.update(kw)
    return N.load().ape_fk_reduce_bodies(a["preds"], a["ring"], a["yy_m"], a["yy_s"], a["bodies"], a["stride"], a["target"], a["O"],
                                         a["B"], a["nF"], a["frame0"], a["sf"], a["n"], a["smooth"], a["msg"], None, None, None, None,
                                         None)


def test_symbols_are_declared_and_bound():
    lib = N.load()
    for name, nargs in (("ape_fk_reduce_bodies", 20), ("ape_pipeline_set_bodies", 3)):
        assert name in N.SYMBOLS
        assert getattr(lib, name).restype is not None and len(getattr(lib, name).argtypes) == nargs
    # the table form takes the arguments of ape_fk_reduce with (bodies, body_stride) in place of body9
    fk, fkb = lib.ape_fk_reduce.argtypes, lib.ape_fk_reduce_bodies.argtypes
    assert fkb[:5] == fk[:5] and fkb[6:] == fk[5:]


CASES = [
    ("no-bodies", dict(bodies=None), BAD),
    ("no-bodies-empty", dict(bodies=None, B=0), BAD),
    ("stride-neg", dict(stride=-1), BAD),
    ("stride-1", dict(stride=1), BAD),
    ("stride-8", dict(stride=8), BAD),
    ("stride-8-empty", dict(stride=8, B=0), BAD),
    # the checks of ape_fk_reduce stay in force
    ("no-preds", dict(preds=None), BAD),
    ("no-msg", dict(msg=None), BAD),
    ("O-mismatch", dict(O=14), BAD),
    ("ring-short", dict(ring=3), BAD),
    ("yy-half", dict(yy_m=512), BAD),
    # accepted; an empty call is done before the device
    ("empty-stride0", dict(B=0, stride=0), OK),
    ("empty-stride9", dict(B=0, stride=9), OK),
    ("empty-stride12", dict(nF=0, stride=12), OK),
]


@pytest.mark.parametrize("kw,want", [c[1:] for c in CASES], ids=[c[0] for c in CASES])
def test_fk_reduce_bodies_refusals_before_the_device(kw, want):
    assert _call(**kw) == want


@pytest.mark.parametrize("stride", [-1, 1, 8])
def test_pipeline_set_bodies_refusals(stride):
    lib = N.load()
    assert lib.ape_pipeline_set_bodies(None, 2048, 9) == BAD            # null pipeline
    assert lib.ape_pipeline_set_bodies(None, None, 0) == BAD
    assert lib.ape_pipeline_set_bodies(4096, 2048, stride) == BAD      # bad stride: refused before the pipeline is looked at


def test_rows_default_skeleton():
    one = body_measurements_row()
    for arg in (None, [None] * 3, [BoneMap()] * 3):
        rows = body_measurements_rows(arg, 3)
        assert rows.shape == (3, 9) and rows.dtype == np.float64
        np.testing.assert_array_equal(rows, np.repeat(one, 3, axis=0))
    assert body_measurements_rows(None, 0).shape == (0, 9)


def test_rows_mixed_entries():
    bm = BoneMap(0.25, 0.30, [-0.2, 0.45, 0.01])
    off_axis = np.array([-0.2, 0.05, 0.03, -0.24, -0.04, 0.06, -0.17, 0.43, -0.01])
    rows = body_measurements_rows([bm, None, off_axis, off_axis.tolist()], 4)
    np.testing.assert_array_equal(rows[0], body_measurements_row(bm)[0])
    np.testing.assert_array_equal(rows[1], body_measurements_row()[0])
    np.testing.assert_array_equal(rows[2], off_axis)                    # bone vectors off the x axis are kept as they are
    np.testing.assert_array_equal(rows[3], off_axis)
    table = np.stack([off_axis, body_measurements_row(bm)[0]])
    np.testing.assert_array_equal(body_measurements_rows(table, 2), table)
    np.testing.assert_array_equal(body_measurements_rows(table.astype(np.float32), 2), table.astype(np.float32))


@pytest.mark.parametrize("arg,n,match", [
    ([None, None], 3, "2 skeletons for 3 streams"),
    (np.zeros((4, 9)), 3, "4 skeletons"),
    ([np.zeros(8)], 1, "got 8"),
    ([np.zeros(10)], 1, "got 10"),
    ([None, [0, 0, 0, 0, 0, 0, 0, 0, np.nan]], 2, "stream 1 is not finite"),
    ([[np.inf] + [0.0] * 8], 1, "stream 0 is not finite"),
    ([BoneMap(left_upper_arm_origin_rh=[0.0, np.nan, 0.0])], 1, "not finite"),
])
def test_rows_refusals(arg, n, match):
    with pytest.raises(UserWarning, match=match):
        body_measurements_rows(arg, n)
