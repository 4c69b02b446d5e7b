"""CPU: the size and shape queries of the tensor-core LSTM kernels, and the refusals of the small-batch cluster kernel that come before
the first CUDA call.

- Every blob, workspace and support query (tc, tcx, tcxs, tcxl, tcxsl, both `_all_steps` forms) answers a grid of shapes, refused ones
  included, exactly as recorded in tests/golden/lstm_queries.json (`PYTHONPATH=. python tests/test_lstm_queries_cabi.py` rewrites that
  file from the library APE_B200_LIB names).
- ape_mc_lstm_tc with tc_flags = 4 refuses the shapes the cluster kernel does not take with APE_ERR_UNSUPPORTED, without a device.
- The tc workspace holds the cluster kernel's buffers for every call of up to 8192 rows: BatchedEstimator sizes its workspace for the
  small-batch path by this query alone.
"""
import ctypes as C
import itertools
import json
from pathlib import Path

import pytest

from arm_pose_estimation_b200 import _native as N

GOLDEN = Path(__file__).resolve().parent / "golden" / "lstm_queries.json"
OK, BAD, UNSUP = N.APE_OK, N.APE_ERR_BAD_ARG, N.APE_ERR_UNSUPPORTED

BLOB = ("ape_lstm_tc_blob_bytes", "ape_lstm_tcx_blob_bytes", "ape_lstm_tcxs_blob_bytes")
SUPPORTED = ("ape_mc_lstm_tc_supported", "ape_mc_lstm_tcx_supported", "ape_mc_lstm_tcxs_supported")
WORKSPACE = ("ape_mc_lstm_tc_workspace_bytes", "ape_mc_lstm_tc_workspace_bytes_all_steps", "ape_mc_lstm_tcx_workspace_bytes",
             "ape_mc_lstm_tcx_workspace_bytes_all_steps", "ape_mc_lstm_tcxs_workspace_bytes", "ape_mc_lstm_tcxs_workspace_bytes_all_steps",
             "ape_mc_lstm_tcxl_workspace_bytes", "ape_mc_lstm_tcxsl_workspace_bytes")

I_SET, H_SET, L_SET, O_SET = (0, 1, 9, 22, 38, 128, 129, 256, 257), (0, 32, 64, 96, 128, 256, 512), (0, 1, 2, 3, 4, 5), (0, 1, 12, 16, 17, 20, 21, 32, 33)


def _workspace_shapes():
    """(I, H, L, T, O, E, n, out): accepted shapes around every limit, then one argument at a time out of range"""
    for H, L, T, E, n in itertools.product((64, 128, 256), (2, 3, 4, 5), (1, 8, 40, 41), (0, 1, 511, 512, 8192, 8193), (1, 100, 128)):
        yield (22, H, L, T, 12, E, n, True)
    for H in (128, 256):
        base = dict(I=22, H=H, L=3, T=6, O=12, E=1, n=100, out=True)
        for k, vals in dict(I=(0, 129, 257), H=(0, 32, 100, 512), L=(0, 1), T=(0, -1), O=(0, 17, 21, 33), E=(-1,), n=(0,),
                            out=(False,)).items():
            for v in vals:
                yield tuple({**base, k: v}.values())


def answers(lib):
    """every query over its grid: the byte count of an accepted shape, minus the return code of a refused one (support: 0 / 1)"""
    res = {}
    for name in BLOB:
        fn, got = getattr(lib, name), []
        for I, H, L in itertools.product(I_SET, H_SET, L_SET):
            v = C.c_int64(0)
            rc = fn(I, H, L, C.byref(v))
            got.append(v.value if rc == OK else -rc)
        got.append(-fn(22, 128, 3, None))
        res[name] = got
    for name in SUPPORTED:
        fn = getattr(lib, name)
        res[name] = [int(fn(I, H, L, O)) for I, H, L, O in itertools.product(I_SET, H_SET, L_SET, O_SET)]
    for name in WORKSPACE:
        fn, got = getattr(lib, name), []
        for I, H, L, T, O, E, n, out in _workspace_shapes():
            v = C.c_uint64(0)
            rc = fn(I, H, L, T, O, E, n, C.byref(v) if out else None)
            got.append(v.value if rc == OK else -rc)
        res[name] = got
    return res


@pytest.mark.parametrize("name", BLOB + SUPPORTED + WORKSPACE)
def test_query_answers_match_the_record(name):
    want = json.loads(GOLDEN.read_text())[name]
    got = answers(N.load())[name]
    assert len(got) == len(want)
    bad = [i for i, (g, w) in enumerate(zip(got, want)) if g != w]
    assert not bad, f"{name}: {len(bad)} answers differ, first at grid index {bad[0]}: {got[bad[0]]} != {want[bad[0]]}"


def _args(**kw):
    a = N.LstmArgs()
    a.weights = a.preds = a.x_dense = a.weights_tc = a.weights_tcx = a.workspace = 256
    a.I, a.H, a.L, a.T, a.O = 22, 128, 3, 6, 12
    a.B, a.nF, a.n_samples = 1, 1, 100
    a.mask_mode, a.pred_ring = N.MASK_NONE, 1
    a.tc_flags = 4
    for k, v in kw.items():
        setattr(a, k, v)
    return a


@pytest.mark.parametrize("kw,want", [
    (dict(all_steps=1), UNSUP),
    (dict(L=5), UNSUP),
    (dict(H=64), UNSUP),
    (dict(layer_begin=0, layer_end=2), UNSUP),
    (dict(B=8193, n_samples=1), UNSUP),
    (dict(B=65, n_samples=128), UNSUP),
    (dict(L=5, layer_begin=2, layer_end=1), BAD),         # an invalid layer range is a bad argument before it is an unsupported shape
], ids=["all-steps", "L5", "H64", "layer-range", "rows-8193", "rows-65x128", "bad-layer-range-L5"])
def test_small_batch_refusals_before_the_device(kw, want):
    assert N.load().ape_mc_lstm_tc(_args(**kw), None) == want


ROWS = 128
SCRATCH_REGION = 160 * ROWS * 256 * 4      # per-CTA cell state of 160 CTAs: the H = 256 streamed-weights kernel, the H = 128 wavefront kernel


@pytest.mark.parametrize("H", (128, 256))
@pytest.mark.parametrize("T", (1, 6, 8, 40))
@pytest.mark.parametrize("L", (2, 3, 4))
def test_tc_workspace_holds_every_cluster(H, T, L):
    scratch = SCRATCH_REGION if H == 256 or L >= 3 else 0
    cluster = (2 + 2 * T) * (H // 8) * ROWS * 16           # exchange buffer of h_t [2] + layer sequences [2][T], fp16 units
    for E, n in ((1, 1), (1, 100), (2, 100), (1, 128), (64, 100), (64, 128), (81, 100), (8191, 1), (8192, 1), (1, 8192)):
        v = C.c_uint64(0)
        assert N.load().ape_mc_lstm_tc_workspace_bytes(22, H, L, T, 12, E, n, C.byref(v)) == OK
        clusters = -(-E * n // ROWS)
        assert v.value >= 255 + 2 * scratch + clusters * cluster, (E, n)


if __name__ == "__main__":
    GOLDEN.write_text(json.dumps(answers(N.load()), separators=(",", ":")) + "\n")
    print("wrote", GOLDEN, "from", N.lib_path())
