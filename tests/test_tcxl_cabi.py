"""CPU: the split-precision small-batch kernel (tc_flags = 5, csrc/ape_lstm_tcxl.cu) - the refusals of ape_mc_lstm_tc, which all come
before the first CUDA call, and its workspace query.  The pointers are placeholders that are never dereferenced."""
import ctypes as C

import pytest

from arm_pose_estimation_b200 import _native as N

OK, BAD, UNSUP = N.APE_OK, N.APE_ERR_BAD_ARG, N.APE_ERR_UNSUPPORTED
ROWS = 128


def _args(**kw):
    a = N.LstmArgs()
    a.weights = a.preds = a.x_dense = a.weights_tc = a.weights_tcx = a.workspace = 256
    a.I, a.H, a.L, a.T, a.O = 38, 128, 3, 6, 14
    a.B, a.nF, a.n_samples = 1, 1, 100
    a.mask_mode, a.pred_ring = N.MASK_NONE, 1
    a.tc_flags = 5
    for k, v in kw.items():
        setattr(a, k, v)
    return a


CASES = [
    ("state", dict(n_samples=1, h0=512, c0=768), UNSUP),
    ("all-steps", dict(all_steps=1), UNSUP),
    ("layer-range-0-1", dict(layer_begin=0, layer_end=1), UNSUP),
    ("layer-range-1-3", dict(layer_begin=1, layer_end=3), UNSUP),
    ("H64", dict(H=64), UNSUP),
    ("H256", dict(H=256), UNSUP),
    ("L1", dict(L=1), UNSUP),
    ("L5", dict(L=5), UNSUP),
    ("O17", dict(O=17), UNSUP),
    ("T41", dict(T=41), UNSUP),
    ("I129", dict(I=129), UNSUP),
    ("rows-8193", dict(B=8193, n_samples=1), UNSUP),
    ("rows-65x128", dict(B=65, n_samples=128), UNSUP),
    ("frames-x-samples", dict(B=2, nF=33, n_samples=128, pred_ring=33), UNSUP),
    # a missing blob or workspace
    ("no-blob", dict(weights_tcx=None), BAD),
    ("no-workspace", dict(workspace=None), BAD),
    ("empty-no-workspace", dict(B=0, workspace=None), BAD),
    ("small-ws-E", dict(B=4, ws_E=2), BAD),
    # the kernel reads only the split blob: no single-pass blob needed; an empty call is done before the device
    ("empty", dict(B=0), OK),
    ("empty-no-single-pass-blob", dict(B=0, weights_tc=None), OK),
    # the largest shapes it takes go on to the device (not reached here): an empty call of them returns OK
    ("empty-L4-T40-O16-I128", dict(B=0, L=4, T=40, O=16, I=128), OK),
    ("empty-L2-T1-I9", dict(B=0, L=2, T=1, I=9), OK),
]


@pytest.mark.parametrize("kw,want", [c[1:] for c in CASES], ids=[c[0] for c in CASES])
def test_tcxl_refusals_before_the_device(kw, want):
    assert N.load().ape_mc_lstm_tc(_args(**kw), None) == want


def test_tcxl_symbol_is_bound():
    assert "ape_mc_lstm_tcxl_workspace_bytes" in N.SYMBOLS and N.load().ape_mc_lstm_tcxl_workspace_bytes is not None


def _query(I=38, H=128, L=3, T=6, O=14, E=1, n=100, out=True):
    v = C.c_uint64(0)
    rc = N.load().ape_mc_lstm_tcxl_workspace_bytes(I, H, L, T, O, E, n, C.byref(v) if out else None)
    return rc, v.value


@pytest.mark.parametrize("kw,want", [
    (dict(out=False), BAD), (dict(T=0), BAD), (dict(E=-1), BAD), (dict(n=0), BAD),
    (dict(H=256), UNSUP), (dict(H=64), UNSUP), (dict(L=1), UNSUP), (dict(L=5), UNSUP), (dict(O=17), UNSUP), (dict(O=0), UNSUP),
    (dict(T=41), UNSUP), (dict(I=129), UNSUP), (dict(I=0), UNSUP), (dict(E=8193, n=1), UNSUP), (dict(E=65, n=128), UNSUP),
])
def test_tcxl_workspace_query_refusals(kw, want):
    assert _query(**kw)[0] == want


@pytest.mark.parametrize("T", [1, 6, 7, 40])
@pytest.mark.parametrize("L", [2, 4])
def test_tcxl_workspace_holds_every_cluster(T, L):
    H, KG = 128, 128 // 8
    last = 0
    for E, n in ((0, 1), (1, 1), (1, 100), (1, 128), (130, 1), (20, 14), (3, 100), (16, 128), (64, 128), (8192, 1)):   # rows ascending
        rc, got = _query(L=L, T=T, E=E, n=n)
        assert rc == OK
        clusters = max(1, -(-E * n // ROWS))
        # per cluster: the exchange buffer [2 parities][hi | lo][H/8][128] and the sequences [2 layer parities][T][hi | lo][H/8][128]
        # of 16-byte units, plus the slack that aligns the base to 256 bytes
        need = clusters * (2 * 2 + 2 * T * 2) * KG * ROWS * 16
        assert got >= need + 255, (E, n, got, need)
        assert got >= last                                   # grows with the rows
        last = got
    assert _query(L=L, T=T, E=64, n=128)[1] > _query(L=L, T=T, E=1, n=100)[1]
    # the query does not depend on the input width or the output count
    assert _query(I=9, L=L, T=T, O=16, E=3, n=100) == _query(I=128, L=L, T=T, O=1, E=3, n=100)


def test_existing_split_queries_keep_their_values():
    # the new kernel adds a query of its own: the split layer kernels' workspace is what it was (their own layout)
    for E, n in ((1, 100), (16, 128)):
        assert N.split_workspace_bytes(38, 128, 3, 6, 14, E, n) == N.tcx_workspace_bytes(38, 128, 3, 6, 14, E, n)
    assert N.tcxl_workspace_bytes(38, 128, 3, 6, 14, 1, 100) == _query()[1]
