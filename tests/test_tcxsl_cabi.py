"""CPU: the H = 256 split-precision small-batch kernel (ape_mc_lstm_tcxsl, csrc/ape_lstm_tcxsl.cu) - its refusals, which all come before
the first CUDA call, its workspace query and its availability query.  The pointers are placeholders that are never dereferenced."""
import ctypes as C

import pytest

from arm_pose_estimation_b200 import _native as N

OK, BAD, UNSUP = N.APE_OK, N.APE_ERR_BAD_ARG, N.APE_ERR_UNSUPPORTED
ROWS = 128


def _args(**kw):
    a = N.LstmArgs()
    a.weights = a.preds = a.x_dense = a.weights_tc = a.weights_tcx = a.workspace = 256
    a.I, a.H, a.L, a.T, a.O = 22, 256, 2, 6, 14                  # the pocket model
    a.B, a.nF, a.n_samples = 1, 1, 100
    a.mask_mode, a.pred_ring = N.MASK_NONE, 1
    a.tc_flags = 5
    for k, v in kw.items():
        setattr(a, k, v)
    return a


CASES = [
    ("flags-3", dict(tc_flags=3), BAD),
    ("flags-0", dict(tc_flags=0), BAD),
    ("state", dict(n_samples=1, h0=512, c0=768), UNSUP),
    ("all-steps", dict(all_steps=1), UNSUP),
    ("layer-range-0-1", dict(layer_begin=0, layer_end=1), UNSUP),
    ("layer-range-1-2", dict(layer_begin=1, layer_end=2), UNSUP),
    ("H128", dict(H=128), UNSUP),
    ("H64", dict(H=64), UNSUP),
    ("L1", dict(L=1), UNSUP),
    ("L5", dict(L=5), UNSUP),
    ("O33", dict(O=33), UNSUP),
    ("T41", dict(T=41), UNSUP),
    ("I257", dict(I=257), UNSUP),
    ("rows-8193", dict(B=8193, n_samples=1), UNSUP),
    ("rows-65x128", dict(B=65, n_samples=128), UNSUP),
    ("frames-x-samples", dict(B=2, nF=33, n_samples=128, pred_ring=33), UNSUP),
    # a missing blob or workspace
    ("no-blob", dict(weights_tcx=None), BAD),
    ("no-workspace", dict(workspace=None), BAD),
    ("empty-no-workspace", dict(B=0, workspace=None), BAD),
    ("small-ws-E", dict(B=4, ws_E=2), BAD),
    # the kernel reads only the split blob; an empty call is done before the device
    ("empty", dict(B=0), OK),
    ("empty-no-single-pass-blob", dict(B=0, weights_tc=None), OK),
    ("empty-L4-T40-O32-I256", dict(B=0, L=4, T=40, O=32, I=256), OK),
    ("empty-L2-T1-I9", dict(B=0, L=2, T=1, I=9), OK),
]


@pytest.mark.parametrize("kw,want", [c[1:] for c in CASES], ids=[c[0] for c in CASES])
def test_tcxsl_refusals_before_the_device(kw, want):
    assert N.load().ape_mc_lstm_tcxsl(_args(**kw), None) == want


def test_tcxsl_null_args_are_refused():
    assert N.load().ape_mc_lstm_tcxsl(None, None) == BAD


def test_tcxsl_symbols_are_bound():
    lib = N.load()
    for name in ("ape_mc_lstm_tcxsl", "ape_mc_lstm_tcxsl_workspace_bytes", "ape_mc_lstm_tcxsl_max_active_clusters"):
        assert name in N.SYMBOLS and getattr(lib, name) is not None


def _query(I=22, H=256, L=2, T=6, O=14, E=1, n=100, out=True):
    v = C.c_uint64(0)
    rc = N.load().ape_mc_lstm_tcxsl_workspace_bytes(I, H, L, T, O, E, n, C.byref(v) if out else None)
    return rc, v.value


@pytest.mark.parametrize("kw,want", [
    (dict(out=False), BAD), (dict(T=0), BAD), (dict(E=-1), BAD), (dict(n=0), BAD),
    (dict(H=128), UNSUP), (dict(H=64), UNSUP), (dict(L=1), UNSUP), (dict(L=5), UNSUP), (dict(O=33), UNSUP), (dict(O=0), UNSUP),
    (dict(T=41), UNSUP), (dict(I=257), UNSUP), (dict(I=0), UNSUP), (dict(E=8193, n=1), UNSUP), (dict(E=65, n=128), UNSUP),
])
def test_tcxsl_workspace_query_refusals(kw, want):
    assert _query(**kw)[0] == want


@pytest.mark.parametrize("T", [1, 6, 8, 40])
@pytest.mark.parametrize("L", [2, 4])
def test_tcxsl_workspace_holds_every_cluster(T, L):
    last = 0
    for E, n in ((0, 1), (1, 1), (1, 100), (1, 128), (130, 1), (20, 14), (3, 100), (8, 128), (16, 128), (64, 128), (8192, 1)):
        rc, got = _query(L=L, T=T, E=E, n=n)
        assert rc == OK
        clusters = max(1, -(-E * n // ROWS))
        # per cluster: the exchange buffer [2 parities][hi | lo][32][128] and the sequences [2 layer parities][T][hi | lo][32][128]
        # of 16-byte units = (2 + 2T) x 128 KB, plus the slack that aligns the base to 256 bytes
        need = clusters * (2 + 2 * T) * 128 * 1024
        assert got >= need + 255, (E, n, got, need)
        assert got >= last                                   # grows with the rows
        last = got
    assert _query(L=L, T=T, E=64, n=128)[1] > _query(L=L, T=T, E=1, n=100)[1]
    # the query does not depend on the input width or the output count
    assert _query(I=9, L=L, T=T, O=32, E=3, n=100) == _query(I=256, L=L, T=T, O=1, E=3, n=100)


def test_existing_queries_keep_their_values():
    # the H = 128 kernel still refuses H = 256, through its query and through ape_mc_lstm_tc with tc_flags = 5
    v = C.c_uint64(0)
    assert N.load().ape_mc_lstm_tcxl_workspace_bytes(22, 256, 2, 6, 14, 1, 100, C.byref(v)) == UNSUP
    assert N.load().ape_mc_lstm_tc(_args(), None) == UNSUP
    # the split layer kernels' workspace at H = 256 is what it was before this kernel existed (their own layout, not the new
    # kernel's): the byte counts the query gave then, for the pocket (I22 T6 O14) and watch-only (I20 T8 O12) models
    for E, n, pocket, watch_only in ((1, 100, 87032320, 88080896), (16, 128, 87032320, 88080896), (1024, 100, 96469504, 100663808)):
        assert N.tcxs_workspace_bytes(22, 256, 2, 6, 14, E, n) == pocket
        assert N.tcxs_workspace_bytes(20, 256, 2, 8, 12, E, n) == watch_only
        assert N.split_workspace_bytes(22, 256, 2, 6, 14, E, n) == pocket
    assert N.tcxsl_workspace_bytes(22, 256, 2, 6, 14, 1, 100) == _query()[1]


def test_availability_query_without_a_device():
    lib = N.load()
    assert lib.ape_mc_lstm_tcxsl_max_active_clusters(None) == BAD
    n = C.c_int(-1)
    rc = lib.ape_mc_lstm_tcxsl_max_active_clusters(C.byref(n))
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        assert rc == OK and n.value >= 0
    else:
        assert rc != OK and n.value == 0                     # an error code, not a crash
