"""ctypes binding of ``libape_b200.so`` - the C ABI declared in ``include/ape_b200.h``.

There is NO fallback: if the shared library is missing or a call returns non-zero, the product path fails
loudly.  Status codes become ``UserWarning`` raised as an exception, the way the reference signals errors
(``nn_models.py:202``, ``:385-387``).  Pointers are raw device addresses (``tensor.data_ptr()``); the library
allocates nothing and enqueues on the stream it is handed (``torch.cuda.current_stream().cuda_stream``).
"""
import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "lib" / "libape_b200.so"

APE_OK, APE_ERR_BAD_ARG, APE_ERR_UNSUPPORTED, APE_ERR_CUDA, APE_ERR_NO_SM100 = 0, 1, 2, 3, 4
KIND_WATCH_ONLY, KIND_POCKET, KIND_UARM = 0, 1, 2
LAYOUT_WATCH_ONLY, LAYOUT_WATCH_PHONE = 0, 1
TARGET_ORI_CAL_LARM_UARM, TARGET_ORI_CAL_LARM_UARM_HIPS, TARGET_ORI_POS_CAL_LARM_UARM_HIPS = 0, 1, 2
MASK_NONE, MASK_INJECTED, MASK_PHILOX = 0, 1, 2
PREC_FP32_FMA, PREC_TC = 0, 1
KSLICE = 16                      # csrc/ape_lstm_pack.h: APE_KSLICE

# every symbol include/ape_b200.h declares (tests/test_cabi.py checks the header against this list and the .so)
SYMBOLS = (
    "ape_abi_version", "ape_last_cuda_error", "ape_device_info", "ape_lstm_blob_floats", "ape_features", "ape_features_push",
    "ape_mc_lstm_workspace_bytes", "ape_mc_lstm_fma", "ape_mc_lstm_tc_supported", "ape_lstm_tc_blob_bytes",
    "ape_mc_lstm_tc_workspace_bytes", "ape_mc_lstm_tc_workspace_bytes_all_steps", "ape_mc_lstm_tc", "ape_mc_lstm_tc_launch_count", "ape_mc_lstm_tcx_supported", "ape_lstm_tcx_blob_bytes", "ape_mc_lstm_tcx_workspace_bytes", "ape_mc_lstm_tcx_workspace_bytes_all_steps", "ape_mc_lstm_tcxs_supported", "ape_lstm_tcxs_blob_bytes", "ape_mc_lstm_tcxs_workspace_bytes",
    "ape_mc_lstm_tcxs_workspace_bytes_all_steps", "ape_mc_lstm_tcxl_workspace_bytes", "ape_mc_lstm_tcxsl", "ape_mc_lstm_tcxsl_workspace_bytes",
    "ape_mc_lstm_tcxsl_max_active_clusters", "ape_philox_masks", "ape_ff_blob_floats", "ape_mc_ff", "ape_mc_ff_ring", "ape_dense_act", "ape_fk_reduce", "ape_fk_reduce_bodies", "ape_msg_from_est",
    "ape_pipeline_create", "ape_pipeline_destroy", "ape_pipeline_submit", "ape_pipeline_wait", "ape_pipeline_query", "ape_pipeline_sync",
    "ape_pipeline_fence", "ape_pipeline_stream", "ape_pipeline_set_bodies",
    "ape_selfcheck_philox", "ape_selfcheck_keep8", "ape_selfcheck_keep_flags", "ape_selfcheck_features", "ape_selfcheck_row_pose", "ape_selfcheck_tcs_schedule",
    "ape_selftest_umma", "ape_selftest_ffma_peak",
)


class LstmArgs(C.Structure):
    """``struct ape_lstm_args`` (include/ape_b200.h)."""
    _fields_ = [
        ("weights", C.c_void_p),
        ("I", C.c_int), ("H", C.c_int), ("L", C.c_int), ("T", C.c_int), ("O", C.c_int),
        ("dropout_p", C.c_float),
        ("x_dense", C.c_void_p),
        ("feat_ring_buf", C.c_void_p),
        ("feat_ring", C.c_int),
        ("B", C.c_int), ("nF", C.c_int), ("frame0", C.c_int),
        ("n_samples", C.c_int),
        ("mask_mode", C.c_int),
        ("masks", C.c_void_p),
        ("philox_seed", C.c_uint64),
        ("stream_id0", C.c_uint32),
        ("workspace", C.c_void_p),
        ("preds", C.c_void_p),
        ("pred_ring", C.c_int),
        ("all_steps", C.c_int),
        ("weights_tc", C.c_void_p),
        ("layer_ms", C.c_void_p),
        ("layer_begin", C.c_int), ("layer_end", C.c_int), ("ws_parity", C.c_int),
        ("trace", C.c_void_p),
        ("trace_layer", C.c_int),
        ("stream_frames", C.c_void_p),
        ("ws_E", C.c_int),
        ("tc_flags", C.c_int),
        ("h0", C.c_void_p),
        ("c0", C.c_void_p),
        ("reserve_sms", C.c_int),
        ("weights_tcx", C.c_void_p),
    ]


PIPELINE_MAX_SLOTS = 8
PIPE_INPUT_PENDING, PIPE_CALLER_WAITS, PIPE_D2H = 1, 2, 4


class PipelineDesc(C.Structure):
    """``struct ape_pipeline_desc`` (include/ape_b200.h)."""
    _fields_ = [
        ("layout", C.c_int), ("kind", C.c_int), ("normalize", C.c_int), ("ncols", C.c_int),
        ("xx_m", C.c_void_p),
        ("xx_s", C.c_void_p),
        ("raw", C.c_void_p),
        ("feats", C.c_void_p),
        ("feat_ring", C.c_int),
        ("lstm", LstmArgs),
        ("lane_workspace", C.c_void_p * 2),
        ("yy_m", C.c_void_p),
        ("yy_s", C.c_void_p),
        ("body9", C.c_void_p),
        ("target", C.c_int), ("smooth", C.c_int), ("emit_samples", C.c_int),
        ("B", C.c_int), ("nF_max", C.c_int), ("n_slots", C.c_int),
        ("out_dev", C.c_void_p * PIPELINE_MAX_SLOTS),
        ("raw_host", C.c_void_p * PIPELINE_MAX_SLOTS),
        ("out_host", C.c_void_p * PIPELINE_MAX_SLOTS),
        ("frames_dev", C.c_void_p * 4),
        ("frames_host", C.c_void_p * PIPELINE_MAX_SLOTS),
    ]


_lib = None


def lib_path():
    return Path(os.environ.get("APE_B200_LIB", LIB_PATH))


def load():
    """Load the shared library (once).  Raises RuntimeError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not path.exists():
        raise RuntimeError(f"{path} is missing - build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback for the estimation path)")
    lib = C.CDLL(str(path))
    vp, i32, u64, u32, f32 = C.c_void_p, C.c_int, C.c_uint64, C.c_uint32, C.c_float
    lib.ape_abi_version.restype = i32
    lib.ape_abi_version.argtypes = []
    lib.ape_last_cuda_error.restype = C.c_char_p
    lib.ape_last_cuda_error.argtypes = []
    lib.ape_device_info.restype = i32
    lib.ape_device_info.argtypes = [C.POINTER(i32)] * 4
    lib.ape_lstm_blob_floats.restype = i32
    lib.ape_lstm_blob_floats.argtypes = [i32, i32, i32, i32, C.POINTER(C.c_int64)]
    lib.ape_features.restype = i32
    lib.ape_features.argtypes = [vp, i32, i32, vp, vp, i32, vp, i32, i32, i32, vp, i32, vp]
    lib.ape_features_push.restype = i32
    lib.ape_features_push.argtypes = [vp, i32, vp, vp, i32, vp, i32, i32, vp, i32, vp]
    lib.ape_mc_lstm_workspace_bytes.restype = i32
    lib.ape_mc_lstm_workspace_bytes.argtypes = [i32, i32, i32, i32, i32, i32, i32, C.POINTER(u64)]
    lib.ape_mc_lstm_fma.restype = i32
    lib.ape_mc_lstm_fma.argtypes = [C.POINTER(LstmArgs), vp]
    lib.ape_mc_lstm_tc_supported.restype = i32
    lib.ape_mc_lstm_tc_supported.argtypes = [i32, i32, i32, i32]
    lib.ape_lstm_tc_blob_bytes.restype = i32
    lib.ape_lstm_tc_blob_bytes.argtypes = [i32, i32, i32, C.POINTER(C.c_int64)]
    lib.ape_mc_lstm_tc_workspace_bytes.restype = i32
    lib.ape_mc_lstm_tc_workspace_bytes.argtypes = [i32, i32, i32, i32, i32, i32, i32, C.POINTER(u64)]
    lib.ape_mc_lstm_tc_workspace_bytes_all_steps.restype = i32
    lib.ape_mc_lstm_tc_workspace_bytes_all_steps.argtypes = [i32, i32, i32, i32, i32, i32, i32, C.POINTER(u64)]
    lib.ape_mc_lstm_tc.restype = i32
    lib.ape_mc_lstm_tc.argtypes = [C.POINTER(LstmArgs), vp]
    lib.ape_mc_lstm_tc_launch_count.restype = i32
    lib.ape_mc_lstm_tc_launch_count.argtypes = [C.POINTER(LstmArgs), C.POINTER(i32)]
    lib.ape_mc_lstm_tcx_supported.restype = i32
    lib.ape_mc_lstm_tcx_supported.argtypes = [i32, i32, i32, i32]
    lib.ape_lstm_tcx_blob_bytes.restype = i32
    lib.ape_lstm_tcx_blob_bytes.argtypes = [i32, i32, i32, C.POINTER(C.c_int64)]
    lib.ape_mc_lstm_tcx_workspace_bytes.restype = i32
    lib.ape_mc_lstm_tcx_workspace_bytes.argtypes = [i32, i32, i32, i32, i32, i32, i32, C.POINTER(u64)]
    lib.ape_mc_lstm_tcx_workspace_bytes_all_steps.restype = i32
    lib.ape_mc_lstm_tcx_workspace_bytes_all_steps.argtypes = [i32, i32, i32, i32, i32, i32, i32, C.POINTER(u64)]
    lib.ape_mc_lstm_tcxs_supported.restype = i32
    lib.ape_mc_lstm_tcxs_supported.argtypes = [i32, i32, i32, i32]
    lib.ape_lstm_tcxs_blob_bytes.restype = i32
    lib.ape_lstm_tcxs_blob_bytes.argtypes = [i32, i32, i32, C.POINTER(C.c_int64)]
    lib.ape_mc_lstm_tcxs_workspace_bytes.restype = i32
    lib.ape_mc_lstm_tcxs_workspace_bytes.argtypes = [i32, i32, i32, i32, i32, i32, i32, C.POINTER(u64)]
    lib.ape_mc_lstm_tcxs_workspace_bytes_all_steps.restype = i32
    lib.ape_mc_lstm_tcxs_workspace_bytes_all_steps.argtypes = [i32, i32, i32, i32, i32, i32, i32, C.POINTER(u64)]
    lib.ape_mc_lstm_tcxl_workspace_bytes.restype = i32
    lib.ape_mc_lstm_tcxl_workspace_bytes.argtypes = [i32, i32, i32, i32, i32, i32, i32, C.POINTER(u64)]
    lib.ape_mc_lstm_tcxsl.restype = i32
    lib.ape_mc_lstm_tcxsl.argtypes = [C.POINTER(LstmArgs), vp]
    lib.ape_mc_lstm_tcxsl_workspace_bytes.restype = i32
    lib.ape_mc_lstm_tcxsl_workspace_bytes.argtypes = [i32, i32, i32, i32, i32, i32, i32, C.POINTER(u64)]
    lib.ape_mc_lstm_tcxsl_max_active_clusters.restype = i32
    lib.ape_mc_lstm_tcxsl_max_active_clusters.argtypes = [C.POINTER(i32)]
    lib.ape_philox_masks.restype = i32
    lib.ape_philox_masks.argtypes = [u64, u32, i32, i32, i32, i32, i32, i32, i32, f32, vp, vp]
    lib.ape_ff_blob_floats.restype = i32
    lib.ape_ff_blob_floats.argtypes = [i32, i32, i32, i32, C.POINTER(C.c_int64)]
    lib.ape_dense_act.restype = i32
    lib.ape_dense_act.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, vp]
    lib.ape_mc_ff.restype = i32
    lib.ape_mc_ff.argtypes = [vp, i32, i32, i32, i32, f32, vp, i32, i32, i32, vp, u64, u32, u32, vp, vp]
    lib.ape_mc_ff_ring.restype = i32
    lib.ape_mc_ff_ring.argtypes = [vp, i32, i32, i32, i32, i32, f32, vp, i32, i32, i32, i32, vp, i32, i32, vp, u64, u32, vp, i32, vp]
    lib.ape_fk_reduce.restype = i32
    lib.ape_fk_reduce.argtypes = [vp, i32, vp, vp, vp, i32, i32, i32, i32, i32, vp, i32, i32, vp, vp, vp, vp, vp, vp]
    lib.ape_fk_reduce_bodies.restype = i32
    lib.ape_fk_reduce_bodies.argtypes = [vp, i32, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, i32, i32, vp, vp, vp, vp, vp, vp]
    lib.ape_msg_from_est.restype = i32
    lib.ape_msg_from_est.argtypes = [vp, i32, vp, i32, i32, i32, vp, vp, vp]
    lib.ape_pipeline_create.restype = i32
    lib.ape_pipeline_create.argtypes = [C.POINTER(PipelineDesc), C.POINTER(vp)]
    lib.ape_pipeline_destroy.restype = i32
    lib.ape_pipeline_destroy.argtypes = [vp]
    lib.ape_pipeline_submit.restype = i32
    lib.ape_pipeline_submit.argtypes = [vp, vp, vp, i32, i32, vp, i32, vp, C.POINTER(i32)]
    lib.ape_pipeline_wait.restype = i32
    lib.ape_pipeline_wait.argtypes = [vp, i32]
    lib.ape_pipeline_query.restype = i32
    lib.ape_pipeline_query.argtypes = [vp, i32, C.POINTER(i32)]
    lib.ape_pipeline_sync.restype = i32
    lib.ape_pipeline_sync.argtypes = [vp]
    lib.ape_pipeline_fence.restype = i32
    lib.ape_pipeline_fence.argtypes = [vp, vp]
    lib.ape_pipeline_stream.restype = i32
    lib.ape_pipeline_stream.argtypes = [vp, i32, C.POINTER(vp)]
    lib.ape_pipeline_set_bodies.restype = i32
    lib.ape_pipeline_set_bodies.argtypes = [vp, vp, i32]
    # host self-check hooks: used by tests/ only
    lib.ape_selfcheck_philox.restype = i32
    lib.ape_selfcheck_philox.argtypes = [C.POINTER(u32), C.POINTER(u32), C.POINTER(u32)]
    lib.ape_selfcheck_keep8.restype = i32
    lib.ape_selfcheck_keep8.argtypes = [u64, u32, u32, u32, u32, u32, u32, f32, C.POINTER(u32)]
    lib.ape_selfcheck_keep_flags.restype = i32
    lib.ape_selfcheck_keep_flags.argtypes = [C.POINTER(u32), i32, u32, C.POINTER(u32)]
    lib.ape_selfcheck_features.restype = i32
    lib.ape_selfcheck_features.argtypes = [i32, i32, C.POINTER(f32), C.POINTER(C.c_double), C.POINTER(i32)]
    lib.ape_selfcheck_row_pose.restype = i32
    lib.ape_selfcheck_row_pose.argtypes = [i32, C.POINTER(C.c_double), C.POINTER(C.c_double), i32, C.POINTER(C.c_double), C.POINTER(i32)]
    lib.ape_selfcheck_tcs_schedule.restype = i32
    lib.ape_selfcheck_tcs_schedule.argtypes = [i32, i32, C.POINTER(u32), i32, C.POINTER(i32)]
    lib.ape_selftest_umma.restype = i32
    lib.ape_selftest_umma.argtypes = [vp, vp, vp, i32, i32, i32, vp]
    lib.ape_selftest_ffma_peak.restype = i32
    lib.ape_selftest_ffma_peak.argtypes = [vp, i32, i32, C.POINTER(f32), vp]
    _lib = lib
    return lib


_ERR_TEXT = {
    APE_ERR_BAD_ARG: "bad argument (null pointer or size out of range)",
    APE_ERR_UNSUPPORTED: "shape not supported by this kernel",
    APE_ERR_NO_SM100: "the current device is not compute capability 10.x",
}


def check(rc, what):
    """Raise ``UserWarning`` (as the reference does) when a C-ABI call did not return APE_OK."""
    if rc == APE_OK:
        return
    if rc == APE_ERR_CUDA:
        raise UserWarning(f"{what}: CUDA error: {load().ape_last_cuda_error().decode()}")
    raise UserWarning(f"{what}: {_ERR_TEXT.get(rc, f'status {rc}')}")


def ptr(t):
    """Device (or host) address of a tensor, ``None`` for ``None``."""
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def blob_floats(I, H, L, O):
    out = C.c_int64(0)
    check(load().ape_lstm_blob_floats(I, H, L, O, C.byref(out)), "ape_lstm_blob_floats")
    return out.value


def workspace_bytes(I, H, L, T, O, E, n, tensor_core=False, all_steps=False):
    out = C.c_uint64(0)
    if tensor_core and all_steps:
        check(load().ape_mc_lstm_tc_workspace_bytes_all_steps(I, H, L, T, O, E, n, C.byref(out)), "ape_mc_lstm_tc_workspace_bytes_all_steps")
    elif tensor_core:
        check(load().ape_mc_lstm_tc_workspace_bytes(I, H, L, T, O, E, n, C.byref(out)), "ape_mc_lstm_tc_workspace_bytes")
    else:
        check(load().ape_mc_lstm_workspace_bytes(I, H, L, T, O, E, n, C.byref(out)), "ape_mc_lstm_workspace_bytes")
    return out.value


def tc_supported(I, H, L, O):
    return bool(load().ape_mc_lstm_tc_supported(I, H, L, O))


def tcx_supported(I, H, L, O):
    return bool(load().ape_mc_lstm_tcx_supported(I, H, L, O))


def tcx_blob_bytes(I, H, L):
    out = C.c_int64(0)
    check(load().ape_lstm_tcx_blob_bytes(I, H, L, C.byref(out)), "ape_lstm_tcx_blob_bytes")
    return out.value


def tcx_workspace_bytes(I, H, L, T, O, E, n, all_steps=False):
    out = C.c_uint64(0)
    name = "ape_mc_lstm_tcx_workspace_bytes" + ("_all_steps" if all_steps else "")
    check(getattr(load(), name)(I, H, L, T, O, E, n, C.byref(out)), name)
    return out.value


def tcxs_supported(I, H, L, O):
    return bool(load().ape_mc_lstm_tcxs_supported(I, H, L, O))


def tcxs_blob_bytes(I, H, L):
    out = C.c_int64(0)
    check(load().ape_lstm_tcxs_blob_bytes(I, H, L, C.byref(out)), "ape_lstm_tcxs_blob_bytes")
    return out.value


def tcxs_workspace_bytes(I, H, L, T, O, E, n, all_steps=False):
    out = C.c_uint64(0)
    name = "ape_mc_lstm_tcxs_workspace_bytes" + ("_all_steps" if all_steps else "")
    check(getattr(load(), name)(I, H, L, T, O, E, n, C.byref(out)), name)
    return out.value


def split_supported(I, H, L, O):
    """A split-precision kernel (tc_flags = 3) takes this shape: ape_lstm_tcx.cu (H = 128) or ape_lstm_tcxs.cu (H = 256)."""
    return tcx_supported(I, H, L, O) or tcxs_supported(I, H, L, O)


def split_blob_bytes(I, H, L):
    return tcxs_blob_bytes(I, H, L) if H == 256 else tcx_blob_bytes(I, H, L)


def split_workspace_bytes(I, H, L, T, O, E, n, all_steps=False):
    """Workspace of a split-precision call; ``all_steps``: a call with per-step outputs (the model API)."""
    fn = tcxs_workspace_bytes if H == 256 else tcx_workspace_bytes
    return fn(I, H, L, T, O, E, n, all_steps)


def tcxl_workspace_bytes(I, H, L, T, O, E, n):
    """Workspace of a call on the split-precision small-batch kernel (tc_flags = 5: H = 128, L <= 4, T <= 40, E * n <= 8192 rows)."""
    out = C.c_uint64(0)
    check(load().ape_mc_lstm_tcxl_workspace_bytes(I, H, L, T, O, E, n, C.byref(out)), "ape_mc_lstm_tcxl_workspace_bytes")
    return out.value


def tcxsl_workspace_bytes(I, H, L, T, O, E, n):
    """Workspace of a call on the H = 256 split-precision small-batch kernel (ape_mc_lstm_tcxsl: L <= 4, T <= 40, O <= 32,
    E * n <= 8192 rows)."""
    out = C.c_uint64(0)
    check(load().ape_mc_lstm_tcxsl_workspace_bytes(I, H, L, T, O, E, n, C.byref(out)), "ape_mc_lstm_tcxsl_workspace_bytes")
    return out.value


def tcxsl_max_active_clusters():
    """16-CTA clusters of the H = 256 split-precision small-batch kernel the current device holds at once (0: it cannot run there)."""
    out = C.c_int(0)
    check(load().ape_mc_lstm_tcxsl_max_active_clusters(C.byref(out)), "ape_mc_lstm_tcxsl_max_active_clusters")
    return out.value


def tc_blob_bytes(I, H, L):
    out = C.c_int64(0)
    check(load().ape_lstm_tc_blob_bytes(I, H, L, C.byref(out)), "ape_lstm_tc_blob_bytes")
    return out.value
