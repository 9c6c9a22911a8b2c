"""ctypes binding of libwmf_b200.so (include/wmf_b200.h). No torch types cross this boundary:
callers pass ``tensor.data_ptr()`` integers and the raw CUDA stream handle.

There is no CPU fallback. If the shared library is missing, or a compute entry point is
called without a B200-class device, this module raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# WMF_B200_LIB (development only): another build of the same sources, e.g. the -DWMF_WATCHDOG variant
LIB_PATH = os.environ.get("WMF_B200_LIB") or os.path.join(_HERE, "csrc", "libwmf_b200.so")

ALGO_AUTO, ALGO_SIMT, ALGO_TCGEN05, ALGO_TCGEN05_DIRECT = 0, 1, 2, 3
PREPROCESS_LOG, PREPROCESS_LINEAR = 0, 1
ERR_NAMES = {1: "INVALID", 2: "WORKSPACE", 3: "CUDA", 4: "NO_DEVICE", 5: "UNSUPPORTED"}
TOPK_MAX = 1024
KNN_SIMILARITIES = {"cosine": 0, "jaccard": 1, "conditional": 2}  # WMF_KNN_COSINE / _JACCARD / _CONDITIONAL
SLIM_K_MAX = 128   # longest candidate list wmf_slim_train keeps on chip

_p, _i64, _i32, _f32, _sz = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_float, ctypes.c_size_t
_f64 = ctypes.c_double

# name -> (restype, argtypes); mirrors include/wmf_b200.h one to one
SIGNATURES = {
    "wmf_last_error": (ctypes.c_char_p, []),
    "wmf_version": (_i32, []),
    "wmf_launch_count": (ctypes.c_longlong, []),
    "wmf_device_check": (_i32, [ctypes.POINTER(ctypes.c_int)]),
    "wmf_preprocess": (_i32, [_p, _i64, _i32, _f32, _f32, _p]),
    "wmf_csr_transpose_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "wmf_csr_transpose": (_i32, [_p, _p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _sz, _p]),
    "wmf_gram_workspace_bytes": (_sz, [_i64, _i32]),
    "wmf_gram": (_i32, [_p, _i64, _i32, _i64, _f32, _i32, _p, _p, _sz, _p]),
    "wmf_gram_block_rows": (_i64, [_i64]),
    "wmf_gram_blocks": (_i64, [_i64]),
    "wmf_gram_partials": (_i32, [_p, _i64, _i64, _i64, _i32, _i64, _i32, _p, _sz, _p]),
    "wmf_gram_reduce": (_i32, [_p, _i64, _i32, _f32, _p, _p]),
    "wmf_peer_broadcast": (_i32, [_p, _sz, _p, _i32, _i32, _sz, _p]),
    "wmf_als_half_step_workspace_bytes": (_sz, [_i64, _i64, _i32, _i32]),
    "wmf_als_dual_max_entries": (_i32, []),
    "wmf_als_half_step_status": (_i32, [_p, _p, _p, _p]),
    "wmf_als_half_step_used_fallback": (_i32, [_p, _p, _p]),
    "wmf_als_half_step_supports": (_i32, [_i32, _i32, _i32]),
    "wmf_rank_ahead": (_i32, [_p, _p, _p, _i64, _i64, _p, _p, _p, _i64, _p, _p]),
    "wmf_als_row_split_entries": (_i32, []),
    "wmf_als_half_step_workspace_bytes_split": (_sz, [_i64, _i64, _i32, _i32, _i64]),
    "wmf_als_half_step": (_i32, [_p, _p, _p, _i64, _i64, _p, _i64, _p, _i64, _i32, _p, _i32, _p, _i64, _i32, _p, _sz, _p]),
    "wmf_sddmm_loss_workspace_bytes": (_sz, [_i64]),
    "wmf_sddmm_loss": (_i32, [_p, _p, _p, _i64, _i64, _p, _i64, _p, _i64, _i32, _i32, _p, _p, _sz, _p]),
    "wmf_predict_pairs": (_i32, [_p, _i64, _p, _i64, _p, _i64, _p, _i64, _i32, _i32, _p, _p]),
    "wmf_score_topk_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "wmf_score_topk": (_i32, [_p, _i64, _p, _i64, _p, _i64, _p, _i64, _i32, _i32, _i32, _p, _p, _p, _sz, _p]),
    "wmf_score_topk_exclude_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "wmf_score_topk_exclude": (_i32, [_p, _i64, _p, _p, _i64, _p, _i64, _p, _i64, _i32, _i32, _i32, _p, _p, _p, _p, _sz,
                                      _p]),
    "wmf_topn_metrics_workspace_bytes": (_sz, [_i64, _i32]),
    "wmf_topn_metrics": (_i32, [_p, _i64, _i32, _p, _p, _p, _p, _p, _i32, _p, _p]),
    "wmf_topn_metrics_reduce": (_i32, [_p, _i64, _i32, _p, _p, _sz, _p]),
    "wmf_inverse_workspace_bytes": (_sz, [_i32]),
    "wmf_inverse": (_i32, [_p, _i32, _p, _p, _sz, _p]),
    "wmf_dense_right_multiply": (_i32, [_p, _i64, _i64, _p, _i32, _p, _i64, _p]),
    "wmf_spmm": (_i32, [_p, _p, _p, _i64, _p, _i64, _i32, _p, _i64, _p]),
    "wmf_ease_workspace_bytes": (_sz, [_i64]),
    "wmf_ease_train": (_i32, [_p, _p, _p, _i64, _i64, _f32, _p, _p, _sz, _p]),
    "wmf_ease_predict": (_i32, [_p, _p, _p, _p, _i64, _p, _i64, _p, _i64, _p, _p]),
    "wmf_ease_score_topk_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "wmf_ease_score_topk": (_i32, [_p, _p, _p, _p, _i64, _p, _i64, _p, _p, _i32, _p, _p, _p, _sz, _p]),
    "wmf_knn_train_workspace_bytes": (_sz, [_i64, _i32]),
    "wmf_knn_train": (_i32, [_p, _p, _i64, _p, _p, _i64, _i32, _i32, _f64, _p, _p, _p, _p, _sz, _p]),
    "wmf_knn_predict": (_i32, [_p, _p, _p, _p, _p, _p, _p, _i64, _p, _i64, _p, _p]),
    "wmf_knn_score_topk_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "wmf_knn_score_topk": (_i32, [_p, _p, _p, _p, _p, _p, _i64, _p, _i64, _p, _p, _i32, _p, _p, _p, _sz, _p]),
    "wmf_userknn_predict": (_i32, [_p, _p, _p, _p, _p, _p, _p, _i64, _p, _i64, _p, _p]),
    "wmf_userknn_score_topk_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "wmf_userknn_score_topk": (_i32, [_p, _p, _p, _p, _p, _p, _i64, _p, _i64, _p, _p, _i32, _p, _p, _p, _sz, _p]),
    "wmf_userknn_fold_in_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "wmf_userknn_fold_in": (_i32, [_p, _p, _i64, _p, _p, _i64, _p, _i64, _i32, _i32, _f64, _p, _p, _p, _p, _sz, _p]),
    "wmf_slim_train_workspace_bytes": (_sz, [_i64, _i32]),
    "wmf_slim_train": (_i32, [_p, _p, _i64, _p, _p, _i64, _p, _p, _i32, _f64, _f64, _i32, _f64, _p, _p, _p, _p, _p, _sz,
                              _p]),
    "wmf_rp3beta_train_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "wmf_rp3beta_train": (_i32, [_p, _p, _i64, _p, _p, _i64, _i64, _p, _p, _p, _i32, _p, _p, _p, _p, _sz, _p]),
}


class WMFLibraryError(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library (once). Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise WMFLibraryError(
            f"{LIB_PATH} is missing. Build it with `python -m recmodel_b200.build` "
            "(nvcc, sm_100a). recmodel_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library drifted apart
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    msg = load().wmf_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc, what):
    if rc != 0:
        raise WMFLibraryError(f"{what} failed: {ERR_NAMES.get(rc, rc)}: {last_error()}")


def require_device():
    """Raise unless an sm_100 device is current. Returns the SM count."""
    sms = ctypes.c_int(0)
    check(load().wmf_device_check(ctypes.byref(sms)), "wmf_device_check")
    return sms.value
