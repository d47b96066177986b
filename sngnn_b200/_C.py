"""ctypes binding of libsng.so (include/sng.h).  No torch types cross the boundary: only raw device
pointers, sizes and the current CUDA stream handle.  There is NO fallback: if the library is missing the
import of any compute path raises, and every non-zero return code becomes a RuntimeError carrying
`sng_last_error()` (the reference raises ordinary Python exceptions from torch, SURVEY.md §8(b))."""
import ctypes
import os

import torch

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libsng.so")
_lib = None

_P, _I64, _I32, _F32, _SZ = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_float, ctypes.c_size_t
_U64 = ctypes.c_uint64

# name -> (restype, argtypes); mirrors include/sng.h one to one (tests/test_abi.py checks the symbol list)
SIGNATURES = {
    "sng_version": (_I32, []),
    "sng_last_error": (ctypes.c_char_p, []),
    "sng_device_info": (_I32, [_P, _P, _P]),
    "sng_set_debug_env": (_I32, [_I32]),
    "sng_rownorm_f32": (_I32, [_P, _I64, _I64, _I64, _P, _I64, _P, _I64, _P, _P]),
    "sng_edge_fwd_workspace_bytes": (_SZ, [_I64, _I64, _I32]),
    "sng_edge_fwd": (_I32, [_P, _I64, _I64, _I64, _I64, _I64, _P, _P, _P, _P, _I64, _P, _P, _I64, _P, _I64, _P, _SZ, _I32, _F32, _P, _I64,
                            _P, _P, _P, _P, _P, _I32, _P, _I64, _P, _P, _P, _P, _P]),
    "sng_edge_fwd_denom": (_I32, [_P, _I64, _I64, _I64, _I64, _I64, _P, _P, _P, _P, _I64, _P, _P, _I64, _P, _I64, _P, _SZ, _I32, _F32, _P,
                                  _I64, _P, _P, _P, _P, _P, _I32, _P, _I64, _P, _P, _P, _P, _I32, _P, _P]),
    "sng_edge_fwd_wide_workspace_bytes": (_SZ, [_I64, _I64, _I64, _I64]),
    "sng_edge_fwd_wide": (_I32, [_P, _I64, _I64, _I64, _I64, _I64, _P, _P, _I64, _P, _I64, _P, _P, _I64, _P, _I64, _P, _SZ, _I32, _I64,
                                 _F32, _P, _I64, _P, _I32, _P, _I32, _P, _I64, _P, _P, _P, _P, _I32, _P, _P]),
    "sng_edge_bwd_wide": (_I32, [_P, _P, _P, _I64, _I64, _I64, _I64, _I64, _I64, _P, _P, _P, _P, _P, _I64, _I64, _P, _P,
                                 _P, _P, _I64, _P, _P, _P, _P, _P, _P, _I64, _P, _I64, _P, _P, _I64, _P, _P]),
    "sng_bn_workspace_bytes": (_SZ, [_I64, _I64]),
    "sng_bn_fwd_stats": (_I32, [_P, _I64, _I64, _I64, _P, _P, _SZ, _P]),
    "sng_bn_fwd_apply": (_I32, [_P, _I64, _I64, _I64, _P, _I64, ctypes.c_double, _P, _P, _P, _P, _P, _I64, _P]),
    "sng_bn_bwd_stats": (_I32, [_P, _P, _I64, _I64, _I64, _I64, _P, _P, _P, _P, _SZ, _P]),
    "sng_bn_bwd_apply": (_I32, [_P, _P, _I64, _I64, _I64, _I64, _P, _I64, _P, _P, _P, _P, _I64, _P]),
    "sng_row_dropout_fwd": (_I32, [_P, _I64, _I64, _I64, _I64, _U64, _U64, _F32, _I32, _P, _I64, _P]),
    "sng_row_dropout_bwd": (_I32, [_P, _P, _I64, _I64, _I64, _I64, _I64, _U64, _U64, _F32, _I32, _P, _I64, _P]),
    "sng_lin_norm_supported": (_I32, [_I64, _I64]),
    "sng_lin_norm_fwd": (_I32, [_P, _I64, _I64, _I64, _P, _I64, _I64, _P, _P, _P, _P]),
    "sng_lin_bwd_supported": (_I32, [_I64, _I64]),
    "sng_lin_bwd_workspace_bytes": (_SZ, [_I64, _I64, _I64]),
    "sng_lin_bwd": (_I32, [_P, _I64, _P, _I64, _I64, _I64, _I64, _P, _I64, _P, _P, _SZ, _P]),
    "sng_edge_bwd": (_I32, [_P, _P, _P, _I64, _I64, _I64, _I64, _I64, _I64, _P, _P, _P, _P, _P, _I64, _I64, _I32, _P, _P, _P, _P,
                            _P, _P, _I64, _P, _P, _P, _P, _P, _P, _I64, _P, _I64, _P, _P, _I64, _P, _P]),
    "sng_edge_bwd_denom": (_I32, [_P, _P, _P, _I64, _I64, _I64, _I64, _I64, _I64, _P, _P, _P, _P, _P, _I64, _I64, _I32, _P, _P, _P, _P,
                                  _P, _P, _I64, _P, _P, _P, _P, _P, _P, _I64, _P, _I64, _P, _P, _I64, _P, _P, _P]),
    "sng_edge_agg_bwd": (_I32, [_P, _P, _P, _I64, _I64, _I64, _I64, _I64, _P, _P, _I32, _P, _P, _P, _P, _P, _P, _P, _P]),
    "sng_list_bwd": (_I32, [_P, _P, _P, _I64, _I64, _I64, _I64, _I64, _I64, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                            _P, _I64, _P, _P, _I64, _P, _P]),
    "sng_list_transpose_workspace_bytes": (_SZ, [_I64, _I64, _I64]),
    "sng_list_transpose": (_I32, [_P, _P, _I64, _I64, _I64, _P, _P, _P, _P, _SZ, _P]),
    "sng_list_agg_fwd": (_I32, [_P, _I64, _I64, _I64, _I32, _P, _P, _P, _P, _P, _I64, _P]),
    "sng_spmm_fwd": (_I32, [_P, _I64, _I64, _I64, _P, _P, _P, _P, _P, _P, _I64, _P]),
    "sng_pp_fuse_fwd": (_I32, [_P, _I64, _I64, _I64, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "sng_pp_beta_grad": (_I32, [_P, _P, _P, _I64, _P, _P, _P]),
    "sng_nll_loss_fwd": (_I32, [_P, _I64, _I64, _I64, _P, _P, _P, _P, _P]),
    "sng_nll_loss_bwd": (_I32, [_I64, _I64, _I64, _P, _P, _P, _P, _P]),
    "sng_knn_to_csr_workspace_bytes": (_SZ, [_I64]),
    "sng_knn_to_csr": (_I32, [_P, _P, _P, _I64, _I32, _P, _P, _P, _P, _SZ, _P]),
    "sng_pp_fuse_bwd": (_I32, [_P, _P, _P, _P, _I64, _I64, _I64, _P, _P, _P, _P, _P, _P, _P, _P]),
    "sng_segment_mean": (_I32, [_P, _P, _I64, _I64, _P, _P, _SZ, _P]),
    "sng_sddmm_dot": (_I32, [_P, _I64, _I64, _I64, _P, _P, _I64, _P, _P]),
    "sng_gemm_nt_f16": (_I32, [_P, _I64, _P, _I64, _I64, _I64, _I64, _P, _P, _P, _I64, _P]),
    "sng_simhist_f16": (_I32, [_P, _I64, _P, _I64, _I64, _I64, _I64, _I64, _F32, _F32, _I32, _P, _P]),
    "sng_sparse_col_cos": (_I32, [_P, _P, _P, _P, _P, _P, _I64, _P, _P]),
    "sng_class_sums_f64": (_I32, [_P, _P, _I64, _I64, _I64, _I32, _P, _P, _P]),
    "sng_graph_prepare_workspace_bytes": (_SZ, [_I64, _I64]),
    "sng_graph_prepare": (_I32, [_P, _I64, _I64, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "sng_simknn_workspace_bytes": (_SZ, [_I64, _I64, _I64, _I32]),
    "sng_simknn_build": (_I32, [_P, _P, _I64, _P, _P, _I64, _I64, _I64, _I64, _I64, _I32, _F32, _I32,
                                _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "sng_simknn_stage1": (_I32, [_P, _P, _I64, _I64, _I64, _I64, _I64, _I32, _F32, _I32, _P, _P, _P, _I32, _I32, _P,
                                 _P, _I32, _I32, _P, _P]),
    "sng_simknn_seed": (_I32, [_P, _P, _I64, _I64, _I64, _I64, _I32, _I32, _P, _P]),
    "sng_simknn_plan": (_I32, [_I64, _I64, _I64, _I32, _P]),
    "sng_simknn_wide_workspace_bytes": (_SZ, [_I64, _I64, _I64, _I64]),
    "sng_simknn_wide_count": (_I32, [_P, _P, _I64, _I64, _I64, _I64, _I64, _I64, _F32, _I32, _P, _P, _SZ, _P]),
    "sng_simknn_wide_select": (_I32, [_P, _P, _I64, _P, _P, _I64, _I64, _I64, _I64, _I64, _I64, _F32, _I32,
                                      _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
}


def lib_path():
    return _LIB_PATH


def lib():
    """Load libsng.so once.  Raises ImportError (loudly) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise ImportError(
                f"sngnn_b200: {_LIB_PATH} is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C sngnn_b200/csrc`.  There is no CPU fallback.")
        L = ctypes.CDLL(_LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def last_error():
    return lib().sng_last_error().decode()


def check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what} failed (rc={rc}): {last_error()}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


PARTIALS = 4096          # SNG_PARTIALS of include/sng.h
MAX_CHANNELS = 512       # SNG_MAX_CHANNELS of include/sng.h
MAX_TOPK = 64            # SNG_MAX_TOPK of include/sng.h: larger top_k take the per-edge form (sng_edge_fwd_wide)
KNN_MAX_TOPK = 64        # SNG_KNN_MAX_TOPK of include/sng.h: larger top_k take the wide all-pairs build (sng_simknn_wide_count)


def stream(t=None):
    """Current CUDA stream handle of the device that owns `t` (default: the current device)."""
    return ctypes.c_void_p(torch.cuda.current_stream(None if t is None else t.device).cuda_stream)


def call(name, anchor, *args):
    """Run the asynchronous entry point `name` on the device that owns the tensor `anchor`, on that device's current
    stream (the stream is always the last C argument), and raise on a non-zero return code.  The library launches on the
    CURRENT device, so the guard matters whenever the tensors do not live on it (model.to('cuda:1') without set_device)."""
    with torch.cuda.device(anchor.device):
        rc = getattr(lib(), name)(*args, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    check(rc, name)


def require_cuda(*tensors):
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("sngnn_b200 runs on CUDA tensors only (there is no CPU path); got a tensor on " + str(t.device))
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"sngnn_b200: tensors on different devices ({dev} and {t.device})")
