"""ctypes binding of libscn_b200.so (C ABI declared in include/scn_b200.h).

This is the whole Python<->native boundary: torch supplies device memory
(``tensor.data_ptr()``) and the current stream, nothing else.  There is NO fallback: if
the library is missing or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SCN_B200_LIB") or os.path.join(_HERE, "lib", "libscn_b200.so")   # override: debug builds

SCN_F32, SCN_BF16 = 0, 1
COORD_CODES = {torch.int64: 0, torch.int32: 1, torch.float32: 2, torch.float64: 3}
PREC_FP32, PREC_BF16, PREC_TF32 = 0, 1, 2

_p, _i, _i64, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t

# name -> (restype, argtypes); mirrors include/scn_b200.h one to one
SIGNATURES = {
    "scn_version": (C.c_char_p, []),
    "scn_launch_count": (C.c_uint64, []),
    "scn_hash_capacity": (_i64, [_i64]),
    "scn_pack_coords_checked": (_i, [_p, _i, _i64, _i, _i, _p, _p, _p]),
    "scn_unpack_keys": (_i, [_p, _i64, _p, _p]),
    "scn_hash_build": (_i, [_p, _i64, _p, _p, _i64, _p]),
    "scn_hash_lookup": (_i, [_p, _i64, _p, _p, _i64, _p, _p]),
    "scn_input_rules_workspace": (_sz, [_i64]),
    "scn_input_layer_rules": (_i, [_p, _i64, _p, _p, _i64, _p, _p, _p, _p, _sz, _p]),
    "scn_subm_rulebook": (_i, [_p, _i64, _p, _p, _i64, _i, _i, _i, _p, _i64, _p]),
    "scn_strided_hash_workspace": (_sz, [_i64]),
    "scn_strided_rulebook_hash": (_i, [_p, _i64, _i, _i, _i, _p, _p, _i64, _p, _p, _p, _p, _p, _sz, _p]),
    "scn_strided_tables": (_i, [_p, _p, _i64, _i, _p, _i64, _p, _i64, _p]),
    "scn_rulebook_workspace": (_sz, [_i, _i64]),
    "scn_rulebook_count": (_i, [_p, _i, _i64, _i64, _p, _p]),
    "scn_rulebook_pairs": (_i, [_p, _i, _i64, _i64, _p, _p, _p, _p, _sz, _p]),
    "scn_conv_prep_weights": (_i, [_p, _i, _i, _i, _i, _i, _i, _i, _p, _p]),
    "scn_conv_prep_weights_batched": (_i, [_p, _i, _i64, _p]),
    "scn_conv_path": (_i, [_i, _i, _i, _i, _i]),
    "scn_conv_prep_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "scn_conv_forward": (_i, [_p, _i, _i64, _p, _i, _i64, _i64, _i, _i, _p, _p, _i, _p, _i, _p]),
    "scn_conv_wgrad": (_i, [_p, _i, _p, _i, _p, _i, _i64, _i64, _i, _i, _i, _p, _p]),
    "scn_col_sum_acc": (_i, [_p, _i, _i64, _i, _p, _p, _i, _p]),
    "scn_conv_module_forward": (_i, [_p, _i, _i64, _p, _i, _i64, _i64, _i, _i, _p, _p, _i, _p, _i, _p, _i, _p]),
    "scn_conv_module_backward_colsum": (_i, [_p, _i, _i64, _p, _i, _i64, _p, _i64, _p, _i64, _i, _i, _i, _p, _i, _i, _p, _i,
                                      _p, _p, _i, _p, _i, _p, _p, _p]),
    "scn_bn_forward": (_i, [_p, _i, _i64, _i, _p, _p, _p, _p, _i, _f, _f, _f, _p, _p, _p, _p, _p]),
    "scn_bn_backward_colsum": (_i, [_p, _p, _i, _i64, _i, _p, _p, _p, _p, _i, _f, _p, _p, _p, _p, _i, _p, _p]),
    "scn_leaky_forward": (_i, [_p, _i, _i64, _f, _p, _p]),
    "scn_leaky_backward": (_i, [_p, _p, _i, _i64, _f, _p, _p]),
    "scn_add_forward": (_i, [_p, _p, _i, _i64, _f, _p, _p]),
    "scn_input_layer_forward": (_i, [_p, _p, _i64, _i64, _i, _i, _p, _i, _p, _p]),
    "scn_rows_gather": (_i, [_p, _i, _p, _i64, _i, _p, _i, _p]),
    "scn_rows_scatter_add": (_i, [_p, _i, _p, _i64, _i, _p, _p]),
    "scn_pool_rows": (_i, [_p, _i, _i, _p, _i, _i64, _i64, _i, _f, _p, _p]),
    "scn_larcv_count": (_i, [_p, _i, _i, _i, _i, _f, _p, _p]),
    "scn_larcv_compact": (_i, [_p, _i, _i, _i, _i, _f, _p, _i, _p, _p, _p]),
    "scn_sparse_to_dense_forward": (_i, [_p, _i, _p, _i64, _i, _i, _i, _i, _i, _p, _p]),
    "scn_sparse_to_dense_backward": (_i, [_p, _p, _i64, _i, _i, _i, _i, _i, _p, _i, _p]),
}

_lib = None


def load(path: str = LIB_PATH):
    """Loads the shared library and binds every symbol; raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(path):
        raise RuntimeError(
            f"libscn_b200.so not found at {path}: build it with `python -m sparseeventid_b200.build` "
            "(there is no CPU or PyTorch fallback for the sparse-convolution path)")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def lib():
    return load()


class ScnError(RuntimeError):
    pass


def check(rc: int, what: str):
    if rc == 0:
        return
    if rc > 0:
        raise ScnError(f"{what}: CUDA error {rc}")
    names = {-1: "SCN_ERR_ARG", -2: "SCN_ERR_UNSUPPORTED", -3: "SCN_ERR_WORKSPACE"}
    raise ScnError(f"{what}: {names.get(rc, rc)}")


def dtype_code(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return SCN_F32
    if t.dtype == torch.bfloat16:
        return SCN_BF16
    raise ScnError(f"unsupported feature dtype {t.dtype}")


def ptr(t):
    if t is None:
        return None
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise ScnError(
            f"{what}: tensor is on {t.device}; the sparse-convolution path runs only on a CUDA device "
            "(no CPU fallback)")
