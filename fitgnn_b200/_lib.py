"""ctypes binding of libfitgnn_b200.so (C ABI declared in include/fitgnn.h).

There is no CPU fallback: if the shared library is missing the import fails loudly, and every entry point
that computes requires CUDA tensors.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FITGNN_B200_LIB", os.path.join(_HERE, "libfitgnn_b200.so"))  # override: kernel tuning only

c_i64, c_i32, c_void, c_size = C.c_int64, C.c_int, C.c_void_p, C.c_size_t


class FitgnnError(RuntimeError):
    pass


class PackStruct(C.Structure):
    _fields_ = [("n_rows", c_i64), ("nnz", c_i64), ("n_sub", c_i64), ("n_core", c_i64), ("n_src", c_i64),
                ("rowptr", c_void), ("col", c_void), ("dinv", c_void), ("gid", c_void), ("sub_ptr", c_void),
                ("core_rows", c_void), ("is_core", c_void), ("mask", c_void)]


class WeightsStruct(C.Structure):
    _fields_ = [("n_layers", C.c_int), ("in_features", C.c_int), ("hidden", C.c_int), ("n_classes", C.c_int),
                ("conv_weight", C.POINTER(c_void)), ("conv_bias", C.POINTER(c_void)), ("lt1_weight", c_void),
                ("lt1_bias", c_void)]


class PlanStruct(C.Structure):
    _fields_ = [("n_rows", c_i64), ("nnz", c_i64), ("n_sub", c_i64), ("n_core", c_i64), ("n_src", c_i64),
                ("fill_ws_bytes", c_i64), ("priv", c_i64 * 27)]


# name -> (restype, argtypes); every symbol include/fitgnn.h declares
SIGNATURES = {
    "fitgnn_abi_version": (c_i32, []),
    "fitgnn_last_error": (c_i32, [C.c_char_p, c_size]),
    "fitgnn_device_info": (c_i32, [C.POINTER(c_i32), C.POINTER(c_i32)]),
    "fitgnn_tuning_set": (c_i32, [C.c_char_p, c_i32]),
    "fitgnn_tuning_get": (c_i32, [C.c_char_p, C.POINTER(c_i32)]),
    "fitgnn_csr_workspace_bytes": (c_size, [c_i64, c_i64]),
    "fitgnn_csr_plan": (c_i32, [c_void, c_i64, c_i64, c_void, c_size, C.POINTER(c_i64), c_void]),
    "fitgnn_csr_fill": (c_i32, [c_i64, c_void, c_size, c_void, c_void, c_void, c_void]),
    "fitgnn_csr_raw_plan": (c_i32, [c_void, c_i64, c_i64, c_void, c_size, C.POINTER(c_i64), c_void]),
    "fitgnn_csr_raw_fill": (c_i32, [c_i64, c_void, c_size, c_void, c_void, c_void]),
    "fitgnn_pack_workspace_bytes": (c_size, [c_i64, c_i64, c_i64, c_i32, c_i64]),
    "fitgnn_pack_plan": (c_i32, [c_void, c_i64, c_i64, c_void, c_i64, c_i32, c_void, c_void, c_i64, c_void, c_size,
                                 C.POINTER(PlanStruct), c_void]),
    "fitgnn_pack_fill": (c_i32, [C.POINTER(PlanStruct), C.POINTER(PackStruct), c_void, c_size, c_void, c_size, c_void]),
    "fitgnn_spmm_symnorm": (c_i32, [c_void, c_void, c_void, c_void, c_i64, c_i32, c_void, c_void, c_i32, c_void, c_i64,
                                    c_void, c_void, c_i64, c_void]),
    "fitgnn_spmm_mean_concat": (c_i32, [c_void, c_void, c_void, c_i64, c_i32, c_i32, c_void, c_void, c_i32, c_void, c_i64,
                                        c_void, c_void, c_i64, c_void]),
    "fitgnn_spmm_mean_root": (c_i32, [c_void, c_void, c_void, c_i64, c_i32, c_i64, c_void, c_void, c_i32, c_void, c_i32,
                                      c_void, c_i64, c_void, c_void, c_i64, c_void]),
    "fitgnn_spmm_symnorm_grouped": (c_i32, [c_void, c_void, c_void, c_void, c_i64, c_i32, c_void, c_i64, c_i32, c_void,
                                            c_void, c_i64, c_i32, C.c_float, c_void]),
    "fitgnn_spmm_symnorm_grouped_f16": (c_i32, [c_void, c_void, c_void, c_void, c_i64, c_i32, c_void, c_i64, c_i32, c_void,
                                                c_i64, c_i32, C.c_float, c_void]),
    "fitgnn_spmm_symnorm_blocked": (c_i32, [c_void, c_void, c_void, c_void, c_i64, c_i32, c_void, c_void, c_i64, c_void,
                                            c_void, c_i32, c_void, c_void, c_i64, c_void]),
    "fitgnn_spmm_symnorm_mma": (c_i32, [c_void, c_void, c_void, c_void, c_i64, c_i32, c_void, c_void, c_i64, c_void,
                                        c_i32, c_void, c_void, c_i64, c_void]),
    "fitgnn_spmm_hubs": (c_i32, [c_void, c_void, c_i64, c_i32, c_void, c_void, c_i32, c_void]),
    "fitgnn_spmm_symnorm_hub": (c_i32, [c_void, c_void, c_void, c_void, c_i64, c_i32, c_void, c_void, c_i32, c_void,
                                        c_i64, c_void, c_void, c_i64, c_void, c_i32, c_i32, c_void]),
    "fitgnn_spmm_symnorm_devhub": (c_i32, [c_void, c_void, c_void, c_void, c_i64, c_i32, c_void, c_void, c_i32, c_void,
                                           c_i64, c_void, c_void, c_i64, c_void, c_void, c_i32, c_i32, c_void]),
    "fitgnn_gcn_forward_workspace_bytes": (c_size, [C.POINTER(PackStruct), C.POINTER(WeightsStruct), c_i32]),
    "fitgnn_gcn_forward": (c_i32, [C.POINTER(PackStruct), c_void, c_i64, C.POINTER(WeightsStruct), c_i32, c_i32, c_void,
                                   c_i64, c_void, c_size, c_void]),
    "fitgnn_gemm_tn_workspace_bytes": (c_size, [c_i64, c_i32, c_i32]),
    "fitgnn_gemm_tn": (c_i32, [c_void, c_i64, c_void, c_i64, c_i64, c_i32, c_i32, c_void, c_i64, c_void, c_size, c_void]),
    "fitgnn_dropout": (c_i32, [c_void, c_i64, c_i64, c_i32, C.c_float, C.c_uint64, C.c_uint64, c_void, c_i64, c_void]),
    "fitgnn_elu_dropout_backward": (c_i32, [c_void, c_i64, c_void, c_i64, c_i64, c_i32, c_i32, C.c_float, C.c_uint64,
                                            C.c_uint64, c_void, c_i64, c_void]),
    "fitgnn_adam_step": (c_i32, [c_void, c_void, c_void, c_void, c_i64, C.c_float, C.c_float, C.c_float, C.c_float,
                                 C.c_float, c_i64, c_void]),
    "fitgnn_spmm_symnorm_f16": (c_i32, [c_void, c_void, c_void, c_void, c_i64, c_i32, c_void, c_void, c_i32, c_void, c_i64,
                                        c_void, c_i64, c_void, c_void, c_i32, c_i32, c_void]),
    "fitgnn_split_f16": (c_i32, [c_void, c_i64, c_i64, c_i32, c_void, c_void, c_i64, c_void]),
    "fitgnn_gemm_f16": (c_i32, [c_void, c_i64, c_void, c_void, c_i64, c_void, c_void, c_i64, c_i32, c_i32, c_i32, c_i32, c_void,
                                c_i64, c_i32, c_void, c_void]),
    "fitgnn_gemm_f16_head_rows_peers": (c_i32, [c_void, c_i64, c_void, c_void, c_i64, c_void, c_i64, c_i32, c_i32, c_i32, c_i32,
                                                c_void, C.POINTER(c_void), c_i32, c_i64, c_void]),
    "fitgnn_gcn_transform_aggregate_f16": (c_i32, [c_i32, c_void, c_void, c_i64, c_void, c_void, c_i64, c_void, c_i64, c_i32,
                                                   c_i32, c_i32, c_void, c_void, c_i32, c_void, c_i64, c_void]),
    "fitgnn_gcn_conv_aligned_f16": (c_i32, [c_void, c_i64, c_void, c_void, c_i64, c_void, c_i64, c_i32, c_i32, c_i32, c_void, c_void,
                                            c_void, c_i64, c_void]),
    "fitgnn_gemm_bias_act": (c_i32, [c_i32, c_void, c_void, c_i64, c_void, c_void, c_i64, c_void, c_i64, c_i32, c_i32,
                                     c_i32, c_i32, c_void, c_i64, c_void]),
    "fitgnn_gemm_bias_act_split": (c_i32, [c_i32, c_void, c_void, c_i64, c_void, c_void, c_i64, c_void, c_i64, c_i32,
                                           c_i32, c_i32, c_i32, c_void, c_void, c_i64, c_void]),
    "fitgnn_gcn_layer_fused": (c_i32, [c_void, c_void, c_void, c_void, c_i64, c_i32, c_void, c_void, c_i64, c_void, c_void,
                                       c_i64, c_void, c_i32, c_i32, c_void, c_void, c_i64, c_void]),
    "fitgnn_pack_align_workspace_bytes": (c_size, [c_i64, c_i64]),
    "fitgnn_pack_align_plan": (c_i32, [C.POINTER(PackStruct), c_i32, c_i32, c_void, C.POINTER(c_i64), C.POINTER(c_i32),
                                       c_void, c_size, c_void]),
    "fitgnn_pack_align_fill": (c_i32, [C.POINTER(PackStruct), c_void, c_i32, c_i64, C.POINTER(PackStruct), c_void, c_void,
                                       c_void, C.POINTER(c_i32), c_void, c_size, c_void]),
    "fitgnn_gcn_transform_aggregate": (c_i32, [c_void, c_void, c_i64, c_void, c_void, c_i64, c_void, c_i64, c_i32, c_i32,
                                               c_i32, c_void, c_void, c_i32, c_void, c_void, c_i64, c_void]),
    "fitgnn_gemm_rowscale_bias_act_split": (c_i32, [c_i32, c_void, c_void, c_i64, c_void, c_void, c_i64, c_void, c_void, c_i64,
                                                    c_i32, c_i32, c_i32, c_i32, c_void, c_void, c_i64, c_void]),
    "fitgnn_gemm_head_rows": (c_i32, [c_void, c_void, c_i64, c_void, c_void, c_i64, c_void, c_i64, c_i32, c_i32, c_i32,
                                      c_i32, c_void, c_void, c_i64, c_void]),
    "fitgnn_gemm_head_rows_peers": (c_i32, [c_void, c_void, c_i64, c_void, c_void, c_i64, c_void, c_i64, c_i32, c_i32, c_i32,
                                            c_i32, c_void, C.POINTER(c_void), c_i32, c_i64, c_void]),
    "fitgnn_peer_push": (c_i32, [c_void, C.POINTER(c_void), c_i32, c_size, c_i32, c_void]),
    "fitgnn_peer_alloc": (c_i32, [c_size, C.POINTER(c_void), C.c_char_p]),
    "fitgnn_peer_open": (c_i32, [C.c_char_p, C.POINTER(c_void)]),
    "fitgnn_peer_close": (c_i32, [c_void]),
    "fitgnn_peer_free": (c_i32, [c_void]),
    "fitgnn_split_bf16": (c_i32, [c_void, c_i64, c_i64, c_i32, c_void, c_void, c_i64, c_void]),
    "fitgnn_segment_pool": (c_i32, [c_void, c_i64, c_i32, c_void, c_void, c_i64, c_i32, c_void, c_i64, c_void]),
    "fitgnn_group_workspace_bytes": (c_size, [c_i64, c_i64]),
    "fitgnn_group_by_part": (c_i32, [c_void, c_i64, c_i64, c_void, c_void, c_void, c_size, c_void]),
    "fitgnn_project_features": (c_i32, [c_void, c_void, c_i64, c_void, c_void, c_i64, c_i32, c_void, c_i64, c_void]),
    "fitgnn_project_adj_workspace_bytes": (c_size, [c_i64]),
    "fitgnn_project_adj_plan": (c_i32, [c_void, c_i64, c_i64, c_void, c_i64, c_void, c_size, C.POINTER(c_i64), c_void]),
    "fitgnn_project_adj_fill": (c_i32, [c_void, c_size, c_i64, c_void, c_void, c_void, c_void, c_void]),
    "fitgnn_sort_workspace_bytes": (c_size, [c_i64]),
    "fitgnn_sort_u64": (c_i32, [c_void, c_void, c_i64, c_i32, c_void, c_size, c_void]),
    "fitgnn_scan_i32": (c_i32, [c_void, c_void, c_i64, c_i32, c_void, c_size, c_void]),
    "fitgnn_scan_workspace_bytes": (c_size, [c_i64]),
}

_lib = None


def lib():
    """The loaded shared library (loaded once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FitgnnError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C fitgnn_b200/csrc`). fitgnn_b200 has no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError here = header/library mismatch
            fn.restype, fn.argtypes = res, args
        if handle.fitgnn_abi_version() != 1:
            raise FitgnnError("libfitgnn_b200.so ABI version mismatch")
        _lib = handle
    return _lib


def last_error() -> str:
    buf = C.create_string_buffer(512)
    lib().fitgnn_last_error(buf, 512)
    return buf.value.decode(errors="replace")


def set_tuning(name: str, value: int) -> int:
    """Set a kernel-tuning switch (include/fitgnn.h fitgnn_tuning_set); returns the previous value."""
    old = C.c_int(0)
    check(lib().fitgnn_tuning_get(name.encode(), C.byref(old)))
    check(lib().fitgnn_tuning_set(name.encode(), int(value)))
    return old.value


_CODES = {-1: "EINVAL", -2: "ECUDA", -3: "ERANGE", -4: "EWS", -5: "EUNSUP"}


def check(rc: int):
    if rc != 0:
        raise FitgnnError(f"fitgnn {_CODES.get(rc, rc)}: {last_error()}")


def ptr(t):
    """Device pointer of a CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise FitgnnError("fitgnn_b200 kernels take CUDA tensors only (there is no CPU path)")
    if not t.is_contiguous():
        raise FitgnnError("tensor must be contiguous")
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
