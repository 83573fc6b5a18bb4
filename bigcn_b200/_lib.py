"""ctypes binding of libbigcn_b200.so (include/bigcn_b200.h).

The library is the product; there is no CPU or PyTorch fallback.  Loading fails
loudly when the shared object is missing, and every compute call fails loudly
when no sm_100 device is present.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbigcn_b200.so")

H = 64
FLAG_EDGE_RANGE, FLAG_BATCH_ORDER, FLAG_ROOT_RANGE = 1, 2, 4
DEG_BY = {"target": 0, "source": 1}
GEMM_MODE = {"fp32": 0, "tf32": 1, "tf32x3": 2, "mixed": 3, "sparse": 4, "tf32x2": 5, "bf16": 6}
FLAG_X_NOT_SPARSE = 8
FLAG_X_CSR_RANGE = 16
FLAG_EDGE_WEIGHT = 32
DIR_TD, DIR_BU = 1, 2

c_f32p = C.c_void_p  # device pointers travel as integers
c_ptr = C.c_void_p


class Dims(C.Structure):
    _fields_ = [("N", C.c_int64), ("B", C.c_int64), ("K", C.c_int64), ("C", C.c_int64),
                ("E_td", C.c_int64), ("E_bu", C.c_int64)]


class BatchPtrs(C.Structure):
    _fields_ = [("x", c_ptr), ("edge_index", c_ptr), ("bu_edge_index", c_ptr), ("batch", c_ptr),
                ("rootindex", c_ptr), ("node_id_base", C.c_int64),
                ("x_ptr", c_ptr), ("x_col", c_ptr), ("x_val", c_ptr), ("prepared", c_ptr),
                ("td_edge_weight", c_ptr), ("bu_edge_weight", c_ptr)]


class Params(C.Structure):
    _fields_ = [(n, c_ptr) for n in ("td_w1", "td_b1", "td_w2", "td_b2",
                                     "bu_w1", "bu_b1", "bu_w2", "bu_b2", "fc_w", "fc_b")]


class Graph(C.Structure):
    _fields_ = [(n, c_ptr) for n in ("in_ptr", "in_idx", "out_ptr", "out_idx", "deg", "dis", "rowsum",
                                     "in_long", "out_long")]


class Opts(C.Structure):
    _fields_ = [("training", C.c_int32), ("p_drop", C.c_float), ("seed", C.c_uint64),
                ("deg_by", C.c_int32), ("gemm_mode", C.c_int32), ("dir_mask", C.c_int32),
                ("bwd_phase", C.c_int32), ("skip_wgrad_prep", C.c_int32), ("fused_tail", C.c_int32),
                ("seed_dev", c_ptr), ("dense_roots", C.c_int32), ("edge_grad", C.c_int32)]


class AsmWeights(C.Structure):
    _fields_ = [(n, c_ptr) for n in ("td_weight", "bu_weight", "edge_weight", "bu_edge_weight")]


class Ebgcn(C.Structure):
    _fields_ = [("N", C.c_int64), ("B", C.c_int64), ("K", C.c_int64), ("E", C.c_int64),
                ("h1", c_ptr), ("x", c_ptr), ("x_ptr", c_ptr), ("x_col", c_ptr), ("x_val", c_ptr),
                ("edge_index", c_ptr), ("edge_weight", c_ptr), ("batch", c_ptr),
                ("rootindex", c_ptr), ("node_ptr", c_ptr), ("bn_weight", c_ptr), ("bn_bias", c_ptr),
                ("running_mean", c_ptr), ("running_var", c_ptr), ("num_batches_tracked", c_ptr),
                ("momentum", C.c_float), ("eps", C.c_float), ("training", C.c_int32), ("deg_by", C.c_int32),
                ("w2", c_ptr), ("b2", c_ptr)]


class BigcnError(RuntimeError):
    pass


_SIGS = {
    "bigcn_last_error": (C.c_char_p, []),
    "bigcn_version": (C.c_int, []),
    "bigcn_join_internal_streams": (C.c_int, [c_ptr]),
    "bigcn_internal_stream": (c_ptr, []),
    "bigcn_device_ok": (C.c_int, []),
    "bigcn_graph_prep_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int64, C.c_int32]),
    "bigcn_graph_prep": (C.c_int, [C.c_int32, C.POINTER(c_ptr), C.POINTER(C.c_int64), C.c_int64, c_ptr,
                                   C.c_int64, C.c_int32, C.POINTER(Graph), c_ptr, c_ptr, c_ptr,
                                   C.c_size_t, c_ptr]),
    "bigcn_xw_scratch_floats": (C.c_size_t, [C.c_int64, C.c_int32]),
    "bigcn_xw": (C.c_int, [c_ptr, C.c_int64, C.c_int64, c_ptr, c_ptr, C.c_int64, c_ptr, C.c_int64, C.c_int32,
                           c_ptr, c_ptr]),
    "bigcn_xw_wgrad_scratch_floats": (C.c_size_t, [C.c_int64, C.c_int64, C.c_int32]),
    "bigcn_xw_wgrad": (C.c_int, [c_ptr, C.c_int64, C.c_int64, c_ptr, C.c_int32, c_ptr, c_ptr, C.c_int64, C.c_int32,
                                 c_ptr, c_ptr]),
    "bigcn_xsparse_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int64]),
    "bigcn_xw_sparse": (C.c_int, [c_ptr, C.c_int64, C.c_int64, c_ptr, c_ptr, C.c_int64, c_ptr, C.c_int64, C.c_int32,
                                  c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "bigcn_x_capture": (C.c_int, [c_ptr, C.c_int64, C.c_int64, C.c_int32, c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "bigcn_xw_wgrad_sparse": (C.c_int, [C.c_int64, C.c_int64, c_ptr, C.c_int32, c_ptr, c_ptr, C.c_int64, c_ptr,
                                        C.c_size_t, c_ptr]),
    "bigcn_xsparse_view": (C.c_int, [C.c_int64, C.c_int64, c_ptr, C.c_size_t] + [C.POINTER(c_ptr)] * 7),
    "bigcn_host_dense_to_csr": (C.c_int64, [c_ptr, C.c_int64, C.c_int64, c_ptr, c_ptr, c_ptr, C.c_int64, C.c_int32]),
    "bigcn_host_read_gbs": (C.c_double, [c_ptr, C.c_int64, C.c_int32, C.c_int32]),
    "bigcn_transpose_weight": (C.c_int, [c_ptr, C.c_int64, C.c_int64, C.c_int64, c_ptr, C.c_int64,
                                         C.c_int64, c_ptr]),
    "bigcn_long_ws_ints": (C.c_size_t, [C.c_int64]),
    "bigcn_propagate": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int64, C.c_int64, c_ptr, c_ptr, C.c_int64, c_ptr,
                                  C.c_int32, c_ptr, C.c_int64, c_ptr]),
    "bigcn_readout_scratch_floats": (C.c_size_t, [C.c_int64, C.c_int64]),
    "bigcn_readout": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int64, C.c_int64, c_ptr, C.c_int64, c_ptr, c_ptr,
                                c_ptr, c_ptr]),
    "bigcn_dropout_mask": (C.c_int, [C.c_uint64, C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.c_float,
                                     c_ptr, c_ptr]),
    "bigcn_gcnconv_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int64, C.c_int64]),
    "bigcn_gcnconv_forward": (C.c_int, [c_ptr, C.c_int64, C.c_int64, c_ptr, C.c_int64, c_ptr, c_ptr,
                                        C.c_int32, C.c_int32, c_ptr, c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "bigcn_gcnconv_backward": (C.c_int, [c_ptr, C.c_int64, C.c_int64, C.c_int64, c_ptr, c_ptr, c_ptr,
                                         C.c_int32, c_ptr, C.c_size_t, c_ptr]),
    "bigcn_gcnconv_csr_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int64, C.c_int64]),
    "bigcn_gcnconv_csr_scratch_bytes": (C.c_size_t, [C.c_int64, C.c_int64]),
    "bigcn_gcnconv_csr_forward": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int64, C.c_int64, c_ptr, C.c_int64, c_ptr, c_ptr,
                                            C.c_int32, c_ptr, c_ptr, c_ptr, C.c_size_t, c_ptr, C.c_size_t, c_ptr]),
    "bigcn_gcnconv_csr_backward": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int64, C.c_int64, C.c_int64, c_ptr, c_ptr, c_ptr,
                                             c_ptr, C.c_size_t, c_ptr, C.c_size_t, c_ptr]),
    "bigcn_features_workspace_bytes": (C.c_size_t, [C.POINTER(Dims)]),
    "bigcn_batch_prepare_bytes": (C.c_size_t, [C.POINTER(Dims)]),
    "bigcn_batch_prepare_edge_bytes": (C.c_size_t, [C.POINTER(Dims)]),
    "bigcn_batch_prepare": (C.c_int, [C.POINTER(Dims), C.POINTER(BatchPtrs), C.POINTER(Opts), c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "bigcn_batch_prepare_join": (C.c_int, [c_ptr]),
    "bigcn_features_forward": (C.c_int, [C.POINTER(Dims), C.POINTER(BatchPtrs), C.POINTER(Params),
                                         C.POINTER(Opts), c_ptr, c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "bigcn_features_backward": (C.c_int, [C.POINTER(Dims), C.POINTER(BatchPtrs), C.POINTER(Params),
                                          C.POINTER(Opts), c_ptr, C.POINTER(Params), c_ptr, C.c_size_t,
                                          c_ptr]),
    "bigcn_features_edge_workspace_bytes": (C.c_size_t, [C.POINTER(Dims), C.c_int32]),
    "bigcn_features_edge_grad": (C.c_int, [C.POINTER(Dims), C.POINTER(BatchPtrs), C.POINTER(Opts), c_ptr, c_ptr, c_ptr,
                                           C.c_size_t, c_ptr]),
    "bigcn_features_x_grad": (C.c_int, [C.POINTER(Dims), C.POINTER(Params), C.POINTER(Opts), c_ptr, c_ptr, c_ptr,
                                        c_ptr, C.c_size_t, c_ptr]),
    "bigcn_x_dgrad_scratch_floats": (C.c_size_t, [C.c_int64, C.c_int64, C.c_int32]),
    "bigcn_x_dgrad": (C.c_int, [c_ptr, C.c_int32, c_ptr, c_ptr, C.c_int64, C.c_int64, C.c_int64, c_ptr, c_ptr, c_ptr,
                                c_ptr]),
    "bigcn_features_x_grad_csr": (C.c_int, [C.POINTER(Dims), C.POINTER(BatchPtrs), C.POINTER(Opts), c_ptr, C.c_int64,
                                            c_ptr, C.c_size_t, c_ptr]),
    "bigcn_x_dgrad_csr_scratch_floats": (C.c_size_t, [C.c_int64, C.c_int32]),
    "bigcn_x_dgrad_csr": (C.c_int, [c_ptr, c_ptr, C.c_int64, C.c_int64, C.c_int64, c_ptr, C.c_int32, c_ptr, c_ptr,
                                    C.c_int64, c_ptr, c_ptr, c_ptr]),
    "bigcn_head_forward": (C.c_int, [c_ptr, C.c_int64, C.c_int64, c_ptr, c_ptr, c_ptr, c_ptr]),
    "bigcn_head_backward_scratch_floats": (C.c_size_t, [C.c_int64, C.c_int64]),
    "bigcn_head_backward": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int64, C.c_int64, c_ptr, c_ptr, c_ptr,
                                      c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "bigcn_head_train_scratch_floats": (C.c_size_t, [C.c_int64, C.c_int64]),
    "bigcn_head_train": (C.c_int, [c_ptr, c_ptr, C.c_int64, C.c_int64, C.c_int64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                   c_ptr, c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "bigcn_gcn_norm_weighted_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int64]),
    "bigcn_gcn_norm_weighted": (C.c_int, [c_ptr, C.c_int64, c_ptr, C.c_int64, C.c_int32, c_ptr, c_ptr, c_ptr, c_ptr,
                                          c_ptr, C.c_size_t, c_ptr]),
    "bigcn_gcnconv_weighted_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int64, C.c_int64]),
    "bigcn_gcnconv_weighted_forward": (C.c_int, [c_ptr, C.c_int64, C.c_int64, c_ptr, C.c_int64, c_ptr, c_ptr, c_ptr,
                                                 C.c_int32, C.c_int32, c_ptr, c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "bigcn_gcnconv_weighted_backward": (C.c_int, [c_ptr, C.c_int64, C.c_int64, c_ptr, C.c_int64, c_ptr, c_ptr, c_ptr,
                                                  c_ptr, c_ptr, c_ptr, c_ptr, C.c_int32, C.c_int32, c_ptr, C.c_size_t,
                                                  c_ptr]),
    "bigcn_ebgcn_conv2_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int64, C.c_int64, C.c_int64]),
    "bigcn_ebgcn_conv2_csr_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int64, C.c_int64, C.c_int64]),
    "bigcn_ebgcn_conv2_forward": (C.c_int, [C.POINTER(Ebgcn), c_ptr, c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "bigcn_ebgcn_conv2_backward": (C.c_int, [C.POINTER(Ebgcn), c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                             c_ptr, C.c_size_t, c_ptr]),
    "bigcn_dense_row_counts": (C.c_int, [c_ptr, C.c_int64, C.c_int64, c_ptr, c_ptr]),
    "bigcn_dense_row_counts_bf16": (C.c_int, [c_ptr, C.c_int64, C.c_int64, c_ptr, c_ptr]),
    "bigcn_dense_rows_to_csr": (C.c_int, [c_ptr, C.c_int64, C.c_int64, c_ptr, C.c_int64, c_ptr, c_ptr, c_ptr, C.c_int64,
                                          c_ptr, c_ptr]),
    "bigcn_readout_backward": (C.c_int, [c_ptr, C.c_int64, c_ptr, c_ptr, C.c_int64, C.c_int64, c_ptr, c_ptr]),
    "bigcn_colsum64_scratch_floats": (C.c_size_t, [C.c_int64]),
    "bigcn_colsum64": (C.c_int, [c_ptr, C.c_int64, c_ptr, c_ptr, c_ptr]),
    "bigcn_train_tail": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                   c_ptr, c_ptr, C.c_size_t, c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "bigcn_eval_counts": (C.c_int, [c_ptr, c_ptr, C.c_int64, C.c_int64, c_ptr, c_ptr, c_ptr]),
    "bigcn_nll_loss": (C.c_int, [c_ptr, c_ptr, C.c_int64, C.c_int64, C.c_int64, c_ptr, c_ptr, c_ptr]),
    "bigcn_assemble_batch": (C.c_int, [c_ptr] * 14 + [C.c_int64, C.c_int64, C.c_int64, C.c_uint64] + [c_ptr] * 9),
    "bigcn_assemble_batch_dense": (C.c_int, [c_ptr] * 10 + [C.c_int64, C.c_int64, C.c_int64, C.c_uint64] + [c_ptr] * 6
                                   + [C.c_int64, C.c_int32, c_ptr, c_ptr]),
    "bigcn_assemble_batch_weighted": (C.c_int, [c_ptr] * 14 + [C.c_int64, C.c_int64, C.c_int64, C.c_uint64]
                                      + [c_ptr] * 8 + [C.POINTER(AsmWeights), c_ptr]),
    "bigcn_assemble_batch_dense_weighted": (C.c_int, [c_ptr] * 10 + [C.c_int64, C.c_int64, C.c_int64, C.c_uint64]
                                            + [c_ptr] * 6 + [C.c_int64, C.c_int32, c_ptr, C.POINTER(AsmWeights), c_ptr]),
    "bigcn_dp_slice": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "bigcn_dp_reduce_adam": (C.c_int, [C.POINTER(c_ptr), C.POINTER(c_ptr), C.c_int32, C.c_int32, c_ptr, c_ptr,
                                       C.c_int64, c_ptr, c_ptr, C.c_int32, C.c_double, C.c_double, C.c_double,
                                       C.c_double, C.c_double, c_ptr, C.POINTER(c_ptr), C.POINTER(c_ptr), c_ptr]),
    "bigcn_dp_stage_chunk": (C.c_int64, [C.c_int64, C.c_int32]),
    "bigcn_adam_step": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int64, c_ptr, c_ptr, C.c_int32,
                                  C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, c_ptr,
                                  c_ptr]),
}

EXPORTS = tuple(_SIGS)
_lib = None


def lib() -> C.CDLL:
    """The loaded library; raises if it has not been built (python -m bigcn_b200.csrc.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BigcnError(
                f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` "
                "(nvcc, sm_100a).  bigcn_b200 has no CPU fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().bigcn_last_error().decode("utf-8", "replace")
        raise BigcnError(f"{what}: {msg}" if what else msg)


def require_device():
    """Fail loudly unless a B200-class (cc 10.x) device is current."""
    import torch
    if not torch.cuda.is_available():
        raise BigcnError("bigcn_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    if not lib().bigcn_device_ok():
        raise BigcnError("bigcn_b200 is built for sm_100a only; the current device is not cc 10.x")
