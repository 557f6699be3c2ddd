"""ctypes binding of libltgnn.so (the C ABI declared in include/ltgnn.h).

There is deliberately no fallback: if the shared library is missing or a call fails, a
``RuntimeError`` is raised.  Build with ``python -m leak_det_gnn_b200.build``.
"""
from __future__ import annotations

import ctypes
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint64, c_void_p
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libltgnn.so"

STATUS = {0: "LTGNN_OK", -1: "LTGNN_E_ARG", -2: "LTGNN_E_SHAPE", -3: "LTGNN_E_ALIGN", -4: "LTGNN_E_CUDA",
          -5: "LTGNN_E_UNSUPPORTED"}

SPMM_AUTO, SPMM_STAGED, SPMM_GATHER = 0, 1, 2

# name -> (restype, argtypes); mirrors include/ltgnn.h one to one (tests/test_abi.py checks
# that every symbol declared in the header is exported and listed here)
SIGNATURES = {
    "ltgnn_version": (c_int, []),
    "ltgnn_last_error": (c_size_t, [c_char_p, c_size_t]),
    "ltgnn_seed_source": (None, [c_void_p]),
    "ltgnn_graph_create": (c_int, [c_int, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, POINTER(c_void_p)]),
    "ltgnn_graph_destroy": (c_int, [c_void_p]),
    "ltgnn_graph_info": (c_int, [c_void_p, POINTER(c_int32), POINTER(c_int32), POINTER(c_int32), POINTER(c_int32)]),
    "ltgnn_spmm": (c_int, [c_void_p, c_int, c_int64, c_int32, c_void_p, c_void_p, c_int, c_void_p]),
    "ltgnn_spmm_ws_floats": (c_int64, [c_void_p]),
    "ltgnn_spmm_fused": (c_int, [c_void_p, c_int, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_int, c_float,
                                 c_uint64, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_spmm_fused_vals": (c_int, [c_void_p, c_int, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_int64, c_int,
                                      c_void_p, c_int, c_float, c_uint64, c_void_p, c_float, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p]),
    "ltgnn_edge_norm_fwd": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p]),
    "ltgnn_edge_norm_bwd": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_gcn_adj_grad": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p,
                                   c_int, c_void_p, c_void_p]),
    "ltgnn_edge_mask_fwd": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_edge_mask_bwd": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_explain_step": (c_int, [c_int, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_double, c_double, c_double, c_double, c_float, c_float, c_int,
                                   c_void_p]),
    "ltgnn_pg_edge_fwd": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_float, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_pg_edge_bwd_ws_floats": (c_int64, [c_int]),
    "ltgnn_pg_edge_bwd": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p]),
    "ltgnn_linear": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p,
                             c_float, c_void_p, c_void_p]),
    "ltgnn_wgrad_ws_floats": (c_int64, [c_int, c_int32, c_int32]),
    "ltgnn_wgrad": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "ltgnn_node_init_fwd": (c_int, [c_int, c_int64, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_float, c_uint64, c_void_p, c_void_p, c_void_p]),
    "ltgnn_node_init_ws_floats": (c_int64, [c_int, c_int64, c_int32, c_int32, c_int32]),
    "ltgnn_node_init_bwd": (c_int, [c_int, c_int64, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p]),
    "ltgnn_node_init_bwd_from_layer": (c_int, [c_int, c_int64, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p,
                                               c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p,
                                               c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_gcn_layer_supported": (c_int, [c_void_p, c_int32, c_int32]),
    "ltgnn_gcn_layer_fwd": (c_int, [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_int, c_float,
                                    c_uint64, c_void_p, c_void_p, c_void_p]),
    "ltgnn_pipe_head_fwd": (c_int, [c_int, c_int64, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_float, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_pipe_head_dx_ws_floats": (c_int64, [c_int, c_int32, c_int32]),
    "ltgnn_pipe_head_bwd_dx": (c_int, [c_int, c_int64, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p,
                                       c_void_p]),
    "ltgnn_mean_pool_fwd": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "ltgnn_mean_pool_bwd_fill": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "ltgnn_tgrad_ws_floats": (c_int64, [c_int, c_int32]),
    "ltgnn_wgrad_tc": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "ltgnn_pipe_head_bwd_w": (c_int, [c_int, c_int64, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p]),
    "ltgnn_pipe_head_ws_floats": (c_int64, [c_int]),
    "ltgnn_tcn_ws_floats": (c_int64, [c_int32]),
    "ltgnn_tcn_conv": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_float, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_tcn_conv_train": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_float, c_void_p, c_void_p, c_float, c_uint64, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p]),
    "ltgnn_tcn_ln_bwd_ws_floats": (c_int64, [c_int]),
    "ltgnn_tcn_ln_bwd": (c_int, [c_int, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
                                 c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_tcn_wgrad": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                c_void_p]),
    "ltgnn_pipe_feat_fwd": (c_int, [c_int, c_int64, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_head_out_fwd": (c_int, [c_int, c_int64, c_int32, c_void_p, c_void_p, c_float, c_uint64, c_void_p, c_void_p]),
    "ltgnn_head_out_ws_floats": (c_int64, [c_int, c_int32]),
    "ltgnn_head_out_bwd": (c_int, [c_int, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p]),
    "ltgnn_head_wide_finish": (c_int, [c_int, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p]),
    "ltgnn_pipe_feat_bwd": (c_int, [c_int, c_int64, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_gru_fwd": (c_int, [c_int, c_int64, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                              c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_gru_bwd_dg_hn": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p]),
    "ltgnn_gru_ws_floats": (c_int64, [c_int]),
    "ltgnn_gru_bwd_w": (c_int, [c_int, c_int64, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_gru_bwd_dx": (c_int, [c_int, c_int64, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_void_p]),
    "ltgnn_gru_layer_fwd": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p]),
    "ltgnn_gru_layer_fwd_train": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_void_p, c_void_p]),
    "ltgnn_gru_layer_bwd": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p]),
    "ltgnn_gru_dropout": (c_int, [c_int, c_int64, c_int32, c_void_p, c_float, c_uint64, c_void_p, c_void_p, c_void_p]),
    "ltgnn_gru_dropout_bwd": (c_int, [c_int, c_int64, c_int32, c_void_p, c_int32, c_void_p, c_float, c_void_p, c_void_p]),
    "ltgnn_gru_sensor_fwd": (c_int, [c_int, c_int64, c_int32, c_int32, c_int64, c_int64, c_int32, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_gru_resident_tiles": (c_int, [c_int, c_void_p]),
    "ltgnn_gru_sensor_bwd_dx": (c_int, [c_int, c_int64, c_int32, c_int32, c_int32, c_int64, c_int64, c_int32, c_void_p,
                                        c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_gru_layer_fwd_windows": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_int64, c_void_p, c_void_p,
                                            c_void_p, c_void_p, c_void_p, c_void_p]),
    "ltgnn_row_gather_sum": (c_int, [c_int, c_int64, c_int32, c_int32, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                     c_int64, c_void_p]),
}

_lib = None


class LtgnnError(RuntimeError):
    def __init__(self, code: int, message: str) -> None:
        super().__init__(f"{STATUS.get(code, code)}: {message}")
        self.code = code


def load() -> ctypes.CDLL:
    """Load (once) and return the library.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA extension has not been built "
                "(run `python -m leak_det_gnn_b200.build`).  There is no CPU fallback.")
        lib = ctypes.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error() -> str:
    buf = ctypes.create_string_buffer(512)
    load().ltgnn_last_error(buf, 512)
    return buf.value.decode(errors="replace")


def check(code: int) -> None:
    if code != 0:
        raise LtgnnError(code, last_error())
