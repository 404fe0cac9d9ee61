"""ctypes binding of libsldm_sage.so (include/sldm_sage.h).

The library is the product: there is no CPU or PyTorch fallback.  If it is missing
this module raises at import time, loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SLDM_LIB_PATH: load another build of the same library (A/B timing of kernel variants); default is the in-tree build
LIB_PATH = os.environ.get("SLDM_LIB_PATH") or os.path.join(_HERE, "lib", "libsldm_sage.so")

OK, EINVAL, ESHAPE, ECUDA, EWORKSPACE, EUNSUPPORTED, ENODEVICE = range(7)
BWD_STAGE_LN, BWD_STAGE_DGRAD, BWD_STAGE_WGRAD, BWD_STAGE_GATHER, BWD_STAGE_ALL = 1, 2, 4, 8, 15
HUB_DEGREE = 256
HUB_CHUNK = 2048
CSR_SECTIONS = ("meta", "rowptr_dst", "col_src", "rowptr_src", "col_dst", "hub_dst", "hub_src", "total")

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build it with `python __graft_entry__.py` (or `make`) first. "
        "sldm_gnn_b200 has no CPU / PyTorch fallback for the SageBlock hot path."
    )

lib = C.CDLL(LIB_PATH)

_p = C.c_void_p
_i64 = C.c_int64
_i32 = C.c_int32
_f = C.c_float

_PROTOS = {
    "sldm_abi_version": (C.c_int, []),
    "sldm_last_error": (C.c_char_p, []),
    "sldm_launch_count": (_i64, []),
    "sldm_device_sm_count": (C.c_int, [C.POINTER(C.c_int)]),
    "sldm_csr_layout": (C.c_int, [_i64, _i64, C.POINTER(_i64)]),
    "sldm_csr_workspace_bytes": (_i64, [_i64, _i64]),
    "sldm_csr_build": (C.c_int, [_p, _i64, _i64, _p, _p, _i64, _p]),
    "sldm_csr_status_async": (C.c_int, [_p, _p, _p]),
    "sldm_csr_build_pairs": (C.c_int, [_p, _p, _i64, _i64, _p, _p, _i64, _p]),
    "sldm_segment_workspace_bytes": (_i64, [_i64, _i64, _i32]),
    "sldm_segment_reduce": (C.c_int, [_p, _i64, _i32, _p, _i64, _i32, _i32, _p, _p, _p, _i64, _p]),
    "sldm_sage_project_workspace_bytes": (_i64, [_i64, _i32, _i32]),
    "sldm_sage_project_forward": (C.c_int, [_p, _p, _i64, _i32, _i32, _p, _p, _p, _p, _p, _f, _f,
                                            _p, _p, _p, _p, _i64, _p]),
    "sldm_sage_layer_fwd_workspace_bytes": (_i64, [_i64, _i64, _i32, _i32]),
    "sldm_sage_layer_forward": (C.c_int, [_p, _i64, _i32, _i32, _p, _i64, _p, _p, _p, _p, _p, _f, _f,
                                          _p, _p, _p, _p, _p, _i64, _p]),
    "sldm_sage_layer_bwd_workspace_bytes": (_i64, [_i64, _i64, _i32, _i32]),
    "sldm_sage_layer_backward": (C.c_int, [_p, _p, _p, _p, _p, _i64, _i32, _i32, _p, _i64, _p, _p, _p, _p, _f,
                                           _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p]),
    "sldm_sage_layer_backward_stages": (C.c_int, [_p, _p, _p, _p, _p, _i64, _i32, _i32, _p, _i64, _p, _p, _p, _p, _f,
                                                  _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p, _i32]),
    "sldm_sage_bf16_supported": (C.c_int, [_i32, _i32]),
    "sldm_segment_mean_bf16": (C.c_int, [_p, _i64, _i32, _p, _i64, _p, _p, _i64, _p]),
    "sldm_sage_project_forward_bf16": (C.c_int, [_p, _p, _i64, _i32, _i32, _p, _p, _p, _p, _p, _f, _f,
                                                 _p, _p, _p, _p, _i64, _p]),
    "sldm_sage_layer_forward_bf16": (C.c_int, [_p, _i64, _i32, _i32, _p, _i64, _p, _p, _p, _p, _p, _f, _f,
                                               _p, _p, _p, _p, _p, _i64, _p]),
    "sldm_sage_layer_backward_bf16": (C.c_int, [_p, _p, _p, _p, _p, _i64, _i32, _i32, _p, _i64, _p, _p, _p, _p, _f,
                                                _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p, _i32]),
    "sldm_readout_workspace_bytes": (_i64, [_i64, _i32]),
    "sldm_readout_forward": (C.c_int, [_p, _i64, _i32, _p, _i64, _i64, _p, _p, _i64, _p]),
    "sldm_readout_backward": (C.c_int, [_p, _i64, _i32, _p, _p, _i64, _i64, _p, _i64, _p, _p, _i64, _p, _p, _i64, _p]),
    "sldm_concat_chunks": (C.c_int, [_p, _i64, _i64, _p, _p]),
    "sldm_collate_graph_index": (C.c_int, [_p, _p, _i64, _i64, _i64, _i64, _p, _p, _p]),
    "sldm_map_attention_workspace_bytes": (_i64, [_i64, _i32]),
    "sldm_map_attention_forward": (C.c_int, [_p, _i64, _p, _i64, _p, _i32, _i32, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p]),
    "sldm_map_grid_bytes": (_i64, [_i64]),
    "sldm_map_grid_build": (C.c_int, [_p, _i64, _p, _i64, _p]),
    "sldm_map_attention_forward_grid": (C.c_int, [_p, _i64, _p, _i64, _i64, _p, _i32, _i32, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p]),
    "sldm_map_attention_backward": (C.c_int, [_p, _i64, _p, _i64, _i32, _i32, _p, _p, _p, _p, _p, _p, _i32, _p, _i64,
                                              _p, _p, _p, _p, _p, _p, _i64, _p]),
    "sldm_edge_build_count": (C.c_int, [_p, _i64, _i32, _i32, _f, _p, _p, _p]),
    "sldm_edge_build_fill": (C.c_int, [_p, _i64, _i32, _i32, _f, _p, _i64, _p, _p, _p]),
    "sldm_gru_supported": (C.c_int, [_i32, _i32, _i32]),
    "sldm_gru_partial_rows": (_i64, [_i64]),
    "sldm_gru_partial_width": (_i64, [_i32]),
    "sldm_gru_forward": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p, _p, _p, _p, _p, _p]),
    "sldm_gru_backward": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p, _p, _p, _p, _p, _i64, _p]),
    "sldm_gru_wgrad_tiles": (_i64, [_i64, _i32]),
    "sldm_gru_wgrad": (C.c_int, [_p, _p, _i64, _i32, _i32, _p, _i64, _p]),
    "sldm_gru_stack_supported": (C.c_int, [_i32, _i32, _i32]),
    "sldm_gru_layer_forward": (C.c_int, [_p, _p, _i64, _i32, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, _p]),
    "sldm_gru_layer_backward": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p]),
    "sldm_gru_project_forward": (C.c_int, [_p, _i64, _i32, _p, _p, _p, _p]),
    "sldm_gru_project_backward": (C.c_int, [_p, _i64, _i32, _p, _p, _p]),
    "sldm_gru_wgrad_strided": (C.c_int, [_p, _p, _i64, _i64, _i32, _i32, _p, _i64, _p]),
    "sldm_gru_projected_supported": (C.c_int, [_i32, _i32]),
    "sldm_gru_input_project_forward": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p, _p, _p]),
    "sldm_gru_input_wgrad": (C.c_int, [_p, _p, _i64, _i32, _i32, _i32, _p, _i64, _p]),
    "sldm_sage_block_forward_host": (C.c_int, [_p, _p, _i64, _i64, C.POINTER(_i32), _i32, C.POINTER(_p), _f, _f, _p]),
    "sldm_sage_block_train_host": (C.c_int, [_p, _p, _i64, _i64, C.POINTER(_i32), _i32, C.POINTER(_p), _f, _f,
                                             _p, _p, _p, C.POINTER(_p)]),
}

EXPORTS = tuple(_PROTOS)

for _name, (_res, _args) in _PROTOS.items():
    _fn = getattr(lib, _name)  # AttributeError here == header and library disagree
    _fn.restype = _res
    _fn.argtypes = _args

if lib.sldm_abi_version() != 1:
    raise ImportError(f"{LIB_PATH}: ABI version {lib.sldm_abi_version()} != 1")


def last_error() -> str:
    msg = lib.sldm_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int) -> None:
    """Map a C return code to the Python exception the reference stack would raise."""
    if rc == OK:
        return
    msg = last_error() or f"libsldm_sage error {rc}"
    if rc == EINVAL:
        raise ValueError(msg)
    if rc == EUNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(msg)


def csr_layout(N: int, E: int) -> dict:
    out = (_i64 * 8)()
    check(lib.sldm_csr_layout(N, E, out))
    return {k: int(out[i]) for i, k in enumerate(CSR_SECTIONS)}
