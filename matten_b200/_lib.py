"""
ctypes binding of the C ABI in include/matten_b200.h.

There is deliberately no fallback: if the shared library cannot be loaded (or
built), importing the compute path raises.  On a machine without an sm_100 GPU the
library loads (so symbols can be checked) but every compute call returns MT_EARCH.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libmatten_b200.so")

MT_F32, MT_F64 = 0, 1
MT_MAX_MLP_LAYERS = 6
FLAG_BAD_SPECIES, FLAG_BAD_INDEX, FLAG_UNSORTED = 1, 2, 4

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)


MT_TC_MAX_PARTS = 4
MT_TC_MAX_BI = 64


class ConvTcPartStruct(C.Structure):
    """mt_conv_tc_part"""
    _fields_ = [
        ("num_tiles", C.c_int32), ("a_rows", C.c_int32), ("num_bi", C.c_int32), ("x_lo", C.c_int32), ("x_cols", C.c_int32),
        ("lmax", C.c_int32), ("cost", C.c_int32), ("q_count", C.c_int32 * 4),
        ("row_wcol", C.c_void_p), ("bi_hdr", C.c_void_p), ("bi_lane", C.c_void_p), ("q_list", C.c_void_p),
    ]


class ConvPlanStruct(C.Structure):
    """mt_conv_plan"""
    _fields_ = [
        ("x_dim", C.c_int32), ("y_dim", C.c_int32), ("out_dim", C.c_int32), ("num_items", C.c_int32),
        ("item_hdr", C.c_void_p), ("slot_tab", C.c_void_p),
        ("mlp_num_layers", C.c_int32), ("mlp_sizes", C.c_int32 * (MT_MAX_MLP_LAYERS + 1)),
        ("mlp_act", C.c_int32), ("mlp_act_cst", C.c_double),
        ("tc_num_parts", C.c_int32), ("tc_y_lmax", C.c_int32), ("tc_parts", ConvTcPartStruct * MT_TC_MAX_PARTS),
        ("bw_num_items", C.c_int32), ("bw_num_paths", C.c_int32),
        ("bw_item_hdr", C.c_void_p), ("bw_lane_tab", C.c_void_p), ("bw_path_tab", C.c_void_p),
    ]


class LinBlockStruct(C.Structure):
    """mt_lin_block"""
    _fields_ = [
        ("in_off", C.c_int32), ("out_off", C.c_int32), ("mul_in", C.c_int32), ("mul_out", C.c_int32),
        ("dim", C.c_int32), ("w_off", C.c_int32), ("scale", C.c_double),
    ]


_V, _I, _L, _D, _Z = C.c_void_p, C.c_int, C.c_int64, C.c_double, C.c_size_t

#: name -> (restype, argtypes); must list every symbol declared in include/matten_b200.h
SIGNATURES = {
    "mt_abi_version": (_I, []),
    "mt_last_error": (C.c_char_p, []),
    "mt_launch_count": (C.c_uint64, []),
    "mt_device_supported": (_I, [_I]),
    "mt_edge_vectors": (_I, [_I, _V, _V, _V, _V, _V, _L, _L, _L, _V, _V, _V, _V]),
    "mt_edge_sh": (_I, [_I, _V, _L, _I, _I, _V, _V]),
    "mt_edge_radial": (_I, [_I, _V, _L, _I, _I, _D, _D, _I, _D, _V, _V, _V]),
    "mt_edge_sh_bwd": (_I, [_I, _V, _V, _L, _I, _I, _V, _V]),
    "mt_edge_radial_bwd": (_I, [_I, _V, _V, _L, _I, _I, _D, _D, _I, _D, _V, _V, _V]),
    "mt_edge_vectors_bwd_workspace_bytes": (_Z, [_I, _L, _L]),
    "mt_edge_vectors_bwd": (_I, [_I, _V, _V, _V, _V, _V, _V, _V, _V, _V, _L, _L, _L, _V, _V, _V, _Z, _V]),
    "mt_csr_workspace_bytes": (_Z, [_L, _L]),
    "mt_csr_by_key": (_I, [_V, _L, _L, _V, _V, _V, _Z, _V, _V]),
    "mt_gather_i64_to_i32": (_I, [_V, _V, _L, _V, _V]),
    "mt_check_sorted": (_I, [_V, _L, _V, _V]),
    "mt_neighbor_workspace_bytes": (_Z, [_L, _L]),
    "mt_neighbor_count": (_I, [_I, _V, _V, _V, _V, _L, _L, _D, _V, _V, _Z, _V]),
    "mt_neighbor_fill": (_I, [_I, _V, _V, _V, _L, _L, _D, _V, _V, _V, _V, _V, _L, _V]),
    "mt_species_embed": (_I, [_I, _V, _I, _V, _L, _L, _I, _I, _V, _V, _L, _V, _V, _V, _V, _V]),
    "mt_conv_fwd_workspace_bytes": (_Z, [C.POINTER(ConvPlanStruct), _I, _L, _L]),
    "mt_conv_fwd": (_I, [C.POINTER(ConvPlanStruct), _I, _V, _V, _V, C.POINTER(_V), _V, _V, _V, _D, _V, _V,
                         _V, _Z, _V, _L, _L, _V]),
    "mt_conv_layout_bytes": (_Z, [_I, _L, _L]),
    "mt_conv_layout_prepare": (_I, [_I, _V, _V, _V, _V, _L, _L, _V, _Z, _V]),
    "mt_conv_select_impl": (_I, [_I]),
    "mt_conv_set_debug_buffer": (None, [_V]),
    "mt_conv_bwd_workspace_bytes": (_Z, [C.POINTER(ConvPlanStruct), _I, _L, _L]),
    "mt_conv_bwd": (_I, [C.POINTER(ConvPlanStruct), _I, _V, _V, _V, C.POINTER(_V), _V, _V, _V, _V, _V, _D, _V, _V, _V,
                         C.POINTER(_V), _V, _Z, _L, _L, _V]),
    "mt_conv_bwd_full": (_I, [C.POINTER(ConvPlanStruct), _I, _V, _V, _V, C.POINTER(_V), _V, _V, _V, _V, _V, _D, _V, _V,
                              _V, C.POINTER(_V), _V, _V, _V, _Z, _L, _L, _V]),
    "mt_linear_bwd_workspace_bytes": (_Z, [_I, _L]),
    "mt_linear_bwd": (_I, [_I, C.POINTER(LinBlockStruct), _I, _I, _I, _I, _L, _V, _V, _V, _V, _V, _V, _I, _V, _I, _V,
                           _Z, _L, _V]),
    "mt_gate_bwd": (_I, [_I, _V, _V, _I, _I, _V, _V, _V, _V, _V, _V, _V, _V, _L, _V]),
    "mt_col_reduce_workspace_bytes": (_Z, [_I, _I]),
    "mt_col_reduce": (_I, [_I, _V, _V, _V, _V, _L, _I, _V, _V, _Z, _V]),
    "mt_affine2": (_I, [_I, _V, _V, _V, _V, _V, _V, _L, _I, _V]),
    "mt_segment_reduce_bwd": (_I, [_I, _V, _V, _I, _L, _L, _I, _V, _V]),
    "mt_segment_sum_gather": (_I, [_I, _V, _V, _V, _I, _L, _L, _V, _V]),
    "mt_mse_loss": (_I, [_I, _V, _V, _L, _D, _V, _V, _V]),
    "mt_adam_step": (_I, [_I, _V, _V, _V, _V, _L, _D, _D, _D, _D, _D, _D, _L, _V]),
    "mt_linear_fwd": (_I, [_I, C.POINTER(LinBlockStruct), _I, _I, _I, _I, _V, _V, _V, _V, _I, _V, _L, _V]),
    "mt_gate_fwd": (_I, [_I, _V, _I, _I, _V, _V, _V, _V, _V, _V, _V, _L, _V]),
    "mt_segment_reduce": (_I, [_I, _V, _V, _I, _L, _I, _V, _V]),
    "mt_segment_extreme_bwd": (_I, [_I, _V, _V, _V, _I, _L, _I, _V, _V]),
    "mt_instance_norm_fwd": (_I, [_I, _V, _V, _L, _I, _I, _V, _V, _V, _V, _V, _D, _I, _I, _V, _V, _V, _V, _V]),
    "mt_instance_norm_bwd": (_I, [_I, _V, _V, _V, _L, _I, _I, _V, _V, _V, _V, _I, _I, _V, _V, _V, _V, _V, _V, _V]),
    "mt_norm_act_fwd": (_I, [_I, _V, _I, _I, _V, _V, _I, _D, _V, _L, _V]),
    "mt_norm_act_bwd": (_I, [_I, _V, _V, _I, _I, _V, _V, _I, _D, _V, _L, _V]),
    "mt_normalize": (_I, [_I, _V, _V, _V, _D, _I, _V, _L, _I, _V]),
}

_lock = threading.Lock()
_lib = None


def load(build_if_missing: bool = True) -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            if not build_if_missing:
                raise RuntimeError(f"{LIB_PATH} is missing; run `python -m matten_b200.build`")
            from . import build as _build

            _build.build(verbose=True)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            try:
                fn = getattr(lib, name)
            except AttributeError as e:
                raise RuntimeError(f"{LIB_PATH} does not export {name}; rebuild it") from e
            fn.restype = res
            fn.argtypes = args
        from . import ABI_VERSION

        if lib.mt_abi_version() != ABI_VERSION:
            raise RuntimeError("libmatten_b200.so ABI version mismatch; rebuild it")
        _lib = lib
        return lib


def check(rc: int):
    if rc != 0:
        msg = load().mt_last_error().decode(errors="replace")
        raise RuntimeError(f"matten_b200 C-ABI call failed ({rc}): {msg}")
