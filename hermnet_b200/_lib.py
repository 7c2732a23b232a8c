"""ctypes binding of ``libhermnet_b200.so`` (the C ABI declared in ``include/hermnet_b200.h``).

There is NO CPU fallback: if the library cannot be loaded, or an op is handed a non-CUDA tensor, the call
raises.  The library is built in-tree by ``hermnet_b200.build`` (nvcc, sm_100a).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int32, c_int64, c_void_p

from . import build as _build

_LIB = None


class EdgeParams(Structure):
    _fields_ = [("n_atoms", c_int32), ("n_rows", c_int32), ("n_modules", c_int32), ("hidden", c_int32),
                ("num_rbf", c_int32), ("env_p", c_int32), ("inv_rc", c_float), ("coeff", c_float), ("variant", c_int32), ("flags", c_int32)]


class P(c_void_p):
    """Argument type of every device pointer: ctypes passes ``None`` (NULL) and ``c_void_p`` through, and the address of
    anything with ``data_ptr()`` (a tensor) as a full-width pointer."""

    @classmethod
    def from_param(cls, obj):
        if obj is None or type(obj) is c_void_p:
            return obj
        try:
            data_ptr = obj.data_ptr
        except AttributeError:
            if isinstance(obj, c_void_p):
                return obj
            raise TypeError(f"expected a tensor, a c_void_p or None for a device pointer, got {type(obj).__name__}") from None
        return c_void_p(data_ptr())     # never a bare int: ctypes would pass it as a 32-bit C int


class TcPlan(Structure):
    """``hn_tc_plan``: tile plan of the tensor-core edge kernels (device pointers)."""
    _fields_ = [("n_blocks", c_int32), ("n_tiles", c_int32), ("blk_info", c_void_p), ("blk_tile", c_void_p),
                ("blk_xoff", c_void_p), ("tile_info", c_void_p), ("tile_win", c_void_p), ("erec", c_void_p), ("tile_geom", c_void_p), ("zero_row", c_void_p), ("blk_order", c_void_p)]


# name -> (restype, argtypes); must list EVERY symbol of include/hermnet_b200.h (checked by tests/test_abi.py)
SIGNATURES = {
    "hn_abi_version": (c_int32, []),
    "hn_last_error": (c_char_p, []),
    "hn_device_sm_count": (c_int32, []),
    "hn_radius_graph_workspace_bytes": (c_int64, [c_int64, c_int32]),
    "hn_radius_graph_count": (c_int32, [P, c_int64, P, P, c_int32, c_double, P, c_int32, c_int32, P, P, c_int64, P]),
    "hn_radius_graph_fill": (c_int32, [P, c_int64, P, P, c_int32, c_double, P, c_int32, c_int32, P, P, P, P, c_int64, P]),
    "hn_sort_by_key_workspace_bytes": (c_int64, [c_int64, c_int32]),
    "hn_sort_by_key": (c_int32, [P, c_int64, c_int32, P, P, P, c_int64, P]),
    "hn_expand_rowptr": (c_int32, [P, c_int32, P, P]),
    "hn_triplets_count": (c_int32, [P, c_int32, P, P, c_int32, c_int32, P, P]),
    "hn_triplets_fill": (c_int32, [P, c_int32, P, P, c_int32, c_int32, P, P, P, P]),
    "hn_triplet_dots": (c_int32, [P, c_int32, P, P, P, c_int32, P, P]),
    "hn_edge_geom_fwd": (c_int32, [P, P, P, P, c_int32, P, P, c_float, c_int64, P, P]),
    "hn_edge_geom_bwd": (c_int32, [P, P, c_int32, P, P, c_int32, P, P, c_float, c_int64, c_int64, P, P, P]),
    "hn_edge_virial_atom": (c_int32, [P, P, P, c_int32, P, P, c_int64, c_int64, P, P]),
    "hn_painn_edge_num_slices": (c_int32, [c_int32, c_int32]),
    "hn_painn_edge_fwd": (c_int32, [POINTER(EdgeParams)] + [P] * 13),
    "hn_painn_edge_bwd_dst": (c_int32, [POINTER(EdgeParams)] + [P] * 13 + [c_int64, P]),
    "hn_painn_edge_bwd_src": (c_int32, [POINTER(EdgeParams)] + [P] * 16),
    "hn_painn_edge_bwd_w": (c_int32, [POINTER(EdgeParams)] + [P] * 13 + [c_int32, P]),
    "hn_tc_supported": (c_int32, [c_int32, c_int32]),
    "hn_tc_block_rows": (c_int32, [c_int32]),
    "hn_tc_tile_edges": (c_int32, []),
    "hn_tc_groups": (c_int32, []),
    "hn_tc_split_weights_elems": (c_int64, [c_int32, c_int32, c_int32]),
    "hn_tc_split_weights": (c_int32, [P, c_int32, c_int32, c_int32, P, P, P]),
    "hn_tc_basis_index": (c_int32, [P, c_int64, c_float, c_int32, P, P]),
    "hn_tc_plan_records": (c_int32, [c_int32, P, P, P, P, P, c_int32, c_int32, P, c_float, c_int32, c_int64, P, P, P, P]),
    "hn_tc_plan_sort": (c_int32, [P, P, P, P, c_int32, c_int32, c_int32, P, P, P, P]),
    "hn_tc_plan_count": (c_int32, [P, P, P, c_int32, c_int32, c_int32, P, P]),
    "hn_tc_plan_fill": (c_int32, [P, P, P, c_int32, c_int32, c_int32, P, P, P]),
    "hn_tc_plan_finalize": (c_int32, [P, P, c_int32, c_int64, P, P, P, P, P]),
    "hn_tc_tile_windows": (c_int32, [POINTER(TcPlan), P, P, c_float, c_int32, P]),
    "hn_tc_edge_fwd": (c_int32, [POINTER(EdgeParams), POINTER(TcPlan)] + [P] * 10 + [c_int64, P]),
    "hn_tc_edge_bwd_dst": (c_int32, [POINTER(EdgeParams), POINTER(TcPlan)] + [P] * 11),
    "hn_tc_edge_bwd_src": (c_int32, [POINTER(EdgeParams), POINTER(TcPlan)] + [P] * 12),
    "hn_gemm_tf32x3": (c_int32, [P, c_int64, c_int64, c_int64, P, P, c_int64, P, P, c_int64, P]),
    "hn_gemm_tf32x3_ex": (c_int32, [P, c_int64, c_int64, c_int64, P, P, c_int64, P, P, c_int64, c_int32, P, c_int64, P, c_int64, P]),
    "hn_node_pre": (c_int32, [c_int64, c_int32, P, P, c_int64, P, P, c_int64, P, P, P]),
    "hn_node_mid": (c_int32, [c_int64, c_int32, P, P, P, P]),
    "hn_node_post": (c_int32, [c_int64, c_int32, P, P, P, P, P, P, P, P]),
    "hn_node_post_bwd": (c_int32, [c_int64, c_int32, P, P, P, P, P, P, P, P, P]),
    "hn_node_mid_bwd": (c_int32, [c_int64, c_int32, P, P, P, P, c_int64, P, P]),
    "hn_node_pre_bwd": (c_int32, [c_int64, c_int32, P, P, P, P, P, P, P]),
    "hn_gather_rows": (c_int32, [P, P, c_int64, c_int32, P, P]),
    "hn_layer0_basis_fwd": (c_int32, [P, P, P, P, P, P, P, c_int32, c_int32, P, P, P]),
    "hn_layer0_basis_bwd": (c_int32, [P, P, P, P, P, P, P, c_int32, c_int32, P, P, P, P]),
    "hn_layernorm_fwd": (c_int32, [P, c_int64, c_int32, c_float, P, P, P, P]),
    "hn_layernorm_bwd": (c_int32, [P, P, P, P, c_int64, c_int32, P, P]),
    "hn_readout_fwd": (c_int32, [P, P, P, P, P, c_int64, c_int32, P, P]),
    "hn_readout_bwd": (c_int32, [P, P, P, P, P, P, c_int64, c_int32, P, P]),
    "hn_halo_pack": (c_int32, [P, P, P, P, P, P, c_int64, c_int32, P]),
    "hn_halo_unpack": (c_int32, [P, P, c_int64, c_int32, P, P, P]),
    "hn_segment_sum_workspace_bytes": (c_int64, [c_int32, c_int32]),
    "hn_segment_sum": (c_int32, [P, P, P, c_int32, c_int32, P, P, c_int64, P]),
    "hn_md_langevin_baoa": (c_int32, [P, P, P, P, P, P, c_int32, P, P, P, c_float, c_float, c_float, c_int64, P]),
    "hn_md_kick": (c_int32, [P, P, P, c_float, c_int64, P, P, P]),
    "hn_md_scr_barostat": (c_int32, [P, P, P, P, P, P, P, P, c_int32, c_float, c_float, P, P, P]),
    "hn_md_affine_scale": (c_int32, [P, P, P, P, c_int64, P]),
    "hn_md_kinetic_tensor": (c_int32, [P, P, c_int64, P, P]),
    "hn_md_scr_barostat_tri": (c_int32, [P, P, P, P, P, P, P, P, c_int32, c_float, c_float, P, P, P, P]),
    "hn_md_affine_deform": (c_int32, [P, P, P, P, P, c_int64, P]),
    "hn_opt_fire_reduce_workspace_bytes": (c_int64, [c_int64, c_int32]),
    "hn_opt_fire_reduce": (c_int32, [P, P, P, P, P, c_int32, c_int64, P, P, c_int64, P]),
    "hn_opt_fire_step": (c_int32, [P] * 14 + [c_int32, c_double, c_double, c_double, c_int32, P, P, P, P]),
    "hn_opt_fire_update": (c_int32, [P] * 9 + [c_int64, P]),
    "hn_neb_reduce_workspace_bytes": (c_int64, [c_int64, c_int32]),
    "hn_neb_reduce": (c_int32, [P] * 7 + [c_int32, c_int32, c_int64, P, P, c_int64, P]),
    "hn_neb_step": (c_int32, [P] * 4 + [c_int32, c_int32, c_int32, P, P, P]),
    "hn_neb_project": (c_int32, [P] * 7 + [c_int32, c_int32, P, c_int64, P]),
}


def lib_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = True):
    """Load (building first when the sources are newer and nvcc is available) and type the library."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if build_if_missing and _build.needs_build():
        try:
            _build.build()
        except Exception as exc:  # no nvcc on the box: use the shipped .so if there is one
            if not os.path.exists(path):
                raise RuntimeError(f"hermnet_b200: cannot build {path} ({exc}); there is no CPU fallback") from exc
    if not os.path.exists(path):
        raise RuntimeError(f"hermnet_b200: {path} is missing -- run `python -m hermnet_b200.build`; "
                           "there is no CPU fallback")
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = ABI mismatch, fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.hn_abi_version() != 2:
        raise RuntimeError("hermnet_b200: ABI version mismatch between _lib.py and the shared library")
    _LIB = lib
    return lib


def check(code: int, what: str):
    if code != 0:
        msg = load().hn_last_error()
        raise RuntimeError(f"{what} failed: {msg.decode() if msg else code}")
