"""Tensor-level wrappers over the C ABI (``include/hermnet_b200.h``).

Each function takes CUDA torch tensors (torch is only the owner of device memory and of the stream),
passes raw pointers + the current stream through ctypes and returns freshly allocated outputs.  There is
no CPU implementation: a non-CUDA tensor raises.  The autograd layer (``functional.py``) and the graph
builder (``graph.py``) call these through the module namespace (``ops.<name>``).
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import EdgeParams

Tensor = torch.Tensor


def _ptr(t: Optional[Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream(dev) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _chk(name: str, *tensors, dtype=None):
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(f"hermnet_b200.{name}: expected a CUDA tensor, got device={t.device}; "
                               "the hot path has no CPU fallback")
        if not t.is_contiguous():
            raise RuntimeError(f"hermnet_b200.{name}: tensors must be contiguous")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"hermnet_b200.{name}: tensors on different devices")
    return dev


def _f32(name, *ts):
    for t in ts:
        if t is not None and t.dtype != torch.float32:
            raise RuntimeError(f"hermnet_b200.{name}: float tensors must be float32 (got {t.dtype})")


def _i32(name, *ts):
    for t in ts:
        if t is not None and t.dtype != torch.int32:
            raise RuntimeError(f"hermnet_b200.{name}: index tensors must be int32 (got {t.dtype})")


def require_cuda(t: Tensor, what: str) -> None:
    """Loud failure for CPU inputs: the product has no CPU path (tests swap this module's functions for an
    emulator that lives under tests/, never the other way round)."""
    if not t.is_cuda:
        raise RuntimeError(f"{what}: data is on {t.device}; the hermnet_b200 hot path runs on CUDA only "
                           "(there is no CPU fallback) -- move the inputs to a CUDA device")


def compute_device(t: Tensor) -> torch.device:
    """Device the kernels will run on for an input living on ``t.device`` (CPU inputs are staged to the GPU)."""
    if t.is_cuda:
        return t.device
    if not torch.cuda.is_available():
        raise RuntimeError("hermnet_b200 needs a CUDA device (there is no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


# ---- instrumentation used by bench.py: per-kernel CUDA-event timing on the launching stream, launch counting ----
TIMERS = None          # set to {} to collect name -> [(start_event, end_event), ...]
GEMM_SHAPES = False    # True: time the tensor-core GEMMs per shape (profiling aid)
LAUNCHES = {"n": 0}    # hand-written kernels launched through this module (cub passes are not counted)


class _timed:
    def __init__(self, name: str, dev, kernels: int = 1):
        self.name, self.dev, self.kernels = name, dev, kernels

    def __enter__(self):
        LAUNCHES["n"] += self.kernels
        if TIMERS is not None:
            self.t0 = torch.cuda.Event(enable_timing=True)
            self.t0.record(torch.cuda.current_stream(self.dev))
        return self

    def __exit__(self, *exc):
        if TIMERS is not None:
            t1 = torch.cuda.Event(enable_timing=True)
            t1.record(torch.cuda.current_stream(self.dev))
            TIMERS.setdefault(self.name, []).append((self.t0, t1))
        return False


def sm_count() -> int:
    return int(_lib.load().hn_device_sm_count())


# ----------------------------------------------------------------------------------------------------
# graph construction
# ----------------------------------------------------------------------------------------------------
def radius_graph(pos: Tensor, cell: Optional[Tensor], graph_ptr: Tensor, rc: float, group: Optional[Tensor] = None,
                 n_groups: int = 1, max_neighbors: int = 0) -> Tuple[Tensor, Tensor, Tensor]:
    """Row CSR of the neighbour list: row ``c*n_groups+g`` = neighbours ``(j, S)`` of centre ``c`` in group ``g``.
    Returns ``rowptr int32 [N*n_groups+1]``, ``col int32 [E]``, ``shift int8 [E,4]``.  One host sync (E)."""
    lib = _lib.load()
    dev = _chk("radius_graph", pos, cell, graph_ptr, group)
    _f32("radius_graph", pos, cell)
    _i32("radius_graph", graph_ptr, group)
    n = pos.size(0)
    n_graphs = graph_ptr.numel() - 1
    with torch.cuda.device(dev):
        ws_bytes = int(lib.hn_radius_graph_workspace_bytes(n, n_graphs))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        counts = torch.empty(n * n_groups, dtype=torch.int32, device=dev)
        st = _stream(dev)
        LAUNCHES["n"] += 6
        _lib.check(lib.hn_radius_graph_count(_ptr(pos), n, _ptr(cell), _ptr(graph_ptr), n_graphs, float(rc), _ptr(group),
                                             n_groups, max_neighbors, _ptr(counts), _ptr(ws), ws_bytes, st),
                   "hn_radius_graph_count")
        rowptr = torch.zeros(n * n_groups + 1, dtype=torch.int32, device=dev)
        torch.cumsum(counts, 0, dtype=torch.int32, out=rowptr[1:])
        n_edges = int(rowptr[-1].item())
        col = torch.empty(n_edges, dtype=torch.int32, device=dev)
        shift = torch.empty((n_edges, 4), dtype=torch.int8, device=dev)
        if n_edges > 0:
            LAUNCHES["n"] += 1
            _lib.check(lib.hn_radius_graph_fill(_ptr(pos), n, _ptr(cell), _ptr(graph_ptr), n_graphs, float(rc), _ptr(group),
                                                n_groups, max_neighbors, _ptr(rowptr), _ptr(col), _ptr(shift), _ptr(ws),
                                                ws_bytes, st), "hn_radius_graph_fill")
    return rowptr, col, shift


def sort_by_key(keys: Tensor, n_keys: int) -> Tuple[Tensor, Tensor]:
    """Stable grouping of ``arange(len(keys))`` by key: ``rowptr int32 [n_keys+1]``, ``order int32 [n]``."""
    lib = _lib.load()
    dev = _chk("sort_by_key", keys)
    _i32("sort_by_key", keys)
    n = keys.numel()
    with torch.cuda.device(dev):
        ws_bytes = int(lib.hn_sort_by_key_workspace_bytes(n, n_keys))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        rowptr = torch.empty(n_keys + 1, dtype=torch.int32, device=dev)
        order = torch.empty(n, dtype=torch.int32, device=dev)
        LAUNCHES["n"] += 1
        _lib.check(lib.hn_sort_by_key(_ptr(keys), n, n_keys, _ptr(rowptr), _ptr(order), _ptr(ws), ws_bytes, _stream(dev)),
                   "hn_sort_by_key")
    return rowptr, order


def expand_rowptr(rowptr: Tensor, n_edges: int) -> Tensor:
    lib = _lib.load()
    dev = _chk("expand_rowptr", rowptr)
    _i32("expand_rowptr", rowptr)
    out = torch.empty(n_edges, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev), _timed("expand_rowptr", dev):
        _lib.check(lib.hn_expand_rowptr(_ptr(rowptr), rowptr.numel() - 1, _ptr(out), _stream(dev)), "hn_expand_rowptr")
    return out


def triplets(rowptr: Tensor, col: Tensor, src_type: Optional[Tensor] = None, type_a: int = -1, type_c: int = -1):
    """Canonical ordered triplets over row-edge ids: ``trip_ptr int64 [R+1]``, ``e1``, ``e2`` int32 [T]."""
    lib = _lib.load()
    dev = _chk("triplets", rowptr, col, src_type)
    _i32("triplets", rowptr, col, src_type)
    n_rows = rowptr.numel() - 1
    with torch.cuda.device(dev):
        counts = torch.empty(n_rows, dtype=torch.int64, device=dev)
        st = _stream(dev)
        _lib.check(lib.hn_triplets_count(_ptr(rowptr), n_rows, _ptr(col), _ptr(src_type), type_a, type_c, _ptr(counts), st),
                   "hn_triplets_count")
        trip_ptr = torch.zeros(n_rows + 1, dtype=torch.int64, device=dev)
        torch.cumsum(counts, 0, out=trip_ptr[1:])
        total = int(trip_ptr[-1].item())
        e1 = torch.empty(total, dtype=torch.int32, device=dev)
        e2 = torch.empty(total, dtype=torch.int32, device=dev)
        if total > 0:
            _lib.check(lib.hn_triplets_fill(_ptr(rowptr), n_rows, _ptr(col), _ptr(src_type), type_a, type_c, _ptr(trip_ptr),
                                            _ptr(e1), _ptr(e2), st), "hn_triplets_fill")
    return trip_ptr, e1, e2


def triplet_dots(m_vec: Tensor, trip_ptr: Tensor, e1: Tensor, e2: Tensor) -> Tensor:
    lib = _lib.load()
    dev = _chk("triplet_dots", m_vec, trip_ptr, e1, e2)
    _f32("triplet_dots", m_vec)
    F = m_vec.size(-1)
    n_rows = trip_ptr.numel() - 1
    out = torch.empty((n_rows, F), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.hn_triplet_dots(_ptr(m_vec), F, _ptr(trip_ptr), _ptr(e1), _ptr(e2), n_rows, _ptr(out), _stream(dev)),
                   "hn_triplet_dots")
    return out


# ----------------------------------------------------------------------------------------------------
# geometry
# ----------------------------------------------------------------------------------------------------
def edge_geom_fwd(pos: Tensor, cell: Optional[Tensor], g) -> Tensor:
    lib = _lib.load()
    dev = _chk("edge_geom_fwd", pos, cell)
    _f32("edge_geom_fwd", pos, cell)
    geom = torch.empty((g.n_edges, 4), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("edge_geom_fwd", dev):
        _lib.check(lib.hn_edge_geom_fwd(_ptr(pos), _ptr(cell), _ptr(g.atom_graph), _ptr(g.edge_row), g.rows_per_atom,
                                        _ptr(g.col), _ptr(g.shift if cell is not None else None), float(g.sign),
                                        g.n_edges, _ptr(geom), _stream(dev)), "hn_edge_geom_fwd")
    return geom


def edge_geom_bwd(geom: Tensor, g_geom: Tensor, g, want_cell: bool):
    """``g_geom`` is ``[n_parts, E, 4]``; returns ``grad_pos [N,3]`` and the per-atom virial partial ``[N,9]``."""
    lib = _lib.load()
    dev = _chk("edge_geom_bwd", geom, g_geom)
    _f32("edge_geom_bwd", geom, g_geom)
    n_parts = g_geom.size(0) if g_geom.dim() == 3 else 1
    grad_pos = torch.empty((g.n_atoms, 3), dtype=torch.float32, device=dev)
    cellw = torch.empty((g.n_atoms, 9), dtype=torch.float32, device=dev) if want_cell else None
    with torch.cuda.device(dev), _timed("edge_geom_bwd", dev):
        _lib.check(lib.hn_edge_geom_bwd(_ptr(geom), _ptr(g_geom), n_parts, _ptr(g.shift), _ptr(g.rowptr), g.rows_per_atom,
                                        _ptr(g.t_rowptr), _ptr(g.t_eid), float(g.sign), g.n_atoms, g.n_edges,
                                        _ptr(grad_pos), _ptr(cellw), _stream(dev)), "hn_edge_geom_bwd")
    return grad_pos, cellw


def edge_virial_atom(geom: Tensor, g_geom: Tensor, g) -> Tensor:
    """Per-atom virial ``[N, 9]`` (internal atom order, row = position component) from ``geom [E,4]`` and its gradient
    ``g_geom [E,4]``: each edge gives ``-1/2 D_e (x) dE/dD_e`` to both of its atoms."""
    lib = _lib.load()
    dev = _chk("edge_virial_atom", geom, g_geom)
    _f32("edge_virial_atom", geom, g_geom)
    if tuple(geom.shape) != (g.n_edges, 4) or tuple(g_geom.shape) != (g.n_edges, 4):
        raise RuntimeError(f"hermnet_b200.edge_virial_atom: geom / g_geom must be [{g.n_edges}, 4]")
    virial = torch.empty((g.n_atoms, 9), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("edge_virial_atom", dev):
        _lib.check(lib.hn_edge_virial_atom(_ptr(geom), _ptr(g_geom), _ptr(g.rowptr), g.rows_per_atom, _ptr(g.t_rowptr),
                                           _ptr(g.t_eid), g.n_atoms, g.n_edges, _ptr(virial), _stream(dev)),
                   "hn_edge_virial_atom")
    return virial


# ----------------------------------------------------------------------------------------------------
# fused PaiNN edge kernels
# ----------------------------------------------------------------------------------------------------
def edge_params(g, n_modules: int, hidden: int, num_rbf: int, env_p: int, rc: float, coeff: float) -> EdgeParams:
    return EdgeParams(g.n_atoms, g.n_rows, n_modules, hidden, num_rbf, env_p, 1.0 / rc, coeff)


def edge_num_slices(hidden: int) -> int:
    n = int(_lib.load().hn_painn_edge_num_slices(hidden, 1 if EDGE_VARIANT["v"] == "row" else 0))
    if n <= 0:
        raise RuntimeError("hermnet_b200: hidden_channels must be a multiple of 32 for the fused edge kernels")
    return n


import os as _os

# 'auto': tensor-core kernels (hn_edge_tc.cu) where supported (F == 128), else the tile-sweep kernels (F % 64 == 0), else
# the row-per-warp kernels; 'quad' / 'row' pin the older families (A/B measurements, tests).  HERMNET_B200_EDGE presets it.
EDGE_VARIANT = {"v": _os.environ.get("HERMNET_B200_EDGE", "auto") if _os.environ.get("HERMNET_B200_EDGE", "auto") in
                ("auto", "tc", "quad", "row") else "auto"}


def edge_set_variant(variant: str) -> None:
    """'auto' / 'tc': tensor-core edge kernels where supported; 'quad': tile-sweep kernels; 'row': row-per-warp kernels."""
    if variant not in ("auto", "tc", "quad", "row"):
        raise ValueError(variant)
    EDGE_VARIANT["v"] = variant      # host-side preference only: every call stamps it into its hn_edge_params.variant


def _stamp(p: EdgeParams) -> EdgeParams:
    p.variant = 1 if EDGE_VARIANT["v"] == "row" else 0
    return p


def edge_use_tc(hidden: int, num_rbf: int) -> bool:
    return EDGE_VARIANT["v"] in ("auto", "tc") and tc_supported(hidden, num_rbf)


def _kernel_geom(name: str, p: EdgeParams, geom):
    """Geometry the row and tile-sweep kernels read: ``geom`` itself, or for a Verlet-skin list (``p.flags`` bit 0) a copy
    whose distance is ``-d`` on the entries ``p.live`` (uint8 [E]) marks dead -- the sign is how the C ABI passes the mask
    (a real distance is >= 1e-6).  The copy is cached on ``p``, keyed on the identity and version of ``geom`` and
    ``p.live``, so that every layer's forward and backward calls of one evaluation share it.  Device ops only: capturable
    in a CUDA graph."""
    import weakref
    if not p.flags & 1:
        return geom
    live = getattr(p, "live", None)
    if not isinstance(live, torch.Tensor) or live.dtype != torch.uint8 or live.numel() != geom.size(0):
        raise TypeError(f"hermnet_b200.{name}: live must be uint8 [E]")
    _chk(name, geom, live)
    stamp = (geom._version, geom.data_ptr(), live._version, live.data_ptr(), tuple(geom.shape))
    hit = getattr(p, "_signed_geom", None)
    if hit is not None and hit[0]() is geom and hit[1]() is live and hit[2] == stamp:
        return hit[3]
    with torch.no_grad():
        signed = geom.detach().clone()
        signed[:, 3] = torch.where(live.bool(), geom[:, 3], -geom[:, 3])
    p._signed_geom = (weakref.ref(geom), weakref.ref(live), stamp, signed)
    return signed


def painn_edge_fwd(p: EdgeParams, xh, vec, geom, g, Wt, bias, offset):
    """A Verlet-skin list (``p.flags`` bit 0) needs ``p.live``, as for ``painn_edge_bwd_w``: entries marked 0 contribute
    nothing, not even the filter bias.  The same holds for ``painn_edge_bwd_dst`` (zero ``g_geom`` rows) and
    ``painn_edge_bwd_src``."""
    geom = _kernel_geom("painn_edge_fwd", p, geom)      # first: a missing mask is the error to report
    lib = _lib.load()
    _stamp(p)
    dev = _chk("painn_edge_fwd", xh, vec, geom, Wt, bias, offset)
    _f32("painn_edge_fwd", xh, vec, geom, Wt, bias, offset)
    F = p.hidden
    dx = torch.empty((p.n_rows, F), dtype=torch.float32, device=dev)
    dvec = torch.empty((p.n_rows, 3, F), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("painn_edge_fwd", dev):
        _lib.check(lib.hn_painn_edge_fwd(ctypes.byref(p), _ptr(xh), _ptr(vec), _ptr(geom), _ptr(g.rowptr), _ptr(g.col),
                                         _ptr(g.row_mod), _ptr(g.row_xoff), _ptr(Wt), _ptr(bias), _ptr(offset), _ptr(dx), _ptr(dvec),
                                         _stream(dev)), "hn_painn_edge_fwd")
    return dx, dvec


def painn_edge_bwd_dst(p: EdgeParams, xh, vec, geom, g, Wt, bias, offset, g_dx, g_dvec):
    geom = _kernel_geom("painn_edge_bwd_dst", p, geom)      # first: a missing mask is the error to report
    lib = _lib.load()
    _stamp(p)
    dev = _chk("painn_edge_bwd_dst", xh, vec, geom, Wt, bias, offset, g_dx, g_dvec)
    _f32("painn_edge_bwd_dst", xh, vec, geom, Wt, bias, offset, g_dx, g_dvec)
    g_geom = torch.empty((edge_num_slices(p.hidden), g.n_edges, 4), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("painn_edge_bwd_dst", dev):
        _lib.check(lib.hn_painn_edge_bwd_dst(ctypes.byref(p), _ptr(xh), _ptr(vec), _ptr(geom), _ptr(g.rowptr), _ptr(g.col),
                                             _ptr(g.row_mod), _ptr(g.row_xoff), _ptr(Wt), _ptr(bias), _ptr(offset), _ptr(g_dx),
                                             _ptr(g_dvec), _ptr(g_geom), g.n_edges, _stream(dev)), "hn_painn_edge_bwd_dst")
    return g_geom


def painn_edge_bwd_src(p: EdgeParams, xh, vec, geom, g, Wt, bias, offset, g_dx, g_dvec):
    geom = _kernel_geom("painn_edge_bwd_src", p, geom)      # first: a missing mask is the error to report
    lib = _lib.load()
    _stamp(p)
    dev = _chk("painn_edge_bwd_src", xh, vec, geom, Wt, bias, offset, g_dx, g_dvec)
    _f32("painn_edge_bwd_src", xh, vec, geom, Wt, bias, offset, g_dx, g_dvec)
    grad_xh = torch.zeros_like(xh)
    grad_vec = torch.empty_like(vec)
    with torch.cuda.device(dev), _timed("painn_edge_bwd_src", dev):
        _lib.check(lib.hn_painn_edge_bwd_src(ctypes.byref(p), _ptr(xh), _ptr(vec), _ptr(geom), _ptr(g.t_rowptr),
                                             _ptr(g.t_eid), _ptr(g.edge_row), _ptr(g.row_mod), _ptr(g.row_xoff), _ptr(Wt), _ptr(bias),
                                             _ptr(offset), _ptr(g_dx), _ptr(g_dvec), _ptr(grad_xh), _ptr(grad_vec),
                                             _stream(dev)), "hn_painn_edge_bwd_src")
    return grad_xh, grad_vec


def painn_edge_bwd_w(p: EdgeParams, xh, vec, geom, g, offset, g_dx, g_dvec):
    """Gradients of the filter projection: ``gWt [M,K,3F]``, ``gb [M,3F]`` (partials reduced in fixed order).  A Verlet-skin
    list (``p.flags`` bit 0) needs ``p.live``, the uint8 [E] mask the model attaches next to the flag: entries marked 0
    contribute nothing."""
    lib = _lib.load()
    live = getattr(p, "live", None) if p.flags & 1 else None
    dev = _chk("painn_edge_bwd_w", xh, vec, geom, offset, g_dx, g_dvec, live)
    _f32("painn_edge_bwd_w", xh, vec, geom, offset, g_dx, g_dvec)
    if live is not None and (live.dtype != torch.uint8 or live.numel() != geom.size(0)):
        raise TypeError("hermnet_b200.painn_edge_bwd_w: live must be uint8 [E]")
    M, K, F3 = p.n_modules, p.num_rbf, 3 * p.hidden
    n_chunks = max(1, min(p.n_rows, (2 * max(sm_count(), 1)) // max(M, 1)))
    gW = torch.empty((n_chunks, M, K, F3), dtype=torch.float32, device=dev)
    gb = torch.empty((n_chunks, M, F3), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("painn_edge_bwd_w", dev):
        _lib.check(lib.hn_painn_edge_bwd_w(ctypes.byref(p), _ptr(xh), _ptr(vec), _ptr(geom), _ptr(g.rowptr), _ptr(g.col),
                                           _ptr(g.row_mod), _ptr(g.row_xoff), _ptr(live), _ptr(offset), _ptr(g_dx), _ptr(g_dvec), _ptr(gW),
                                           _ptr(gb), n_chunks, _stream(dev)), "hn_painn_edge_bwd_w")
    return gW.sum(0), gb.sum(0)


# ----------------------------------------------------------------------------------------------------
# gather / segmented sum
# ----------------------------------------------------------------------------------------------------
def gather_rows(X: Tensor, idx: Tensor) -> Tensor:
    lib = _lib.load()
    dev = _chk("gather_rows", X, idx)
    _f32("gather_rows", X)
    _i32("gather_rows", idx)
    C = X.size(1)
    out = torch.empty((idx.numel(), C), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("gather_rows", dev):
        _lib.check(lib.hn_gather_rows(_ptr(X), _ptr(idx), idx.numel(), C, _ptr(out), _stream(dev)), "hn_gather_rows")
    return out


def layer0_row_len(n_elem: int, num_rbf: int) -> int:
    """Length of a basis-sum row of the first-layer pass: ``n_elem * (K + 1)`` sums, padded to a GEMM-friendly multiple."""
    pad = int(_os.environ.get("HERMNET_B200_L0_PAD", "128"))
    return (n_elem * (num_rbf + 1) + pad - 1) // pad * pad


def layer0_basis_fwd(p: EdgeParams, g, geom: Tensor, live: Optional[Tensor], offset: Tensor, n_elem: int, kp: int):
    """``(Sa [R,kp], Sc [R,3,kp])``: per-(destination row, source element) sums of the radial basis (``hn_layer0_basis_fwd``);
    ``g.col`` holds the element index of every row-edge's source."""
    lib = _lib.load()
    dev = _chk("layer0_basis_fwd", g.rowptr, g.col, g.row_mod, geom, live, offset)
    _i32("layer0_basis_fwd", g.rowptr, g.col, g.row_mod)
    _f32("layer0_basis_fwd", geom, offset)
    R = int(p.n_rows)
    Sa = torch.empty((R, kp), dtype=torch.float32, device=dev)
    Sc = torch.empty((R, 3, kp), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("layer0_basis_fwd", dev):
        _lib.check(lib.hn_layer0_basis_fwd(ctypes.byref(p), _ptr(g.rowptr), _ptr(g.col), _ptr(g.row_mod), _ptr(geom), _ptr(live),
                                           _ptr(offset), int(n_elem), int(kp), _ptr(Sa), _ptr(Sc), _stream(dev)), "hn_layer0_basis_fwd")
    return Sa, Sc


def layer0_basis_bwd(p: EdgeParams, g, geom: Tensor, live: Optional[Tensor], offset: Tensor, n_elem: int, kp: int, g_Sa: Tensor,
                     g_Sc: Tensor) -> Tensor:
    lib = _lib.load()
    dev = _chk("layer0_basis_bwd", g.rowptr, g.col, g.row_mod, geom, live, offset, g_Sa, g_Sc)
    _f32("layer0_basis_bwd", geom, offset, g_Sa, g_Sc)
    g_geom = torch.empty((geom.size(0), 4), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("layer0_basis_bwd", dev):
        _lib.check(lib.hn_layer0_basis_bwd(ctypes.byref(p), _ptr(g.rowptr), _ptr(g.col), _ptr(g.row_mod), _ptr(geom), _ptr(live),
                                           _ptr(offset), int(n_elem), int(kp), _ptr(g_Sa), _ptr(g_Sc), _ptr(g_geom), _stream(dev)),
                   "hn_layer0_basis_bwd")
    return g_geom


def layernorm_fwd(x: Tensor, eps: float):
    """``(xhat, mean [n], rstd [n])`` of the affine-free LayerNorm over the last dimension (``hn_layernorm_fwd``)."""
    lib = _lib.load()
    dev = _chk("layernorm_fwd", x)
    _f32("layernorm_fwd", x)
    n, F = x.shape
    xhat = torch.empty_like(x)
    mean = torch.empty(n, dtype=torch.float32, device=dev)
    rstd = torch.empty(n, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("node_elementwise", dev):
        _lib.check(lib.hn_layernorm_fwd(_ptr(x), n, F, float(eps), _ptr(xhat), _ptr(mean), _ptr(rstd), _stream(dev)), "hn_layernorm_fwd")
    return xhat, mean, rstd


def layernorm_bwd(g_xhat: Tensor, x: Tensor, mean: Tensor, rstd: Tensor) -> Tensor:
    lib = _lib.load()
    dev = _chk("layernorm_bwd", g_xhat, x, mean, rstd)
    _f32("layernorm_bwd", g_xhat, x, mean, rstd)
    n, F = x.shape
    g_x = torch.empty_like(x)
    with torch.cuda.device(dev), _timed("node_elementwise", dev):
        _lib.check(lib.hn_layernorm_bwd(_ptr(g_xhat), _ptr(x), _ptr(mean), _ptr(rstd), n, F, _ptr(g_x), _stream(dev)), "hn_layernorm_bwd")
    return g_x


def readout_fwd(x: Tensor, W1: Tensor, b1: Tensor, W2: Tensor, b2: Tensor) -> Tensor:
    """``e_atom [N,1] = W2 . ssilu(W1 x + b1) + b2`` in plain fp32 (hn_readout_fwd)."""
    lib = _lib.load()
    dev = _chk("readout_fwd", x, W1, b1, W2, b2)
    _f32("readout_fwd", x, W1, b1, W2, b2)
    out = torch.empty((x.size(0), 1), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("readout", dev):
        _lib.check(lib.hn_readout_fwd(_ptr(x), _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), x.size(0), x.size(1), _ptr(out), _stream(dev)),
                   "hn_readout_fwd")
    return out


def readout_bwd(x: Tensor, W1: Tensor, b1: Tensor, W2: Tensor, b2: Tensor, g_e: Tensor) -> Tensor:
    lib = _lib.load()
    dev = _chk("readout_bwd", x, W1, b1, W2, b2, g_e)
    _f32("readout_bwd", x, W1, b1, W2, b2, g_e)
    g_x = torch.empty_like(x)
    with torch.cuda.device(dev), _timed("readout", dev):
        _lib.check(lib.hn_readout_bwd(_ptr(x), _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), _ptr(g_e), x.size(0), x.size(1), _ptr(g_x),
                                      _stream(dev)), "hn_readout_bwd")
    return g_x


def halo_pack(x: Tensor, vec: Tensor, src_idx: Tensor, row_peer: Tensor, row_slot: Tensor, dst_base: Tensor) -> None:
    """Rows ``[x | vec]`` of the atoms ``src_idx`` stored at ``dst_base[row_peer[i]] + row_slot[i] * 4F`` floats (device
    addresses: peers' landing buffers over NVLink, or slices of a local send buffer)."""
    lib = _lib.load()
    dev = _chk("halo_pack", x, vec, src_idx, row_peer, row_slot, dst_base)
    _f32("halo_pack", x, vec)
    _i32("halo_pack", src_idx, row_peer, row_slot)
    if dst_base.dtype != torch.int64:
        raise TypeError("hermnet_b200.halo_pack: dst_base must be int64 device addresses")
    with torch.cuda.device(dev), _timed("halo_pack", dev):
        _lib.check(lib.hn_halo_pack(_ptr(x), _ptr(vec), _ptr(src_idx), _ptr(row_peer), _ptr(row_slot), _ptr(dst_base),
                                    src_idx.numel(), x.size(1), _stream(dev)), "hn_halo_pack")


def halo_unpack(buf: Tensor, dst_idx: Tensor, x: Tensor, vec: Tensor) -> None:
    """Row ``i`` of ``buf [n, 4F]`` -> ``x[dst_idx[i]]``, ``vec[dst_idx[i]]`` (in place)."""
    lib = _lib.load()
    dev = _chk("halo_unpack", buf, dst_idx, x, vec)
    _f32("halo_unpack", buf, x, vec)
    _i32("halo_unpack", dst_idx)
    with torch.cuda.device(dev), _timed("halo_unpack", dev):
        _lib.check(lib.hn_halo_unpack(_ptr(buf), _ptr(dst_idx), dst_idx.numel(), x.size(1), _ptr(x), _ptr(vec), _stream(dev)),
                   "hn_halo_unpack")


def segment_sum(Y: Tensor, rowptr: Tensor, perm: Optional[Tensor], n_rows: int) -> Tensor:
    lib = _lib.load()
    dev = _chk("segment_sum", Y, rowptr, perm)
    _f32("segment_sum", Y)
    _i32("segment_sum", rowptr, perm)
    C = Y.size(1)
    out = torch.empty((n_rows, C), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("segment_sum", dev):
        ws_bytes = int(lib.hn_segment_sum_workspace_bytes(n_rows, C))      # chunk partials of long rows: caller-owned
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
        _lib.check(lib.hn_segment_sum(_ptr(Y), _ptr(rowptr), _ptr(perm), n_rows, C, _ptr(out), _ptr(ws), ws_bytes, _stream(dev)),
                   "hn_segment_sum")
    return out


# ----------------------------------------------------------------------------------------------------
# Langevin and constant-pressure MD steps (csrc/hn_md.cu)
# ----------------------------------------------------------------------------------------------------
def _i64(name, *ts):
    for t in ts:
        if t is not None and t.dtype != torch.int64:
            raise RuntimeError(f"hermnet_b200.{name}: seed / step tensors must be int64 (got {t.dtype})")


def _md_shapes(name, n: int, vel: Tensor, force: Tensor, inv_mass: Tensor):
    if tuple(vel.shape) != (n, 3) or tuple(force.shape) != (n, 3) or inv_mass.numel() != n:
        raise RuntimeError(f"hermnet_b200.{name}: expected vel / force [{n},3] and inv_mass [{n}]")


def md_langevin_baoa(pos: Tensor, vel: Tensor, force: Tensor, inv_mass: Tensor, replica: Tensor, replica_ptr: Tensor,
                     kT: Tensor, seed: Tensor, step: Tensor, c1: float, c2: float, dt: float) -> None:
    """B-A-O-A half of a BAOAB Langevin step, in place on ``pos`` / ``vel [N,3]`` (``hn_md_langevin_baoa``): ``replica int32
    [N]``, ``replica_ptr int32 [G+1]`` (contiguous replicas), per-replica ``kT float32 [G]`` (eV) and ``seed int64 [G]``,
    ``step int64 [1]`` (read, not advanced).  ``c1 = exp(-gamma dt)``, ``c2 = sqrt(1 - c1^2)``."""
    lib = _lib.load()
    dev = _chk("md_langevin_baoa", pos, vel, force, inv_mass, replica, replica_ptr, kT, seed, step)
    _f32("md_langevin_baoa", pos, vel, force, inv_mass, kT)
    _i32("md_langevin_baoa", replica, replica_ptr)
    _i64("md_langevin_baoa", seed, step)
    n, G = pos.size(0), replica_ptr.numel() - 1
    _md_shapes("md_langevin_baoa", n, vel, force, inv_mass)
    if tuple(pos.shape) != (n, 3) or replica.numel() != n or kT.numel() != G or seed.numel() != G or step.numel() != 1:
        raise RuntimeError(f"hermnet_b200.md_langevin_baoa: expected pos [N,3], replica [N], kT / seed [G={G}], step [1]")
    with torch.cuda.device(dev), _timed("md_langevin_baoa", dev):
        _lib.check(lib.hn_md_langevin_baoa(_ptr(pos), _ptr(vel), _ptr(force), _ptr(inv_mass), _ptr(replica), _ptr(replica_ptr), G,
                                           _ptr(kT), _ptr(seed), _ptr(step), float(c1), float(c2), float(dt), n, _stream(dev)),
                   "hn_md_langevin_baoa")
    # written through raw pointers: version-keyed caches (graphs, signed geometry, tile windows) must see the change
    torch.autograd.graph.increment_version(pos)
    torch.autograd.graph.increment_version(vel)


def md_kick(vel: Tensor, force: Tensor, inv_mass: Tensor, half_dt: float, kinetic: Optional[Tensor], step: Tensor) -> None:
    """Closing B of a BAOAB step, in place on ``vel [N,3]`` (``hn_md_kick``); ``kinetic [N]`` (optional) receives
    ``1/2 |v_i|^2 / inv_m_i`` in eV; ``step int64 [1]`` is advanced by one."""
    lib = _lib.load()
    dev = _chk("md_kick", vel, force, inv_mass, kinetic, step)
    _f32("md_kick", vel, force, inv_mass, kinetic)
    _i64("md_kick", step)
    n = vel.size(0)
    _md_shapes("md_kick", n, vel, force, inv_mass)
    if (kinetic is not None and kinetic.numel() != n) or step.numel() != 1:
        raise RuntimeError(f"hermnet_b200.md_kick: expected kinetic [{n}] and step [1]")
    with torch.cuda.device(dev), _timed("md_kick", dev):
        _lib.check(lib.hn_md_kick(_ptr(vel), _ptr(force), _ptr(inv_mass), float(half_dt), n, _ptr(kinetic), _ptr(step), _stream(dev)),
                   "hn_md_kick")
    for t in (vel, kinetic, step):
        if t is not None:
            torch.autograd.graph.increment_version(t)


def md_scr_barostat(cell: Tensor, kinetic: Tensor, virial: Tensor, P0: Tensor, kT: Tensor, beta: Tensor, seed: Tensor,
                    step: Tensor, dt: float, tau_p: float, mu: Tensor, pressure: Tensor) -> None:
    """Stochastic cell rescaling of ``G`` replicas (``hn_md_scr_barostat``): ``cell [G,3,3]`` is scaled in place by
    ``mu [G]`` (written), from the per-replica kinetic energy ``kinetic [G]`` (eV), ``virial [G,3,3]`` (eV), target
    pressure ``P0 [G]`` (eV/A^3), ``kT [G]`` (eV), compressibility ``beta [G]`` (A^3/eV, >= 0), ``seed int64 [G]`` and
    ``step int64 [1]`` (read).  ``pressure [G]`` receives the internal pressure (eV/A^3) of the unscaled cell."""
    lib = _lib.load()
    dev = _chk("md_scr_barostat", cell, kinetic, virial, P0, kT, beta, seed, step, mu, pressure)
    _f32("md_scr_barostat", cell, kinetic, virial, P0, kT, beta, mu, pressure)
    _i64("md_scr_barostat", seed, step)
    G = kinetic.numel()
    if (tuple(cell.shape) != (G, 3, 3) or tuple(virial.shape) != (G, 3, 3) or step.numel() != 1
            or any(t.numel() != G for t in (P0, kT, beta, seed, mu, pressure))):
        raise RuntimeError(f"hermnet_b200.md_scr_barostat: expected cell / virial [G={G},3,3], kinetic / P0 / kT / beta / seed / "
                           "mu / pressure [G] and step [1]")
    with torch.cuda.device(dev), _timed("md_scr_barostat", dev):
        _lib.check(lib.hn_md_scr_barostat(_ptr(cell), _ptr(kinetic), _ptr(virial), _ptr(P0), _ptr(kT), _ptr(beta), _ptr(seed),
                                          _ptr(step), G, float(dt), float(tau_p), _ptr(mu), _ptr(pressure), _stream(dev)),
                   "hn_md_scr_barostat")
    for t in (cell, mu, pressure):
        torch.autograd.graph.increment_version(t)


def md_affine_scale(pos: Tensor, vel: Tensor, replica: Tensor, mu: Tensor) -> None:
    """``pos *= mu[replica]``, ``vel /= mu[replica]`` in place on ``[N,3]`` (``hn_md_affine_scale``; ``replica int32 [N]``)."""
    lib = _lib.load()
    dev = _chk("md_affine_scale", pos, vel, replica, mu)
    _f32("md_affine_scale", pos, vel, mu)
    _i32("md_affine_scale", replica)
    n = pos.size(0)
    if tuple(pos.shape) != (n, 3) or tuple(vel.shape) != (n, 3) or replica.numel() != n:
        raise RuntimeError(f"hermnet_b200.md_affine_scale: expected pos / vel [{n},3] and replica [{n}]")
    with torch.cuda.device(dev), _timed("md_affine_scale", dev):
        _lib.check(lib.hn_md_affine_scale(_ptr(pos), _ptr(vel), _ptr(replica), _ptr(mu), n, _stream(dev)), "hn_md_affine_scale")
    torch.autograd.graph.increment_version(pos)
    torch.autograd.graph.increment_version(vel)


# ----------------------------------------------------------------------------------------------------
# FIRE structure relaxation (csrc/hn_opt.cu)
# ----------------------------------------------------------------------------------------------------
def _f64(name, *ts):
    for t in ts:
        if t is not None and t.dtype != torch.float64:
            raise RuntimeError(f"hermnet_b200.{name}: optimizer state tensors must be float64 (got {t.dtype})")


def _g9(name, G: int, *ts):
    for t in ts:
        if t is not None and t.numel() != 9 * G:
            raise RuntimeError(f"hermnet_b200.{name}: expected [G={G},3,3] (or [G,9]) matrices, got {tuple(t.shape)}")


def opt_fire_reduce(force: Tensor, vel: Tensor, A: Optional[Tensor], replica: Tensor, replica_ptr: Tensor) -> Tensor:
    """Per-replica float64 ``[G,4]``: ``(sum F'.v, sum |F'|^2, sum |v|^2, max |F'_i|^2)`` over the atoms with ``F'_i = f_i A^T``
    (``hn_opt_fire_reduce``; ``A float64 [G,3,3]`` or ``None`` for ``A = I``).  Deterministic (fixed summation order)."""
    lib = _lib.load()
    dev = _chk("opt_fire_reduce", force, vel, A, replica, replica_ptr)
    _f32("opt_fire_reduce", force, vel)
    _f64("opt_fire_reduce", A)
    _i32("opt_fire_reduce", replica, replica_ptr)
    n, G = force.size(0), replica_ptr.numel() - 1
    if tuple(force.shape) != (n, 3) or tuple(vel.shape) != (n, 3) or replica.numel() != n:
        raise RuntimeError(f"hermnet_b200.opt_fire_reduce: expected force / vel [{n},3] and replica [{n}]")
    _g9("opt_fire_reduce", G, A)
    sums = (torch.empty if n else torch.zeros)((G, 4), dtype=torch.float64, device=dev)      # (n == 0: the launch is a no-op)
    with torch.cuda.device(dev), _timed("opt_fire_reduce", dev, kernels=2):
        ws_bytes = int(lib.hn_opt_fire_reduce_workspace_bytes(n, G))        # per-chunk partials: caller-owned
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
        _lib.check(lib.hn_opt_fire_reduce(_ptr(force), _ptr(vel), _ptr(A), _ptr(replica), _ptr(replica_ptr), G, n, _ptr(sums),
                                          _ptr(ws), ws_bytes, _stream(dev)), "hn_opt_fire_reduce")
    return sums


def opt_fire_step(sums: Tensor, virial: Optional[Tensor], cell: Optional[Tensor], h0: Optional[Tensor], A: Optional[Tensor],
                  A_prev: Optional[Tensor], vcell: Optional[Tensor], P0: Optional[Tensor], cell_factor: Optional[Tensor],
                  dt: Tensor, alpha: Tensor, n_pos: Tensor, steps: Tensor, converged: Tensor, fmax: float, dt_max: float,
                  max_step: float, move: bool, coef: Tensor, fmax_out: Tensor, n_active: Tensor) -> None:
    """One FIRE step of ``G`` replicas in float64 (``hn_opt_fire_step``): convergence test, mixing, ``dt`` / ``alpha`` /
    ``n_pos`` logic and the closed-form ``max_step`` cap; with ``A`` the three cell rows from ``virial [G,3,3]`` (fp32), the
    cell ``[G,3,3]`` (fp32, rewritten in place as ``h0 A``), target pressure ``P0 [G]`` (eV/A^3) and ``cell_factor [G]``.
    Writes ``coef [G,3]`` (for ``opt_fire_update``), ``fmax_out [G]`` and ``n_active int32 [1]``; ``move=False`` runs the
    convergence test only.  State: ``dt``, ``alpha`` float64 ``[G]``, ``n_pos``, ``steps``, ``converged`` int32 ``[G]``,
    ``A``, ``A_prev``, ``vcell``, ``h0`` float64 ``[G,3,3]``."""
    lib = _lib.load()
    dev = _chk("opt_fire_step", sums, virial, cell, h0, A, A_prev, vcell, P0, cell_factor, dt, alpha, n_pos, steps, converged, coef,
               fmax_out, n_active)
    G = dt.numel()
    _f64("opt_fire_step", sums, h0, A, A_prev, vcell, P0, cell_factor, dt, alpha, coef, fmax_out)
    _f32("opt_fire_step", virial, cell)
    _i32("opt_fire_step", n_pos, steps, converged, n_active)
    if (sums.numel() != 4 * G or coef.numel() != 3 * G or n_active.numel() != 1
            or any(t.numel() != G for t in (alpha, n_pos, steps, converged, fmax_out))):
        raise RuntimeError(f"hermnet_b200.opt_fire_step: expected sums [G={G},4], coef [G,3], dt / alpha / n_pos / steps / "
                           "converged / fmax_out [G] and n_active [1]")
    if A is not None:
        if any(t is None for t in (virial, cell, h0, A_prev, vcell, P0, cell_factor)):
            raise RuntimeError("hermnet_b200.opt_fire_step: the cell rows need virial, cell, h0, A_prev, vcell, P0 and cell_factor")
        _g9("opt_fire_step", G, virial, cell, h0, A, A_prev, vcell)
        if P0.numel() != G or cell_factor.numel() != G:
            raise RuntimeError(f"hermnet_b200.opt_fire_step: expected P0 / cell_factor [G={G}]")
    with torch.cuda.device(dev), _timed("opt_fire_step", dev):
        _lib.check(lib.hn_opt_fire_step(_ptr(sums), _ptr(virial), _ptr(cell), _ptr(h0), _ptr(A), _ptr(A_prev), _ptr(vcell), _ptr(P0),
                                        _ptr(cell_factor), _ptr(dt), _ptr(alpha), _ptr(n_pos), _ptr(steps), _ptr(converged), G,
                                        float(fmax), float(dt_max), float(max_step), int(bool(move)), _ptr(coef), _ptr(fmax_out),
                                        _ptr(n_active), _stream(dev)), "hn_opt_fire_step")
    for t in (dt, alpha, n_pos, steps, converged, coef, fmax_out, n_active) + ((cell, A, A_prev, vcell) if A is not None else ()):
        torch.autograd.graph.increment_version(t)


def opt_fire_update(x: Optional[Tensor], rp: Tensor, vel: Tensor, force: Tensor, A_prev: Optional[Tensor], A: Optional[Tensor],
                    replica: Tensor, converged: Tensor, coef: Tensor) -> None:
    """Atom rows of a FIRE step in place (``hn_opt_fire_update``), for atoms of replicas not converged:
    ``vel = c_v vel + c_f' f A_prev^T``, ``rp += s dt vel``, ``x = rp A``.  ``A = None``: positions only, ``rp`` is the
    positions and ``x`` / ``A_prev`` are unused."""
    lib = _lib.load()
    dev = _chk("opt_fire_update", x, rp, vel, force, A_prev, A, replica, converged, coef)
    _f32("opt_fire_update", x, rp, vel, force)
    _f64("opt_fire_update", A_prev, A, coef)
    _i32("opt_fire_update", replica, converged)
    n, G = rp.size(0), converged.numel()
    if (tuple(rp.shape) != (n, 3) or tuple(vel.shape) != (n, 3) or tuple(force.shape) != (n, 3) or replica.numel() != n
            or coef.numel() != 3 * G):
        raise RuntimeError(f"hermnet_b200.opt_fire_update: expected rp / vel / force [{n},3], replica [{n}] and coef [G={G},3]")
    if A is not None:
        if x is None or A_prev is None or tuple(x.shape) != (n, 3):
            raise RuntimeError(f"hermnet_b200.opt_fire_update: A needs x [{n},3] and A_prev")
        _g9("opt_fire_update", G, A, A_prev)
    with torch.cuda.device(dev), _timed("opt_fire_update", dev):
        _lib.check(lib.hn_opt_fire_update(_ptr(x if A is not None else None), _ptr(rp), _ptr(vel), _ptr(force), _ptr(A_prev),
                                          _ptr(A), _ptr(replica), _ptr(converged), _ptr(coef), n, _stream(dev)),
                   "hn_opt_fire_update")
    for t in (rp, vel) + ((x,) if A is not None else ()):
        torch.autograd.graph.increment_version(t)


# ----------------------------------------------------------------------------------------------------
# tensor-core dense layer (3xTF32 split on tcgen05)
# ----------------------------------------------------------------------------------------------------
def split_tf32(w: Tensor) -> Tuple[Tensor, Tensor]:
    """``w = hi + lo`` with ``hi`` exactly representable in TF32 (low 13 mantissa bits cleared)."""
    w = w.detach().contiguous()
    hi = (w.view(torch.int32) & -8192).view(torch.float32)
    return hi, w - hi


def gemm_supported(K: int, N: int) -> bool:
    return K >= 32 and K % 32 == 0 and N >= 64 and N % 64 == 0


def gemm_tf32x3(a: Tensor, w_hi: Tensor, w_lo: Tensor, bias: Optional[Tensor]) -> Tensor:
    """``a [M,K] @ (w_hi + w_lo)[N,K]^T + bias`` on the tensor cores; ``a`` may be a column slice (row pitch)."""
    lib = _lib.load()
    if a.dim() != 2 or a.stride(1) != 1 or a.stride(0) % 4 != 0 or a.data_ptr() % 16 != 0:
        a = a.contiguous()
    dev = _chk("gemm_tf32x3", w_hi, w_lo, bias)
    require_cuda(a, "gemm_tf32x3")
    _f32("gemm_tf32x3", a, w_hi, w_lo, bias)
    M, K = a.shape
    N = w_hi.size(0)
    out = torch.empty((M, N), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("gemm_tf32x3", dev):
        _lib.check(lib.hn_gemm_tf32x3(_ptr(a), M, K, a.stride(0), _ptr(w_hi), _ptr(w_lo), N, _ptr(bias), _ptr(out), N,
                                      _stream(dev)), "hn_gemm_tf32x3")
    return out


def _rowmajor(name: str, t: Tensor):
    """A 2-D float32 CUDA view whose rows are contiguous (row pitch may exceed the row length)."""
    if t.dim() != 2 or t.stride(1) != 1 or t.stride(0) % 4 != 0 or t.data_ptr() % 16 != 0:
        raise RuntimeError(f"hermnet_b200.{name}: expected a 16-byte aligned 2-D view with contiguous rows")
    require_cuda(t, name)
    _f32(name, t)
    return t


def gemm_tf32x3_ex(a: Tensor, w_hi: Tensor, w_lo: Tensor, bias: Optional[Tensor], out: Optional[Tensor] = None, mode: int = 0,
                   aux: Optional[Tensor] = None, out2: Optional[Tensor] = None) -> Tensor:
    """``epilogue(a @ (w_hi + w_lo)^T + bias)`` written into ``out`` (a row-major view, e.g. a column block of a wider
    buffer); ``mode`` 0 identity / 1 ScaledSiLU with the pre-activation stored in ``out2`` / 2 multiply by
    ScaledSiLU'(``aux``).  All operands may be row-pitched views."""
    lib = _lib.load()
    dev = _chk("gemm_tf32x3_ex", w_hi, w_lo, bias)
    a = _rowmajor("gemm_tf32x3_ex", a)
    M, K = a.shape
    N = w_hi.size(0)
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=dev)
    _rowmajor("gemm_tf32x3_ex", out)
    if aux is not None:
        _rowmajor("gemm_tf32x3_ex", aux)
    if out2 is not None:
        _rowmajor("gemm_tf32x3_ex", out2)
    tname = f"gemm_tf32x3[{M}x{K}->{N},mode{mode}]" if GEMM_SHAPES else "gemm_tf32x3"
    with torch.cuda.device(dev), _timed(tname, dev):
        _lib.check(lib.hn_gemm_tf32x3_ex(_ptr(a), M, K, a.stride(0), _ptr(w_hi), _ptr(w_lo), N, _ptr(bias), _ptr(out), out.stride(0),
                                         int(mode), _ptr(aux), 4 if aux is None else aux.stride(0), _ptr(out2),
                                         4 if out2 is None else out2.stride(0), _stream(dev)), "hn_gemm_tf32x3_ex")
    return out


# ----------------------------------------------------------------------------------------------------
# fused element-wise stages of the node update (csrc/hn_node.cu); every tensor is a contiguous row range
# ----------------------------------------------------------------------------------------------------
def node_pre(x, dx, vec, dvec, xcat, vecp):
    """``dx [n,F]`` / ``dvec [n,3,F]`` may be row-pitched views (slot of ``[N,R,F]`` / ``[N,R,3,F]``)."""
    lib = _lib.load()
    dev = _chk("node_pre", x, vec, xcat, vecp)
    n, F = x.shape
    with torch.cuda.device(dev), _timed("node_elementwise", dev):
        _lib.check(lib.hn_node_pre(n, F, _ptr(x), _ptr(dx), dx.stride(0), _ptr(vec), _ptr(dvec), dvec.stride(0), _ptr(xcat),
                                   _ptr(vecp), _stream(dev)), "hn_node_pre")


def node_mid(v12, vdot, xcat):
    lib = _lib.load()
    dev = _chk("node_mid", v12, vdot, xcat)
    n, F = vdot.shape
    with torch.cuda.device(dev), _timed("node_elementwise", dev):
        _lib.check(lib.hn_node_mid(n, F, _ptr(v12), _ptr(vdot), _ptr(xcat), _stream(dev)), "hn_node_mid")


def node_post(xcat, a, vdot, vecp, v12, x_out, vec_out):
    lib = _lib.load()
    dev = _chk("node_post", xcat, a, vdot, vecp, v12, x_out, vec_out)
    n, F = vdot.shape
    with torch.cuda.device(dev), _timed("node_elementwise", dev):
        _lib.check(lib.hn_node_post(n, F, _ptr(xcat), _ptr(a), _ptr(vdot), _ptr(vecp), _ptr(v12), _ptr(x_out), _ptr(vec_out),
                                    _stream(dev)), "hn_node_post")


def node_post_bwd(g_x, g_vec, a, vdot, v12, g_a, g_vdot, g_v12):
    lib = _lib.load()
    dev = _chk("node_post_bwd", g_x, g_vec, a, vdot, v12, g_a, g_vdot, g_v12)
    n, F = vdot.shape
    with torch.cuda.device(dev), _timed("node_elementwise", dev):
        _lib.check(lib.hn_node_post_bwd(n, F, _ptr(g_x), _ptr(g_vec), _ptr(a), _ptr(vdot), _ptr(v12), _ptr(g_a), _ptr(g_vdot),
                                        _ptr(g_v12), _stream(dev)), "hn_node_post_bwd")


def node_mid_bwd(g_vdot, g_cat, v12, vn, g_v12):
    """``vn`` may be the second half of the saved ``xcat`` (row pitch 2F)."""
    lib = _lib.load()
    dev = _chk("node_mid_bwd", g_vdot, g_cat, v12, g_v12)
    n, F = g_vdot.shape
    with torch.cuda.device(dev), _timed("node_elementwise", dev):
        _lib.check(lib.hn_node_mid_bwd(n, F, _ptr(g_vdot), _ptr(g_cat), _ptr(v12), _ptr(vn), vn.stride(0), _ptr(g_v12),
                                       _stream(dev)), "hn_node_mid_bwd")


def node_pre_bwd(g_xn, g_cat, g_vecn, g_vecp, g_x, g_vec):
    lib = _lib.load()
    dev = _chk("node_pre_bwd", g_xn, g_cat, g_vecn, g_vecp, g_x, g_vec)
    n, F = g_xn.shape
    with torch.cuda.device(dev), _timed("node_elementwise", dev):
        _lib.check(lib.hn_node_pre_bwd(n, F, _ptr(g_xn), _ptr(g_cat), _ptr(g_vecn), _ptr(g_vecp), _ptr(g_x), _ptr(g_vec),
                                       _stream(dev)), "hn_node_pre_bwd")


# ----------------------------------------------------------------------------------------------------
# tensor-core edge kernels (csrc/hn_edge_tc.cu): tile plan, weight split, forward / backward
# ----------------------------------------------------------------------------------------------------
def tc_supported(hidden: int, num_rbf: int) -> bool:
    return bool(_lib.load().hn_tc_supported(int(hidden), int(num_rbf)))


def tc_block_rows(src_major: bool = False) -> int:
    return int(_lib.load().hn_tc_block_rows(1 if src_major else 0))


def tc_groups() -> int:
    return int(_lib.load().hn_tc_groups())


def tc_split_weights(Wt: Tensor):
    """``Wt [M,K,3F]`` -> fp16 (hi | lo) rows ``[M*3F, 2, K32]`` scaled by a per-module power of two, ``wscale [M]``."""
    lib = _lib.load()
    dev = _chk("tc_split_weights", Wt)
    _f32("tc_split_weights", Wt)
    M, K, F3 = Wt.shape
    n = int(lib.hn_tc_split_weights_elems(M, F3 // 3, K))
    wsplit = torch.empty(n, dtype=torch.float16, device=dev)
    wscale = torch.empty(M, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("tc_split_weights", dev):
        _lib.check(lib.hn_tc_split_weights(_ptr(Wt), M, K, F3 // 3, _ptr(wsplit), _ptr(wscale), _stream(dev)), "hn_tc_split_weights")
    return wsplit, wscale


def tc_basis_index(geom: Tensor, inv_rc: float, num_rbf: int) -> Tensor:
    lib = _lib.load()
    dev = _chk("tc_basis_index", geom)
    kc = torch.empty(geom.size(0), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev), _timed("tc_plan", dev):
        _lib.check(lib.hn_tc_basis_index(_ptr(geom), geom.size(0), float(inv_rc), int(num_rbf), _ptr(kc), _stream(dev)),
                   "hn_tc_basis_index")
    return kc


def tc_plan_records(g, geom: Tensor, inv_rc: float, num_rbf: int, src_major: bool, atom_local: Optional[Tensor], src_block: int):
    """``(rec int32 [E,4], kc int32 [E], sub int32 [E])`` of a plan in one pass over the row-edges (``hn_tc_plan_records``)."""
    lib = _lib.load()
    dev = _chk("tc_plan_records", g.edge_row, g.col, g.row_xoff, g.row_mod, atom_local, geom)
    _i32("tc_plan_records", g.edge_row, g.col, g.row_mod, atom_local)
    E = int(g.n_edges)
    rec = torch.empty((max(E, 1), 4), dtype=torch.int32, device=dev)
    kc = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
    sub = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev), _timed("tc_plan", dev):
        _lib.check(lib.hn_tc_plan_records(int(bool(src_major)), _ptr(g.edge_row), _ptr(g.col), _ptr(g.row_xoff), _ptr(g.row_mod),
                                          _ptr(atom_local), int(g.rows_per_atom), int(src_block), _ptr(geom), float(inv_rc),
                                          int(num_rbf), E, _ptr(rec), _ptr(kc), _ptr(sub), _stream(dev)), "hn_tc_plan_records")
    return rec[:E], kc[:E], sub[:E]


def tc_plan_sort(in_ptr: Tensor, ids: Optional[Tensor], kc: Tensor, sub: Optional[Tensor], n_seg: int, n_sub: int, num_rbf: int):
    """Segment-local sort of the plan builder (``hn_tc_plan_sort``): returns ``(order int32 [n_live], grp_ptr int32
    [n_seg * n_sub + 1])`` -- edge ids ordered by (segment, sub, kc) without the dropped (sub < 0) entries, and the start of
    every (segment, sub) group in it.  One host-free count pass, a cumsum, one fill pass."""
    lib = _lib.load()
    dev = _chk("tc_plan_sort", in_ptr, ids, kc, sub)
    _i32("tc_plan_sort", in_ptr, ids, kc, sub)
    counts = torch.zeros(max(n_seg * n_sub, 1), dtype=torch.int32, device=dev)
    grp_ptr = torch.zeros(n_seg * n_sub + 1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev), _timed("tc_plan", dev):
        _lib.check(lib.hn_tc_plan_sort(_ptr(in_ptr), _ptr(ids), _ptr(kc), _ptr(sub), n_seg, n_sub, int(num_rbf), _ptr(counts), None, None,
                                       _stream(dev)), "hn_tc_plan_sort")
        torch.cumsum(counts[: n_seg * n_sub], 0, dtype=torch.int32, out=grp_ptr[1:])
        out_base = grp_ptr[:: n_sub][:n_seg].contiguous()
        order = torch.empty(max(int(kc.numel()), 1), dtype=torch.int32, device=dev)
        _lib.check(lib.hn_tc_plan_sort(_ptr(in_ptr), _ptr(ids), _ptr(kc), _ptr(sub), n_seg, n_sub, int(num_rbf), None, _ptr(out_base),
                                       _ptr(order), _stream(dev)), "hn_tc_plan_sort")
    return order, grp_ptr


def tc_plan_count(order: Tensor, kc: Tensor, grp_ptr: Tensor, n_groups: int, num_rbf: int, window: int = 32) -> Tensor:
    lib = _lib.load()
    dev = _chk("tc_plan_count", order, kc, grp_ptr)
    _i32("tc_plan_count", order, kc, grp_ptr)
    counts = torch.zeros(n_groups, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev), _timed("tc_plan", dev):
        _lib.check(lib.hn_tc_plan_count(_ptr(order), _ptr(kc), _ptr(grp_ptr), n_groups, int(num_rbf), int(window), _ptr(counts), _stream(dev)),
                   "hn_tc_plan_count")
    return counts


def tc_plan_fill(order: Tensor, kc: Tensor, grp_ptr: Tensor, n_groups: int, num_rbf: int, grp_tile: Tensor, n_tiles: int,
                 window: int = 32) -> Tensor:
    lib = _lib.load()
    dev = _chk("tc_plan_fill", order, kc, grp_ptr, grp_tile)
    _i32("tc_plan_fill", order, kc, grp_ptr, grp_tile)
    tile_start = torch.empty(max(n_tiles, 1), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev), _timed("tc_plan", dev):
        _lib.check(lib.hn_tc_plan_fill(_ptr(order), _ptr(kc), _ptr(grp_ptr), n_groups, int(num_rbf), int(window), _ptr(grp_tile), _ptr(tile_start),
                                       _stream(dev)), "hn_tc_plan_fill")
    return tile_start


def tc_plan_finalize(order: Tensor, tile_start: Tensor, n_tiles: int, n_edges: int, rec: Tensor, tile_mod: Tensor):
    lib = _lib.load()
    dev = _chk("tc_plan_finalize", order, tile_start, rec, tile_mod)
    _i32("tc_plan_finalize", order, tile_start, rec, tile_mod)
    erec = torch.empty((max(n_edges, 1), 4), dtype=torch.int32, device=dev)
    tile_info = torch.empty((max(n_tiles, 1), 4), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev), _timed("tc_plan", dev):
        _lib.check(lib.hn_tc_plan_finalize(_ptr(order), _ptr(tile_start), n_tiles, n_edges, _ptr(rec), _ptr(tile_mod), _ptr(erec),
                                           _ptr(tile_info), _stream(dev)), "hn_tc_plan_finalize")
    return erec, tile_info


def tc_tile_windows(plan, geom: Tensor, inv_rc: float, num_rbf: int, live: Optional[Tensor] = None) -> None:
    lib = _lib.load()
    dev = _chk("tc_tile_windows", geom, live)
    if live is not None and (live.dtype != torch.uint8 or live.numel() != geom.size(0)):
        raise TypeError("hermnet_b200.tc_tile_windows: live must be uint8 [E]")
    with torch.cuda.device(dev), _timed("tc_tile_windows", dev):
        _lib.check(lib.hn_tc_tile_windows(ctypes.byref(plan.cstruct()), _ptr(geom), _ptr(live), float(inv_rc), int(num_rbf),
                                          _stream(dev)), "hn_tc_tile_windows")


def tc_edge_fwd(p: EdgeParams, plan, xh, vec, geom, wsplit, wscale, bias, offset, n_rows: int, debug_phi: bool = False):
    lib = _lib.load()
    dev = _chk("tc_edge_fwd", xh, vec, geom, wsplit, wscale, bias, offset)
    _f32("tc_edge_fwd", xh, vec, geom, wscale, bias, offset)
    F = p.hidden
    dx = torch.empty((n_rows, F), dtype=torch.float32, device=dev)
    dvec = torch.empty((n_rows, 3, F), dtype=torch.float32, device=dev)
    E = geom.size(0)
    dbg = torch.zeros(2 * E * 3 * F + 14336, dtype=torch.float32, device=dev) if debug_phi else None
    with torch.cuda.device(dev), _timed("painn_edge_fwd", dev):
        _lib.check(lib.hn_tc_edge_fwd(ctypes.byref(p), ctypes.byref(plan.cstruct()), _ptr(xh), _ptr(vec), _ptr(geom), _ptr(wsplit),
                                      _ptr(wscale), _ptr(bias), _ptr(offset), _ptr(dx), _ptr(dvec), _ptr(dbg), E, _stream(dev)),
                   "hn_tc_edge_fwd")
    return (dx, dvec, dbg) if debug_phi else (dx, dvec)


def tc_edge_bwd_dst(p: EdgeParams, plan, xh, vec, geom, wsplit, wscale, bias, offset, g_dx, g_dvec):
    lib = _lib.load()
    dev = _chk("tc_edge_bwd_dst", xh, vec, geom, wsplit, wscale, bias, offset, g_dx, g_dvec)
    _f32("tc_edge_bwd_dst", xh, vec, geom, wscale, bias, offset, g_dx, g_dvec)
    alloc = torch.zeros if plan.has_inactive else torch.empty
    g_geom = alloc((1, geom.size(0), 4), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("painn_edge_bwd_dst", dev):
        _lib.check(lib.hn_tc_edge_bwd_dst(ctypes.byref(p), ctypes.byref(plan.cstruct()), _ptr(xh), _ptr(vec), _ptr(geom), _ptr(wsplit),
                                          _ptr(wscale), _ptr(bias), _ptr(offset), _ptr(g_dx), _ptr(g_dvec), _ptr(g_geom),
                                          _stream(dev)), "hn_tc_edge_bwd_dst")
    return g_geom


def tc_edge_bwd_src(p: EdgeParams, plan, xh, vec, geom, wsplit, wscale, bias, offset, g_dx, g_dvec):
    lib = _lib.load()
    dev = _chk("tc_edge_bwd_src", xh, vec, geom, wsplit, wscale, bias, offset, g_dx, g_dvec)
    _f32("tc_edge_bwd_src", xh, vec, geom, wscale, bias, offset, g_dx, g_dvec)
    grad_xh = torch.zeros_like(xh)
    grad_vec = torch.empty_like(vec)
    with torch.cuda.device(dev), _timed("painn_edge_bwd_src", dev):
        _lib.check(lib.hn_tc_edge_bwd_src(ctypes.byref(p), ctypes.byref(plan.cstruct()), _ptr(xh), _ptr(vec), _ptr(geom), _ptr(wsplit),
                                          _ptr(wscale), _ptr(bias), _ptr(offset), _ptr(g_dx), _ptr(g_dvec), _ptr(grad_xh),
                                          _ptr(grad_vec), _stream(dev)), "hn_tc_edge_bwd_src")
    return grad_xh, grad_vec
