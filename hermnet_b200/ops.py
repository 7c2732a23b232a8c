"""Tensor-level wrappers over the C ABI (``include/hermnet_b200.h``).

Each function takes CUDA torch tensors (torch is only the owner of device memory and of the stream),
passes raw pointers + the current stream through ctypes and returns freshly allocated outputs.  There is
no CPU implementation: a non-CUDA tensor raises.  The autograd layer (``functional.py``) and the graph
builder (``graph.py``) call these through the module namespace (``ops.<name>``).
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import EdgeParams

Tensor = torch.Tensor


def _stream(dev) -> ctypes.c_void_p:
    # the raw handle of torch.cuda.current_stream(dev), without building a torch Stream object (about 2.5 us of host time a call)
    return ctypes.c_void_p(torch._C._cuda_getCurrentRawStream(dev.index))


_DTYPE_RULE = {torch.float32: "float tensors must be float32", torch.int32: "index tensors must be int32",
               torch.int64: "seed / step tensors must be int64", torch.float64: "optimizer state tensors must be float64"}


def _chk(name: str, *tensors, f32=(), i32=(), i64=(), f64=()):
    """Device of the CUDA tensors ``tensors``, ``f32``, ``i32``, ``i64`` and ``f64`` (``None`` entries are skipped): all must
    be contiguous and on one device, and those of a dtype group must have that dtype."""
    dev = None
    for dtype, group in ((None, tensors), (torch.float32, f32), (torch.int32, i32), (torch.int64, i64), (torch.float64, f64)):
        for t in group:
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
            if dtype is not None and t.dtype != dtype:
                raise RuntimeError(f"hermnet_b200.{name}: {_DTYPE_RULE[dtype]} (got {t.dtype})")
    return dev


def _live(name: str, live, n_edges: int) -> None:
    """The mask of a Verlet-skin list: uint8 [E], 0 marks an entry the kernels must skip."""
    if not isinstance(live, torch.Tensor) or live.dtype != torch.uint8 or live.numel() != n_edges:
        raise TypeError(f"hermnet_b200.{name}: live must be uint8 [E]")


def _bump(*tensors) -> None:
    """Tensors a kernel wrote through raw pointers: version-keyed caches (graphs, signed geometry, tile windows) must see the
    change."""
    for t in tensors:
        if t is not None:
            torch.autograd.graph.increment_version(t)


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


def _call(sym: str, dev, *args) -> None:
    """``sym(*args, stream)`` on the current stream of ``dev``; a non-zero return raises with the library's message."""
    _lib.check(getattr(_lib.load(), sym)(*args, _stream(dev)), sym)


def _launch(sym: str, dev, timer: str, *args, kernels: int = 1) -> None:
    """``_call`` on device ``dev``, counted as ``kernels`` launches and timed under ``timer`` (``TIMERS``, ``LAUNCHES``)."""
    with torch.cuda.device(dev), _timed(timer, dev, kernels):
        _call(sym, dev, *args)


def sm_count() -> int:
    return int(_lib.load().hn_device_sm_count())


# ----------------------------------------------------------------------------------------------------
# graph construction
# ----------------------------------------------------------------------------------------------------
def radius_graph(pos: Tensor, cell: Optional[Tensor], graph_ptr: Tensor, rc: float, group: Optional[Tensor] = None,
                 n_groups: int = 1, max_neighbors: int = 0) -> Tuple[Tensor, Tensor, Tensor]:
    """Row CSR of the neighbour list: row ``c*n_groups+g`` = neighbours ``(j, S)`` of centre ``c`` in group ``g``.
    Returns ``rowptr int32 [N*n_groups+1]``, ``col int32 [E]``, ``shift int8 [E,4]``.  One host sync (E)."""
    dev = _chk("radius_graph", f32=(pos, cell), i32=(graph_ptr, group))
    n = pos.size(0)
    n_graphs = graph_ptr.numel() - 1
    with torch.cuda.device(dev):
        ws_bytes = int(_lib.load().hn_radius_graph_workspace_bytes(n, n_graphs))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        counts = torch.empty(n * n_groups, dtype=torch.int32, device=dev)
        LAUNCHES["n"] += 6
        _call("hn_radius_graph_count", dev, pos, n, cell, graph_ptr, n_graphs, float(rc), group, n_groups, max_neighbors, counts,
              ws, ws_bytes)
        rowptr = torch.zeros(n * n_groups + 1, dtype=torch.int32, device=dev)
        torch.cumsum(counts, 0, dtype=torch.int32, out=rowptr[1:])
        n_edges = int(rowptr[-1].item())
        col = torch.empty(n_edges, dtype=torch.int32, device=dev)
        shift = torch.empty((n_edges, 4), dtype=torch.int8, device=dev)
        if n_edges > 0:
            LAUNCHES["n"] += 1
            _call("hn_radius_graph_fill", dev, pos, n, cell, graph_ptr, n_graphs, float(rc), group, n_groups, max_neighbors, rowptr,
                  col, shift, ws, ws_bytes)
    return rowptr, col, shift


def sort_by_key(keys: Tensor, n_keys: int) -> Tuple[Tensor, Tensor]:
    """Stable grouping of ``arange(len(keys))`` by key: ``rowptr int32 [n_keys+1]``, ``order int32 [n]``."""
    dev = _chk("sort_by_key", i32=(keys,))
    n = keys.numel()
    with torch.cuda.device(dev):
        ws_bytes = int(_lib.load().hn_sort_by_key_workspace_bytes(n, n_keys))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        rowptr = torch.empty(n_keys + 1, dtype=torch.int32, device=dev)
        order = torch.empty(n, dtype=torch.int32, device=dev)
        LAUNCHES["n"] += 1
        _call("hn_sort_by_key", dev, keys, n, n_keys, rowptr, order, ws, ws_bytes)
    return rowptr, order


def expand_rowptr(rowptr: Tensor, n_edges: int) -> Tensor:
    dev = _chk("expand_rowptr", i32=(rowptr,))
    out = torch.empty(n_edges, dtype=torch.int32, device=dev)
    _launch("hn_expand_rowptr", dev, "expand_rowptr", rowptr, rowptr.numel() - 1, out)
    return out


def triplets(rowptr: Tensor, col: Tensor, src_type: Optional[Tensor] = None, type_a: int = -1, type_c: int = -1):
    """Canonical ordered triplets over row-edge ids: ``trip_ptr int64 [R+1]``, ``e1``, ``e2`` int32 [T]."""
    dev = _chk("triplets", i32=(rowptr, col, src_type))
    n_rows = rowptr.numel() - 1
    with torch.cuda.device(dev):
        counts = torch.empty(n_rows, dtype=torch.int64, device=dev)
        _call("hn_triplets_count", dev, rowptr, n_rows, col, src_type, type_a, type_c, counts)
        trip_ptr = torch.zeros(n_rows + 1, dtype=torch.int64, device=dev)
        torch.cumsum(counts, 0, out=trip_ptr[1:])
        total = int(trip_ptr[-1].item())
        e1 = torch.empty(total, dtype=torch.int32, device=dev)
        e2 = torch.empty(total, dtype=torch.int32, device=dev)
        if total > 0:
            _call("hn_triplets_fill", dev, rowptr, n_rows, col, src_type, type_a, type_c, trip_ptr, e1, e2)
    return trip_ptr, e1, e2


def triplet_dots(m_vec: Tensor, trip_ptr: Tensor, e1: Tensor, e2: Tensor) -> Tensor:
    dev = _chk("triplet_dots", trip_ptr, e1, e2, f32=(m_vec,))
    F = m_vec.size(-1)
    n_rows = trip_ptr.numel() - 1
    out = torch.empty((n_rows, F), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _call("hn_triplet_dots", dev, m_vec, F, trip_ptr, e1, e2, n_rows, out)
    return out


# ----------------------------------------------------------------------------------------------------
# geometry
# ----------------------------------------------------------------------------------------------------
def edge_geom_fwd(pos: Tensor, cell: Optional[Tensor], g) -> Tensor:
    dev = _chk("edge_geom_fwd", f32=(pos, cell))
    geom = torch.empty((g.n_edges, 4), dtype=torch.float32, device=dev)
    _launch("hn_edge_geom_fwd", dev, "edge_geom_fwd", pos, cell, g.atom_graph, g.edge_row, g.rows_per_atom, g.col,
            g.shift if cell is not None else None, float(g.sign), g.n_edges, geom)
    return geom


def edge_geom_bwd(geom: Tensor, g_geom: Tensor, g, want_cell: bool):
    """``g_geom`` is ``[n_parts, E, 4]``; returns ``grad_pos [N,3]`` and the per-atom virial partial ``[N,9]``."""
    dev = _chk("edge_geom_bwd", f32=(geom, g_geom))
    n_parts = g_geom.size(0) if g_geom.dim() == 3 else 1
    grad_pos = torch.empty((g.n_atoms, 3), dtype=torch.float32, device=dev)
    cellw = torch.empty((g.n_atoms, 9), dtype=torch.float32, device=dev) if want_cell else None
    _launch("hn_edge_geom_bwd", dev, "edge_geom_bwd", geom, g_geom, n_parts, g.shift, g.rowptr, g.rows_per_atom, g.t_rowptr,
            g.t_eid, float(g.sign), g.n_atoms, g.n_edges, grad_pos, cellw)
    return grad_pos, cellw


def edge_virial_atom(geom: Tensor, g_geom: Tensor, g) -> Tensor:
    """Per-atom virial ``[N, 9]`` (internal atom order, row = position component) from ``geom [E,4]`` and its gradient
    ``g_geom [E,4]``: each edge gives ``-1/2 D_e (x) dE/dD_e`` to both of its atoms."""
    dev = _chk("edge_virial_atom", f32=(geom, g_geom))
    if tuple(geom.shape) != (g.n_edges, 4) or tuple(g_geom.shape) != (g.n_edges, 4):
        raise RuntimeError(f"hermnet_b200.edge_virial_atom: geom / g_geom must be [{g.n_edges}, 4]")
    virial = torch.empty((g.n_atoms, 9), dtype=torch.float32, device=dev)
    _launch("hn_edge_virial_atom", dev, "edge_virial_atom", geom, g_geom, g.rowptr, g.rows_per_atom, g.t_rowptr, g.t_eid,
            g.n_atoms, g.n_edges, virial)
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


# 'auto': tensor-core kernels (hn_edge_tc.cu) where supported (F == 128), else the tile-sweep kernels (F % 64 == 0), else
# the row-per-warp kernels; 'quad' / 'row' pin the older families (A/B measurements, tests).  HERMNET_B200_EDGE presets it.
_EDGE_VARIANTS = ("auto", "tc", "quad", "row")
EDGE_VARIANT = {"v": os.environ["HERMNET_B200_EDGE"] if os.environ.get("HERMNET_B200_EDGE") in _EDGE_VARIANTS else "auto"}


def edge_set_variant(variant: str) -> None:
    """'auto' / 'tc': tensor-core edge kernels where supported; 'quad': tile-sweep kernels; 'row': row-per-warp kernels."""
    if variant not in _EDGE_VARIANTS:
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
    _live(name, live, geom.size(0))
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
    _stamp(p)
    dev = _chk("painn_edge_fwd", f32=(xh, vec, geom, Wt, bias, offset))
    F = p.hidden
    dx = torch.empty((p.n_rows, F), dtype=torch.float32, device=dev)
    dvec = torch.empty((p.n_rows, 3, F), dtype=torch.float32, device=dev)
    _launch("hn_painn_edge_fwd", dev, "painn_edge_fwd", ctypes.byref(p), xh, vec, geom, g.rowptr, g.col, g.row_mod, g.row_xoff, Wt,
            bias, offset, dx, dvec)
    return dx, dvec


def painn_edge_bwd_dst(p: EdgeParams, xh, vec, geom, g, Wt, bias, offset, g_dx, g_dvec):
    geom = _kernel_geom("painn_edge_bwd_dst", p, geom)      # first: a missing mask is the error to report
    _stamp(p)
    dev = _chk("painn_edge_bwd_dst", f32=(xh, vec, geom, Wt, bias, offset, g_dx, g_dvec))
    g_geom = torch.empty((edge_num_slices(p.hidden), g.n_edges, 4), dtype=torch.float32, device=dev)
    _launch("hn_painn_edge_bwd_dst", dev, "painn_edge_bwd_dst", ctypes.byref(p), xh, vec, geom, g.rowptr, g.col, g.row_mod,
            g.row_xoff, Wt, bias, offset, g_dx, g_dvec, g_geom, g.n_edges)
    return g_geom


def painn_edge_bwd_src(p: EdgeParams, xh, vec, geom, g, Wt, bias, offset, g_dx, g_dvec):
    geom = _kernel_geom("painn_edge_bwd_src", p, geom)      # first: a missing mask is the error to report
    _stamp(p)
    dev = _chk("painn_edge_bwd_src", f32=(xh, vec, geom, Wt, bias, offset, g_dx, g_dvec))
    grad_xh = torch.zeros_like(xh)
    grad_vec = torch.empty_like(vec)
    _launch("hn_painn_edge_bwd_src", dev, "painn_edge_bwd_src", ctypes.byref(p), xh, vec, geom, g.t_rowptr, g.t_eid, g.edge_row,
            g.row_mod, g.row_xoff, Wt, bias, offset, g_dx, g_dvec, grad_xh, grad_vec)
    return grad_xh, grad_vec


def painn_edge_bwd_w(p: EdgeParams, xh, vec, geom, g, offset, g_dx, g_dvec):
    """Gradients of the filter projection: ``gWt [M,K,3F]``, ``gb [M,3F]`` (partials reduced in fixed order).  A Verlet-skin
    list (``p.flags`` bit 0) needs ``p.live``, the uint8 [E] mask the model attaches next to the flag: entries marked 0
    contribute nothing."""
    live = getattr(p, "live", None) if p.flags & 1 else None
    dev = _chk("painn_edge_bwd_w", live, f32=(xh, vec, geom, offset, g_dx, g_dvec))
    if live is not None:
        _live("painn_edge_bwd_w", live, geom.size(0))
    M, K, F3 = p.n_modules, p.num_rbf, 3 * p.hidden
    n_chunks = max(1, min(p.n_rows, (2 * max(sm_count(), 1)) // max(M, 1)))
    gW = torch.empty((n_chunks, M, K, F3), dtype=torch.float32, device=dev)
    gb = torch.empty((n_chunks, M, F3), dtype=torch.float32, device=dev)
    _launch("hn_painn_edge_bwd_w", dev, "painn_edge_bwd_w", ctypes.byref(p), xh, vec, geom, g.rowptr, g.col, g.row_mod, g.row_xoff,
            live, offset, g_dx, g_dvec, gW, gb, n_chunks)
    return gW.sum(0), gb.sum(0)


# ----------------------------------------------------------------------------------------------------
# gather / segmented sum
# ----------------------------------------------------------------------------------------------------
def gather_rows(X: Tensor, idx: Tensor) -> Tensor:
    dev = _chk("gather_rows", f32=(X,), i32=(idx,))
    C = X.size(1)
    out = torch.empty((idx.numel(), C), dtype=torch.float32, device=dev)
    _launch("hn_gather_rows", dev, "gather_rows", X, idx, idx.numel(), C, out)
    return out


def layer0_row_len(n_elem: int, num_rbf: int) -> int:
    """Length of a basis-sum row of the first-layer pass: ``n_elem * (K + 1)`` sums, padded to a GEMM-friendly multiple."""
    pad = int(os.environ.get("HERMNET_B200_L0_PAD", "128"))
    return (n_elem * (num_rbf + 1) + pad - 1) // pad * pad


def _params_ptr(p: EdgeParams) -> ctypes.c_void_p:
    """Address of ``p`` for the ``hn_layer0_basis_*`` entry points, whose ctypes table types the params as a plain pointer."""
    return ctypes.c_void_p(ctypes.addressof(p))


def layer0_basis_fwd(p: EdgeParams, g, geom: Tensor, live: Optional[Tensor], offset: Tensor, n_elem: int, kp: int):
    """``(Sa [R,kp], Sc [R,3,kp])``: per-(destination row, source element) sums of the radial basis (``hn_layer0_basis_fwd``);
    ``g.col`` holds the element index of every row-edge's source."""
    dev = _chk("layer0_basis_fwd", live, i32=(g.rowptr, g.col, g.row_mod), f32=(geom, offset))
    R = int(p.n_rows)
    Sa = torch.empty((R, kp), dtype=torch.float32, device=dev)
    Sc = torch.empty((R, 3, kp), dtype=torch.float32, device=dev)
    _launch("hn_layer0_basis_fwd", dev, "layer0_basis_fwd", _params_ptr(p), g.rowptr, g.col, g.row_mod, geom, live, offset,
            int(n_elem), int(kp), Sa, Sc)
    return Sa, Sc


def layer0_basis_bwd(p: EdgeParams, g, geom: Tensor, live: Optional[Tensor], offset: Tensor, n_elem: int, kp: int, g_Sa: Tensor,
                     g_Sc: Tensor) -> Tensor:
    dev = _chk("layer0_basis_bwd", g.rowptr, g.col, g.row_mod, live, f32=(geom, offset, g_Sa, g_Sc))
    g_geom = torch.empty((geom.size(0), 4), dtype=torch.float32, device=dev)
    _launch("hn_layer0_basis_bwd", dev, "layer0_basis_bwd", _params_ptr(p), g.rowptr, g.col, g.row_mod, geom, live, offset,
            int(n_elem), int(kp), g_Sa, g_Sc, g_geom)
    return g_geom


def layernorm_fwd(x: Tensor, eps: float):
    """``(xhat, mean [n], rstd [n])`` of the affine-free LayerNorm over the last dimension (``hn_layernorm_fwd``)."""
    dev = _chk("layernorm_fwd", f32=(x,))
    n, F = x.shape
    xhat = torch.empty_like(x)
    mean = torch.empty(n, dtype=torch.float32, device=dev)
    rstd = torch.empty(n, dtype=torch.float32, device=dev)
    _launch("hn_layernorm_fwd", dev, "node_elementwise", x, n, F, float(eps), xhat, mean, rstd)
    return xhat, mean, rstd


def layernorm_bwd(g_xhat: Tensor, x: Tensor, mean: Tensor, rstd: Tensor) -> Tensor:
    dev = _chk("layernorm_bwd", f32=(g_xhat, x, mean, rstd))
    n, F = x.shape
    g_x = torch.empty_like(x)
    _launch("hn_layernorm_bwd", dev, "node_elementwise", g_xhat, x, mean, rstd, n, F, g_x)
    return g_x


def readout_fwd(x: Tensor, W1: Tensor, b1: Tensor, W2: Tensor, b2: Tensor) -> Tensor:
    """``e_atom [N,1] = W2 . ssilu(W1 x + b1) + b2`` in plain fp32 (hn_readout_fwd)."""
    dev = _chk("readout_fwd", f32=(x, W1, b1, W2, b2))
    out = torch.empty((x.size(0), 1), dtype=torch.float32, device=dev)
    _launch("hn_readout_fwd", dev, "readout", x, W1, b1, W2, b2, x.size(0), x.size(1), out)
    return out


def readout_bwd(x: Tensor, W1: Tensor, b1: Tensor, W2: Tensor, b2: Tensor, g_e: Tensor) -> Tensor:
    dev = _chk("readout_bwd", f32=(x, W1, b1, W2, b2, g_e))
    g_x = torch.empty_like(x)
    _launch("hn_readout_bwd", dev, "readout", x, W1, b1, W2, b2, g_e, x.size(0), x.size(1), g_x)
    return g_x


def halo_pack(x: Tensor, vec: Tensor, src_idx: Tensor, row_peer: Tensor, row_slot: Tensor, dst_base: Tensor) -> None:
    """Rows ``[x | vec]`` of the atoms ``src_idx`` stored at ``dst_base[row_peer[i]] + row_slot[i] * 4F`` floats (device
    addresses: peers' landing buffers over NVLink, or slices of a local send buffer)."""
    dev = _chk("halo_pack", dst_base, f32=(x, vec), i32=(src_idx, row_peer, row_slot))
    if dst_base.dtype != torch.int64:
        raise TypeError("hermnet_b200.halo_pack: dst_base must be int64 device addresses")
    _launch("hn_halo_pack", dev, "halo_pack", x, vec, src_idx, row_peer, row_slot, dst_base, src_idx.numel(), x.size(1))


def halo_unpack(buf: Tensor, dst_idx: Tensor, x: Tensor, vec: Tensor) -> None:
    """Row ``i`` of ``buf [n, 4F]`` -> ``x[dst_idx[i]]``, ``vec[dst_idx[i]]`` (in place)."""
    dev = _chk("halo_unpack", f32=(buf, x, vec), i32=(dst_idx,))
    _launch("hn_halo_unpack", dev, "halo_unpack", buf, dst_idx, dst_idx.numel(), x.size(1), x, vec)


def segment_sum(Y: Tensor, rowptr: Tensor, perm: Optional[Tensor], n_rows: int) -> Tensor:
    dev = _chk("segment_sum", f32=(Y,), i32=(rowptr, perm))
    C = Y.size(1)
    out = torch.empty((n_rows, C), dtype=torch.float32, device=dev)
    ws_bytes = int(_lib.load().hn_segment_sum_workspace_bytes(n_rows, C))      # chunk partials of long rows: caller-owned
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
    _launch("hn_segment_sum", dev, "segment_sum", Y, rowptr, perm, n_rows, C, out, ws, ws_bytes)
    return out


# ----------------------------------------------------------------------------------------------------
# Langevin and constant-pressure MD steps (csrc/hn_md.cu)
# ----------------------------------------------------------------------------------------------------
def _md_shapes(name, n: int, vel: Tensor, force: Tensor, inv_mass: Tensor):
    if tuple(vel.shape) != (n, 3) or tuple(force.shape) != (n, 3) or inv_mass.numel() != n:
        raise RuntimeError(f"hermnet_b200.{name}: expected vel / force [{n},3] and inv_mass [{n}]")


def md_langevin_baoa(pos: Tensor, vel: Tensor, force: Tensor, inv_mass: Tensor, replica: Tensor, replica_ptr: Tensor,
                     kT: Tensor, seed: Tensor, step: Tensor, c1: float, c2: float, dt: float) -> None:
    """B-A-O-A half of a BAOAB Langevin step, in place on ``pos`` / ``vel [N,3]`` (``hn_md_langevin_baoa``): ``replica int32
    [N]``, ``replica_ptr int32 [G+1]`` (contiguous replicas), per-replica ``kT float32 [G]`` (eV) and ``seed int64 [G]``,
    ``step int64 [1]`` (read, not advanced).  ``c1 = exp(-gamma dt)``, ``c2 = sqrt(1 - c1^2)``."""
    dev = _chk("md_langevin_baoa", f32=(pos, vel, force, inv_mass, kT), i32=(replica, replica_ptr), i64=(seed, step))
    n, G = pos.size(0), replica_ptr.numel() - 1
    _md_shapes("md_langevin_baoa", n, vel, force, inv_mass)
    if tuple(pos.shape) != (n, 3) or replica.numel() != n or kT.numel() != G or seed.numel() != G or step.numel() != 1:
        raise RuntimeError(f"hermnet_b200.md_langevin_baoa: expected pos [N,3], replica [N], kT / seed [G={G}], step [1]")
    _launch("hn_md_langevin_baoa", dev, "md_langevin_baoa", pos, vel, force, inv_mass, replica, replica_ptr, G, kT, seed, step,
            float(c1), float(c2), float(dt), n)
    _bump(pos, vel)


def md_kick(vel: Tensor, force: Tensor, inv_mass: Tensor, half_dt: float, kinetic: Optional[Tensor], step: Tensor) -> None:
    """Closing B of a BAOAB step, in place on ``vel [N,3]`` (``hn_md_kick``); ``kinetic [N]`` (optional) receives
    ``1/2 |v_i|^2 / inv_m_i`` in eV; ``step int64 [1]`` is advanced by one."""
    dev = _chk("md_kick", f32=(vel, force, inv_mass, kinetic), i64=(step,))
    n = vel.size(0)
    _md_shapes("md_kick", n, vel, force, inv_mass)
    if (kinetic is not None and kinetic.numel() != n) or step.numel() != 1:
        raise RuntimeError(f"hermnet_b200.md_kick: expected kinetic [{n}] and step [1]")
    _launch("hn_md_kick", dev, "md_kick", vel, force, inv_mass, float(half_dt), n, kinetic, step)
    _bump(vel, kinetic, step)


def md_scr_barostat(cell: Tensor, kinetic: Tensor, virial: Tensor, P0: Tensor, kT: Tensor, beta: Tensor, seed: Tensor,
                    step: Tensor, dt: float, tau_p: float, mu: Tensor, pressure: Tensor) -> None:
    """Stochastic cell rescaling of ``G`` replicas (``hn_md_scr_barostat``): ``cell [G,3,3]`` is scaled in place by
    ``mu [G]`` (written), from the per-replica kinetic energy ``kinetic [G]`` (eV), ``virial [G,3,3]`` (eV), target
    pressure ``P0 [G]`` (eV/A^3), ``kT [G]`` (eV), compressibility ``beta [G]`` (A^3/eV, >= 0), ``seed int64 [G]`` and
    ``step int64 [1]`` (read).  ``pressure [G]`` receives the internal pressure (eV/A^3) of the unscaled cell."""
    dev = _chk("md_scr_barostat", f32=(cell, kinetic, virial, P0, kT, beta, mu, pressure), i64=(seed, step))
    G = kinetic.numel()
    if (tuple(cell.shape) != (G, 3, 3) or tuple(virial.shape) != (G, 3, 3) or step.numel() != 1
            or any(t.numel() != G for t in (P0, kT, beta, seed, mu, pressure))):
        raise RuntimeError(f"hermnet_b200.md_scr_barostat: expected cell / virial [G={G},3,3], kinetic / P0 / kT / beta / seed / "
                           "mu / pressure [G] and step [1]")
    _launch("hn_md_scr_barostat", dev, "md_scr_barostat", cell, kinetic, virial, P0, kT, beta, seed, step, G, float(dt),
            float(tau_p), mu, pressure)
    _bump(cell, mu, pressure)


def md_affine_scale(pos: Tensor, vel: Tensor, replica: Tensor, mu: Tensor) -> None:
    """``pos *= mu[replica]``, ``vel /= mu[replica]`` in place on ``[N,3]`` (``hn_md_affine_scale``; ``replica int32 [N]``)."""
    dev = _chk("md_affine_scale", f32=(pos, vel, mu), i32=(replica,))
    n = pos.size(0)
    if tuple(pos.shape) != (n, 3) or tuple(vel.shape) != (n, 3) or replica.numel() != n:
        raise RuntimeError(f"hermnet_b200.md_affine_scale: expected pos / vel [{n},3] and replica [{n}]")
    _launch("hn_md_affine_scale", dev, "md_affine_scale", pos, vel, replica, mu, n)
    _bump(pos, vel)


def md_kinetic_tensor(vel: Tensor, inv_mass: Tensor) -> Tensor:
    """Per-atom kinetic tensors ``[N,6]``: the lower triangle ``(00, 10, 11, 20, 21, 22)`` of ``m v (x) v`` (eV) with
    ``m = 1 / inv_mass`` (``hn_md_kinetic_tensor``)."""
    dev = _chk("md_kinetic_tensor", f32=(vel, inv_mass))
    n = vel.size(0)
    if tuple(vel.shape) != (n, 3) or inv_mass.numel() != n:
        raise RuntimeError(f"hermnet_b200.md_kinetic_tensor: expected vel [{n},3] and inv_mass [{n}]")
    out = torch.empty((n, 6), dtype=torch.float32, device=dev)
    _launch("hn_md_kinetic_tensor", dev, "md_kinetic_tensor", vel, inv_mass, n, out)
    return out


def md_scr_barostat_tri(cell: Tensor, kin6: Tensor, virial: Tensor, P0: Tensor, kT: Tensor, beta: Tensor, seed: Tensor,
                        step: Tensor, dt: float, tau_p: float, mu: Tensor, mu_inv_t: Tensor, pressure: Tensor) -> None:
    """Triclinic stochastic cell rescaling of ``G`` lower-triangular cells (``hn_md_scr_barostat_tri``): ``cell [G,3,3]`` is
    deformed in place to ``cell mu``; ``mu``, ``mu_inv_t`` (``mu^-T``) and ``pressure`` (the internal pressure tensor of the
    undeformed cell, eV/A^3) ``[G,3,3]`` are written.  Inputs: per-replica kinetic tensors ``kin6 [G,6]`` (eV, packed lower
    triangle), ``virial [G,3,3]`` (eV, lower triangle read), ``P0 [G]`` (eV/A^3), ``kT [G]`` (eV), ``beta [G]`` (A^3/eV,
    >= 0), ``seed int64 [G]`` and ``step int64 [1]`` (read)."""
    dev = _chk("md_scr_barostat_tri", f32=(cell, kin6, virial, P0, kT, beta, mu, mu_inv_t, pressure), i64=(seed, step))
    G = P0.numel()
    if (any(tuple(t.shape) != (G, 3, 3) for t in (cell, virial, mu, mu_inv_t, pressure)) or tuple(kin6.shape) != (G, 6)
            or step.numel() != 1 or any(t.numel() != G for t in (kT, beta, seed))):
        raise RuntimeError(f"hermnet_b200.md_scr_barostat_tri: expected cell / virial / mu / mu_inv_t / pressure [G={G},3,3], "
                           "kin6 [G,6], P0 / kT / beta / seed [G] and step [1]")
    _launch("hn_md_scr_barostat_tri", dev, "md_scr_barostat_tri", cell, kin6, virial, P0, kT, beta, seed, step, G, float(dt),
            float(tau_p), mu, mu_inv_t, pressure)
    _bump(cell, mu, mu_inv_t, pressure)


def md_affine_deform(pos: Tensor, vel: Tensor, replica: Tensor, mu: Tensor, mu_inv_t: Tensor) -> None:
    """``pos = pos mu[replica]``, ``vel = vel mu_inv_t[replica]`` in place on ``[N,3]`` (row vectors; ``hn_md_affine_deform``;
    ``replica int32 [N]``, ``mu`` / ``mu_inv_t [G,3,3]``)."""
    dev = _chk("md_affine_deform", f32=(pos, vel, mu, mu_inv_t), i32=(replica,))
    n = pos.size(0)
    if (tuple(pos.shape) != (n, 3) or tuple(vel.shape) != (n, 3) or replica.numel() != n or mu.dim() != 3
            or tuple(mu.shape[1:]) != (3, 3) or mu_inv_t.shape != mu.shape):
        raise RuntimeError(f"hermnet_b200.md_affine_deform: expected pos / vel [{n},3], replica [{n}] and mu / mu_inv_t [G,3,3]")
    _launch("hn_md_affine_deform", dev, "md_affine_deform", pos, vel, replica, mu, mu_inv_t, n)
    _bump(pos, vel)


# ----------------------------------------------------------------------------------------------------
# FIRE structure relaxation (csrc/hn_opt.cu)
# ----------------------------------------------------------------------------------------------------
def _g9(name, G: int, *ts):
    for t in ts:
        if t is not None and t.numel() != 9 * G:
            raise RuntimeError(f"hermnet_b200.{name}: expected [G={G},3,3] (or [G,9]) matrices, got {tuple(t.shape)}")


def opt_fire_reduce(force: Tensor, vel: Tensor, A: Optional[Tensor], replica: Tensor, replica_ptr: Tensor) -> Tensor:
    """Per-replica float64 ``[G,4]``: ``(sum F'.v, sum |F'|^2, sum |v|^2, max |F'_i|^2)`` over the atoms with ``F'_i = f_i A^T``
    (``hn_opt_fire_reduce``; ``A float64 [G,3,3]`` or ``None`` for ``A = I``).  Deterministic (fixed summation order)."""
    dev = _chk("opt_fire_reduce", f32=(force, vel), f64=(A,), i32=(replica, replica_ptr))
    n, G = force.size(0), replica_ptr.numel() - 1
    if tuple(force.shape) != (n, 3) or tuple(vel.shape) != (n, 3) or replica.numel() != n:
        raise RuntimeError(f"hermnet_b200.opt_fire_reduce: expected force / vel [{n},3] and replica [{n}]")
    _g9("opt_fire_reduce", G, A)
    sums = (torch.empty if n else torch.zeros)((G, 4), dtype=torch.float64, device=dev)      # (n == 0: the launch is a no-op)
    ws_bytes = int(_lib.load().hn_opt_fire_reduce_workspace_bytes(n, G))        # per-chunk partials: caller-owned
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
    _launch("hn_opt_fire_reduce", dev, "opt_fire_reduce", force, vel, A, replica, replica_ptr, G, n, sums, ws, ws_bytes, kernels=2)
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
    dev = _chk("opt_fire_step", f64=(sums, h0, A, A_prev, vcell, P0, cell_factor, dt, alpha, coef, fmax_out), f32=(virial, cell),
               i32=(n_pos, steps, converged, n_active))
    G = dt.numel()
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
    _launch("hn_opt_fire_step", dev, "opt_fire_step", sums, virial, cell, h0, A, A_prev, vcell, P0, cell_factor, dt, alpha, n_pos,
            steps, converged, G, float(fmax), float(dt_max), float(max_step), int(bool(move)), coef, fmax_out, n_active)
    _bump(dt, alpha, n_pos, steps, converged, coef, fmax_out, n_active, *((cell, A, A_prev, vcell) if A is not None else ()))


def opt_fire_update(x: Optional[Tensor], rp: Tensor, vel: Tensor, force: Tensor, A_prev: Optional[Tensor], A: Optional[Tensor],
                    replica: Tensor, converged: Tensor, coef: Tensor) -> None:
    """Atom rows of a FIRE step in place (``hn_opt_fire_update``), for atoms of replicas not converged:
    ``vel = c_v vel + c_f' f A_prev^T``, ``rp += s dt vel``, ``x = rp A``.  ``A = None``: positions only, ``rp`` is the
    positions and ``x`` / ``A_prev`` are unused."""
    dev = _chk("opt_fire_update", f32=(x, rp, vel, force), f64=(A_prev, A, coef), i32=(replica, converged))
    n, G = rp.size(0), converged.numel()
    if (tuple(rp.shape) != (n, 3) or tuple(vel.shape) != (n, 3) or tuple(force.shape) != (n, 3) or replica.numel() != n
            or coef.numel() != 3 * G):
        raise RuntimeError(f"hermnet_b200.opt_fire_update: expected rp / vel / force [{n},3], replica [{n}] and coef [G={G},3]")
    if A is not None:
        if x is None or A_prev is None or tuple(x.shape) != (n, 3):
            raise RuntimeError(f"hermnet_b200.opt_fire_update: A needs x [{n},3] and A_prev")
        _g9("opt_fire_update", G, A, A_prev)
    x = x if A is not None else None
    _launch("hn_opt_fire_update", dev, "opt_fire_update", x, rp, vel, force, A_prev, A, replica, converged, coef, n)
    _bump(rp, vel, x)


# ----------------------------------------------------------------------------------------------------
# nudged elastic band forces (csrc/hn_neb.cu)
# ----------------------------------------------------------------------------------------------------
def _neb_layout(name: str, pos: Tensor, initial: Tensor, final: Tensor, image: Tensor, image_ptr: Tensor, band_ptr: Tensor,
                n_images: int):
    """``(M, B)`` of the band-major layout: ``pos [M,3]`` with ``M = K N``, endpoints ``[N,3]``, ``image [M]``,
    ``image_ptr [B K + 1]``, ``band_ptr [B+1]``."""
    m, B, K = pos.size(0), band_ptr.numel() - 1, int(n_images)
    n = initial.size(0)
    if (K < 1 or tuple(pos.shape) != (m, 3) or tuple(initial.shape) != (n, 3) or tuple(final.shape) != (n, 3) or m != K * n
            or image.numel() != m or image_ptr.numel() != B * K + 1):
        raise RuntimeError(f"hermnet_b200.{name}: expected pos [K N,3], initial / final [N,3], image [K N], "
                           f"image_ptr [B K+1] and band_ptr [B+1] with K = n_images >= 1 (got K={K}, pos {tuple(pos.shape)}, "
                           f"initial {tuple(initial.shape)}, final {tuple(final.shape)}, image {image.numel()}, "
                           f"image_ptr {image_ptr.numel()}, band_ptr {band_ptr.numel()})")
    return m, B


def neb_reduce(pos: Tensor, force: Tensor, initial: Tensor, final: Tensor, image: Tensor, image_ptr: Tensor, band_ptr: Tensor,
               n_images: int) -> Tensor:
    """Per-image float64 ``[B K,5]``: ``(|D+|^2, |D-|^2, D+.D-, F.D+, F.D-)`` of the band-major images (``hn_neb_reduce``;
    ``D+ = R_{k+1} - R_k``, ``D- = R_k - R_{k-1}``, endpoints from ``initial`` / ``final``).  Deterministic."""
    dev = _chk("neb_reduce", f32=(pos, force, initial, final), i32=(image, image_ptr, band_ptr))
    m, B = _neb_layout("neb_reduce", pos, initial, final, image, image_ptr, band_ptr, n_images)
    if tuple(force.shape) != (m, 3):
        raise RuntimeError(f"hermnet_b200.neb_reduce: expected force [{m},3], got {tuple(force.shape)}")
    n_img = B * int(n_images)
    sums = (torch.empty if m else torch.zeros)((n_img, 5), dtype=torch.float64, device=dev)
    ws_bytes = int(_lib.load().hn_neb_reduce_workspace_bytes(m, n_img))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
    _launch("hn_neb_reduce", dev, "neb_reduce", pos, force, initial, final, image, image_ptr, band_ptr, B, int(n_images), m, sums,
            ws, ws_bytes, kernels=2)
    return sums


def neb_step(sums: Tensor, energy: Tensor, end_energy: Tensor, spring: Tensor, climb: bool, coef: Tensor, imax: Tensor) -> None:
    """Tangent weights, climbing image and projection coefficients of ``B`` bands of ``K`` images (``hn_neb_step``, float64):
    ``sums [B K,5]`` of ``neb_reduce``, image energies ``energy [B K]`` and ``end_energy [B,2]`` (fp32), ``spring [B]``
    (eV/A^2, float64).  Writes ``coef [B K,2]`` (float64) and ``imax [B]`` (int32, the first highest image, 1..K)."""
    dev = _chk("neb_step", f32=(energy, end_energy), f64=(sums, spring, coef), i32=(imax,))
    B = spring.numel()
    n_img = energy.numel()
    if (B == 0 and n_img) or (B and n_img % B) or end_energy.numel() != 2 * B or imax.numel() != B \
            or sums.numel() != 5 * n_img or coef.numel() != 2 * n_img:
        raise RuntimeError(f"hermnet_b200.neb_step: expected sums [B K,5], energy [B K], end_energy [B,2], spring / imax [B] "
                           f"and coef [B K,2] (got B={B}, energy {n_img}, sums {sums.numel()}, coef {coef.numel()})")
    K = n_img // B if B else 1
    _launch("hn_neb_step", dev, "neb_step", sums, energy, end_energy, spring, int(bool(climb)), B, K, coef, imax)
    _bump(coef, imax)


def neb_project(force: Tensor, pos: Tensor, initial: Tensor, final: Tensor, image: Tensor, image_ptr: Tensor, band_ptr: Tensor,
                n_images: int, coef: Tensor) -> None:
    """``force <- force + coef[g,0] D+ + coef[g,1] D-`` in place for every atom of the band-major images (``hn_neb_project``;
    float64 arithmetic, fp32 storage)."""
    dev = _chk("neb_project", f32=(force, pos, initial, final), f64=(coef,), i32=(image, image_ptr, band_ptr))
    m, B = _neb_layout("neb_project", pos, initial, final, image, image_ptr, band_ptr, n_images)
    if tuple(force.shape) != (m, 3) or coef.numel() != 2 * B * int(n_images):
        raise RuntimeError(f"hermnet_b200.neb_project: expected force [{m},3] and coef [B K,2]")
    _launch("hn_neb_project", dev, "neb_project", force, pos, initial, final, image, image_ptr, band_ptr, B, int(n_images), coef, m)
    _bump(force)


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


def _pitched_f32(name: str, t: Tensor) -> Tensor:
    """A float32 CUDA operand the kernel reads through its row pitch (so it need not be contiguous)."""
    require_cuda(t, name)
    if t.dtype != torch.float32:
        raise RuntimeError(f"hermnet_b200.{name}: float tensors must be float32 (got {t.dtype})")
    return t


def gemm_tf32x3(a: Tensor, w_hi: Tensor, w_lo: Tensor, bias: Optional[Tensor]) -> Tensor:
    """``a [M,K] @ (w_hi + w_lo)[N,K]^T + bias`` on the tensor cores; ``a`` may be a column slice (row pitch)."""
    if a.dim() != 2 or a.stride(1) != 1 or a.stride(0) % 4 != 0 or a.data_ptr() % 16 != 0:
        a = a.contiguous()
    dev = _chk("gemm_tf32x3", f32=(w_hi, w_lo, bias))
    _pitched_f32("gemm_tf32x3", a)
    M, K = a.shape
    N = w_hi.size(0)
    out = torch.empty((M, N), dtype=torch.float32, device=dev)
    _launch("hn_gemm_tf32x3", dev, "gemm_tf32x3", a, M, K, a.stride(0), w_hi, w_lo, N, bias, out, N)
    return out


def _rowmajor(name: str, t: Tensor):
    """A 2-D float32 CUDA view whose rows are contiguous (row pitch may exceed the row length)."""
    if t.dim() != 2 or t.stride(1) != 1 or t.stride(0) % 4 != 0 or t.data_ptr() % 16 != 0:
        raise RuntimeError(f"hermnet_b200.{name}: expected a 16-byte aligned 2-D view with contiguous rows")
    return _pitched_f32(name, t)


def gemm_tf32x3_ex(a: Tensor, w_hi: Tensor, w_lo: Tensor, bias: Optional[Tensor], out: Optional[Tensor] = None, mode: int = 0,
                   aux: Optional[Tensor] = None, out2: Optional[Tensor] = None) -> Tensor:
    """``epilogue(a @ (w_hi + w_lo)^T + bias)`` written into ``out`` (a row-major view, e.g. a column block of a wider
    buffer); ``mode`` 0 identity / 1 ScaledSiLU with the pre-activation stored in ``out2`` / 2 multiply by
    ScaledSiLU'(``aux``).  All operands may be row-pitched views."""
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
    _launch("hn_gemm_tf32x3_ex", dev, tname, a, M, K, a.stride(0), w_hi, w_lo, N, bias, out, out.stride(0), int(mode), aux,
            4 if aux is None else aux.stride(0), out2, 4 if out2 is None else out2.stride(0))
    return out


# ----------------------------------------------------------------------------------------------------
# fused element-wise stages of the node update (csrc/hn_node.cu); every tensor is a contiguous row range
# ----------------------------------------------------------------------------------------------------
def node_pre(x, dx, vec, dvec, xcat, vecp):
    """``dx [n,F]`` / ``dvec [n,3,F]`` may be row-pitched views (slot of ``[N,R,F]`` / ``[N,R,3,F]``)."""
    dev = _chk("node_pre", x, vec, xcat, vecp)
    n, F = x.shape
    _launch("hn_node_pre", dev, "node_elementwise", n, F, x, dx, dx.stride(0), vec, dvec, dvec.stride(0), xcat, vecp)


def node_mid(v12, vdot, xcat):
    dev = _chk("node_mid", v12, vdot, xcat)
    n, F = vdot.shape
    _launch("hn_node_mid", dev, "node_elementwise", n, F, v12, vdot, xcat)


def node_post(xcat, a, vdot, vecp, v12, x_out, vec_out):
    dev = _chk("node_post", xcat, a, vdot, vecp, v12, x_out, vec_out)
    n, F = vdot.shape
    _launch("hn_node_post", dev, "node_elementwise", n, F, xcat, a, vdot, vecp, v12, x_out, vec_out)


def node_post_bwd(g_x, g_vec, a, vdot, v12, g_a, g_vdot, g_v12):
    dev = _chk("node_post_bwd", g_x, g_vec, a, vdot, v12, g_a, g_vdot, g_v12)
    n, F = vdot.shape
    _launch("hn_node_post_bwd", dev, "node_elementwise", n, F, g_x, g_vec, a, vdot, v12, g_a, g_vdot, g_v12)


def node_mid_bwd(g_vdot, g_cat, v12, vn, g_v12):
    """``vn`` may be the second half of the saved ``xcat`` (row pitch 2F)."""
    dev = _chk("node_mid_bwd", g_vdot, g_cat, v12, g_v12)
    n, F = g_vdot.shape
    _launch("hn_node_mid_bwd", dev, "node_elementwise", n, F, g_vdot, g_cat, v12, vn, vn.stride(0), g_v12)


def node_pre_bwd(g_xn, g_cat, g_vecn, g_vecp, g_x, g_vec):
    dev = _chk("node_pre_bwd", g_xn, g_cat, g_vecn, g_vecp, g_x, g_vec)
    n, F = g_xn.shape
    _launch("hn_node_pre_bwd", dev, "node_elementwise", n, F, g_xn, g_cat, g_vecn, g_vecp, g_x, g_vec)


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
    dev = _chk("tc_split_weights", f32=(Wt,))
    M, K, F3 = Wt.shape
    n = int(_lib.load().hn_tc_split_weights_elems(M, F3 // 3, K))
    wsplit = torch.empty(n, dtype=torch.float16, device=dev)
    wscale = torch.empty(M, dtype=torch.float32, device=dev)
    _launch("hn_tc_split_weights", dev, "tc_split_weights", Wt, M, K, F3 // 3, wsplit, wscale)
    return wsplit, wscale


def tc_basis_index(geom: Tensor, inv_rc: float, num_rbf: int) -> Tensor:
    dev = _chk("tc_basis_index", geom)
    kc = torch.empty(geom.size(0), dtype=torch.int32, device=dev)
    _launch("hn_tc_basis_index", dev, "tc_plan", geom, geom.size(0), float(inv_rc), int(num_rbf), kc)
    return kc


def tc_plan_records(g, geom: Tensor, inv_rc: float, num_rbf: int, src_major: bool, atom_local: Optional[Tensor], src_block: int):
    """``(rec int32 [E,4], kc int32 [E], sub int32 [E])`` of a plan in one pass over the row-edges (``hn_tc_plan_records``)."""
    dev = _chk("tc_plan_records", g.row_xoff, geom, i32=(g.edge_row, g.col, g.row_mod, atom_local))
    E = int(g.n_edges)
    rec = torch.empty((max(E, 1), 4), dtype=torch.int32, device=dev)
    kc = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
    sub = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
    _launch("hn_tc_plan_records", dev, "tc_plan", int(bool(src_major)), g.edge_row, g.col, g.row_xoff, g.row_mod, atom_local,
            int(g.rows_per_atom), int(src_block), geom, float(inv_rc), int(num_rbf), E, rec, kc, sub)
    return rec[:E], kc[:E], sub[:E]


def tc_plan_sort(in_ptr: Tensor, ids: Optional[Tensor], kc: Tensor, sub: Optional[Tensor], n_seg: int, n_sub: int, num_rbf: int):
    """Segment-local sort of the plan builder (``hn_tc_plan_sort``): returns ``(order int32 [n_live], grp_ptr int32
    [n_seg * n_sub + 1])`` -- edge ids ordered by (segment, sub, kc) without the dropped (sub < 0) entries, and the start of
    every (segment, sub) group in it.  One host-free count pass, a cumsum, one fill pass."""
    dev = _chk("tc_plan_sort", i32=(in_ptr, ids, kc, sub))
    counts = torch.zeros(max(n_seg * n_sub, 1), dtype=torch.int32, device=dev)
    grp_ptr = torch.zeros(n_seg * n_sub + 1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev), _timed("tc_plan", dev):
        _call("hn_tc_plan_sort", dev, in_ptr, ids, kc, sub, n_seg, n_sub, int(num_rbf), counts, None, None)
        torch.cumsum(counts[: n_seg * n_sub], 0, dtype=torch.int32, out=grp_ptr[1:])
        out_base = grp_ptr[:: n_sub][:n_seg].contiguous()
        order = torch.empty(max(int(kc.numel()), 1), dtype=torch.int32, device=dev)
        _call("hn_tc_plan_sort", dev, in_ptr, ids, kc, sub, n_seg, n_sub, int(num_rbf), None, out_base, order)
    return order, grp_ptr


def tc_plan_count(order: Tensor, kc: Tensor, grp_ptr: Tensor, n_groups: int, num_rbf: int, window: int = 32) -> Tensor:
    dev = _chk("tc_plan_count", i32=(order, kc, grp_ptr))
    counts = torch.zeros(n_groups, dtype=torch.int32, device=dev)
    _launch("hn_tc_plan_count", dev, "tc_plan", order, kc, grp_ptr, n_groups, int(num_rbf), int(window), counts)
    return counts


def tc_plan_fill(order: Tensor, kc: Tensor, grp_ptr: Tensor, n_groups: int, num_rbf: int, grp_tile: Tensor, n_tiles: int,
                 window: int = 32) -> Tensor:
    dev = _chk("tc_plan_fill", i32=(order, kc, grp_ptr, grp_tile))
    tile_start = torch.empty(max(n_tiles, 1), dtype=torch.int32, device=dev)
    _launch("hn_tc_plan_fill", dev, "tc_plan", order, kc, grp_ptr, n_groups, int(num_rbf), int(window), grp_tile, tile_start)
    return tile_start


def tc_plan_finalize(order: Tensor, tile_start: Tensor, n_tiles: int, n_edges: int, rec: Tensor, tile_mod: Tensor):
    dev = _chk("tc_plan_finalize", i32=(order, tile_start, rec, tile_mod))
    erec = torch.empty((max(n_edges, 1), 4), dtype=torch.int32, device=dev)
    tile_info = torch.empty((max(n_tiles, 1), 4), dtype=torch.int32, device=dev)
    _launch("hn_tc_plan_finalize", dev, "tc_plan", order, tile_start, n_tiles, n_edges, rec, tile_mod, erec, tile_info)
    return erec, tile_info


def tc_tile_windows(plan, geom: Tensor, inv_rc: float, num_rbf: int, live: Optional[Tensor] = None) -> None:
    dev = _chk("tc_tile_windows", geom, live)
    if live is not None:
        _live("tc_tile_windows", live, geom.size(0))
    _launch("hn_tc_tile_windows", dev, "tc_tile_windows", ctypes.byref(plan.cstruct()), geom, live, float(inv_rc), int(num_rbf))


def tc_edge_fwd(p: EdgeParams, plan, xh, vec, geom, wsplit, wscale, bias, offset, n_rows: int, debug_phi: bool = False):
    dev = _chk("tc_edge_fwd", wsplit, f32=(xh, vec, geom, wscale, bias, offset))
    F = p.hidden
    dx = torch.empty((n_rows, F), dtype=torch.float32, device=dev)
    dvec = torch.empty((n_rows, 3, F), dtype=torch.float32, device=dev)
    E = geom.size(0)
    dbg = torch.zeros(2 * E * 3 * F + 14336, dtype=torch.float32, device=dev) if debug_phi else None
    _launch("hn_tc_edge_fwd", dev, "painn_edge_fwd", ctypes.byref(p), ctypes.byref(plan.cstruct()), xh, vec, geom, wsplit, wscale,
            bias, offset, dx, dvec, dbg, E)
    return (dx, dvec, dbg) if debug_phi else (dx, dvec)


def tc_edge_bwd_dst(p: EdgeParams, plan, xh, vec, geom, wsplit, wscale, bias, offset, g_dx, g_dvec):
    dev = _chk("tc_edge_bwd_dst", wsplit, f32=(xh, vec, geom, wscale, bias, offset, g_dx, g_dvec))
    alloc = torch.zeros if plan.has_inactive else torch.empty
    g_geom = alloc((1, geom.size(0), 4), dtype=torch.float32, device=dev)
    _launch("hn_tc_edge_bwd_dst", dev, "painn_edge_bwd_dst", ctypes.byref(p), ctypes.byref(plan.cstruct()), xh, vec, geom, wsplit,
            wscale, bias, offset, g_dx, g_dvec, g_geom)
    return g_geom


def tc_edge_bwd_src(p: EdgeParams, plan, xh, vec, geom, wsplit, wscale, bias, offset, g_dx, g_dvec):
    dev = _chk("tc_edge_bwd_src", wsplit, f32=(xh, vec, geom, wscale, bias, offset, g_dx, g_dvec))
    grad_xh = torch.zeros_like(xh)
    grad_vec = torch.empty_like(vec)
    _launch("hn_tc_edge_bwd_src", dev, "painn_edge_bwd_src", ctypes.byref(p), ctypes.byref(plan.cstruct()), xh, vec, geom, wsplit,
            wscale, bias, offset, g_dx, g_dvec, grad_xh, grad_vec)
    return grad_xh, grad_vec
