"""Autograd layer over the CUDA kernels.

Two formulations of the same arithmetic (HermNet/hermnet.py:133-152, rmnet.py:51-73):

* **fused** (inference / first-order): ``EdgeGeometry`` and ``PaiNNEdge`` call the fused kernels and their
  hand-written backward kernels (forces, virial, feature and filter-weight gradients).  Marked
  ``once_differentiable``.
* **composite** (training with a force loss needs ``create_graph=True`` -> double backward, SURVEY F10):
  the same maths expressed with ``gather_rows`` / ``segment_sum`` -- two mutually adjoint linear kernels, so the
  formulation is differentiable to any order -- plus ordinary torch elementwise ops and GEMMs.

Neither uses torch_scatter / PyG / atomics; there is no CPU implementation.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import ops, tileplan
from .graph import RowGraph, Segments

Tensor = torch.Tensor


# ----------------------------------------------------------------------------------------------------
# adjoint pair: gather rows  <->  segmented sum
# ----------------------------------------------------------------------------------------------------
class _GatherRows(Function):
    @staticmethod
    def forward(ctx, X: Tensor, seg: Segments):
        ctx.seg = seg
        ctx.shape = X.shape
        cols = math.prod(X.shape[1:])          # (explicit sizes: -1 is ambiguous for empty tensors, e.g. a graph without edges)
        return ops.gather_rows(X.reshape(X.size(0), cols).contiguous(), seg.index).view((seg.index.numel(),) + tuple(X.shape[1:]))

    @staticmethod
    def backward(ctx, g):
        return segment_sum(g, ctx.seg), None


class _SegmentSum(Function):
    @staticmethod
    def forward(ctx, Y: Tensor, seg: Segments):
        ctx.seg = seg
        out = ops.segment_sum(Y.reshape(Y.size(0), math.prod(Y.shape[1:])).contiguous(), seg.rowptr, seg.perm, seg.n_rows)
        return out.view((seg.n_rows,) + tuple(Y.shape[1:]))

    @staticmethod
    def backward(ctx, g):
        return gather_rows(g, ctx.seg), None


def gather_rows(X: Tensor, seg: Segments) -> Tensor:
    """``out[i] = X[seg.index[i]]`` (rows of X = rows of the segmentation)."""
    return _GatherRows.apply(X, seg)


def segment_sum(Y: Tensor, seg: Segments) -> Tensor:
    """``out[r] = sum of Y[i] over the items i of row r`` -- deterministic, no atomics."""
    return _SegmentSum.apply(Y, seg)


# ----------------------------------------------------------------------------------------------------
# fused formulation
# ----------------------------------------------------------------------------------------------------
class _EdgeGeometry(Function):
    @staticmethod
    def forward(ctx, pos: Tensor, cell: Optional[Tensor], g: RowGraph):
        geom = ops.edge_geom_fwd(pos.contiguous(), None if cell is None else cell.contiguous(), g)
        ctx.g = g
        ctx.has_cell = cell is not None
        ctx.save_for_backward(geom)
        return geom

    @staticmethod
    @once_differentiable
    def backward(ctx, g_geom):
        (geom,) = ctx.saved_tensors
        g = ctx.g
        want_cell = ctx.has_cell and ctx.needs_input_grad[1]
        grad_pos, cellw = ops.edge_geom_bwd(geom, g_geom.contiguous().view(1, -1, 4), g, want_cell)
        grad_cell = None
        if want_cell:
            sb = g.seg_batch
            grad_cell = ops.segment_sum(cellw, sb.rowptr, sb.perm, sb.n_rows).view(-1, 3, 3)[: g.n_graphs]
        return grad_pos, grad_cell, None


def edge_geometry(pos: Tensor, cell: Optional[Tensor], g: RowGraph) -> Tensor:
    """``geom[e] = (ux, uy, uz, d)`` for every row-edge (internal atom order)."""
    return _EdgeGeometry.apply(pos, cell, g)


class _PaiNNEdge(Function):
    """Edge side of one layer.  F == 128: the tensor-core kernels of csrc/hn_edge_tc.cu over the graph's tile plans
    (``tileplan``); otherwise the C ABI picks the tile-sweep kernels (F in {64, 256, 512}) or the row-per-warp kernels
    (any F % 32 == 0).  Every family takes Verlet-skin superset lists (``p.flags`` bit 0 with the ``p.live`` mask): the
    entries marked dead contribute nothing, not even the filter bias -- the tensor-core kernels through the tile plans'
    windows, the others through the signed geometry ``ops`` builds once per evaluation."""

    @staticmethod
    def forward(ctx, xh, vec, geom, Wt, bias, offset, g: RowGraph, p, vec_zero=False):
        xh, vec, geom, Wt, bias = xh.contiguous(), vec.contiguous(), geom.contiguous(), Wt.contiguous(), bias.contiguous()
        # vec == 0 identically (first layer, hermnet.py:124): the kernels take NULL and skip the vec gathers and the F:2F
        # part of the filter in the forward and the destination-major backward
        ctx.vec_null = bool(vec_zero)
        ctx.tc = ops.edge_use_tc(p.hidden, p.num_rbf) and g.n_edges > 0
        if ctx.tc:
            dst, _ = tileplan.plans_of(g, geom, p.inv_rc, p.num_rbf, want_src=False)
            dst.update_windows(geom, p.inv_rc, p.num_rbf, getattr(p, "live", None))
            wsplit, wscale = _tc_split_cached(Wt)
            dx, dvec = ops.tc_edge_fwd(p, dst, xh, None if ctx.vec_null else vec, geom, wsplit, wscale, bias, offset, p.n_rows)
            ctx.wsplit = (wsplit, wscale)
        else:
            dx, dvec = ops.painn_edge_fwd(p, xh, None if ctx.vec_null else vec, geom, g, Wt, bias, offset)
        ctx.g, ctx.p = g, p
        ctx.save_for_backward(xh, vec, geom, Wt, bias, offset)
        return dx, dvec

    @staticmethod
    @once_differentiable
    def backward(ctx, g_dx, g_dvec):
        xh, vec, geom, Wt, bias, offset = ctx.saved_tensors
        g, p = ctx.g, ctx.p
        g_dx, g_dvec = g_dx.contiguous(), g_dvec.contiguous()
        need = ctx.needs_input_grad
        grad_xh = grad_vec = grad_geom = grad_W = grad_b = None
        tc_src = ctx.tc and getattr(g, "_tc_parent", None) is None      # the element-table graph has no source-major plan
        if ctx.tc:
            wsplit, wscale = ctx.wsplit
            dst, src = tileplan.plans_of(g, geom, p.inv_rc, p.num_rbf, want_src=tc_src and (need[0] or need[1]))
        if need[2]:
            if ctx.tc:
                dst.update_windows(geom, p.inv_rc, p.num_rbf, getattr(p, "live", None))
                parts = ops.tc_edge_bwd_dst(p, dst, xh, None if ctx.vec_null else vec, geom, wsplit, wscale, bias, offset, g_dx, g_dvec)
            else:
                parts = ops.painn_edge_bwd_dst(p, xh, None if ctx.vec_null else vec, geom, g, Wt, bias, offset, g_dx, g_dvec)
            grad_geom = parts[0] if parts.size(0) == 1 else parts.sum(0)
        if need[0] or need[1]:
            if tc_src:
                src.update_windows(geom, p.inv_rc, p.num_rbf, getattr(p, "live", None))
                grad_xh, grad_vec = ops.tc_edge_bwd_src(p, src, xh, vec, geom, wsplit, wscale, bias, offset, g_dx, g_dvec)
            else:
                grad_xh, grad_vec = ops.painn_edge_bwd_src(p, xh, vec, geom, g, Wt, bias, offset, g_dx, g_dvec)
        if need[3] or need[4]:
            grad_W, grad_b = ops.painn_edge_bwd_w(p, xh, vec, geom, g, offset, g_dx, g_dvec)
        return grad_xh, grad_vec, grad_geom, grad_W, grad_b, None, None, None, None


_TC_SPLIT = {}


def _tc_split_cached(Wt: Tensor):
    """fp16 hi / lo split of the stacked filter weights for the tensor-core edge kernels, cached per live tensor object,
    version and storage (the frozen-parameter path hands the same stacked tensor to every evaluation)."""
    import weakref
    key = id(Wt)
    stamp = (Wt._version, Wt.data_ptr(), str(Wt.device), tuple(Wt.shape))
    hit = _TC_SPLIT.get(key)
    if hit is not None and hit[0]() is Wt and hit[1] == stamp:
        return hit[2], hit[3]
    wsplit, wscale = ops.tc_split_weights(Wt)
    if Wt.requires_grad or Wt.grad_fn is not None:
        return wsplit, wscale                       # a per-step tensor of the autograd graph: nothing to cache
    if len(_TC_SPLIT) > 256:
        _TC_SPLIT.clear()
    _TC_SPLIT[key] = (weakref.ref(Wt), stamp, wsplit, wscale)
    return wsplit, wscale


def painn_edge(xh, vec, geom, Wt, bias, offset, g: RowGraph, p, vec_zero=False):
    """Fused gather -> filter -> message -> segmented reduction.  Returns ``dx [R,F]``, ``dvec [R,3,F]``.
    ``vec_zero``: the caller guarantees ``vec == 0`` (first layer); lets the kernels skip everything that multiplies it."""
    return _PaiNNEdge.apply(xh, vec, geom, Wt, bias, offset, g, p, vec_zero)


# ----------------------------------------------------------------------------------------------------
# node-side dense layers on the tensor cores (fused path)
# ----------------------------------------------------------------------------------------------------
_SPLIT_CACHE = {}


def _split_cached(w: Tensor, transposed: bool):
    """(hi, lo) TF32 split of a weight (or of its transpose), cached per live tensor object and version (addresses and
    ids are recycled by the allocator, so the entry keeps a weak reference and is only trusted for the same object)."""
    import weakref
    key = (id(w), transposed)
    hit = _SPLIT_CACHE.get(key)
    stamp = (w._version, w.data_ptr(), str(w.device))      # .data / .to() updates do not bump _version: also key on storage
    if hit is not None and hit[0]() is w and hit[1] == stamp:
        return hit[2], hit[3]
    hi, lo = ops.split_tf32(w.detach().t().contiguous() if transposed else w.detach())
    if len(_SPLIT_CACHE) > 1024:
        _SPLIT_CACHE.clear()
    _SPLIT_CACHE[key] = (weakref.ref(w), stamp, hi, lo)
    return hi, lo


class _LinearTC(Function):
    """``x @ W^T + b`` through ``hn_gemm_tf32x3`` (tcgen05, 3xTF32).  Backward: the data gradient uses the same kernel
    with the transposed weight; weight / bias gradients (only when parameters require grad) are plain torch GEMMs."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        hi, lo = _split_cached(weight, False)
        x2 = x.reshape(-1, x.size(-1))
        out = ops.gemm_tf32x3(x2, hi, lo, None if bias is None else bias.detach().contiguous())
        return out.view(tuple(x.shape[:-1]) + (weight.size(0),))

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        x, weight = ctx.saved_tensors
        gx = gw = gb = None
        g2 = g.reshape(-1, g.size(-1))
        if ctx.needs_input_grad[0]:
            if ops.gemm_supported(weight.size(0), weight.size(1)):
                hi, lo = _split_cached(weight, True)
                gx = ops.gemm_tf32x3(g2.contiguous(), hi, lo, None).view(x.shape)
            else:
                gx = (g2 @ weight).view(x.shape)
        if ctx.needs_input_grad[1]:
            gw = g2.t() @ x.reshape(-1, x.size(-1))
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = g2.sum(0)
        return gx, gw, gb


def linear(x: Tensor, weight: Tensor, bias: Optional[Tensor], tensor_cores: bool) -> Tensor:
    """nn.Linear forward; on the fused path (fp32, K % 32 == 0, N % 64 == 0) it runs on the tensor cores."""
    if tensor_cores and x.dtype == torch.float32 and ops.gemm_supported(weight.size(1), weight.size(0)) and x.numel() > 0:
        return _LinearTC.apply(x, weight, bias)
    return torch.nn.functional.linear(x, weight, bias)


class _Readout(Function):
    """Readout MLP of frozen parameters (hermnet.py:129) in plain fp32 through ``hn_readout_{fwd,bwd}``."""

    @staticmethod
    def forward(ctx, x, W1, b1, W2, b2):
        x = x.contiguous()
        b2 = b2.detach().reshape(-1).contiguous()            # stays on the device: no host read-back (CUDA-graph capturable)
        ctx.save_for_backward(x, W1, b1, W2, b2)
        return ops.readout_fwd(x, W1.detach().contiguous(), b1.detach().contiguous(), W2.detach().reshape(-1).contiguous(), b2)

    @staticmethod
    @once_differentiable
    def backward(ctx, g_e):
        x, W1, b1, W2, b2 = ctx.saved_tensors
        g_x = ops.readout_bwd(x, W1.detach().contiguous(), b1.detach().contiguous(), W2.detach().reshape(-1).contiguous(), b2,
                              g_e.reshape(-1).contiguous())
        return g_x, None, None, None, None


def readout(x: Tensor, lin0, lin2) -> Tensor:
    """``e_atom [N,1]`` of the readout ``Sequential(Linear(F, F/2), ScaledSiLU, Linear(F/2, 1))`` with frozen parameters."""
    return _Readout.apply(x, lin0.weight, lin0.bias, lin2.weight, lin2.bias)


# ----------------------------------------------------------------------------------------------------
# fused node side of one HVNet layer (frozen parameters): two autograd nodes per layer instead of ~60
# ----------------------------------------------------------------------------------------------------
def node_fusable(hidden: int) -> bool:
    """The fused node path chains tensor-core GEMMs with K, N in {F, 2F, 3F, T*F}: needs F % 64 == 0."""
    return hidden % 64 == 0


def _wsplit(w: Tensor, transposed: bool = False):
    return _split_cached(w, transposed)


_XPROJ = {}


def _xproj_folded(mods):
    """First Linear of every sub-network with its LayerNorm affine folded in (W1.diag(gamma), b1 + W1.beta), concatenated
    over the sub-networks, plus the TF32 hi / lo splits of it and of its transpose; cached per layer for frozen parameters
    (the fused node path only runs with frozen parameters)."""
    ps = [q for m in mods for q in (m.x_proj[0].weight, m.x_proj[0].bias, m.x_layernorm.weight, m.x_layernorm.bias)]
    stamp = tuple((q._version, q.data_ptr(), str(q.device)) for q in ps)
    key = id(mods[0])
    hit = _XPROJ.get(key)
    if hit is not None and hit[0] == stamp and hit[1]() is mods[0]:
        return hit[2]
    import weakref
    w1 = torch.cat([m.x_proj[0].weight * m.x_layernorm.weight[None, :] for m in mods], 0).detach()
    b1 = torch.cat([m.x_proj[0].bias + m.x_proj[0].weight @ m.x_layernorm.bias for m in mods]).detach().contiguous()
    w1_hi, w1_lo = ops.split_tf32(w1)
    w1t_hi, w1t_lo = ops.split_tf32(w1.t().contiguous())
    out = (w1, b1, w1_hi, w1_lo, w1t_hi, w1t_lo)
    if len(_XPROJ) > 256:
        _XPROJ.clear()
    _XPROJ[key] = (stamp, weakref.ref(mods[0]), out)
    return out


class _XProjHV(Function):
    """``xh[m] = x_proj_m(LayerNorm_m(x))`` for every sub-network m of an HVNet layer (rmnet.py:52 run per element,
    hermnet.py:51-59), written straight into the flat ``[M*N, 3F]`` buffer the edge kernel reads.  The normalisation is
    computed once (its affine part folded into the first Linear of every sub-network), the first Linears of all
    sub-networks are one GEMM with the ScaledSiLU in its epilogue, and the backward is hand-written."""

    @staticmethod
    def forward(ctx, x, mods, eps):
        N, F = x.shape
        M = len(mods)
        x = x.contiguous()
        xhat, mean, rstd = ops.layernorm_fwd(x, eps)
        w1, b1, w1_hi, w1_lo, w1t_hi, w1t_lo = _xproj_folded(mods)
        hpre = torch.empty((N, M * F), dtype=x.dtype, device=x.device)
        h = torch.empty_like(hpre)
        ops.gemm_tf32x3_ex(xhat, w1_hi, w1_lo, b1, out=h, mode=1, out2=hpre)
        xh = torch.empty((M * N, 3 * F), dtype=x.dtype, device=x.device)
        for m, mod in enumerate(mods):
            hi, lo = _wsplit(mod.x_proj[2].weight)
            ops.gemm_tf32x3_ex(h[:, m * F:(m + 1) * F], hi, lo, mod.x_proj[2].bias.detach(), out=xh[m * N:(m + 1) * N])
        ctx.mods, ctx.w1t = mods, (w1t_hi, w1t_lo)
        ctx.save_for_backward(x, mean, rstd, hpre)
        return xh

    @staticmethod
    @once_differentiable
    def backward(ctx, g_xh):
        x, mean, rstd, hpre = ctx.saved_tensors
        mods = ctx.mods
        N, F = x.shape
        g_xh = g_xh.contiguous()
        g_pre = torch.empty_like(hpre)
        for m, mod in enumerate(mods):
            hi, lo = _wsplit(mod.x_proj[2].weight, True)                      # [F, 3F]: g_h = g_xh . W2
            ops.gemm_tf32x3_ex(g_xh[m * N:(m + 1) * N], hi, lo, None, out=g_pre[:, m * F:(m + 1) * F], mode=2,
                               aux=hpre[:, m * F:(m + 1) * F])
        hi, lo = ctx.w1t                                                      # [F, M*F]
        g_xhat = ops.gemm_tf32x3_ex(g_pre, hi, lo, None)
        g_x = ops.layernorm_bwd(g_xhat, x, mean, rstd)
        return g_x, None, None


def xproj_hv(x: Tensor, mods, eps: float) -> Tensor:
    return _XProjHV.apply(x, mods, eps)


class _NodeUpdateHV(Function):
    """Residual + update block of every sub-network of an HVNet layer on its own destination rows (rmnet.py:24-32,
    94-107; hermnet.py:60-61 keeps only those rows): three fused element-wise kernels and three tensor-core GEMMs per
    element forward, the mirror image backward.  Rows of elements without an active sub-network, of unknown elements and
    ghost rows stay zero (hermnet.py:56-57)."""

    @staticmethod
    def forward(ctx, x, vec, dx, dvec, g: RowGraph, mods):
        N, F = x.shape
        x, vec = x.contiguous(), vec.contiguous()
        dx2, dvec2 = dx.reshape(N, F), dvec.reshape(N, 3 * F)
        T = len(mods)
        covered = sum((g.dst_slice(t).stop - g.dst_slice(t).start) for t in range(T) if g.mod_active_host[t])
        alloc = torch.empty if covered == N else torch.zeros
        x_new = alloc((N, F), dtype=x.dtype, device=x.device)
        vec_new = alloc((N, 3, F), dtype=x.dtype, device=x.device)
        saved, spans = [], []
        for t in range(T):
            sl = g.dst_slice(t)
            n = sl.stop - sl.start
            if n <= 0 or not g.mod_active_host[t]:
                continue
            upd = mods[t].update_layer
            xcat = torch.empty((n, 2 * F), dtype=x.dtype, device=x.device)
            vecp = torch.empty((n, 3, F), dtype=x.dtype, device=x.device)
            ops.node_pre(x[sl], dx2[sl], vec[sl], dvec2[sl], xcat, vecp)
            hi, lo = _wsplit(upd.vec_proj.weight)
            v12 = ops.gemm_tf32x3_ex(vecp.view(3 * n, F), hi, lo, None)                       # [3n, 2F]
            vdot = torch.empty((n, F), dtype=x.dtype, device=x.device)
            ops.node_mid(v12, vdot, xcat)
            pre2 = torch.empty((n, F), dtype=x.dtype, device=x.device)
            hi, lo = _wsplit(upd.xvec_proj[0].weight)
            h2 = ops.gemm_tf32x3_ex(xcat, hi, lo, upd.xvec_proj[0].bias.detach(), mode=1, out2=pre2)
            hi, lo = _wsplit(upd.xvec_proj[2].weight)
            a = ops.gemm_tf32x3_ex(h2, hi, lo, upd.xvec_proj[2].bias.detach())                # [n, 3F]
            ops.node_post(xcat, a, vdot, vecp, v12, x_new[sl], vec_new[sl])
            saved += [v12, xcat, vdot, a, pre2]
            spans.append((t, sl))
        ctx.spans, ctx.mods, ctx.full = spans, mods, covered == N
        ctx.shapes = (dx.shape, dvec.shape)
        ctx.save_for_backward(*saved)
        return x_new, vec_new

    @staticmethod
    @once_differentiable
    def backward(ctx, g_xn, g_vecn):
        saved = ctx.saved_tensors
        g_xn, g_vecn = g_xn.contiguous(), g_vecn.contiguous()
        N, F = g_xn.shape
        alloc = torch.empty if ctx.full else torch.zeros
        g_x = alloc((N, F), dtype=g_xn.dtype, device=g_xn.device)
        g_vec = alloc((N, 3, F), dtype=g_xn.dtype, device=g_xn.device)
        for i, (t, sl) in enumerate(ctx.spans):
            v12, xcat, vdot, a, pre2 = saved[5 * i:5 * i + 5]
            n = sl.stop - sl.start
            upd = ctx.mods[t].update_layer
            g_a = torch.empty((n, 3 * F), dtype=g_xn.dtype, device=g_xn.device)
            g_vdot = torch.empty((n, F), dtype=g_xn.dtype, device=g_xn.device)
            g_v12 = torch.empty((3 * n, 2 * F), dtype=g_xn.dtype, device=g_xn.device)
            ops.node_post_bwd(g_xn[sl], g_vecn[sl], a, vdot, v12, g_a, g_vdot, g_v12)
            hi, lo = _wsplit(upd.xvec_proj[2].weight, True)                                   # [F, 3F]
            g_pre2 = ops.gemm_tf32x3_ex(g_a, hi, lo, None, mode=2, aux=pre2)
            hi, lo = _wsplit(upd.xvec_proj[0].weight, True)                                   # [2F, F]
            g_cat = ops.gemm_tf32x3_ex(g_pre2, hi, lo, None)
            ops.node_mid_bwd(g_vdot, g_cat, v12, xcat[:, F:], g_v12)
            hi, lo = _wsplit(upd.vec_proj.weight, True)                                       # [F, 2F]
            g_vecp = ops.gemm_tf32x3_ex(g_v12, hi, lo, None)                                  # [3n, F]
            ops.node_pre_bwd(g_xn[sl], g_cat, g_vecn[sl], g_vecp, g_x[sl], g_vec[sl])
        dx_shape, dvec_shape = ctx.shapes
        return g_x, g_vec, g_x.view(dx_shape), g_vec.view(dvec_shape), None, None


def node_update_hv(x, vec, dx, dvec, g: RowGraph, mods):
    return _NodeUpdateHV.apply(x, vec, dx, dvec, g, mods)


def _layer0_weights(xh_tab: Tensor, Wt: Tensor, bias: Tensor, M: int, nz: int, F: int, K: int, KP: int):
    """``BigA, BigC [M, F, KP]`` of include/hermnet_b200.h (hn_layer0_basis_*): the first-layer filter with the element table of
    projected source features folded in; column ``z*K + k`` = ``x[m][z][f] * W[m][k][f]``, column ``nz*K + z`` = ``x[m][z][f] * b[m][f]``."""
    tab = xh_tab.view(M, nz, 3 * F)

    def big(x, W, b):
        out = torch.zeros((M, F, KP), dtype=x.dtype, device=x.device)
        out[:, :, :nz * K] = torch.einsum("mzf,mkf->mfzk", x, W).reshape(M, F, nz * K)
        out[:, :, nz * K:nz * K + nz] = (x * b[:, None, :]).transpose(1, 2)
        return out

    c2 = 1.0 / math.sqrt(F)
    return big(tab[:, :, :F], Wt[:, :, :F], bias[:, :F]), big(tab[:, :, 2 * F:] * c2, Wt[:, :, 2 * F:], bias[:, 2 * F:])


class _Layer0HV(Function):
    """Edge side of the FIRST HVNet layer (x = Embedding[Z], vec = 0; hermnet.py:123-124, rmnet.py:55-73) by basis aggregation:
    per-(destination, source element) sums of the radial basis (``hn_layer0_basis_fwd``: 12 Gaussians x 4 weights per edge instead
    of 3F channels), then one tensor-core GEMM per destination element and output; the backward mirrors it (GEMMs, then
    ``hn_layer0_basis_bwd`` -> per-edge geometry gradient).  Frozen parameters only (no gradient for the table / filter)."""

    @staticmethod
    def forward(ctx, geom, xh_tab, Wt, bias, offset, g0: RowGraph, p0, n_elem: int):
        F, K, M = int(p0.hidden), int(p0.num_rbf), int(p0.n_modules)
        KP = ops.layer0_row_len(n_elem, K)
        geom = geom.contiguous()
        live = getattr(p0, "live", None)
        Sa, Sc = ops.layer0_basis_fwd(p0, g0, geom, live, offset, n_elem, KP)
        bigA, bigC = _layer0_weights(xh_tab.detach(), Wt.detach(), bias.detach(), M, n_elem, F, K, KP)
        a_hi, a_lo = ops.split_tf32(bigA.view(M * F, KP))
        c_hi, c_lo = ops.split_tf32(bigC.view(M * F, KP))
        R = int(p0.n_rows)
        spans = []
        for t in range(M):
            sl = g0.dst_slice(t)
            if sl.stop - sl.start > 0 and g0.mod_active_host[t]:
                spans.append((t, sl))
        covered = sum(sl.stop - sl.start for _, sl in spans)
        alloc = torch.empty if covered == R else torch.zeros
        dx = alloc((R, F), dtype=geom.dtype, device=geom.device)
        dvec = alloc((R, 3, F), dtype=geom.dtype, device=geom.device)
        for t, sl in spans:
            n = sl.stop - sl.start
            w = slice(t * F, (t + 1) * F)
            ops.gemm_tf32x3_ex(Sa[sl], a_hi[w], a_lo[w], None, out=dx[sl])
            ops.gemm_tf32x3_ex(Sc[sl].view(3 * n, KP), c_hi[w], c_lo[w], None, out=dvec[sl].view(3 * n, F))
        ctx.g0, ctx.p0, ctx.spans, ctx.dims, ctx.live = g0, p0, spans, (F, K, M, KP, n_elem), live
        ctx.save_for_backward(geom, offset, bigA, bigC)
        return dx, dvec

    @staticmethod
    @once_differentiable
    def backward(ctx, g_dx, g_dvec):
        geom, offset, bigA, bigC = ctx.saved_tensors
        F, K, M, KP, n_elem = ctx.dims
        g_dx, g_dvec = g_dx.contiguous(), g_dvec.contiguous()
        R = g_dx.size(0)
        at_hi, at_lo = ops.split_tf32(bigA.transpose(1, 2).reshape(M * KP, F))
        ct_hi, ct_lo = ops.split_tf32(bigC.transpose(1, 2).reshape(M * KP, F))
        gSa = torch.empty((R, KP), dtype=g_dx.dtype, device=g_dx.device)
        gSc = torch.empty((R, 3, KP), dtype=g_dx.dtype, device=g_dx.device)
        for t, sl in ctx.spans:
            n = sl.stop - sl.start
            w = slice(t * KP, (t + 1) * KP)
            ops.gemm_tf32x3_ex(g_dx[sl], at_hi[w], at_lo[w], None, out=gSa[sl])
            ops.gemm_tf32x3_ex(g_dvec[sl].view(3 * n, F), ct_hi[w], ct_lo[w], None, out=gSc[sl].view(3 * n, KP))
        g_geom = ops.layer0_basis_bwd(ctx.p0, ctx.g0, geom, ctx.live, offset, n_elem, KP, gSa, gSc)
        return g_geom, None, None, None, None, None, None, None


def layer0_fusable(hidden: int, num_rbf: int, n_elem: int) -> bool:
    """The aggregated first-layer pass needs GEMM-shaped outputs (F % 64 == 0) and a row of sums that fits shared memory."""
    return hidden % 64 == 0 and ops.layer0_row_len(n_elem, num_rbf) <= 3072


def layer0_edge(geom, xh_tab, Wt, bias, offset, g0: RowGraph, p0, n_elem: int):
    return _Layer0HV.apply(geom, xh_tab, Wt, bias, offset, g0, p0, n_elem)


# ----------------------------------------------------------------------------------------------------
# composite (any-order differentiable) formulation
# ----------------------------------------------------------------------------------------------------
def edge_geometry_composite(pos: Tensor, cell: Optional[Tensor], g: RowGraph) -> Tensor:
    ps = gather_rows(pos, g.seg_src)
    pr = gather_rows(pos, g.seg_dst_atom)
    D = ps - pr
    if cell is not None:
        ce = gather_rows(cell.reshape(-1, 9), g.seg_edge_graph).view(-1, 3, 3)
        S = g.shift[:, :3].to(pos.dtype) * g.sign
        D = D + (S.unsqueeze(2) * ce).sum(1)
    d = D.norm(dim=-1)
    d = torch.where(d <= 1.0e-6, torch.full_like(d, 1.0e-6), d)
    return torch.cat([D / d[:, None], d[:, None]], dim=1)


def painn_edge_composite_flat(xh, vec, geom, Wt, bias, radial_basis, g: RowGraph, live_mask: Optional[Tensor] = None):
    """Same contract as ``painn_edge`` (``xh`` is the flat ``[rows, 3F]`` buffer of ``graph.xh_sources``) built from
    differentiable pieces; materialises per-edge tensors, so it is meant for training-size batches."""
    F3 = xh.size(1)
    F = F3 // 3
    M = Wt.size(0)
    P = gather_rows(xh, g.seg_xh)
    V = gather_rows(vec.reshape(-1, F3), g.seg_src).view(-1, 3, F)
    emb = radial_basis(geom[:, 3])
    phi = torch.zeros((g.n_edges, F3), dtype=xh.dtype, device=xh.device)
    for m in range(M):
        idx = g.module_edges(m)
        if idx.numel():
            phi = phi.index_copy(0, idx, emb[idx] @ Wt[m] + bias[m])
    a, b, c = torch.split(P * phi, F, dim=-1)
    m_vec = V * (b * (1 / math.sqrt(3.0)))[:, None, :] + c[:, None, :] * geom[:, :3, None]
    m_vec = m_vec * (1 / math.sqrt(F))
    live = g.edge_mod >= 0
    if live_mask is not None:     # Verlet-skin superset list: dead entries are not edges of the reference
        live = live & live_mask.bool()
    live = live.to(xh.dtype)[:, None]
    dx = segment_sum(a * live, g.seg_dst)
    dvec = segment_sum((m_vec * live[:, :, None]).reshape(-1, F3), g.seg_dst).view(-1, 3, F)
    return dx, dvec
