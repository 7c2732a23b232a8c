"""CPU emulation of ``hermnet_b200.ops`` for the ``-m "not gpu"`` suite (TEST INFRASTRUCTURE).

The product has no CPU path.  To exercise the HOST logic (graph building, row layouts, autograd wiring, model
classes, DDP / halo plumbing under gloo) without a GPU, ``install(monkeypatch)`` swaps every function of
``hermnet_b200.ops`` for a torch-CPU function with the same contract.  The emulated edge / geometry backward
functions follow the formulas of the CUDA kernels (csrc/hn_edge.cu, hn_geom.cu) line by line -- including the
12-wide Gaussian band -- so that the maths of the hand-written backward is checked against autograd of the
oracle on the CPU; the kernels themselves are checked on the GPU by the ``-m gpu`` tests.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from hermnet_b200 import ops
from hermnet_b200._lib import EdgeParams
from oracle import neighbor_oracle as NO


def _rows(rowptr):
    lens = (rowptr[1:] - rowptr[:-1]).long()
    return torch.repeat_interleave(torch.arange(lens.numel()), lens)


def radius_graph(pos, cell, graph_ptr, rc, group=None, n_groups=1, max_neighbors=0):
    pos_np = pos.detach().numpy().astype(np.float32)
    gp = graph_ptr.tolist()
    rows = []
    for g in range(len(gp) - 1):
        a0, a1 = gp[g], gp[g + 1]
        if cell is None:
            ei = NO.radius_graph_nonpbc(pos_np[a0:a1], rc, max_neighbors if max_neighbors > 0 else 10 ** 9)
            i, j, S = ei[1], ei[0], np.zeros((ei.shape[1], 3), np.int64)
        else:
            i, j, S = NO.neighbor_list_pbc(pos_np[a0:a1], cell[g].numpy(), rc)
        rows.append(np.concatenate([(i + a0)[:, None], (j + a0)[:, None], S], 1))
    allr = np.concatenate(rows, 0) if rows else np.zeros((0, 5), np.int64)
    grp = np.zeros(len(allr), np.int64) if group is None else group.numpy()[allr[:, 1]]
    key = allr[:, 0] * n_groups + grp
    order = np.lexsort((allr[:, 4], allr[:, 3], allr[:, 2], allr[:, 1], key))
    allr, key = allr[order], key[order]
    n = pos.size(0)
    counts = np.bincount(key, minlength=n * n_groups)
    rowptr = torch.zeros(n * n_groups + 1, dtype=torch.int32)
    rowptr[1:] = torch.from_numpy(np.cumsum(counts)).to(torch.int32)
    col = torch.from_numpy(allr[:, 1]).to(torch.int32)
    shift = torch.zeros((len(allr), 4), dtype=torch.int8)
    shift[:, :3] = torch.from_numpy(allr[:, 2:5]).to(torch.int8)
    return rowptr, col, shift


def sort_by_key(keys, n_keys):
    order = torch.sort(keys.long(), stable=True).indices
    counts = torch.bincount(keys.long(), minlength=n_keys)
    rowptr = torch.zeros(n_keys + 1, dtype=torch.int32)
    rowptr[1:] = torch.cumsum(counts, 0).to(torch.int32)
    return rowptr, order.to(torch.int32)


def expand_rowptr(rowptr, n_edges):
    return _rows(rowptr).to(torch.int32)


def triplets(rowptr, col, src_type=None, type_a=-1, type_c=-1):
    rows = NO.triplets_bruteforce(rowptr.numpy(), col.numpy(), None if src_type is None else src_type.numpy(),
                                  None if type_a < 0 else type_a, None if type_c < 0 else type_c)
    n_rows = rowptr.numel() - 1
    counts = np.bincount(rows[:, 1], minlength=n_rows) if len(rows) else np.zeros(n_rows, np.int64)
    # row of a triplet = row of e1 (rows may be (atom, slot) rows: recover from e1)
    er = _rows(rowptr).numpy()
    counts = np.bincount(er[rows[:, 3]], minlength=n_rows) if len(rows) else np.zeros(n_rows, np.int64)
    tp = torch.zeros(n_rows + 1, dtype=torch.int64)
    tp[1:] = torch.from_numpy(np.cumsum(counts))
    return tp, torch.from_numpy(rows[:, 3]).to(torch.int32), torch.from_numpy(rows[:, 4]).to(torch.int32)


def triplet_dots(m_vec, trip_ptr, e1, e2):
    n_rows = trip_ptr.numel() - 1
    out = torch.zeros((n_rows, m_vec.size(-1)), dtype=m_vec.dtype)
    row = _rows(trip_ptr)
    out.index_add_(0, row, (m_vec[e1.long()] * m_vec[e2.long()]).sum(1))
    return out


# ---------------------------------------------------------------------------------------------------------
def _grad_D(geom, g_geom):
    t = g_geom.sum(0) if g_geom.dim() == 3 else g_geom
    u, d = geom[:, :3], geom[:, 3:4]
    clamped = (d == 1.0e-6)
    dot = (t[:, :3] * u).sum(1, keepdim=True)
    free = t[:, 3:4] * u + (t[:, :3] - dot * u) / d
    return torch.where(clamped, t[:, :3] / d, free)


def edge_geom_fwd(pos, cell, g):
    s, r = g.col.long(), torch.div(g.edge_row.long(), g.rows_per_atom, rounding_mode="floor")
    D = pos[s] - pos[r]
    if cell is not None:
        S = g.shift[:, :3].to(pos.dtype) * g.sign
        D = D + torch.einsum("ni,nij->nj", S, cell[g.atom_graph[s].long()])
    d = D.norm(dim=-1)
    d = torch.where(d <= 1.0e-6, torch.full_like(d, 1.0e-6), d)
    return torch.cat([D / d[:, None], d[:, None]], 1).contiguous()


def edge_geom_bwd(geom, g_geom, g, want_cell):
    gD = _grad_D(geom, g_geom)
    s, r = g.col.long(), torch.div(g.edge_row.long(), g.rows_per_atom, rounding_mode="floor")
    grad_pos = torch.zeros((g.n_atoms, 3), dtype=geom.dtype)
    grad_pos.index_add_(0, s, gD)
    grad_pos.index_add_(0, r, -gD)
    cellw = None
    if want_cell:
        S = g.shift[:, :3].to(geom.dtype) * g.sign
        cellw = torch.zeros((g.n_atoms, 9), dtype=geom.dtype)
        cellw.index_add_(0, r, (S[:, :, None] * gD[:, None, :]).reshape(-1, 9))
    return grad_pos, cellw


def edge_params(g, n_modules, hidden, num_rbf, env_p, rc, coeff):
    return EdgeParams(g.n_atoms, g.n_rows, n_modules, hidden, num_rbf, env_p, 1.0 / rc, coeff)


def edge_num_slices(hidden):
    return 1


def _band(p, geom, offset, deriv=False):
    """val[e, k] (and dval) with the kernel's 12-wide band; zeros outside the band / beyond the cutoff."""
    K = p.num_rbf
    u = geom[:, 3] * p.inv_rc
    nb = min(12, K)
    kc = torch.floor(u * (K - 1)).long()
    k0 = (kc - 5).clamp(min=0).clamp(max=K - nb)
    k = torch.arange(K)[None, :]
    inband = (k >= k0[:, None]) & (k < k0[:, None] + nb) & (u < 1)[:, None]
    pp = p.env_p
    a, b, c = -0.5 * (pp + 1) * (pp + 2), float(pp * (pp + 2)), -0.5 * pp * (pp + 1)
    env = 1 + a * u ** pp + b * u ** (pp + 1) + c * u ** (pp + 2)
    diff = u[:, None] - offset[None, :]
    gk = torch.exp(p.coeff * diff * diff)
    val = torch.where(inband, env[:, None] * gk, torch.zeros_like(gk))
    if not deriv:
        return val
    denv = a * pp * u ** (pp - 1) + b * (pp + 1) * u ** pp + c * (pp + 2) * u ** (pp + 1)
    dval = (denv[:, None] * gk + env[:, None] * gk * (2 * p.coeff * diff)) * p.inv_rc
    return val, torch.where(inband, dval, torch.zeros_like(dval))


def _edge_common(p, xh, vec, geom, g, Wt, bias, offset, deriv=False):
    F = p.hidden
    row = g.edge_row.long()
    m = g.row_mod.long()[row]
    live = m >= 0
    mm = m.clamp(min=0)
    s = g.col.long()
    P = xh[(g.row_xoff[row] + s).clamp(min=0)]
    V = vec[s]
    band = _band(p, geom, offset, deriv)
    val = band[0] if deriv else band
    phi = torch.einsum("ek,ekc->ec", val, Wt[mm]) + bias[mm]
    dphi = torch.einsum("ek,ekc->ec", band[1], Wt[mm]) if deriv else None
    return F, row, mm, live, s, P, V, val, phi, dphi


def painn_edge_fwd(p, xh, vec, geom, g, Wt, bias, offset):
    if vec is None:                      # NULL = identically zero (include/hermnet_b200.h)
        vec = torch.zeros((p.n_atoms, 3, p.hidden), dtype=xh.dtype)
    F, row, mm, live, s, P, V, val, phi, _ = _edge_common(p, xh, vec, geom, g, Wt, bias, offset)
    c1, c2 = 1 / math.sqrt(3.0 * F), 1 / math.sqrt(F)
    a, b, c = torch.split(P * phi, F, dim=-1)
    mv = V * (b * c1)[:, None, :] + (c * c2)[:, None, :] * geom[:, :3, None]
    lv = live.to(xh.dtype)
    dx = torch.zeros((p.n_rows, F), dtype=xh.dtype).index_add_(0, row, a * lv[:, None])
    dvec = torch.zeros((p.n_rows, 3, F), dtype=xh.dtype).index_add_(0, row, mv * lv[:, None, None])
    return dx, dvec


def _t_terms(p, V, geom, g_dvec, row, F):
    c1, c2 = 1 / math.sqrt(3.0 * F), 1 / math.sqrt(F)
    gv = g_dvec[row]                                    # [E,3,F]
    tb = (gv * V).sum(1) * c1
    tc = (gv * geom[:, :3, None]).sum(1) * c2
    return gv, tb, tc, c1, c2


def painn_edge_bwd_dst(p, xh, vec, geom, g, Wt, bias, offset, g_dx, g_dvec):
    if vec is None:
        vec = torch.zeros((p.n_atoms, 3, p.hidden), dtype=xh.dtype)
    F, row, mm, live, s, P, V, val, phi, dphi = _edge_common(p, xh, vec, geom, g, Wt, bias, offset, deriv=True)
    gv, tb, tc, c1, c2 = _t_terms(p, V, geom, g_dvec, row, F)
    Pa, Pb, Pc = torch.split(P, F, dim=-1)
    da, db, dc = torch.split(dphi, F, dim=-1)
    gd = (g_dx[row] * Pa * da + tb * Pb * db + tc * Pc * dc).sum(1)
    cphi = Pc * phi[:, 2 * F:] * c2
    gu = (gv * cphi[:, None, :]).sum(2)
    out = torch.cat([gu, gd[:, None]], 1) * live.to(xh.dtype)[:, None]
    return out.view(1, -1, 4).contiguous()


def painn_edge_bwd_src(p, xh, vec, geom, g, Wt, bias, offset, g_dx, g_dvec):
    F, row, mm, live, s, P, V, val, phi, _ = _edge_common(p, xh, vec, geom, g, Wt, bias, offset)
    gv, tb, tc, c1, c2 = _t_terms(p, V, geom, g_dvec, row, F)
    fa, fb, fc = torch.split(phi, F, dim=-1)
    lv = live.to(xh.dtype)[:, None]
    gP = torch.cat([g_dx[row] * fa, tb * fb, tc * fc], 1) * lv
    grad_xh = torch.zeros_like(xh).index_add_(0, (g.row_xoff[row] + s).clamp(min=0), gP)
    bphi = P[:, F:2 * F] * fb * c1 * lv
    grad_vec = torch.zeros_like(vec).index_add_(0, s, gv * bphi[:, None, :])
    return grad_xh, grad_vec


def painn_edge_bwd_w(p, xh, vec, geom, g, offset, g_dx, g_dvec):
    F = p.hidden
    row = g.edge_row.long()
    m = g.row_mod.long()[row]
    act = m >= 0
    if p.flags & 1:                      # Verlet-skin superset list: dead entries feed neither gW nor gb
        act = act & p.live.bool()
    lv = act.to(xh.dtype)[:, None]
    mm = m.clamp(min=0)
    s = g.col.long()
    P = xh[(g.row_xoff[row] + s).clamp(min=0)]
    V = vec[s]
    gv, tb, tc, c1, c2 = _t_terms(p, V, geom, g_dvec, row, F)
    gphi = torch.cat([g_dx[row] * P[:, :F], tb * P[:, F:2 * F], tc * P[:, 2 * F:]], 1) * lv
    val = _band(p, geom, offset)
    gW = torch.zeros((p.n_modules, p.num_rbf, 3 * F), dtype=xh.dtype)
    gW.index_add_(0, mm, val[:, :, None] * gphi[:, None, :])
    gb = torch.zeros((p.n_modules, 3 * F), dtype=xh.dtype).index_add_(0, mm, gphi)
    return gW, gb


# ---------------------------------------------------------------------------------------------------------
# tensor-core edge kernels (csrc/hn_edge_tc.cu): the plan builders follow the CUDA kernels step by step and the
# edge passes walk the PLAN (blocks -> tiles -> edge records, basis restricted to the tile's window), so the host logic
# of hermnet_b200/tileplan.py and the plan layout are exercised on the CPU
# ---------------------------------------------------------------------------------------------------------
TC_TN, TC_KC, TC_ROWS_DST, TC_ROWS_SRC, TC_NG = 64, 32, 12, 32, 3


def tc_supported(hidden, num_rbf):
    return hidden == 128 and 2 <= num_rbf <= 256


def tc_block_rows(src_major=False):
    return TC_ROWS_SRC if src_major else TC_ROWS_DST


def tc_groups():
    return TC_NG


def tc_split_weights(Wt):
    return Wt.detach().clone(), torch.ones(Wt.size(0), dtype=torch.float32)


def tc_basis_index(geom, inv_rc, num_rbf):
    u = geom.detach()[:, 3] * inv_rc
    kc = torch.clamp((u * (num_rbf - 1)).to(torch.int32), max=num_rbf - 1)
    return torch.where(u < 1, kc, torch.full_like(kc, num_rbf - 1)).to(torch.int32)


def _tc_fits(kc, k0, K, W=32):
    return kc >= K - 1 or min(kc + 6, K - 1) <= k0 + W - 1


def _tc_window_start(kc, K):
    return 0 if kc >= K - 1 else (max(kc - 5, 0) & ~7)


def _tc_tiles_of_group(ks, K, W=32):
    starts, start, k0 = [], 0, 0
    for i, k in enumerate(ks):
        if i == start:
            k0 = _tc_window_start(k, K)
        elif i - start >= TC_TN or not _tc_fits(k, k0, K, W):
            starts.append(start)
            start = i
            k0 = _tc_window_start(k, K)
    if len(ks):
        starts.append(start)
    return starts


def tc_plan_records(g, geom, inv_rc, num_rbf, src_major, atom_local, src_block):
    row, col = g.edge_row.long(), g.col.long()
    m = g.row_mod.long()[row]
    xr = (g.row_xoff[row] + col).to(torch.int32)
    eid = torch.arange(g.n_edges, dtype=torch.int32)
    kc = tc_basis_index(geom, inv_rc, num_rbf)
    if src_major:
        rec = torch.stack([g.edge_row, xr, (col % src_block).to(torch.int32), eid], 1)
        sub = m.to(torch.int32)
    else:
        atom = torch.div(row, g.rows_per_atom, rounding_mode="floor")
        rec = torch.stack([xr, g.col, atom_local[atom].to(torch.int32), eid], 1)
        sub = torch.where(m >= 0, torch.zeros_like(m), torch.full_like(m, -1)).to(torch.int32)
    return rec.contiguous(), kc, sub.contiguous()


def tc_plan_sort(in_ptr, ids, kc, sub, n_seg, n_sub, num_rbf):
    ip = in_ptr.tolist()
    order, counts = [], torch.zeros(n_seg * n_sub, dtype=torch.int32)
    for sg in range(n_seg):
        items = torch.arange(ip[sg], ip[sg + 1])
        e = items if ids is None else ids[items].long()
        sb = torch.zeros_like(e) if sub is None else sub[e].long()
        keep = sb >= 0
        e, sb = e[keep], sb[keep]
        o = torch.sort(sb * num_rbf + kc[e].long(), stable=True).indices
        order.append(e[o])
        counts[sg * n_sub:(sg + 1) * n_sub] = torch.bincount(sb, minlength=n_sub).to(torch.int32)
    grp_ptr = torch.zeros(n_seg * n_sub + 1, dtype=torch.int32)
    grp_ptr[1:] = torch.cumsum(counts, 0).to(torch.int32)
    order = torch.cat(order).to(torch.int32) if order else torch.zeros(0, dtype=torch.int32)
    return order, grp_ptr


def tc_plan_count(order, kc, grp_ptr, n_groups, num_rbf, window=32):
    kk = kc[order.long()].tolist()
    gp = grp_ptr.tolist()
    return torch.tensor([len(_tc_tiles_of_group(kk[gp[g]:gp[g + 1]], num_rbf, window)) for g in range(n_groups)], dtype=torch.int32)


def tc_plan_fill(order, kc, grp_ptr, n_groups, num_rbf, grp_tile, n_tiles, window=32):
    kk = kc[order.long()].tolist()
    gp = grp_ptr.tolist()
    out = []
    for g in range(n_groups):
        out += [gp[g] + s for s in _tc_tiles_of_group(kk[gp[g]:gp[g + 1]], num_rbf, window)]
    assert len(out) == n_tiles
    return torch.tensor(out + ([0] if not out else []), dtype=torch.int32)


def tc_plan_finalize(order, tile_start, n_tiles, n_edges, rec, tile_mod):
    erec = torch.zeros((max(n_edges, 1), 4), dtype=torch.int32)
    info = torch.zeros((max(n_tiles, 1), 4), dtype=torch.int32)
    ts = tile_start.tolist()
    for t in range(n_tiles):
        e0, e1 = ts[t], (ts[t + 1] if t + 1 < n_tiles else n_edges)
        r = rec[order[e0:e1].long()]
        key = ((r[:, 2] % TC_NG) << 16) | r[:, 2]
        o = torch.sort(key, stable=True).indices
        erec[e0:e1] = r[o]
        split = sum(int(((r[:, 2] % TC_NG) <= gq).sum()) << (8 * gq) for gq in range(TC_NG - 1))
        info[t] = torch.tensor([e0, e1 - e0, split, int(tile_mod[t])], dtype=torch.int32)
    return erec, info


def tc_tile_windows(plan, geom, inv_rc, num_rbf, live=None):
    K = num_rbf
    u = geom.detach()[:, 3] * inv_rc
    for t in range(plan.n_tiles):
        e0, cnt = int(plan.tile_info[t, 0]), int(plan.tile_info[t, 1])
        ue = u[plan.erec[e0:e0 + cnt, 3].long()]
        ue = ue[ue < 1]
        k0, nchunk = 0, 1
        if ue.numel():
            kc = torch.clamp((ue * (K - 1)).to(torch.int32), max=K - 1)
            k0 = max(int(kc.min()) - 5, 0) & ~7
            hi = min(int(kc.max()) + 6, K - 1)
            nchunk = (hi - k0 + TC_KC) // TC_KC
        plan.tile_win[t, 0], plan.tile_win[t, 1] = k0, nchunk
        eid = plan.erec[e0:e0 + cnt, 3].long()
        tg = geom.detach()[eid].clone()
        if live is not None:
            tg[:, 3] = torch.where(live[eid].bool(), tg[:, 3], -tg[:, 3])
        plan.tile_geom[e0:e0 + cnt] = tg


def _tc_records(plan):
    """Flattened view of a plan: per record (block, tile, window lo, window hi)."""
    nt = plan.n_tiles
    info, win = plan.tile_info[:nt].long(), plan.tile_win[:nt].long()
    cnt = info[:, 1]
    n = int(cnt.sum())
    tile_of = torch.repeat_interleave(torch.arange(nt), cnt)
    assert n == 0 or bool((info[:, 0] == torch.cumsum(cnt, 0) - cnt).all()), "tiles must be contiguous"
    bt = plan.blk_tile.long()
    blk_of_tile = torch.repeat_interleave(torch.arange(plan.n_blocks), bt[1:] - bt[:-1])
    return n, tile_of, blk_of_tile[tile_of], win[tile_of, 0], win[tile_of, 0] + TC_KC * win[tile_of, 1], info[tile_of, 3]


def _tc_phi(p, plan, geom, Wt, bias, offset, eid, mod, lo, hi, deriv=False):
    K = p.num_rbf
    dead = geom[:, 3] < 0                 # tc_tile_windows stores -d for the dead entries of a superset list
    u = geom[:, 3].abs() * p.inv_rc
    pp = p.env_p
    a, b, c = -0.5 * (pp + 1) * (pp + 2), float(pp * (pp + 2)), -0.5 * pp * (pp + 1)
    env = 1 + a * u ** pp + b * u ** (pp + 1) + c * u ** (pp + 2)
    diff = u[:, None] - offset[None, :]
    gk = torch.exp(p.coeff * diff * diff)
    k = torch.arange(K)[None, :]
    inwin = (k >= lo[:, None]) & (k < hi[:, None]) & (u < 1)[:, None]
    val = torch.where(inwin, env[:, None] * gk, torch.zeros_like(gk))
    phi = torch.einsum("ek,ekc->ec", val, Wt[mod]) + bias[mod]
    if getattr(p, "flags", 0) & 1:       # Verlet-skin superset list: dead entries contribute nothing
        phi = torch.where(dead[:, None], torch.zeros_like(phi), phi)
    if not deriv:
        return phi, None
    denv = a * pp * u ** (pp - 1) + b * (pp + 1) * u ** pp + c * (pp + 2) * u ** (pp + 1)
    dval = torch.where(inwin, (denv[:, None] * gk + env[:, None] * gk * (2 * p.coeff * diff)) * p.inv_rc, torch.zeros_like(gk))
    dphi = torch.einsum("ek,ekc->ec", dval, Wt[mod])
    if getattr(p, "flags", 0) & 1:
        dphi = torch.where(dead[:, None], torch.zeros_like(dphi), dphi)
    return phi, dphi


def tc_edge_fwd(p, plan, xh, vec, geom, wsplit, wscale, bias, offset, n_rows, debug_phi=False):
    F = p.hidden
    assert plan.kind == "dst"
    if vec is None:
        vec = torch.zeros((p.n_atoms, 3, F), dtype=xh.dtype)
    n, tile_of, blk, lo, hi, mod = _tc_records(plan)
    er = plan.erec[:n].long()
    bi = plan.blk_info.long()
    row = bi[blk, 0] + er[:, 2] * bi[blk, 1]
    assert bool((er[:, 2] < bi[blk, 2]).all()) and bool((mod == bi[blk, 3]).all())
    tg = plan.tile_geom[:n]                      # the kernels read the geometry in record order (hn_tc_tile_windows)
    phi, _ = _tc_phi(p, plan, tg, wsplit, bias, offset, er[:, 3], mod, lo, hi)
    c1, c2 = 1 / math.sqrt(3.0 * F), 1 / math.sqrt(F)
    xrow = plan.blk_xoff.long()[blk] + er[:, 1]              # the kernels index xh with (block offset + source index)
    a, b, c = torch.split(xh[xrow] * phi, F, dim=-1)
    mv = vec[er[:, 1]] * (b * c1)[:, None, :] + (c * c2)[:, None, :] * tg[:, :3, None]
    dx = torch.zeros((n_rows, F), dtype=xh.dtype).index_add_(0, row, a)
    dvec = torch.zeros((n_rows, 3, F), dtype=xh.dtype).index_add_(0, row, mv)
    return dx, dvec


def tc_edge_bwd_dst(p, plan, xh, vec, geom, wsplit, wscale, bias, offset, g_dx, g_dvec):
    F = p.hidden
    if vec is None:
        vec = torch.zeros((p.n_atoms, 3, F), dtype=xh.dtype)
    n, tile_of, blk, lo, hi, mod = _tc_records(plan)
    er = plan.erec[:n].long()
    bi = plan.blk_info.long()
    row = bi[blk, 0] + er[:, 2] * bi[blk, 1]
    gm = plan.tile_geom[:n]
    phi, dphi = _tc_phi(p, plan, gm, wsplit, bias, offset, er[:, 3], mod, lo, hi, deriv=True)
    gv, tb, tc, c1, c2 = _t_terms(p, vec[er[:, 1]], gm, g_dvec, row, F)
    Pa, Pb, Pc = torch.split(xh[plan.blk_xoff.long()[blk] + er[:, 1]], F, dim=-1)
    da, db, dc = torch.split(dphi, F, dim=-1)
    gd = (g_dx[row] * Pa * da + tb * Pb * db + tc * Pc * dc).sum(1)
    gu = (gv * (Pc * phi[:, 2 * F:] * c2)[:, None, :]).sum(2)
    out = torch.zeros((1, geom.size(0), 4), dtype=xh.dtype)
    out[0, er[:, 3]] = torch.cat([gu, gd[:, None]], 1)
    return out


def tc_edge_bwd_src(p, plan, xh, vec, geom, wsplit, wscale, bias, offset, g_dx, g_dvec):
    F = p.hidden
    assert plan.kind == "src"
    n, tile_of, blk, lo, hi, mod = _tc_records(plan)
    er = plan.erec[:n].long()
    bi = plan.blk_info.long()
    s = bi[blk, 0] + er[:, 2]
    row = er[:, 0]
    gm = plan.tile_geom[:n]
    phi, _ = _tc_phi(p, plan, gm, wsplit, bias, offset, er[:, 3], mod, lo, hi)
    gv, tb, tc, c1, c2 = _t_terms(p, vec[s], gm, g_dvec, row, F)
    fa, fb, fc = torch.split(phi, F, dim=-1)
    gP = torch.cat([g_dx[row] * fa, tb * fb, tc * fc], 1)
    grad_xh = torch.zeros_like(xh).index_add_(0, er[:, 1], gP)
    bphi = xh[er[:, 1]][:, F:2 * F] * fb * c1
    grad_vec = torch.zeros_like(vec).index_add_(0, s, gv * bphi[:, None, :])
    return grad_xh, grad_vec


def _layer0_terms(p, g, geom, live, offset, deriv=False):
    row = g.edge_row.long()
    act = g.row_mod.long()[row] >= 0
    if live is not None and (p.flags & 1):
        act = act & live.bool()
    band = _band(p, geom, offset, deriv)
    w = torch.cat([torch.ones_like(geom[:, :1]), geom[:, :3]], 1)          # weights (1, ux, uy, uz)
    return row, act, band, w


def layer0_basis_fwd(p, g, geom, live, offset, n_elem, kp):
    K = p.num_rbf
    row, act, val, w = _layer0_terms(p, g, geom, live, offset)
    z = g.col.long()
    S = torch.zeros((p.n_rows, 4, kp), dtype=geom.dtype)
    a = act.to(geom.dtype)
    contrib = (w[:, :, None] * val[:, None, :]) * a[:, None, None]         # [E,4,K]
    flat = S.view(p.n_rows, 4, kp)
    for zz in range(n_elem):
        sel = (z == zz)
        if sel.any():
            flat[:, :, zz * K:(zz + 1) * K].index_add_(0, row[sel], contrib[sel])
            cnt = torch.zeros((p.n_rows, 4), dtype=geom.dtype).index_add_(0, row[sel], w[sel] * a[sel, None])
            flat[:, :, n_elem * K + zz] += cnt
    return S[:, 0].contiguous(), S[:, 1:].contiguous()


def layer0_basis_bwd(p, g, geom, live, offset, n_elem, kp, g_Sa, g_Sc):
    K = p.num_rbf
    row, act, (val, dval), w = _layer0_terms(p, g, geom, live, offset, deriv=True)
    z = g.col.long()
    G = torch.cat([g_Sa[:, None, :], g_Sc], 1)                              # [R,4,kp]
    E = geom.size(0)
    idx = (z[:, None] * K + torch.arange(K)[None, :])                       # [E,K]
    Ge = G[row]                                                             # [E,4,kp]
    Gk = torch.gather(Ge, 2, idx[:, None, :].expand(E, 4, K))               # [E,4,K]
    Gc = torch.gather(Ge, 2, (n_elem * K + z)[:, None, None].expand(E, 4, 1)).squeeze(2)   # [E,4]
    gd = ((Gk * w[:, :, None]).sum(1) * dval).sum(1)
    gu = (Gk[:, 1:, :] * val[:, None, :]).sum(2) + Gc[:, 1:]
    out = torch.cat([gu, gd[:, None]], 1) * act.to(geom.dtype)[:, None]
    return out.contiguous()


def layernorm_fwd(x, eps):
    mean = x.mean(1)
    var = ((x - mean[:, None]) ** 2).mean(1)
    rstd = 1.0 / torch.sqrt(var + eps)
    return (x - mean[:, None]) * rstd[:, None], mean, rstd


def layernorm_bwd(g_xhat, x, mean, rstd):
    xhat = (x - mean[:, None]) * rstd[:, None]
    return rstd[:, None] * (g_xhat - g_xhat.mean(1, keepdim=True) - xhat * (g_xhat * xhat).mean(1, keepdim=True))


def readout_fwd(x, W1, b1, W2, b2):
    h = x @ W1.t() + b1
    return (_ssilu(h) @ W2.reshape(-1, 1)) + b2


def readout_bwd(x, W1, b1, W2, b2, g_e):
    h = x @ W1.t() + b1
    sg = torch.sigmoid(h)
    dh = sg * (1 + h * (1 - sg)) / 0.6
    return ((g_e.reshape(-1, 1) * W2.reshape(1, -1)) * dh) @ W1


def gather_rows(X, idx):
    return X[idx.long()].contiguous()


def segment_sum(Y, rowptr, perm, n_rows):
    items = torch.arange(Y.size(0)) if perm is None else perm.long()
    row = _rows(rowptr)
    return torch.zeros((n_rows, Y.size(1)), dtype=Y.dtype).index_add_(0, row, Y[items])


def gemm_tf32x3(a, w_hi, w_lo, bias):
    out = a @ (w_hi + w_lo).t()
    return out if bias is None else out + bias


def _ssilu(z):
    return torch.nn.functional.silu(z) / 0.6


def _dssilu(z):
    sg = torch.sigmoid(z)
    return sg * (1 + z * (1 - sg)) / 0.6


def gemm_tf32x3_ex(a, w_hi, w_lo, bias, out=None, mode=0, aux=None, out2=None):
    acc = a @ (w_hi + w_lo).t()
    if bias is not None:
        acc = acc + bias
    if mode == 1:
        if out2 is not None:
            out2.copy_(acc)
        acc = _ssilu(acc)
    elif mode == 2:
        acc = acc * _dssilu(aux)
    if out is None:
        return acc
    out.copy_(acc)
    return out


# fused element-wise stages of the node update (csrc/hn_node.cu), same in-place output contract
def node_pre(x, dx, vec, dvec, xcat, vecp):
    F = x.size(1)
    xcat[:, :F] = (x + dx) * (1 / math.sqrt(2.0))
    vecp.copy_(vec + dvec.reshape(vec.shape))


def node_mid(v12, vdot, xcat):
    n, F = vdot.shape
    v = v12.view(n, 3, 2 * F)
    v1, v2 = v[:, :, :F], v[:, :, F:]
    vdot.copy_((v1 * v2).sum(1) / math.sqrt(F))
    xcat[:, F:] = torch.sqrt((v2 * v2).sum(1) + 1e-8)


def node_post(xcat, a, vdot, vecp, v12, x_out, vec_out):
    n, F = vdot.shape
    a1, a2, a3 = a[:, :F], a[:, F:2 * F], a[:, 2 * F:]
    x_out.copy_(xcat[:, :F] + (a1 + a2 * vdot) * (1 / math.sqrt(2.0)))
    vec_out.copy_(vecp + a3[:, None, :] * v12.view(n, 3, 2 * F)[:, :, :F])


def node_post_bwd(g_x, g_vec, a, vdot, v12, g_a, g_vdot, g_v12):
    n, F = vdot.shape
    c = 1 / math.sqrt(2.0)
    v1 = v12.view(n, 3, 2 * F)[:, :, :F]
    g_a[:, :F] = g_x * c
    g_a[:, F:2 * F] = g_x * c * vdot
    g_a[:, 2 * F:] = (g_vec * v1).sum(1)
    g_vdot.copy_(g_x * c * a[:, F:2 * F])
    g_v12.view(n, 3, 2 * F)[:, :, :F] = g_vec * a[:, None, 2 * F:]


def node_mid_bwd(g_vdot, g_cat, v12, vn, g_v12):
    n, F = g_vdot.shape
    v = v12.view(n, 3, 2 * F)
    v1, v2 = v[:, :, :F], v[:, :, F:]
    gd = g_vdot / math.sqrt(F)
    gv = g_v12.view(n, 3, 2 * F)
    gv[:, :, :F] += gd[:, None, :] * v2
    gv[:, :, F:] = (g_cat[:, F:] / vn)[:, None, :] * v2 + gd[:, None, :] * v1


def node_pre_bwd(g_xn, g_cat, g_vecn, g_vecp, g_x, g_vec):
    F = g_xn.size(1)
    g_x.copy_((g_xn + g_cat[:, :F]) * (1 / math.sqrt(2.0)))
    g_vec.copy_(g_vecn + g_vecp.view(g_vecn.shape))


def split_tf32(w):
    w = w.detach().contiguous()
    hi = (w.view(torch.int32) & -8192).view(torch.float32)
    return hi, w - hi


def install(monkeypatch):
    """Swap ``hermnet_b200.ops`` for the CPU emulation (pytest ``monkeypatch`` restores it afterwards)."""
    for name in ("radius_graph", "sort_by_key", "expand_rowptr", "triplets", "triplet_dots", "edge_geom_fwd",
                 "edge_geom_bwd", "edge_params", "edge_num_slices", "painn_edge_fwd", "painn_edge_bwd_dst",
                 "painn_edge_bwd_src", "painn_edge_bwd_w", "gemm_tf32x3_ex", "node_pre", "node_mid", "node_post",
                 "node_post_bwd", "node_mid_bwd", "node_pre_bwd", "gather_rows", "segment_sum", "gemm_tf32x3", "split_tf32",
                 "tc_supported", "tc_block_rows", "tc_groups", "tc_split_weights", "tc_basis_index", "tc_plan_count", "tc_plan_fill",
                 "tc_plan_records", "tc_plan_sort", "tc_plan_finalize", "tc_tile_windows", "tc_edge_fwd", "tc_edge_bwd_dst", "tc_edge_bwd_src", "layer0_basis_fwd", "layer0_basis_bwd", "layernorm_fwd", "layernorm_bwd", "readout_fwd", "readout_bwd"):
        monkeypatch.setattr(ops, name, globals()[name])
    monkeypatch.setattr(ops, "require_cuda", lambda t, what: None)
    monkeypatch.setattr(ops, "compute_device", lambda t: t.device)
    monkeypatch.setattr(ops, "sm_count", lambda: 148)


def install_plain():
    """Same as ``install`` for spawned worker processes (no pytest monkeypatch there)."""
    class _MP:
        @staticmethod
        def setattr(obj, name, value):
            setattr(obj, name, value)
    install(_MP)
