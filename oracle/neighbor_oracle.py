"""Brute-force neighbour-list / triplet oracle (TEST INFRASTRUCTURE, numpy, CPU).

Restates the contract of ``/root/reference/HermNet/data.py:14-24``:

* periodic branch (data.py:18-24): ASE ``primitive_neighbor_list('ijS', pbc=[T,T,T], cell, positions,
  cutoff=rc)`` [upstream, unverified here] -- the set
  ``{(i, j, S) : || pos_j - pos_i + S.cell || < rc, not (i == j and S == 0)}``.
  Arithmetic restated from ASE: ``float32(pos_j - pos_i)`` promoted to float64, plus
  ``S.dot(cell)`` in float64 (int64 x float32 -> float64), squared, summed over the 3 components
  left to right, ``sqrt``, strict ``<`` against the Python float ``rc``.  Positions need not lie
  inside the cell.  The reference then stores ``edge_index = [i; j]``, ``edge_shift = S``.
* non-periodic branch (data.py:15-17): torch_cluster ``radius_graph(pos, rc)`` [upstream]:
  float32 squared distance ``< rc*rc``, no self loops, at most ``max_num_neighbors=32`` neighbours
  per centre (first 32 by ascending neighbour index -- the CUDA implementation's choice),
  ``edge_index[0]`` = neighbour, ``edge_index[1]`` = centre.

Lists are compared as canonically sorted sets -- never by order (SURVEY.md 8c).
"""
from __future__ import annotations

import numpy as np


def _wrap_info(pos: np.ndarray, cell: np.ndarray):
    c64 = cell.astype(np.float64)
    frac = np.linalg.solve(c64.T, pos.astype(np.float64).T).T
    w = np.floor(frac).astype(np.int64)
    return c64, frac - w, w


def _image_range(c64: np.ndarray, rc: float) -> np.ndarray:
    vol = abs(np.linalg.det(c64))
    cross = np.stack([np.cross(c64[1], c64[2]), np.cross(c64[2], c64[0]), np.cross(c64[0], c64[1])])
    heights = vol / np.linalg.norm(cross, axis=1)
    return np.ceil(rc / heights).astype(int) + 1


def neighbor_list_pbc(pos: np.ndarray, cell: np.ndarray, rc: float, centres=None):
    """Return ``(i, j, S)`` (int64, int64, int64[.,3]) canonically sorted by (i, j, Sx, Sy, Sz)."""
    pos = np.ascontiguousarray(pos, dtype=np.float32)
    cell = np.ascontiguousarray(cell, dtype=np.float32).reshape(3, 3)
    n = pos.shape[0]
    c64, fw, w = _wrap_info(pos, cell)
    m = _image_range(c64, rc)
    cart_w = fw @ c64
    centres = np.arange(n) if centres is None else np.asarray(centres)
    # the exact test rounds pos_j - pos_i to fp32 (up to 2^-23 max|pos| per component): the screen must not be tighter
    margin = 1e-3 + 2.0 ** -21 * float(np.abs(pos).max(initial=0.0))
    out_i, out_j, out_s = [], [], []
    sig = np.array([(a, b, c) for a in range(-m[0], m[0] + 1) for b in range(-m[1], m[1] + 1)
                    for c in range(-m[2], m[2] + 1)], dtype=np.int64)
    chunk = max(1, int(2_000_000 // max(n, 1)))
    for s in sig:
        off = s.astype(np.float64) @ c64
        for a in range(0, len(centres), chunk):
            ci = centres[a:a + chunk]
            # cheap float64 screen in wrapped coordinates with a safety margin
            d = cart_w[None, :, :] + off[None, None, :] - cart_w[ci][:, None, :]
            cand = np.argwhere((d * d).sum(-1) < (rc + margin) ** 2)
            if cand.size == 0:
                continue
            ii = ci[cand[:, 0]]
            jj = cand[:, 1]
            S = s[None, :] - w[jj] + w[ii]
            # exact test in the ASE arithmetic on the ORIGINAL float32 positions
            dv = (pos[jj] - pos[ii]).astype(np.float64) + S.astype(np.float64) @ c64
            dist = np.sqrt(dv[:, 0] * dv[:, 0] + dv[:, 1] * dv[:, 1] + dv[:, 2] * dv[:, 2])
            keep = (dist < rc) & ~((ii == jj) & (S == 0).all(1))
            out_i.append(ii[keep]); out_j.append(jj[keep]); out_s.append(S[keep])
    if not out_i:
        z = np.zeros(0, dtype=np.int64)
        return z, z.copy(), np.zeros((0, 3), dtype=np.int64)
    i = np.concatenate(out_i); j = np.concatenate(out_j); S = np.concatenate(out_s)
    order = np.lexsort((S[:, 2], S[:, 1], S[:, 0], j, i))
    return i[order], j[order], S[order]


def neighbor_list_pbc_binned(pos: np.ndarray, cell: np.ndarray, rc: float):
    """Same contract and exact test as ``neighbor_list_pbc`` at the cost of a production CPU list (what ASE's binning
    achieves): candidates from a periodic k-d tree (scipy), then the ASE arithmetic on the original float32 positions.
    Orthorhombic cells with every edge > 2 (rc + 1e-3) only (then an atom pair has at most one image in range).  Used by the
    CPU-baseline leg of bench.py so that the reference arm is not charged for a brute-force list."""
    from scipy.spatial import cKDTree
    pos = np.ascontiguousarray(pos, dtype=np.float32)
    cell = np.ascontiguousarray(cell, dtype=np.float32).reshape(3, 3)
    c64 = cell.astype(np.float64)
    L = np.diag(c64)
    if np.abs(c64 - np.diag(L)).max() != 0.0 or (L <= 2 * (rc + 1e-3)).any():
        raise ValueError("neighbor_list_pbc_binned: orthorhombic cell with edges > 2 rc required")
    wrapped = np.mod(pos.astype(np.float64), L)
    wrapped[wrapped >= L] = 0.0
    tree = cKDTree(wrapped, boxsize=L)
    pairs = tree.query_pairs(rc + 1e-3, output_type="ndarray").astype(np.int64)
    ii = np.concatenate([pairs[:, 0], pairs[:, 1]])
    jj = np.concatenate([pairs[:, 1], pairs[:, 0]])
    d0 = (pos[jj] - pos[ii]).astype(np.float64)
    S = -np.round(d0 / L).astype(np.int64)
    dv = d0 + S.astype(np.float64) @ c64
    dist = np.sqrt(dv[:, 0] * dv[:, 0] + dv[:, 1] * dv[:, 1] + dv[:, 2] * dv[:, 2])
    keep = dist < rc
    i, j, S = ii[keep], jj[keep], S[keep]
    order = np.lexsort((S[:, 2], S[:, 1], S[:, 0], j, i))
    return i[order], j[order], S[order]


def radius_graph_nonpbc(pos: np.ndarray, rc: float, max_num_neighbors: int = 32, batch=None):
    """Return ``edge_index`` int64 ``[2,E]`` (row 0 = neighbour, row 1 = centre), sorted by (centre, neighbour)."""
    pos = np.ascontiguousarray(pos, dtype=np.float32)
    n = pos.shape[0]
    r2 = np.float32(rc) * np.float32(rc)
    src, dst = [], []
    for i in range(n):
        d = pos - pos[i]
        d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        ok = d2 < r2
        ok[i] = False
        if batch is not None:
            ok &= (batch == batch[i])
        nb = np.nonzero(ok)[0][:max_num_neighbors]
        src.append(nb); dst.append(np.full(nb.shape, i, dtype=np.int64))
    if not src:
        return np.zeros((2, 0), dtype=np.int64)
    return np.stack([np.concatenate(src), np.concatenate(dst)]).astype(np.int64)


def canonical_edges(edge_index, edge_shift=None) -> np.ndarray:
    """Canonical sorted array of rows ``(dst, src, Sx, Sy, Sz)`` used to compare edge SETS bit-exactly."""
    ei = np.asarray(edge_index).astype(np.int64)
    e = ei.shape[1]
    S = np.zeros((e, 3), dtype=np.int64) if edge_shift is None else np.rint(np.asarray(edge_shift)).astype(np.int64)
    rows = np.concatenate([ei[1][:, None], ei[0][:, None], S], axis=1)
    order = np.lexsort((rows[:, 4], rows[:, 3], rows[:, 2], rows[:, 1], rows[:, 0]))
    return rows[order]


def triplets_bruteforce(rowptr: np.ndarray, col: np.ndarray, src_type=None, type_a=None, type_c=None):
    """Canonical ordered triplet list over CSR edge ids (SURVEY.md A.3): all ``(e1, e2)`` with the same
    destination and ``e1 != e2``, sorted by ``(i, e1, e2)``; optional typed filter ``Z[j]==A, Z[k]==C``.
    Returns int64 ``[T,5]`` rows ``(j, i, k, e1, e2)``."""
    out = []
    n = len(rowptr) - 1
    for i in range(n):
        for e1 in range(rowptr[i], rowptr[i + 1]):
            if src_type is not None and type_a is not None and src_type[col[e1]] != type_a:
                continue
            for e2 in range(rowptr[i], rowptr[i + 1]):
                if e1 == e2:
                    continue
                if src_type is not None and type_c is not None and src_type[col[e2]] != type_c:
                    continue
                out.append((col[e1], i, col[e2], e1, e2))
    return np.asarray(out, dtype=np.int64).reshape(-1, 5)
