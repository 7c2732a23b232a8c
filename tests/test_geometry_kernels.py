"""Neighbour search (csrc/hn_graph.cu) and edge geometry (csrc/hn_geom.cu) against brute-force float64 references, at the
cells and positions the barostat, the cell relaxation and long unwrapped trajectories produce: general shears, left-handed
and thin cells, bin widths at rc, atoms far outside the cell or on a face, pairs within one fp32 step of the cutoff,
batches, source-element groups and capped non-periodic rows.  ``-m gpu``.

Bars: neighbour lists are bit-exact SETS against ``oracle.neighbor_oracle`` (ASE arithmetic on the original fp32
positions); geometry within a few fp32 ulps of its condition-aware scale (sum of absolute values)."""
import numpy as np
import pytest
import torch

import hermnet_b200 as H
from hermnet_b200 import ops
from hermnet_b200.graph import GraphBuilder
from oracle import hermnet_oracle as O
from oracle import neighbor_oracle as NO
from tests import util

pytestmark = pytest.mark.gpu
DEV = "cuda"
EPS32 = 2.0 ** -23
f32 = np.float32


# ---- helpers ---------------------------------------------------------------------------------------------------------
def _t(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a)).to(DEV, dtype).contiguous()


def _device_list(pos, cell, gptr, rc, group=None, n_groups=1, cap=0):
    """``ops.radius_graph`` as canonical rows ``(row, j, Sx, Sy, Sz)`` plus the raw ``(rowptr, col, shift)``."""
    raw = ops.radius_graph(_t(pos), None if cell is None else _t(np.reshape(cell, (-1, 3, 3))), _t(gptr, torch.int32),
                           rc, None if group is None else _t(group, torch.int32), n_groups, cap)
    rowptr, col, shift = (x.cpu().numpy().astype(np.int64) for x in raw)
    row = np.repeat(np.arange(len(rowptr) - 1), np.diff(rowptr))
    return NO.canonical_edges(np.stack([col, row]), shift[:, :3]), raw


def _oracle_pbc(pos, cell, gptr, rc):
    cell = np.reshape(cell, (-1, 3, 3))
    rows = []
    for g in range(len(gptr) - 1):
        a0, a1 = gptr[g], gptr[g + 1]
        if a1 > a0:
            i, j, S = NO.neighbor_list_pbc(pos[a0:a1], cell[g], rc)
            rows.append(NO.canonical_edges(np.stack([j + a0, i + a0]), S))
    rows = np.concatenate(rows) if rows else np.zeros((0, 5), np.int64)
    return rows[np.lexsort((rows[:, 4], rows[:, 3], rows[:, 2], rows[:, 1], rows[:, 0]))]


def _check_pbc(pos, cell, rc, min_edges=1):
    pos = np.asarray(pos, f32)
    gptr = np.array([0, len(pos)])
    got, _ = _device_list(pos, cell, gptr, rc)
    ref = _oracle_pbc(pos, cell, gptr, rc)
    assert len(ref) >= min_edges
    assert np.array_equal(got, ref), (len(got), len(ref))
    return got


def _random_in_cell(cell, n, rng, lo=0.0, hi=1.0):
    return (rng.uniform(lo, hi, (n, 3)) @ np.asarray(cell, np.float64)).astype(f32)


def _ase_d(pi, pj, S, cell):
    """The oracle's exact test: float32(pos_j - pos_i) promoted, plus S.cell in float64."""
    dv = (pj - pi).astype(np.float64) + np.asarray(S, np.float64) @ np.asarray(cell, f32).astype(np.float64)
    return np.sqrt(dv[0] * dv[0] + dv[1] * dv[1] + dv[2] * dv[2])


def _straddle(pi, pj, S, cell, rc, ax):
    """fp32 copies of ``pj`` one step apart along axis ``ax`` around the cutoff of the pair ``(pi, pj, S)``: the two
    outermost the oracle keeps (rc - 1, rc - 0) and the two innermost it drops (rc + 0, rc + 1)."""
    D = (pj - pi).astype(np.float64) + np.asarray(S, np.float64) @ np.asarray(cell, f32).astype(np.float64)
    out_dir, in_dir = (f32(np.inf), f32(-np.inf)) if D[ax] > 0 else (f32(-np.inf), f32(np.inf))

    def step(p, d):
        q = p.copy()
        q[ax] = np.nextafter(q[ax], d)
        return q

    p = np.asarray(pj, f32).copy()
    for _ in range(100000):
        if _ase_d(pi, p, S, cell) < rc:
            break
        p = step(p, in_dir)
    for _ in range(100000):
        if _ase_d(pi, p, S, cell) >= rc:
            break
        p = step(p, out_dir)
    out0 = p
    in0 = step(out0, in_dir)
    in1, out1 = step(in0, in_dir), step(out0, out_dir)
    assert _ase_d(pi, in1, S, cell) < rc and _ase_d(pi, in0, S, cell) < rc
    assert _ase_d(pi, out0, S, cell) >= rc and _ase_d(pi, out1, S, cell) >= rc
    return np.stack([in1, in0, out0, out1])


def _shear(a, b, c, t, left=False):
    """Triclinic cell with rows a x, t0 a x + b y, t1 a x + t2 b y + c z (left: last row mirrored, det < 0)."""
    cell = np.array([[a, 0, 0], [t[0] * a, b, 0], [t[1] * a, t[2] * b, c]], np.float64)
    if left:
        cell[2, 2] = -cell[2, 2]
    return cell.astype(f32)


def _heights(cell):
    c = np.asarray(cell, np.float64)
    vol = abs(np.linalg.det(c))
    return vol / np.linalg.norm(np.stack([np.cross(c[1], c[2]), np.cross(c[2], c[0]), np.cross(c[0], c[1])]), axis=1)


# ---- 1. cell shapes ----------------------------------------------------------------------------------------------
CELLS = {
    "tilt+0.9": _shear(11.0, 12.0, 13.0, (0.9, 0.7, 0.8)),
    "tilt-0.9": _shear(11.0, 12.0, 13.0, (-0.9, -0.6, 0.85)),
    "tilt-mixed": _shear(14.0, 10.5, 12.5, (0.45, -0.9, -0.3)),
    "left-handed": _shear(11.0, 12.0, 13.0, (0.3, -0.5, 0.2), left=True),
    "left-handed-swap": _shear(12.0, 11.0, 13.0, (0.0, 0.0, 0.0))[[1, 0, 2]],
    "thin-one": _shear(3.1, 12.0, 12.5, (0.0, 0.2, -0.1)),
    "thin-all": _shear(3.3, 2.9, 4.1, (0.2, -0.1, 0.3)),
    "needle": _shear(1.7, 11.0, 11.0, (0.0, 0.0, 0.0)),
}


@pytest.mark.parametrize("rc", [5.0, 4.7, 5.3, 5.0 + 0.5, 6.0])
@pytest.mark.parametrize("name", list(CELLS))
def test_cell_shapes_vs_oracle(name, rc):
    cell = CELLS[name]
    rng = np.random.default_rng([list(CELLS).index(name), int(rc * 10)])
    h = _heights(cell)
    n = int(np.clip(0.05 * np.prod(h), 6, 120))
    got = _check_pbc(_random_in_cell(cell, n, rng), cell, rc)
    if name.startswith("thin") or name == "needle":
        assert np.abs(got[:, 2:]).max() >= 2              # images beyond the first shell are in the list


@pytest.mark.parametrize("rc", [5.0, 4.7, 5.3])
@pytest.mark.parametrize("k", [1, 2, 3, 5])
@pytest.mark.parametrize("rel", [-3e-7, 0.0, 3e-7])
def test_heights_at_bin_boundaries(k, rel, rc):
    """Heights just below, at and just above k * rc * (1 + 1e-6): the bin count floor(h / rcs) changes there and the bin
    width is within a few 1e-6 A of the search radius."""
    L = f32(k * rc * (1 + 1e-6) * (1 + rel))
    cell = np.diag([L, f32(2.0 * rc + 0.7), L]).astype(f32)
    rng = np.random.default_rng([k, int(rel * 1e7) + 10, int(rc * 10)])
    _check_pbc(_random_in_cell(cell, 40, rng), cell, rc)


def test_vacuum_slab_bin_cap():
    """1 000 A of vacuum on z: the bin count hits the 2 N cap and the reduction loop of the set-up kernel."""
    cell = np.diag([14.0, 15.0, 1010.0]).astype(f32)
    rng = np.random.default_rng(5)
    pos = (rng.uniform(0, 1, (90, 3)) * [14.0, 15.0, 9.0] + [0, 0, 500.0]).astype(f32)
    _check_pbc(pos, cell, 5.0)


# ---- 2. positions: unwrapped, on a face, coincident ----------------------------------------------------------------
def _grid_cell():
    """Sheared cell and positions on a 2^-10 grid: pos + k.cell stays exact in fp32 for |k| <= 50, so the wrapped and the
    unwrapped configuration have bit-identical pair geometry."""
    cell = np.array([[12.5, 0.0, 0.0], [5.25, 11.75, 0.0], [-4.5, 3.125, 13.0]], f32)
    rng = np.random.default_rng(11)
    pos = np.round((rng.uniform(0.02, 0.98, (70, 3)) @ cell.astype(np.float64)) * 1024.0) / 1024.0
    pos = np.concatenate([pos, pos[:3]])                 # three coincident pairs
    return cell, pos.astype(f32), rng


@pytest.mark.parametrize("kmax", [1, 7, 50])
def test_unwrapped_positions_vs_oracle_and_wrapped(kmax):
    cell, pos, rng = _grid_cell()
    k = rng.integers(-kmax, kmax + 1, (len(pos), 3))
    pos_u = (pos.astype(np.float64) + k @ cell.astype(np.float64)).astype(f32)
    assert np.array_equal(pos_u.astype(np.float64), pos.astype(np.float64) + k @ cell.astype(np.float64))
    got_w = _check_pbc(pos, cell, 5.0)
    got_u = _check_pbc(pos_u, cell, 5.0)
    # row c, entry (j, S): pos_u_j - pos_u_c + S.cell = pos_j - pos_c + (S + k_j - k_c).cell
    fixed = got_u.copy()
    fixed[:, 2:] += k[got_u[:, 1]] - k[got_u[:, 0]]
    fixed = fixed[np.lexsort((fixed[:, 4], fixed[:, 3], fixed[:, 2], fixed[:, 1], fixed[:, 0]))]
    assert np.array_equal(fixed, got_w)
    coincident = (got_w[:, 0] >= 70) & (got_w[:, 1] == got_w[:, 0] - 70) & (np.abs(got_w[:, 2:]).sum(1) == 0)
    assert coincident.sum() == 3


def test_atoms_on_faces():
    """Fractional coordinates exactly 0, exactly 1 and 1 - ulp, on every axis, in an orthorhombic and a sheared cell
    (the floor and the clamp of the binning)."""
    L = f32(13.0)
    below = np.nextafter(L, f32(0))
    ortho = np.diag([L, L, L]).astype(f32)
    pts = []
    for v in (f32(0.0), below, L, f32(-0.0), np.nextafter(f32(0), f32(1))):
        for ax in range(3):
            p = np.full(3, 6.5, f32)
            p[ax] = v
            pts.append(p)
    pts += [np.zeros(3, f32), np.full(3, below, f32), np.full(3, L, f32)]
    rng = np.random.default_rng(2)
    pos = np.concatenate([np.stack(pts), _random_in_cell(ortho, 30, rng)])
    _check_pbc(pos, ortho, 5.0)
    cell, _, _ = _grid_cell()
    c = cell.astype(np.float64)
    faces = [c[1] * 0.5 + c[2] * 0.25, c[0] * 0.5 + c[2] * 0.5, c[0] * 0.25 + c[1] * 0.75, c[0] + c[1] * 0.5,
             c[0] + c[1] + c[2], np.zeros(3), c[2]]
    pos = np.concatenate([np.asarray(faces, f32), _random_in_cell(cell, 30, rng)])
    pos = np.concatenate([pos, np.nextafter(pos[:4], f32(-np.inf))])
    _check_pbc(pos, cell, 5.0)


# ---- 3. pairs within one fp32 step of the cutoff -------------------------------------------------------------------
def _straddle_system(cell, pi, pj_target, S, rc, ax, fill, seed):
    parts = _straddle(pi, pj_target, S, cell, rc, ax)
    rng = np.random.default_rng(seed)
    pos = np.concatenate([pi[None], parts, _random_in_cell(cell, fill, rng, 0.3, 0.7)]).astype(f32)
    got = _check_pbc(pos, cell, rc)
    mine = got[(got[:, 0] == 0) & (got[:, 1] >= 1) & (got[:, 1] <= 4) & (got[:, 2:] == S).all(1)]
    assert sorted(mine[:, 1].tolist()) == [1, 2]          # rc - 1 and rc - 0 kept, rc + 0 and rc + 1 dropped


@pytest.mark.parametrize("rc", [5.0, 4.7, 5.3])
def test_cutoff_pairs_inside_the_box(rc):
    cell = _shear(17.0, 18.0, 19.0, (0.3, -0.2, 0.1))
    pi = np.array([6.1, 7.3, 8.2], f32)
    u = np.array([0.48, -0.6, 0.64])
    _straddle_system(cell, pi, (pi + rc * u).astype(f32), np.zeros(3, np.int64), rc, 2, 10, 1)


@pytest.mark.parametrize("rc", [5.0, 4.7, 5.3])
def test_cutoff_pairs_across_a_face(rc):
    cell = _shear(15.0, 16.0, 17.0, (0.5, 0.3, -0.4))
    pi = np.array([0.7, 1.1, 0.9], f32)
    S = np.array([-1, 0, 0], np.int64)                  # partner just inside the opposite face, seen through -x
    u = np.array([-0.8, 0.36, 0.48])
    pj = pi.astype(np.float64) + rc * u - S @ cell.astype(np.float64)
    _straddle_system(cell, pi, pj.astype(f32), S, rc, 0, 10, 2)


@pytest.mark.parametrize("rc", [5.0, 4.7])
def test_cutoff_pairs_through_the_image_of_a_large_box(rc):
    """|pos_j - pos_i| >= 128 A: the fp32 difference the oracle takes is rounded to 2^-16."""
    cell = np.diag([136.0, 9.5, 9.5]).astype(f32)
    pi = np.array([1.3, 4.0, 4.0], f32)
    S = np.array([-1, 0, 0], np.int64)
    pj = pi.astype(np.float64) + np.array([-rc, 0.0, 0.0]) - S @ cell.astype(np.float64)
    _straddle_system(cell, pi, pj.astype(f32), S, rc, 0, 30, 3)


@pytest.mark.parametrize("rc", [5.0, 5.3])
def test_cutoff_pairs_of_unwrapped_atoms(rc):
    cell = _shear(15.0, 16.0, 17.0, (0.2, -0.3, 0.4))
    pi = np.array([3.2, 4.1, 5.3], f32)
    K = np.array([23, -17, 31], np.int64)
    S = -K
    u = np.array([0.6, 0.0, 0.8])
    pj = pi.astype(np.float64) + rc * u + K @ cell.astype(np.float64)
    _straddle_system(cell, pi, pj.astype(f32), S, rc, 2, 10, 4)


@pytest.mark.parametrize("rc", [5.0, 4.7])
@pytest.mark.parametrize("k", [3, 5])
def test_cutoff_pairs_at_heights_just_below_k_rc(k, rc):
    """Height k rc (1 - 4e-6): k bins would each be narrower than rc.  A pair just inside rc from the top of the first
    bin reaches the bottom of the third one, so only bins at least rc wide (k - 1 of them) keep it."""
    L = f32(k * rc * (1 - 4e-6))
    cell = np.diag([L, f32(11.0), f32(11.0)]).astype(f32)
    w = float(L) / k
    pi = np.array([w - 5e-6, 5.5, 5.5], f32)
    pj = np.array([float(pi[0]) + rc, 5.5, 5.5], f32)
    assert float(pj[0]) > 2 * w
    _straddle_system(cell, pi, pj, np.zeros(3, np.int64), rc, 0, 10, k)


def _band_pair(rc, nb):
    """A periodic box whose x bins are within 1e-5 A of rc (1 + 1e-6) wide, an atom just above the lower face of bin k,
    shifted by K cells, and a wrapped atom just below the upper face of bin k - 2: two bins apart and more than one bin
    width apart in exact arithmetic, yet the oracle's fp32 difference (|pos_j - pos_i| >= 128 A) puts them inside rc."""
    rcs = rc * (1 + 1e-6)
    L = f32(nb * rcs)
    while float(L) / nb < rcs:
        L = np.nextafter(L, f32(np.inf))
    Ld = float(L)
    w = Ld / nb
    assert int(np.floor(Ld / rcs)) == nb and w - rcs < 1e-5
    k = np.arange(nb)[:, None]
    K = np.arange(-50, 51)[None, :]
    face_i = k * w
    xi = (face_i + K * Ld).astype(f32)
    for _ in range(2):
        xi = np.where(xi.astype(np.float64) - K * Ld < face_i + 1e-9, np.nextafter(xi, f32(np.inf)), xi)
    face_j = (k - 1 + nb) * w
    xj = np.broadcast_to(face_j, xi.shape).astype(f32)
    xj = np.where(xj.astype(np.float64) > face_j - 1e-9, np.nextafter(xj, f32(-np.inf)), xj)
    S = K - 1
    d32 = np.abs((xj - xi).astype(np.float64) + S * Ld)
    dex = np.abs(xj.astype(np.float64) - xi.astype(np.float64) + S * Ld)
    hits = np.argwhere((d32 < rc) & (dex > w) & (np.abs(xj - xi) >= 128))
    assert len(hits) > 0
    a, b = hits[len(hits) // 2]
    return L, float(xi[a, b]), float(xj[a, b]), int(S[0, b]), w


@pytest.mark.parametrize("rc,nb", [(5.0, 27), (4.7, 29), (5.0 + 0.5, 26)])
def test_cutoff_band_two_bins_apart(rc, nb):
    """The band where the 1e-6 relative bin margin alone is too thin: bin width within 1e-5 A of rc (1 + 1e-6), the
    fp32 difference of the positions >= 128 A (rounding up to half of 2^-16 A, far more for unwrapped atoms), and the
    pair two bins apart.  On the B200, before the bins were widened by the fp32 bound of that difference
    (2^-22 max|pos| per graph, graph_setup_kernel), the device list missed these pairs; they are kept now."""
    L, xi, xj, S, w = _band_pair(rc, nb)
    cell = np.diag([L, f32(9.0), f32(9.0)]).astype(f32)
    pi = np.array([xi, 4.5, 4.5], f32)
    pj = np.array([xj, 4.5, 4.5], f32)
    Sv = np.array([S, 0, 0], np.int64)
    assert _ase_d(pi, pj, Sv, cell) < rc
    assert abs(float(pj[0]) - float(pi[0]) + S * float(L)) > w
    parts = _straddle(pi, pj, Sv, cell, rc, 0)
    rng = np.random.default_rng(nb)
    fill = _random_in_cell(cell, 24, rng)
    fill[:, 0] = rng.uniform(0.3, 0.7, 24) * float(L)
    pos = np.concatenate([pi[None], pj[None], parts, fill]).astype(f32)
    got = _check_pbc(pos, cell, rc)
    hit = (got[:, 0] == 0) & (got[:, 1] == 1) & (got[:, 2:] == Sv).all(1)
    assert hit.sum() == 1


# ---- 4. batches, groups, capped non-periodic rows -------------------------------------------------------------------
def _mixed_batch(rng):
    cells, pos = [], []
    specs = [("one", 4.0), ("one", 12.0), ("far", 30.0), ("tiny", 3.0), ("big", 22.0), ("one", 2.5), ("sheared", 9.0),
             ("far", 40.0), ("big", 18.0), ("tiny", 2.2), ("one", 7.0), ("sheared", 13.0), ("square", 11.0),
             ("big", 16.0), ("one", 5.0), ("tiny", 4.4), ("sheared", 6.0), ("far", 25.0), ("big", 20.0), ("one", 60.0)]
    for kind, a in specs:
        if kind == "sheared":
            c = _shear(a, a * 1.1, a * 0.9, tuple(rng.uniform(-0.9, 0.9, 3)), left=bool(rng.integers(2)))
        else:
            c = np.diag([a, a * 1.05, a * 0.95]).astype(f32)
        n = {"one": 1, "far": 2, "tiny": 3, "big": 150, "sheared": 25, "square": 4}[kind]
        p = _random_in_cell(c, n, rng)
        if kind == "far":
            p = np.array([[0.1, 0.1, 0.1], [a / 2, a / 2, a / 2]], f32)
        if kind == "square":
            p = np.array([[1.0, 1.0, 1.0], [1.0, 6.0, 1.0], [6.0, 1.0, 6.0], [6.0, 6.0, 1.0]], f32) * 0.9
        cells.append(c)
        pos.append(p)
    gptr = np.concatenate([[0], np.cumsum([len(p) for p in pos])])
    return np.concatenate(pos).astype(f32), np.stack(cells).astype(f32), gptr


@pytest.mark.parametrize("rc", [5.0, 5.5])
def test_mixed_batch_vs_oracle(rc):
    rng = np.random.default_rng(21)
    pos, cells, gptr = _mixed_batch(rng)
    got, _ = _device_list(pos, cells, gptr, rc)
    ref = _oracle_pbc(pos, cells, gptr, rc)
    assert np.array_equal(got, ref)
    centre_graph = np.searchsorted(gptr, ref[:, 0], side="right") - 1
    per_graph = np.bincount(centre_graph, minlength=len(gptr) - 1)
    assert (per_graph == 0).any() and (per_graph > 0).any()   # graphs without edges next to graphs with edges
    one = np.diff(gptr) == 1
    assert (per_graph[one] > 0).any()                          # one-atom graphs with self images


@pytest.mark.parametrize("n_groups", [2, 5, 16])
def test_groups_vs_oracle(n_groups):
    cell = _shear(13.0, 12.0, 14.0, (0.4, -0.3, 0.6))
    rng = np.random.default_rng(n_groups)
    pos = _random_in_cell(cell, 160, rng)
    group = rng.integers(0, n_groups, len(pos)).astype(np.int32)
    gptr = np.array([0, len(pos)])
    got, (rowptr, _, _) = _device_list(pos, cell, gptr, 5.0, group, n_groups)
    assert rowptr.numel() == len(pos) * n_groups + 1
    ref = _oracle_pbc(pos, cell, gptr, 5.0)
    ref[:, 0] = ref[:, 0] * n_groups + group[ref[:, 1]]
    ref = ref[np.lexsort((ref[:, 4], ref[:, 3], ref[:, 2], ref[:, 1], ref[:, 0]))]
    assert np.array_equal(got, ref)


def _open_batch(rng):
    blob = rng.uniform(0, 8.0, (90, 3))                             # dense: > 64 neighbours per centre
    plane = np.concatenate([rng.uniform(0, 12, (40, 2)), np.full((40, 1), 3.0)], 1)
    line = np.stack([np.linspace(0, 30, 50), np.full(50, 1.0), np.full(50, -2.0)], 1)
    single = np.array([[5.0, 5.0, 5.0]])
    parts = [blob, plane, single, line, blob[:7] + 100.0]
    gptr = np.concatenate([[0], np.cumsum([len(p) for p in parts])])
    return np.concatenate(parts).astype(f32), gptr


@pytest.mark.parametrize("cap", [1, 32, 64])
def test_open_boundary_capped_rows_vs_oracle(cap):
    rng = np.random.default_rng(cap)
    pos, gptr = _open_batch(rng)
    batch = np.repeat(np.arange(len(gptr) - 1), np.diff(gptr))
    got, (rowptr, _, _) = _device_list(pos, None, gptr, 5.0, cap=cap)
    ref = NO.canonical_edges(NO.radius_graph_nonpbc(pos, 5.0, cap, batch=batch))
    assert np.array_equal(got, ref)
    assert int((rowptr[1:] - rowptr[:-1]).max()) == cap           # the cap is reached


def test_list_is_deterministic():
    rng = np.random.default_rng(8)
    pos, cells, gptr = _mixed_batch(rng)
    a = ops.radius_graph(_t(pos), _t(cells), _t(gptr, torch.int32), 5.0)
    b = ops.radius_graph(_t(pos), _t(cells), _t(gptr, torch.int32), 5.0)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    cell = _shear(13.0, 12.0, 14.0, (0.4, -0.3, 0.6))
    p = _random_in_cell(cell, 200, rng)
    grp = rng.integers(0, 5, len(p)).astype(np.int32)
    args = (_t(p), _t(cell[None]), _t(np.array([0, len(p)]), torch.int32), 5.0, _t(grp, torch.int32), 5)
    a, b = ops.radius_graph(*args), ops.radius_graph(*args)
    assert all(torch.equal(x, y) for x, y in zip(a, b))


def test_neighbor_search_on_unwrapped_sheared_cell():
    """The public entry point (data.py contract) on the same inputs as the kernels above."""
    cell, pos, rng = _grid_cell()
    k = rng.integers(-20, 21, (len(pos), 3))
    pos_u = (pos.astype(np.float64) + k @ cell.astype(np.float64)).astype(f32)
    ei, es = H.neighbor_search(torch.from_numpy(pos_u).to(DEV), 5.0, torch.from_numpy(cell)[None].to(DEV))
    i, j, S = NO.neighbor_list_pbc(pos_u, cell, 5.0)
    assert np.array_equal(NO.canonical_edges(ei.cpu().numpy(), es.cpu().numpy()), NO.canonical_edges(np.stack([i, j]), S))


# ---- 6. edge geometry on those graphs ---------------------------------------------------------------------------------
def _geom_system(which):
    cell, pos, rng = _grid_cell()
    if which == "single":
        k = rng.integers(-6, 7, (len(pos), 3))
        k[70:] = k[:3]                                   # the coincident pairs stay coincident
        pos =(pos.astype(np.float64) + k @ cell.astype(np.float64)).astype(f32)
        return pos, cell[None], None
    parts, cells = [pos], [cell]
    for a, t in ((7.5, (0.8, -0.7, 0.5)), (3.4, (-0.3, 0.2, 0.1))):
        c = _shear(a, a * 1.1, a * 0.9, t, left=a < 5)
        p = _random_in_cell(c, 20, rng)
        parts.append(np.concatenate([p, p[:2]]))
        cells.append(c)
    batch = np.repeat(np.arange(3), [len(p) for p in parts])
    return np.concatenate(parts).astype(f32), np.stack(cells).astype(f32), batch


def _graph(kind, sign, which):
    pos, cell, batch = _geom_system(which)
    Z = np.where(np.arange(len(pos)) % 3 == 0, 8, 1)
    b = GraphBuilder(kind, ["H", "O"], 5.0, pbc_shift=sign)
    g = b.from_positions(_t(pos), torch.from_numpy(Z).to(DEV), _t(cell),
                         None if batch is None else torch.from_numpy(batch).to(DEV))
    pos_i = _t(pos)[g.perm].contiguous()
    return g, pos_i, _t(cell)


def _geom_reference(g, pos_i, cell):
    """float64 D = pos[src] - pos[dst] + sign S.cell, per-destination-atom copies of the cell (their gradient is cellw)."""
    P = pos_i.double().cpu().requires_grad_(True)
    C = cell.double().cpu()
    r = (g.edge_row.long() // g.rows_per_atom).cpu()
    s = g.col.long().cpu()
    S = g.shift[:, :3].double().cpu()
    CA = C[g.atom_graph.long().cpu()].clone().requires_grad_(True)
    D = P[s] - P[r] + g.sign * torch.einsum("ea,eab->eb", S, CA[r])
    scale = (P[s].abs() + P[r].abs() + torch.einsum("ea,eab->eb", S.abs(), C[g.atom_graph.long().cpu()][r].abs())).detach()
    return P, CA, D, r, s, S, scale


@pytest.mark.parametrize("which", ["single", "batch"])
@pytest.mark.parametrize("sign", ["reference", "physical"])
@pytest.mark.parametrize("kind", ["HVNet", "HPNet"])
def test_edge_geom_fwd_vs_fp64(kind, sign, which):
    g, pos_i, cell = _graph(kind, sign, which)
    geom = ops.edge_geom_fwd(pos_i, cell, g).double().cpu()
    _, _, D, _, _, _, scale = _geom_reference(g, pos_i, cell)
    D = D.detach()
    d = D.norm(dim=1)
    zero = d == 0
    assert int(zero.sum()) >= 2 and int((g.shift[:, :3] != 0).any(1).sum()) > 0
    assert torch.equal(geom[zero], torch.tensor([0.0, 0.0, 0.0, 1e-6], dtype=torch.float32).double().expand(int(zero.sum()), 4))
    live = ~zero
    sn = scale[live].norm(dim=1)
    assert ((geom[live, 3] - d[live]).abs() / sn).max().item() < 8 * EPS32
    u_err = (geom[live, :3] - D[live] / d[live, None]).abs().max(1).values
    assert (u_err * d[live] / sn).max().item() < 16 * EPS32


@pytest.mark.parametrize("n_parts", [1, 3])
@pytest.mark.parametrize("which", ["single", "batch"])
@pytest.mark.parametrize("sign", ["reference", "physical"])
@pytest.mark.parametrize("kind", ["HVNet", "HPNet"])
def test_edge_geom_bwd_vs_fp64_autograd(kind, sign, which, n_parts):
    g, pos_i, cell = _graph(kind, sign, which)
    geom = ops.edge_geom_fwd(pos_i, cell, g)
    gen = torch.Generator().manual_seed(n_parts * 31 + len(kind) + len(sign))
    gg = torch.randn(n_parts, g.n_edges, 4, generator=gen)
    grad_pos, cellw = ops.edge_geom_bwd(geom, gg.to(DEV).contiguous(), g, True)
    P, CA, D, r, s, S, scale = _geom_reference(g, pos_i, cell)
    clamped = D.detach().norm(dim=1) <= 1e-6
    dn = torch.where(clamped[:, None], torch.ones_like(D), D).norm(dim=1)   # no 0/0 in the unselected branch
    d_c = torch.where(clamped, torch.full_like(dn, 1e-6), dn)
    u = D / d_c[:, None]
    t = gg.double().sum(0)
    L = (t[:, :3] * u).sum() + (t[:, 3] * d_c).sum()
    ref_pos, ref_cw = torch.autograd.grad(L, (P, CA))
    # condition-aware scale: |dL/dD_e| terms, times the relative conditioning of the fp32 geometry of the edge
    ta = gg.double().abs().sum(0)
    dd = d_c.detach()
    a_e = (ta[:, 3] + 2 * ta[:, :3].sum(1) / dd) * (scale.norm(dim=1) / dd + 4)
    n = g.n_atoms
    bound_pos = torch.zeros(n, dtype=torch.float64).index_add_(0, r, a_e).index_add_(0, s, a_e)
    bound_cw = torch.zeros(n, dtype=torch.float64).index_add_(0, r, a_e * S.abs().max(1).values)
    err_pos = (grad_pos.double().cpu() - ref_pos).abs().max(1).values
    err_cw = (cellw.double().cpu().view(n, 3, 3) - ref_cw).abs().flatten(1).max(1).values
    assert (err_pos <= 16 * EPS32 * bound_pos + 1e-30).all(), (err_pos / bound_pos).max().item()
    assert (err_cw <= 16 * EPS32 * bound_cw + 1e-30).all(), (err_cw / bound_cw.clamp(min=1e-300)).max().item()
    assert float(ref_cw.abs().max()) > 0                      # image edges present: the cell partial is exercised
    grad_pos1, cellw1 = ops.edge_geom_bwd(geom, gg.sum(0, keepdim=True).to(DEV).contiguous(), g, True)
    if n_parts > 1:   # the part sum equals one call with the summed gradient, to fp32 rounding
        assert ((grad_pos1.double() - grad_pos.double()).abs().cpu().max(1).values <= 16 * EPS32 * bound_pos + 1e-30).all()


# ---- 7. end to end: unwrapped sheared cell ------------------------------------------------------------------------------
def test_hvnet_unwrapped_sheared_cell_matches_wrapped_and_fp64():
    cfg = dict(elems=["H", "O"], rc=5.0, num_layers=2, hidden_channels=32, num_rbf=32)
    model, _ = util.make_model("HVNet", cfg, 5, DEV, pbc_shift="physical")
    for p in model.parameters():
        p.requires_grad_(False)
    cell, pos, rng = _grid_cell()
    pos, n = pos[:70], 70
    Z = np.where(np.arange(n) % 3 == 0, 8, 1)
    k = rng.integers(-40, 41, (n, 3))
    pos_u = (pos.astype(np.float64) + k @ cell.astype(np.float64)).astype(f32)

    def run(p):
        d = H.Data(pos=torch.from_numpy(p).to(DEV).requires_grad_(True), atomic_number=torch.from_numpy(Z).to(DEV),
                   batch=torch.zeros(n, dtype=torch.long, device=DEV), cell=torch.from_numpy(cell)[None].to(DEV))
        e, f, _ = util.energy_forces(model, d)
        return e.double().cpu(), f.double().cpu()

    e_w, f_w = run(pos)
    e_u, f_u = run(pos_u)
    assert util.rel_err(e_u, e_w) <= 1e-5 and float((f_u - f_w).abs().max()) <= 1e-4
    i, j, S = NO.neighbor_list_pbc(pos, cell, 5.0)
    sd64 = O.make_state_dict("HVNet", cfg, 5, dtype=torch.float64)
    p64 = torch.from_numpy(pos).double().requires_grad_(True)
    e64 = O.FORWARDS["HVNet"](sd64, cfg, p64, torch.from_numpy(Z), torch.from_numpy(np.stack([j, i])),
                              torch.from_numpy(cell).double()[None], -torch.from_numpy(S).double(),
                              torch.zeros(n, dtype=torch.long), pbc_shift="physical")
    (g64,) = torch.autograd.grad(e64.sum(), p64)
    assert util.rel_err(e_w, e64.detach()) <= 1e-5 and float((f_w + g64).abs().max()) <= 1e-4
    assert util.rel_err(e_u, e64.detach()) <= 1e-5 and float((f_u + g64).abs().max()) <= 1e-4
