"""Quad-tile edge kernels (csrc/hn_edge_quad.cu, the default for F % 64 == 0) against the row-per-warp kernels of
csrc/hn_edge.cu on identical inputs, and both against a dense float64 evaluation of the reference formula
(rmnet.py:55-73 with the full K-term Gaussian sum of rmnet.py:168-193).  Covers HVNet / HPNet / HTNet row layouts,
F = 64 / 128 / 256, small K, rows that are not distance-sorted (graph re-used after the atoms moved, edges crossing the
cutoff) and rows longer than one tile sweep."""
import numpy as np
import pytest
import torch

from hermnet_b200 import ops
from tests.util import edge_inputs as _edge_inputs, frozen_model as _model, lattice_system as _system

pytestmark = pytest.mark.gpu

CASES = [
    ("HVNet", ["Li", "Al", "Si", "O"], [3, 13, 14, 8], 128, 128, 7),
    ("HVNet", ["H", "O"], [1, 8], 64, 20, 6),
    ("HVNet", ["Cr", "Fe", "Ni"], [24, 26, 28], 256, 128, 6),
    ("HPNet", ["Li", "O"], [3, 8], 64, 50, 6),
    ("HTNet", ["H", "O"], [1, 8], 128, 128, 6),
    ("HVNet", ["H", "O"], [1, 8, 6], 128, 32, 6),      # atoms of an element the model does not know: inactive rows
]


def _close(a, b, what, tol):
    scale = float(b.abs().max()) + 1e-12
    err = float((a - b).abs().max())
    assert err <= tol * scale, (what, err, scale)


def _run(variant, g, p, geom, xh, vec, Wt, bias, off, g_dx, g_dvec):
    ops.edge_set_variant(variant)
    try:
        dx, dv = ops.painn_edge_fwd(p, xh, vec, geom, g, Wt, bias, off)
        gg = ops.painn_edge_bwd_dst(p, xh, vec, geom, g, Wt, bias, off, g_dx, g_dvec).sum(0)
        gxh, gvec = ops.painn_edge_bwd_src(p, xh, vec, geom, g, Wt, bias, off, g_dx, g_dvec)
    finally:
        ops.edge_set_variant("auto")
    return dx, dv, gg, gxh, gvec


def _dense_reference(g, p, geom, xh, vec, Wt, bias, off, g_dx, g_dvec, filter_grads=False):
    """float64, all K basis functions, autograd for the three gradients (``filter_grads``: and for ``Wt`` / ``bias``,
    appended to the result)."""
    F = p.hidden
    dd = lambda t: t.detach().double()
    xh64, vec64, geom64 = dd(xh).requires_grad_(True), dd(vec).requires_grad_(True), dd(geom).requires_grad_(True)
    Wt64, bias64 = dd(Wt).requires_grad_(filter_grads), dd(bias).requires_grad_(filter_grads)
    row = g.edge_row.long()
    mod = g.row_mod.long()[row]
    live = mod >= 0
    m = mod.clamp(min=0)
    u = geom64[:, 3] * float(p.inv_rc)
    pe = p.env_p
    a, b, c = -(pe + 1) * (pe + 2) / 2, pe * (pe + 2), -pe * (pe + 1) / 2
    env = torch.where(u < 1, 1 + a * u ** pe + b * u ** (pe + 1) + c * u ** (pe + 2), torch.zeros_like(u))
    emb = env[:, None] * torch.exp(float(p.coeff) * (u[:, None] - dd(off)[None, :]) ** 2)
    phi = torch.einsum("ek,ekc->ec", emb, Wt64[m]) + bias64[m]
    P = xh64[g.row_xoff.long()[row] + g.col.long()]
    V = vec64[g.col.long()]
    A, B, C = torch.split(P * phi, F, dim=-1)
    mv = (V * (B / 3 ** 0.5)[:, None, :] + C[:, None, :] * geom64[:, :3, None]) / F ** 0.5
    w = live.double()[:, None]
    dx = torch.zeros((g.n_rows, F), dtype=torch.float64, device=xh.device).index_add_(0, row, A * w)
    dv = torch.zeros((g.n_rows, 3, F), dtype=torch.float64, device=xh.device).index_add_(0, row, mv * w[:, :, None])
    loss = (dx * dd(g_dx)).sum() + (dv * dd(g_dvec)).sum()
    if filter_grads:
        gxh, gvec, gg, gW, gb = torch.autograd.grad(loss, [xh64, vec64, geom64, Wt64, bias64])
        return dx.detach(), dv.detach(), gg, gxh, gvec, gW, gb
    gxh, gvec, gg = torch.autograd.grad(loss, [xh64, vec64, geom64])
    return dx.detach(), dv.detach(), gg, gxh, gvec


def _compare(model, g, pos, cell, dense=True, tol=2e-5):
    args = _edge_inputs(model, g, pos, cell)
    row = _run("row", g, *args)
    quad = _run("auto", g, *args)
    names = ("dx", "dvec", "g_geom", "grad_xh", "grad_vec")
    for n, a, b in zip(names, quad, row):
        _close(a, b.view_as(a), n + " quad vs row", tol)
    if dense:
        ref = _dense_reference(g, *args)
        for n, a, b, r in zip(names, quad, row, ref):
            _close(a.double(), r.view_as(a), n + " quad vs float64", tol)
            # the quad kernels keep the terms the 12-wide band drops: never (materially) worse than the row kernels
            eq = float((a.double() - r.view_as(a)).abs().max())
            er = float((b.view_as(a).double() - r.view_as(a)).abs().max())
            assert eq <= 2.0 * er + 1e-6 * float(r.abs().max()), (n, eq, er)


@pytest.mark.parametrize("kind,elems,zs,F,K,n_side", CASES)
def test_quad_kernels_match_row_kernels_and_float64(kind, elems, zs, F, K, n_side):
    dev = "cuda:0"
    pos, Z, cell = _system(n_side, zs, 5)
    pos, Z, cell = pos.to(dev), Z.to(dev), cell.to(dev)
    model = _model(kind, elems, F, K, dev)
    g = model.build_graph(pos, Z, cell)
    _compare(model, g, pos, cell)


def test_quad_kernels_on_unsorted_rows_and_edges_beyond_the_cutoff():
    """Graph built for one configuration, kernels run after the atoms moved: rows are no longer distance-sorted (tiles get
    cut where the union of bands would exceed the table) and some edges lie beyond rc (filter = bias)."""
    dev = "cuda:0"
    pos, Z, cell = _system(8, [3, 13, 14, 8], 31)
    pos, Z, cell = pos.to(dev), Z.to(dev), cell.to(dev)
    model = _model("HVNet", ["Li", "Al", "Si", "O"], 128, 128, dev)
    g = model.build_graph(pos, Z, cell)
    gen = torch.Generator().manual_seed(1)
    moved = pos + (torch.rand(pos.shape, generator=gen).to(dev) - 0.5) * 1.6
    d_new = ops.edge_geom_fwd(moved[g.perm].contiguous(), cell, g)[:, 3]
    assert int((d_new >= 5.0).sum()) > 100
    _compare(model, g, moved, cell)


def test_quad_kernels_long_rows_dense_system():
    """rc = 5 on a compressed lattice: ~150 edges per row, many tiles per row."""
    dev = "cuda:0"
    rng = np.random.default_rng(3)
    n_side, a = 8, 1.45
    grid = np.stack(np.meshgrid(*[np.arange(n_side)] * 3, indexing="ij"), -1).reshape(-1, 3)
    pos = torch.from_numpy((grid * a + rng.normal(0, 0.05, grid.shape)).astype(np.float32)).to(dev)
    Z = torch.from_numpy(rng.choice(np.array([1, 8]), size=len(grid))).long().to(dev)
    cell = torch.from_numpy((np.eye(3) * n_side * a).astype(np.float32)[None]).to(dev)
    model = _model("HVNet", ["H", "O"], 128, 128, dev)
    g = model.build_graph(pos, Z, cell)
    assert g.n_edges / g.n_atoms > 120
    _compare(model, g, pos, cell)


@pytest.mark.parametrize("variant", ["auto", "row"])
@pytest.mark.parametrize("F,K", [(128, 128), (64, 20), (256, 128)])
def test_null_vec_equals_zero_vec(variant, F, K):
    """vec = NULL (first layer: vec == 0, hermnet.py:124) must give exactly what a zero tensor gives."""
    dev = "cuda:0"
    pos, Z, cell = _system(6, [1, 8], 9)
    pos, Z, cell = pos.to(dev), Z.to(dev), cell.to(dev)
    model = _model("HVNet", ["H", "O"], F, K, dev)
    g = model.build_graph(pos, Z, cell)
    p, geom, xh, vec, Wt, bias, off, g_dx, g_dvec = _edge_inputs(model, g, pos, cell)
    zero = torch.zeros_like(vec)
    ops.edge_set_variant(variant)
    try:
        dx0, dv0 = ops.painn_edge_fwd(p, xh, zero, geom, g, Wt, bias, off)
        dx1, dv1 = ops.painn_edge_fwd(p, xh, None, geom, g, Wt, bias, off)
        gg0 = ops.painn_edge_bwd_dst(p, xh, zero, geom, g, Wt, bias, off, g_dx, g_dvec).sum(0)
        gg1 = ops.painn_edge_bwd_dst(p, xh, None, geom, g, Wt, bias, off, g_dx, g_dvec).sum(0)
    finally:
        ops.edge_set_variant("auto")
    _close(dx1, dx0, "dx", 1e-6)
    _close(dv1, dv0, "dvec", 1e-6)
    _close(gg1, gg0, "g_geom", 1e-6)


@pytest.mark.parametrize("F,K,exponent", [(64, 200, 3), (128, 256, 7), (128, 12, 5)])
def test_other_envelope_exponents_and_basis_sizes(F, K, exponent):
    """Polynomial envelope with p != 5 (rmnet.py:183-193 is generic in p), K > 128 and K at the band width."""
    import hermnet_b200 as H
    dev = "cuda:0"
    pos, Z, cell = _system(6, [1, 8], 11)
    pos, Z, cell = pos.to(dev), Z.to(dev), cell.to(dev)
    torch.manual_seed(5)
    model = H.HVNet(elems=["H", "O"], rc=5.0, num_layers=2, hidden_channels=F, num_rbf=K,
                    envelope={"name": "polynomial", "exponent": exponent}).to(dev).eval()
    for p in model.parameters():
        p.requires_grad_(False)
    g = model.build_graph(pos, Z, cell)
    _compare(model, g, pos, cell)


@pytest.mark.parametrize("name", ["triclinic_multi_image", "cluster_nonpbc_capped", "batch3_mixed"])
@pytest.mark.parametrize("F", [64, 128])
def test_sweep_kernels_on_the_golden_geometries(name, F):
    """The golden systems' geometries (5-atom triclinic cell with rc > L/2: several images of the same pair, self edges;
    a capped non-periodic cluster; a mixed batch) through the sweep kernels, against the row kernels and float64."""
    from tests import util
    case = util.load_case(name)
    dev = "cuda:0"
    elems = case["cfg"]["elems"]
    model = _model("HVNet", elems, F, 24, dev)
    pos, Z = case["pos"].to(dev), case["Z"].to(dev)
    cell = None if case["cell"] is None else case["cell"].to(dev)
    batch = case["batch"].to(dev)
    g = model.builder.from_positions(pos, Z, cell, batch)
    _compare(model, g, pos, cell)
