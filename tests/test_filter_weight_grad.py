"""Filter-weight gradient of the fused edge path (``hn_painn_edge_bwd_w``, csrc/hn_edge.cu: the gradient of
``rbf_proj.weight`` / ``rbf_proj.bias``, rmnet.py:45,55) against a float64 evaluation of the same sums over the full
K-term radial basis, at the production width (F = 128: one full 384-column slice), several column slices (3F > 384, the
last one partly filled; K so large that the shared-memory accumulator needs narrower slices), HPNet / HTNet row layouts,
inactive rows, edges beyond the cutoff, Verlet-skin live masks, the golden geometries and a mid-size graph with long fp32
chunk sums.  The kernel also runs for eval-mode models whose parameters still require grad: any force evaluation calls it,
so the model-level cases compare such a model's fused path with the composite formulation."""
import pytest
import torch

import hermnet_b200 as H
from hermnet_b200 import ops
from tests import util
from tests.test_sweep_kernels import _dense_reference
from tests.util import edge_inputs, frozen_model, lattice_system

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
REL = 1e-5          # of the condition number cond_W of dense_filter_grad (fp32 products, fp32 chunk sums)
BAND = 2e-8         # the kernel's 12-wide Gaussian band drops terms below exp(-18) = 1.5e-8 of |gphi| (env <= 1)


def dense_filter_grad(g, p, geom, xh, vec, offset, g_dx, g_dvec, live=None):
    """float64 ``(gW [M,K,3F], gb [M,3F], cond_W [M,K,3F], sum |gphi| [M,3F])``.  ``gphi [E,3F]`` = dL/dphi of the message
    formula (rmnet.py:61-67, the terms of ``_dense_reference``), zero for entries of inactive rows and for dead entries
    (``live == 0``); ``emb [E,K]`` = envelope x all K Gaussians; one matmul per module.

    ``u = d / rc`` is taken as the fp32 product the model computes (a Gaussian of width 1/(K-1) turns its half-ulp rounding
    into up to K * 6e-8 of relative change).  ``cond_W = |emb|^T . |gphi|`` with the envelope's terms summed in absolute
    value: near the cutoff the envelope 1 + a u^p + b u^(p+1) + c u^(p+2) is a cancelling sum, which fp32 evaluates to
    eps * (1 + |a| + |b| + |c|) absolute, not relative, accuracy."""
    F, K, M = p.hidden, p.num_rbf, p.n_modules
    dd = lambda t: t.detach().double()
    row = g.edge_row.long()
    mod = g.row_mod.long()[row]
    act = mod >= 0
    if live is not None:
        act = act & live.bool()
    e = torch.nonzero(act).squeeze(1)
    row, mod, s = row[e], mod[e], g.col.long()[e]
    P = dd(xh)[g.row_xoff.long()[row] + s]
    gv = dd(g_dvec)[row]                                                   # [e,3,F]
    gm = dd(geom)[e]
    tb = (gv * dd(vec)[s]).sum(1) / (3 * F) ** 0.5
    tc = (gv * gm[:, :3, None]).sum(1) / F ** 0.5
    gphi = torch.cat([dd(g_dx)[row], tb, tc], 1) * P
    del P, gv, tb, tc
    u = (geom[e, 3] * torch.tensor(p.inv_rc, dtype=torch.float32)).double()
    pe = p.env_p
    a, b, c = -(pe + 1) * (pe + 2) / 2, pe * (pe + 2), -pe * (pe + 1) / 2
    inside = u < 1
    env = torch.where(inside, 1 + a * u ** pe + b * u ** (pe + 1) + c * u ** (pe + 2), torch.zeros_like(u))
    env_abs = torch.where(inside, 1 + abs(a) * u ** pe + b * u ** (pe + 1) + abs(c) * u ** (pe + 2), torch.zeros_like(u))
    gauss = torch.exp(float(p.coeff) * (u[:, None] - dd(offset)[None, :]) ** 2)
    emb, emb_abs = env[:, None] * gauss, env_abs[:, None] * gauss
    gW = torch.zeros((M, K, 3 * F), dtype=torch.float64, device=xh.device)
    cW = torch.zeros_like(gW)
    gb = torch.zeros((M, 3 * F), dtype=torch.float64, device=xh.device)
    cb = torch.zeros_like(gb)
    for m in range(M):
        sel = mod == m
        em, gm_ = emb[sel], gphi[sel]
        gW[m], cW[m] = em.t() @ gm_, emb_abs[sel].t() @ gm_.abs()
        gb[m], cb[m] = gm_.sum(0), gm_.abs().sum(0)
    return gW, gb, cW, cb


def _within(got, ref, bound, what):
    err = (got.double() - ref).abs()
    ratio = err / bound.clamp(min=1e-300)
    i = int(ratio.argmax())
    assert bool((err <= bound).all()), (what, float(err.flatten()[i]), float(bound.flatten()[i]), float(ratio.max()))


def _check(g, p, geom, xh, vec, off, g_dx, g_dvec, xcheck=None):
    """Kernel vs float64 under the condition-aware bound, bitwise-equal repeat; ``xcheck = (Wt, bias)``: also compare the
    float64 sums with autograd of ``_dense_reference`` (small cases: it materialises ``[E,K,3F]``).  With ``p.flags`` bit 0
    the mask ``p.live`` applies."""
    gW, gb = ops.painn_edge_bwd_w(p, xh, vec, geom, g, off, g_dx, g_dvec)
    gW2, gb2 = ops.painn_edge_bwd_w(p, xh, vec, geom, g, off, g_dx, g_dvec)
    assert torch.equal(gW, gW2) and torch.equal(gb, gb2), "fixed-order reduction: two calls must agree bitwise"
    live = p.live if p.flags & 1 else None
    rW, rb, cW, cb = dense_filter_grad(g, p, geom, xh, vec, off, g_dx, g_dvec, live)
    assert float(rW.abs().max()) > 0 and float(rb.abs().max()) > 0
    _within(gW, rW, REL * cW + BAND * cb[:, None, :], "gW")
    _within(gb, rb, REL * cb, "gb")
    if xcheck is not None:
        assert live is None
        *_, aW, ab = _dense_reference(g, p, geom, xh, vec, *xcheck, off, g_dx, g_dvec, filter_grads=True)
        # _dense_reference takes u in float64: the Gaussians differ by (x - k) * K * 6e-8 relative, x = u (K - 1)
        _within(rW, aW, 1e-4 * cW + BAND * cb[:, None, :], "float64 gW vs autograd")
        _within(rb, ab, 1e-10 * cb, "float64 gb vs autograd")


def _inputs(model, g, pos, cell):
    p, geom, xh, vec, Wt, bias, off, g_dx, g_dvec = edge_inputs(model, g, pos, cell)
    return (g, p, geom, xh, vec, off, g_dx, g_dvec), (Wt, bias)


CASES = [   # kind, elements, atomic numbers in the lattice, F, K, lattice side, cross-check with autograd
    ("HVNet", ["Li", "Al", "Si", "O"], [3, 13, 14, 8], 128, 128, 7, False),
    ("HVNet", ["H", "O"], [1, 8], 64, 20, 6, True),
    ("HVNet", ["H", "O"], [1, 8, 6], 32, 8, 6, True),               # Z = 6 is not a model element: inactive rows
    ("HVNet", ["H", "O"], [1, 8], 160, 50, 6, True),                # 3F = 480: two slices, the second 96 of 384 live
    ("HPNet", ["Li", "O"], [3, 8], 64, 50, 6, True),
    ("HTNet", ["H", "O"], [1, 8], 128, 128, 6, False),
    ("HVNet", ["Cr", "Fe", "Ni"], [24, 26, 28], 128, 200, 6, False),  # [200][384] fp32 > 227 KB: narrower slices
    ("HVNet", ["Cr", "Fe", "Ni"], [24, 26, 28], 256, 256, 6, False),  # four 224-column slices, the last 96 live
]


@pytest.mark.parametrize("kind,elems,zs,F,K,n_side,xcheck", CASES)
def test_filter_weight_grad_matches_float64(kind, elems, zs, F, K, n_side, xcheck):
    pos, Z, cell = (t.to(DEV) for t in lattice_system(n_side, zs, 5))
    model = frozen_model(kind, elems, F, K, DEV)
    g = model.build_graph(pos, Z, cell)
    args, filt = _inputs(model, g, pos, cell)
    _check(*args, xcheck=filt if xcheck else None)


@pytest.mark.parametrize("name", ["triclinic_multi_image", "cluster_nonpbc_capped", "batch3_mixed"])
def test_filter_weight_grad_on_the_golden_geometries(name):
    """5-atom triclinic cell with rc > L/2 (several images of one pair, self-image edges), a capped non-periodic cluster, a
    mixed batch: fewer rows than the 2 x SMs / M row chunks of a large graph, so one or two rows per chunk."""
    case = util.load_case(name)
    model = frozen_model("HVNet", case["cfg"]["elems"], 128, 24, DEV)
    pos, Z = case["pos"].to(DEV), case["Z"].to(DEV)
    cell = None if case["cell"] is None else case["cell"].to(DEV)
    g = model.builder.from_positions(pos, Z, cell, case["batch"].to(DEV))
    args, filt = _inputs(model, g, pos, cell)
    _check(*args, xcheck=filt)


def test_filter_weight_grad_with_edges_beyond_the_cutoff():
    """Graph built for one configuration, kernel run after the atoms moved by up to 0.8 A: entries at or beyond rc have no
    basis term and feed only the bias gradient."""
    pos, Z, cell = (t.to(DEV) for t in lattice_system(8, [3, 13, 14, 8], 31))
    model = frozen_model("HVNet", ["Li", "Al", "Si", "O"], 128, 128, DEV)
    g = model.build_graph(pos, Z, cell)
    gen = torch.Generator().manual_seed(1)
    moved = pos + (torch.rand(pos.shape, generator=gen).to(DEV) - 0.5) * 1.6
    args, _ = _inputs(model, g, moved, cell)
    assert int((args[2][:, 3] >= model.rc).sum()) > 100
    _check(*args)


def test_filter_weight_grad_with_a_live_mask():
    """Verlet-skin list (p.flags bit 0): entries with live == 0 feed neither gW nor gb; the mask is required with the flag
    and ignored without it."""
    pos, Z, cell = (t.to(DEV) for t in lattice_system(6, [3, 13, 14, 8], 5))
    model = frozen_model("HVNet", ["Li", "Al", "Si", "O"], 128, 128, DEV)
    g = model.build_graph(pos, Z, cell)
    args, _ = _inputs(model, g, pos, cell)
    g, p, geom, xh, vec, off, g_dx, g_dvec = args
    gen = torch.Generator().manual_seed(1)
    live = (torch.rand(g.n_edges, generator=gen) > 0.2).to(torch.uint8).to(DEV)
    run = lambda: ops.painn_edge_bwd_w(p, xh, vec, geom, g, off, g_dx, g_dvec)
    full = run()
    p.live = live
    plain = run()                                                       # flags == 0: the mask is ignored
    assert torch.equal(plain[0], full[0]) and torch.equal(plain[1], full[1])
    p.flags, p.live = 1, None
    with pytest.raises(RuntimeError, match="live mask"):
        run()
    p.live = live
    _check(*args)


def test_filter_weight_grad_mid_size():
    """20^3 lattice (8000 atoms, ~3.4e5 edges), F = 128, K = 128: row chunks of ~1000 edges per module summed in fp32."""
    pos, Z, cell = (t.to(DEV) for t in lattice_system(20, [3, 13, 14, 8], 17))
    model = frozen_model("HVNet", ["Li", "Al", "Si", "O"], 128, 128, DEV)
    g = model.build_graph(pos, Z, cell)
    assert g.n_edges > 250_000
    args, _ = _inputs(model, g, pos, cell)
    _check(*args)


@pytest.mark.parametrize("elems,zs,F,K", [(["Li", "Al", "Si", "O"], [3, 13, 14, 8], 128, 200),    # tensor-core forward
                                          (["Cr", "Fe", "Ni"], [24, 26, 28], 256, 160)])          # tile-sweep forward
def test_eval_mode_model_with_trainable_parameters(elems, zs, F, K):
    """model.eval() without freezing (validation loops, MD drivers): every backward runs the filter-weight kernel, even for
    forces alone.  Fused path == composite formulation for energies, forces and rbf_proj gradients."""
    pos, Z, cell = (t.to(DEV) for t in lattice_system(6, zs, 13))
    torch.manual_seed(7)
    model = H.HVNet(elems=elems, rc=5.0, num_layers=2, hidden_channels=F, num_rbf=K).to(DEV).eval()
    assert all(q.requires_grad for q in model.parameters())
    model.store_features = True
    out = {}
    for path in ("fused", "composite"):
        model.edge_path = path
        model.zero_grad()
        d = H.Data(pos=pos.clone().requires_grad_(True), atomic_number=Z, cell=cell.clone())
        e = model(d)
        (gp,) = torch.autograd.grad(e.sum(), [d.pos], retain_graph=True)       # forces alone: runs the kernel as well
        e.sum().backward()
        out[path] = (e.detach(), -gp, {k: q.grad.clone() for k, q in model.named_parameters() if "rbf_proj" in k})
    (ef, ff, wf), (ec, fc, wc) = out["fused"], out["composite"]
    # random weights: the readout e_atom = W2 . h + b2 cancels (|e_atom| ~ 0.05 from terms of ~1), so the energy bar is
    # relative to sum_atoms |W2| . |h|, the size of the terms whose fp32 rounding the two formulations do differently
    lin1, act, lin2 = model.out_energy
    with torch.no_grad():
        e_cond = float((act(lin1(d.x)).abs() @ lin2.weight.abs().t()).sum())
    assert float((ef - ec).abs().max()) < 1e-5 * e_cond
    assert float((ff - fc).abs().max()) < 1e-4 * max(1.0, float(fc.abs().max()))
    assert len(wc) == 4 * len(elems)
    for k, ref in wc.items():
        assert float((wf[k] - ref).abs().max()) < 2e-4 * (float(ref.abs().max()) + 1e-6) + 1e-6, k
