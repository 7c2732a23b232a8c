"""Verlet-skin superset lists (``build_graph(skin=...)``, ``md.VerletGraph``, ``NNCalculator(skin=...)``) on the row-per-warp
and tile-sweep edge kernels, i.e. at every hidden width other than the tensor-core one (F = 128).

A skin list is searched with ``rc + skin`` and re-used after the atoms moved; with ``p.flags`` bit 0 the entries ``p.live``
marks dead must contribute nothing (not even the filter bias), their ``g_geom`` rows are exact zeros, and they take no
gathers.  Kernel level: every output against a float64 dense evaluation with the mask as a factor on each entry, bitwise
checks of determinism, of the all-live mask against an unmasked call and (row kernels) of a masked list against the same
list with its dead entries removed.  Model level: energies / forces / cell gradients on a re-used list equal those of a
fresh list, and the MD drivers follow the rebuild-every-step trajectory."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import hermnet_b200 as H
from hermnet_b200 import functional as Fn
from hermnet_b200 import ops, synthetic
from tests import util
from tests.util import edge_inputs, frozen_model, lattice_system

DEV = "cuda:0"
NAMES = ("dx", "dvec", "g_geom", "grad_xh", "grad_vec")


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def _masked(p, live):
    q = ops.EdgeParams(p.n_atoms, p.n_rows, p.n_modules, p.hidden, p.num_rbf, p.env_p, p.inv_rc, p.coeff, p.variant, 1)
    q.live = live
    return q


def _unmasked(p):
    return ops.EdgeParams(p.n_atoms, p.n_rows, p.n_modules, p.hidden, p.num_rbf, p.env_p, p.inv_rc, p.coeff, p.variant, 0)


def _run(variant, g, p, geom, xh, vec, Wt, bias, off, g_dx, g_dvec):
    """(dx, dvec, g_geom planes [n_slices, E, 4], grad_xh, grad_vec) of the three ops on one kernel family."""
    ops.edge_set_variant(variant)
    try:
        dx, dv = ops.painn_edge_fwd(p, xh, vec, geom, g, Wt, bias, off)
        parts = ops.painn_edge_bwd_dst(p, xh, vec, geom, g, Wt, bias, off, g_dx, g_dvec)
        gxh, gvec = ops.painn_edge_bwd_src(p, xh, vec, geom, g, Wt, bias, off, g_dx, g_dvec)
    finally:
        ops.edge_set_variant("auto")
    torch.cuda.synchronize()
    return dx, dv, parts, gxh, gvec


def _dense_reference(g, p, geom, xh, vec, Wt, bias, off, g_dx, g_dvec, mask):
    """float64 over all K basis functions, each entry's contribution multiplied by ``mask`` (and by its row being active);
    autograd for the three gradients.  One matmul per module."""
    F = p.hidden
    dd = lambda t: t.detach().double()
    xh64, vec64, geom64 = dd(xh).requires_grad_(True), dd(vec).requires_grad_(True), dd(geom).requires_grad_(True)
    row = g.edge_row.long()
    mod = g.row_mod.long()[row]
    w = ((mod >= 0) & mask.bool()).double()[:, None]
    u = geom64[:, 3] * float(p.inv_rc)
    pe = p.env_p
    a, b, c = -(pe + 1) * (pe + 2) / 2, pe * (pe + 2), -pe * (pe + 1) / 2
    env = torch.where(u < 1, 1 + a * u ** pe + b * u ** (pe + 1) + c * u ** (pe + 2), torch.zeros_like(u))
    emb = env[:, None] * torch.exp(float(p.coeff) * (u[:, None] - dd(off)[None, :]) ** 2)
    phi = torch.zeros((geom.size(0), 3 * F), dtype=torch.float64, device=geom.device)
    for m in range(p.n_modules):
        sel = mod == m
        phi[sel] = emb[sel] @ dd(Wt[m]) + dd(bias[m])
    P = xh64[g.row_xoff.long()[row] + g.col.long()] if g.n_edges else xh64[:0]
    V = vec64[g.col.long()]
    A, B, C = torch.split(P * phi, F, dim=-1)
    mv = (V * (B / 3 ** 0.5)[:, None, :] + C[:, None, :] * geom64[:, :3, None]) / F ** 0.5
    dx = torch.zeros((g.n_rows, F), dtype=torch.float64, device=xh.device).index_add_(0, row, A * w)
    dv = torch.zeros((g.n_rows, 3, F), dtype=torch.float64, device=xh.device).index_add_(0, row, mv * w[:, :, None])
    loss = (dx * dd(g_dx)).sum() + (dv * dd(g_dvec)).sum()
    gxh, gvec, gg = torch.autograd.grad(loss, [xh64, vec64, geom64])
    return dx.detach(), dv.detach(), gg, gxh, gvec


def _close(a, b, what, tol=2e-5):
    scale = float(b.abs().max()) + 1e-12
    err = float((a.double() - b.double()).abs().max())
    assert err <= tol * scale, (what, err, scale)


def _bits(t):
    return t.contiguous().view(torch.int32)


def _skin_case(kind, elems, zs, F, K, n_side, seed=5):
    """A frozen model, a skin list (skin 0.8) built on a lattice, and random edge-kernel inputs after every atom moved by
    less than skin / 2: some superset entries are now beyond rc, the rows are no longer distance-sorted."""
    pos, Z, cell = lattice_system(n_side, zs, seed)
    pos, Z, cell = pos.to(DEV), Z.to(DEV), cell.to(DEV)
    model = frozen_model(kind, elems, F, K, DEV)
    g = model.build_graph(pos, Z, cell, skin=0.8)
    assert g.masked
    gen = torch.Generator().manual_seed(seed + 1)
    moved = pos + (0.38 * (2 * torch.rand(pos.shape, generator=gen) - 1) / 3 ** 0.5).to(DEV)
    args = edge_inputs(model, g, moved, cell)
    return model, g, moved, cell, args


def _mask(kind, model, g, moved, cell, geom):
    if kind == "physical":
        m = model._live_mask(moved[g.perm], cell, g, geom)
        assert 0 < int((m == 0).sum()) < g.n_edges
        return m
    gen = torch.Generator().manual_seed(17)
    return (torch.rand(g.n_edges, generator=gen) >= 0.2).to(torch.uint8).to(DEV)


def _compact(g, keep):
    """The row CSR / transposed view of ``g`` with the entries ``keep == 0`` removed and the order kept."""
    kb = keep.bool()
    dev = kb.device
    newid = torch.cumsum(kb.long(), 0) - 1
    n_rows, n_src = g.rowptr.numel() - 1, g.t_rowptr.numel() - 1
    per_row = torch.zeros(n_rows, dtype=torch.long, device=dev).index_add_(0, g.edge_row.long(), kb.long())
    t_eid = g.t_eid.long()
    t_src = torch.repeat_interleave(torch.arange(n_src, device=dev), (g.t_rowptr[1:] - g.t_rowptr[:-1]).long())
    t_keep = kb[t_eid]
    per_src = torch.zeros(n_src, dtype=torch.long, device=dev).index_add_(0, t_src[t_keep], torch.ones_like(t_src[t_keep]))
    ptr = lambda c: torch.cat([torch.zeros(1, dtype=torch.long, device=dev), torch.cumsum(c, 0)]).int().contiguous()
    return SimpleNamespace(rowptr=ptr(per_row), col=g.col[kb].contiguous(), edge_row=g.edge_row[kb].contiguous(), row_mod=g.row_mod,
                           row_xoff=g.row_xoff, t_rowptr=ptr(per_src), t_eid=newid[t_eid[t_keep]].int().contiguous(),
                           n_edges=int(kb.sum()))


# ---------------------------------------------------------------------------------------------------------------------
# kernel level (GPU)
# ---------------------------------------------------------------------------------------------------------------------
KCASES = [
    pytest.param("HVNet", ["Li", "Al", "Si", "O"], [3, 13, 14, 8], 256, 128, 6, id="HVNet-F256-K128"),
    pytest.param("HVNet", ["H", "O"], [1, 8], 64, 20, 6, id="HVNet-F64-K20"),
    pytest.param("HVNet", ["H", "O"], [1, 8], 96, 40, 6, id="HVNet-F96-K40"),
    pytest.param("HVNet", ["Cr", "Fe", "Ni"], [24, 26, 28], 512, 64, 5, id="HVNet-F512-K64"),
    pytest.param("HPNet", ["Li", "O"], [3, 8], 64, 50, 6, id="HPNet-F64-K50"),
    pytest.param("HTNet", ["H", "O"], [1, 8], 256, 128, 5, id="HTNet-F256-K128"),
    pytest.param("HVNet", ["H", "O"], [1, 8, 6], 64, 32, 6, id="HVNet-F64-inactive-rows"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("mask_kind", ["physical", "random"])
@pytest.mark.parametrize("variant", ["auto", "row"])
@pytest.mark.parametrize("kind,elems,zs,F,K,n_side", KCASES)
def test_masked_edge_kernels_match_float64(kind, elems, zs, F, K, n_side, variant, mask_kind):
    """dx, dvec, g_geom (summed over slices), grad_xh and grad_vec of a masked skin list against float64 with the mask as a
    factor; dead g_geom rows are bitwise zero in every slice plane; two calls agree bitwise."""
    if F == 96 and variant == "auto":
        pytest.skip("F = 96 has only the row kernels: covered by variant='row'")
    model, g, moved, cell, args = _skin_case(kind, elems, zs, F, K, n_side)
    p, geom, rest = args[0], args[1], args[2:]
    live = _mask(mask_kind, model, g, moved, cell, geom)
    q = _masked(p, live)
    out = _run(variant, g, q, geom, *rest)
    again = _run(variant, g, _masked(p, live), geom, *rest)
    for n, a, b in zip(NAMES, out, again):
        assert torch.equal(_bits(a), _bits(b)), n + ": two calls differ"
    dead = live == 0
    assert int(dead.sum()) > 0
    assert int(_bits(out[2][:, dead]).abs().sum()) == 0, "g_geom of dead entries is not exactly zero"
    ref = _dense_reference(g, p, geom, *rest, live)
    got = (out[0], out[1], out[2].sum(0), out[3], out[4])
    for n, a, r in zip(NAMES, got, ref):
        _close(a, r.view_as(a), f"{n} ({variant}, {mask_kind} mask) vs float64")


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["auto", "row"])
@pytest.mark.parametrize("F,K", [(64, 20), (96, 40), (256, 128), (512, 64)])
def test_all_live_mask_equals_unmasked_call_bitwise(F, K, variant):
    """flags bit 0 with every entry live runs the MASKED kernels on the same sums: bitwise the results of flags 0."""
    model, g, moved, cell, args = _skin_case("HVNet", ["H", "O"], [1, 8], F, K, 5)
    p, geom, rest = args[0], args[1], args[2:]
    ones = torch.ones(g.n_edges, dtype=torch.uint8, device=DEV)
    a = _run(variant, g, _masked(p, ones), geom, *rest)
    b = _run(variant, g, _unmasked(p), geom, *rest)
    for n, x, y in zip(NAMES, a, b):
        assert torch.equal(_bits(x), _bits(y)), n


@pytest.mark.gpu
@pytest.mark.parametrize("F,K", [(64, 20), (96, 40), (256, 128)])
@pytest.mark.parametrize("kind,elems,zs", [("HVNet", ["H", "O"], [1, 8]), ("HTNet", ["H", "O"], [1, 8])])
def test_row_kernels_masked_list_equals_compacted_list_bitwise(kind, elems, zs, F, K):
    """Row kernels: a masked superset list gives bitwise the results of the same CSR with the dead entries removed (order
    kept) -- dead entries are skipped, the per-row and per-source summation order is unchanged."""
    model, g, moved, cell, args = _skin_case(kind, elems, zs, F, K, 5)
    p, geom, rest = args[0], args[1], args[2:]
    live = _mask("random", model, g, moved, cell, geom)
    keep = live.bool()
    a = _run("row", g, _masked(p, live), geom, *rest)
    gc = _compact(g, live)
    b = _run("row", gc, _unmasked(p), geom[keep].contiguous(), *rest)
    assert torch.equal(_bits(a[0]), _bits(b[0])), "dx"
    assert torch.equal(_bits(a[1]), _bits(b[1])), "dvec"
    assert torch.equal(_bits(a[2][:, keep]), _bits(b[2])), "g_geom"
    assert torch.equal(_bits(a[3]), _bits(b[3])), "grad_xh"
    assert torch.equal(_bits(a[4]), _bits(b[4])), "grad_vec"


@pytest.mark.gpu
def test_three_families_agree_on_one_masked_list():
    """F = 128, K = 64: tensor-core, tile-sweep and row kernels on one masked superset list, through the autograd layer."""
    model, g, moved, cell, args = _skin_case("HVNet", ["Li", "Al", "Si", "O"], [3, 13, 14, 8], 128, 64, 6)
    p, geom, xh, vec, Wt, bias, off, g_dx, g_dvec = args
    live = _mask("physical", model, g, moved, cell, geom)
    outs = {}
    for fam in ("tc", "quad", "row"):
        ops.edge_set_variant(fam)
        try:
            xh_, vec_, geom_ = xh.clone().requires_grad_(True), vec.clone().requires_grad_(True), geom.clone().requires_grad_(True)
            dx, dv = Fn.painn_edge(xh_, vec_, geom_, Wt, bias, off, g, _masked(p, live))
            gxh, gvec, gg = torch.autograd.grad((dx * g_dx).sum() + (dv * g_dvec).sum(), [xh_, vec_, geom_])
        finally:
            ops.edge_set_variant("auto")
        outs[fam] = (dx.detach(), dv.detach(), gg, gxh, gvec)
    ref = _dense_reference(g, p, geom, xh, vec, Wt, bias, off, g_dx, g_dvec, live)
    for i, n in enumerate(NAMES):
        for fam in ("quad", "row"):
            _close(outs[fam][i], outs["tc"][i], f"{n}: {fam} vs tc")
        _close(outs["tc"][i], ref[i].view_as(outs["tc"][i]), f"{n}: tc vs float64")


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["auto", "row"])
def test_missing_or_malformed_live_mask_raises_on_gpu(variant):
    model, g, moved, cell, args = _skin_case("HVNet", ["H", "O"], [1, 8], 64, 20, 4)
    p, geom, xh, vec, Wt, bias, off, g_dx, g_dvec = args
    calls = [lambda q: ops.painn_edge_fwd(q, xh, vec, geom, g, Wt, bias, off),
             lambda q: ops.painn_edge_bwd_dst(q, xh, vec, geom, g, Wt, bias, off, g_dx, g_dvec),
             lambda q: ops.painn_edge_bwd_src(q, xh, vec, geom, g, Wt, bias, off, g_dx, g_dvec)]
    ops.edge_set_variant(variant)
    try:
        for live in (None, torch.ones(g.n_edges, dtype=torch.int32, device=DEV), torch.ones(3, dtype=torch.uint8, device=DEV)):
            for call in calls:
                with pytest.raises(TypeError, match="live must be uint8"):
                    call(_masked(p, live))
    finally:
        ops.edge_set_variant("auto")


# ---------------------------------------------------------------------------------------------------------------------
# model level (GPU)
# ---------------------------------------------------------------------------------------------------------------------
MCASES = [
    pytest.param("HVNet", 256, 128, "reference", True, False, id="HVNet-F256-K128"),
    pytest.param("HVNet", 512, 128, "reference", True, False, id="HVNet-F512-K128"),
    pytest.param("HVNet", 96, 32, "reference", True, False, id="HVNet-F96"),
    pytest.param("HVNet", 256, 64, "physical", False, False, id="HVNet-F256-no-layer0-basis-physical"),
    pytest.param("HPNet", 64, 50, "reference", True, False, id="HPNet-F64"),
    pytest.param("HTNet", 64, 64, "reference", True, False, id="HTNet-F64"),
    pytest.param("HVNet", 256, 128, "reference", True, True, id="HVNet-F256-K128-trainable"),
    pytest.param("HTNet", 64, 64, "reference", True, True, id="HTNet-F64-trainable"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,F,K,pbc_shift,layer0_basis,trainable", MCASES)
def test_verlet_skin_list_reuse_at_other_widths(kind, F, K, pbc_shift, layer0_basis, trainable):
    """A skin list re-used after the atoms moved (< skin / 2) gives the energies / forces / cell gradient of a fresh list;
    with trainable parameters (filter-weight backward running alongside) the rbf_proj gradients agree too."""
    pos, Z, cell = synthetic.water_box(5, seed=9)
    pos, Z, cell = torch.from_numpy(pos).to(DEV), torch.from_numpy(Z).to(DEV), torch.from_numpy(cell)[None].to(DEV)
    torch.manual_seed(11)
    model = getattr(H, kind)(elems=["H", "O"], rc=4.5, num_layers=2, hidden_channels=F, num_rbf=K, pbc_shift=pbc_shift).to(DEV).eval()
    model.layer0_basis = layer0_basis
    for q in model.parameters():
        q.requires_grad_(trainable)
    g_skin = model.build_graph(pos, Z, cell, skin=0.8)
    assert g_skin.masked and g_skin.n_edges > model.build_graph(pos, Z, cell).n_edges
    gen = torch.Generator().manual_seed(1)
    pos2 = pos + (0.38 * (2 * torch.rand(pos.shape, generator=gen) - 1) / 3 ** 0.5).to(DEV)
    out, wgrads = [], []
    for graph in (g_skin, None):
        d = H.Data(pos=pos2.clone().requires_grad_(True), atomic_number=Z, cell=cell.clone().requires_grad_(True))
        if graph is not None:
            d.graph = graph
        e = model(d)
        gp, gcell = torch.autograd.grad(e.sum(), [d.pos, d.cell], retain_graph=trainable)
        out.append((e.detach(), gp, gcell))
        if trainable:
            model.zero_grad()
            e.sum().backward()
            wgrads.append({k: q.grad.clone() for k, q in model.named_parameters() if "rbf_proj" in k})
    assert util.rel_err(out[0][0], out[1][0]) < 3e-6
    assert float((out[0][1] - out[1][1]).abs().max()) < 3e-5 * max(1.0, float(out[1][1].abs().max()))
    assert float((out[0][2] - out[1][2]).abs().max()) < 3e-4 * max(1.0, float(out[1][2].abs().max()))
    if trainable:
        assert len(wgrads[1]) >= 8
        for k, ref in wgrads[1].items():
            assert float((wgrads[0][k] - ref).abs().max()) < 3e-4 * float(ref.abs().max()), k


@pytest.mark.gpu
def test_device_md_reuses_the_list_at_f256_eager_and_graphed():
    """velocity_verlet_device at F = 256 (tile-sweep kernels): skin 0.8 re-uses one list for 8 steps and follows the
    rebuild-every-step trajectory; the same loop with the evaluation captured as a CUDA graph matches the eager loop."""
    from hermnet_b200.plugin import md
    pos, Z, cell = synthetic.water_box(5, seed=9)
    torch.manual_seed(11)
    model = H.HVNet(elems=["H", "O"], rc=4.5, num_layers=2, hidden_channels=256, num_rbf=128).to(DEV).eval()
    for q in model.parameters():
        q.requires_grad_(False)
    v0 = 0.003 * torch.randn(pos.shape, generator=torch.Generator().manual_seed(2)).numpy()
    runs = {}
    for skin, cg in ((0.0, False), (0.8, False), (0.8, True)):
        st = {}
        p1, _, e1 = md.velocity_verlet_device(model, Z, pos, cell, v0, steps=8, dt_fs=0.5, device=DEV, skin=skin, stats=st,
                                              cuda_graph=cg)
        runs[(skin, cg)] = (p1, e1, st)
    assert runs[(0.0, False)][2] == {"builds": 9, "reuses": 0}
    assert runs[(0.8, False)][2]["builds"] == 1 and runs[(0.8, False)][2]["reuses"] == 8
    assert float((runs[(0.0, False)][0] - runs[(0.8, False)][0]).abs().max()) < 1e-4
    assert util.rel_err(runs[(0.8, False)][1], runs[(0.0, False)][1]) < 1e-5
    assert runs[(0.8, True)][2] == runs[(0.8, False)][2]
    assert float((runs[(0.8, True)][0] - runs[(0.8, False)][0]).abs().max()) < 1e-5
    assert util.rel_err(runs[(0.8, True)][1], runs[(0.8, False)][1]) < 1e-6


@pytest.mark.gpu
def test_calculator_with_skin_on_the_reference_default_model():
    """NNCalculator(HVNet(hidden_channels=512, num_rbf=128), skin=0.5) driven by the host-side velocity Verlet loop: the
    re-used list gives the trajectory of a fresh list per call."""
    from hermnet_b200.plugin import NNCalculator, md
    pos, Z, cell = synthetic.water_box(4, seed=4)
    runs = {}
    for skin in (0.0, 0.5):
        torch.manual_seed(3)
        model = H.HVNet(elems=["H", "O"], hidden_channels=512, num_rbf=128)
        calc = NNCalculator(model, None, trn_mean=0.0, device_=DEV, skin=skin)
        atoms = md.SimpleAtoms(Z, pos, cell)
        atoms.calc = calc
        md.maxwell_boltzmann(atoms, 300.0, seed=5)
        energies = md.velocity_verlet(atoms, steps=6, dt_fs=0.5)
        runs[skin] = (atoms.positions.copy(), np.array(energies), calc.verlet.builds, calc.verlet.reuses)
    assert runs[0.5][2] == 1 and runs[0.5][3] >= 6
    assert float(np.abs(runs[0.5][0] - runs[0.0][0]).max()) < 1e-4
    assert float(np.abs(runs[0.5][1] - runs[0.0][1]).max()) < 1e-5 * max(1.0, float(np.abs(runs[0.0][1]).max()))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: host logic over the kernel emulator, and the ops-level mask check
# ---------------------------------------------------------------------------------------------------------------------
def _emu_masked(fn):
    """An emulated edge op with the Verlet-skin contract of ``ops``: with ``p.flags`` bit 0 it needs ``p.live`` and gives
    what the same op gives on the list with the dead entries removed (zero ``g_geom`` rows for them)."""
    def call(p, xh, vec, geom, g, *rest):
        if not p.flags & 1:
            return fn(p, xh, vec, geom, g, *rest)
        live = getattr(p, "live", None)
        if not isinstance(live, torch.Tensor) or live.dtype != torch.uint8 or live.numel() != geom.size(0):
            raise TypeError("hermnet_b200.painn_edge_*: live must be uint8 [E]")
        keep = live.bool()
        out = fn(p, xh, vec, geom[keep].contiguous(), _compact(g, live), *rest)
        if fn.__name__ != "painn_edge_bwd_dst":
            return out
        full = torch.zeros((out.size(0), geom.size(0), 4), dtype=out.dtype, device=out.device)
        full[:, keep] = out
        return full
    return call


@pytest.fixture
def emu_skin(emu, monkeypatch):
    """The CPU kernel emulator with the row / tile-sweep edge ops honouring Verlet-skin masks."""
    for name in ("painn_edge_fwd", "painn_edge_bwd_dst", "painn_edge_bwd_src"):
        monkeypatch.setattr(ops, name, _emu_masked(getattr(emu, name)))
    return emu


@pytest.mark.parametrize("F", [64, 96])
def test_verlet_skin_list_on_the_fused_path_without_tensor_cores(emu_skin, F):
    """edge_path = 'fused' at F != 128 (row / tile-sweep kernels): a re-used skin list gives the energies and forces of a
    fresh list."""
    pos, Z, cell = lattice_system(5, [3, 8], 21)
    torch.manual_seed(5)
    model = H.HVNet(elems=["Li", "O"], rc=4.0, num_layers=2, hidden_channels=F, num_rbf=32).eval()
    for q in model.parameters():
        q.requires_grad_(False)
    model.edge_path = "fused"
    g_skin = model.build_graph(pos, Z, cell, skin=0.6)
    assert g_skin.masked and g_skin.n_edges > model.build_graph(pos, Z, cell).n_edges
    gen = torch.Generator().manual_seed(1)
    pos2 = pos + 0.28 * (2 * torch.rand(pos.shape, generator=gen) - 1) / 3 ** 0.5
    out = []
    for graph in (g_skin, None):
        d = H.Data(pos=pos2.clone().requires_grad_(True), atomic_number=Z, cell=cell.clone().requires_grad_(True))
        if graph is not None:
            d.graph = graph
        e = model(d)
        gp, gcell = torch.autograd.grad(e.sum(), [d.pos, d.cell])
        out.append((e.detach(), gp, gcell))
    assert util.rel_err(out[0][0], out[1][0]) < 2e-6
    assert float((out[0][1] - out[1][1]).abs().max()) < 2e-5 * max(1.0, float(out[1][1].abs().max()))
    assert float((out[0][2] - out[1][2]).abs().max()) < 2e-4 * max(1.0, float(out[1][2].abs().max()))


@pytest.mark.parametrize("name", ["painn_edge_fwd", "painn_edge_bwd_dst", "painn_edge_bwd_src"])
def test_ops_without_live_mask_raise(name):
    """flags bit 0 without p.live (or with a mask of the wrong dtype / length) is refused before anything runs."""
    E = 10
    p = ops.EdgeParams(4, 4, 1, 64, 16, 5, 0.2, -10.0, 0, 1)
    geom = torch.ones((E, 4))
    t = torch.zeros(1)
    fn = getattr(ops, name)
    extra = [] if name == "painn_edge_fwd" else [t, t]
    for live in (None, torch.ones(E, dtype=torch.bool), torch.ones(E + 1, dtype=torch.uint8)):
        p.live = live
        with pytest.raises(TypeError, match="live must be uint8"):
            fn(p, t, t, geom, None, t, t, t, *extra)
