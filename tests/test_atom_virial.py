"""Per-atom energies and virials from the force pass: ``hn_edge_virial_atom`` (``ops.edge_virial_atom``),
``_HermNet.energy_forces_virial``, the calculator's ``energies`` / ``stresses`` and the virial trace of the device MD loop.

Kernel level: a float64 ``index_add`` over both endpoints of every edge, from the same fp32 geometry and gradient.
Model level: a float64 oracle whose edge vectors are kept as autograd leaves (``with_edge`` wrapped below), and the per-graph
virial of the existing cell-gradient route.  The CPU cases run over the kernel emulator with an ``index_add`` emulation of
``ops.edge_virial_atom``."""
import numpy as np
import pytest
import torch

import hermnet_b200 as H
from hermnet_b200 import ops, synthetic
from oracle import hermnet_oracle as O
from tests import util
from tests.util import frozen_model, lattice_system

DEV = "cuda:0"


def _grad_D64(geom, g_geom):
    """``edge_grad_D`` of csrc/hn_geom.cu in float64 (the clamped branch is decided on the fp32 distance)."""
    g, t = geom.double(), g_geom.double()
    u, d = g[:, :3], g[:, 3:4]
    dot = (t[:, :3] * u).sum(1, keepdim=True)
    return torch.where(geom[:, 3:4] == 1.0e-6, t[:, :3] / d, t[:, 3:4] * u + (t[:, :3] - dot * u) / d)


def _ends(g):
    return g.col.long(), torch.div(g.edge_row.long(), g.rows_per_atom, rounding_mode="floor")


def _ref_virial(geom, g_geom, g):
    """float64 per-atom virial ``[N,9]`` and its per-atom bound scale ``sum_{e at i} |D_e| |gD_e|``."""
    gD = _grad_D64(geom, g_geom)
    D = geom[:, :3].double() * geom[:, 3:4].double()
    w = -0.5 * (D[:, :, None] * gD[:, None, :]).reshape(-1, 9)
    s, r = _ends(g)
    ref = torch.zeros((g.n_atoms, 9), dtype=torch.float64, device=geom.device).index_add_(0, r, w).index_add_(0, s, w)
    m = D.norm(dim=1) * gD.norm(dim=1)
    scale = torch.zeros(g.n_atoms, dtype=torch.float64, device=geom.device).index_add_(0, r, m).index_add_(0, s, m)
    return ref, scale


def _emu_edge_virial_atom(geom, g_geom, g):
    """CPU stand-in of ``ops.edge_virial_atom`` (same contract, torch ``index_add``)."""
    ref, _ = _ref_virial(geom, g_geom, g)
    return ref.to(geom.dtype)


@pytest.fixture
def emu_virial(emu, monkeypatch):
    monkeypatch.setattr(ops, "edge_virial_atom", _emu_edge_virial_atom)
    return emu


# ---------------------------------------------------------------------------------------------------------------------
# kernel level (GPU)
# ---------------------------------------------------------------------------------------------------------------------
KCASES = [
    pytest.param("HVNet", 4, True, False, id="HVNet-R1-periodic"),
    pytest.param("HPNet", 4, True, False, id="HPNet-R2-periodic"),
    pytest.param("HTNet", 4, True, False, id="HTNet-R3-periodic"),
    pytest.param("HVNet", 2, True, False, id="HVNet-self-images"),
    pytest.param("HTNet", 2, True, False, id="HTNet-self-images"),
    pytest.param("HVNet", 4, False, True, id="HVNet-cluster-isolated-atoms"),
    pytest.param("HPNet", 4, False, True, id="HPNet-cluster-isolated-atoms"),
    pytest.param("HVNet", 20, True, False, id="HVNet-8000-atoms"),
]


def _kernel_case(kind, n_side, periodic, isolated, seed=3):
    pos, Z, cell = lattice_system(n_side, [3, 8], seed)
    if isolated:                                  # atoms with no neighbour at all
        far = torch.tensor([[60.0, 60.0, 60.0], [-60.0, 0.0, 0.0]])
        pos, Z = torch.cat([pos, far]), torch.cat([Z, torch.tensor([3, 8])])
    pos, Z = pos.to(DEV), Z.to(DEV)
    cell = cell.to(DEV) if periodic else None
    model = frozen_model(kind, ["Li", "O"], 32, 16, DEV)
    g = model.build_graph(pos, Z, cell)
    geom = ops.edge_geom_fwd(pos[g.perm].contiguous(), cell, g)
    gen = torch.Generator().manual_seed(seed)
    g_geom = torch.randn((g.n_edges, 4), generator=gen).to(DEV)
    E = g.n_edges
    if E >= 40:
        idx = torch.randperm(E, generator=gen)[:E // 10].to(DEV)
        g_geom[idx[: len(idx) // 2]] = 0.0        # dead Verlet-skin entries / unused edges
        k = idx[len(idx) // 2:]                   # clamped edges: |D| <= 1e-6, d = 1e-6, u = D * 1e6
        v = torch.randn((k.numel(), 3), generator=gen).to(DEV)
        geom[k, :3] = 0.5 * v / v.norm(dim=1, keepdim=True)
        geom[k, 3] = 1.0e-6
    return g, geom.contiguous(), g_geom.contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n_side,periodic,isolated", KCASES)
def test_edge_virial_atom_matches_float64_and_is_deterministic(kind, n_side, periodic, isolated):
    g, geom, g_geom = _kernel_case(kind, n_side, periodic, isolated)
    assert (g.rows_per_atom == 1) == (kind == "HVNet")
    if n_side == 2:
        s, r = _ends(g)
        assert bool((s == r).any())               # periodic self-images
    if n_side == 20:
        assert g.n_atoms == 8000 and g.n_edges > 250_000
    W = ops.edge_virial_atom(geom, g_geom, g)
    ref, scale = _ref_virial(geom, g_geom, g)
    err = (W.double() - ref).abs().max(dim=1).values
    assert bool((err <= 1e-6 * scale).all()), float((err / scale.clamp(min=1e-30)).max())
    if isolated:
        s, r = _ends(g)
        lone = torch.ones(g.n_atoms, dtype=torch.bool, device=DEV)
        lone[s] = False
        lone[r] = False
        assert int(lone.sum()) >= 2 and float(W[lone].abs().max()) == 0.0
    assert torch.equal(W, ops.edge_virial_atom(geom, g_geom, g))
    # summed over the atoms: W = -sum_e D_e (x) gD_e
    D = geom[:, :3].double() * geom[:, 3:4].double()
    tot = -(D[:, :, None] * _grad_D64(geom, g_geom)[:, None, :]).sum(0).reshape(9)
    assert float((W.double().sum(0) - tot).abs().max()) <= 1e-6 * float(scale.sum())


@pytest.mark.gpu
def test_edge_virial_atom_without_edges_writes_zeros():
    pos, Z, cell = lattice_system(3, [3, 8], 4, a=6.0, jitter=0.0)
    model = H.HVNet(elems=["Li", "O"], rc=3.0, num_layers=1, hidden_channels=32, num_rbf=16).to(DEV)
    g = model.build_graph(pos.to(DEV), Z.to(DEV), cell.to(DEV))
    assert g.n_edges == 0
    empty = torch.zeros((0, 4), device=DEV)
    W = ops.edge_virial_atom(empty, empty, g)
    assert W.shape == (27, 9) and float(W.abs().max()) == 0.0


# ---------------------------------------------------------------------------------------------------------------------
# model level: float64 oracle
# ---------------------------------------------------------------------------------------------------------------------
def _oracle(case, monkeypatch, intensive=False, pbc_shift="reference"):
    """float64 oracle: ``energy [G]``, per-atom ``energies [N]`` and ``virials [N,3,3]`` (same 1/2 + 1/2 split)."""
    kind, cfg = case["kind"], dict(case["cfg"], intensive=intensive)
    sd = {k: (v.double() if v.is_floating_point() else v) for k, v in O.make_state_dict(kind, cfg, case["seed"]).items()}
    keep = {}
    orig = O.with_edge

    def with_edge(pos, edge_index, cell, edge_shift, batch, pbc_shift="reference"):
        # the oracle's own edge vectors, made autograd leaves; the norm / clamp / unit vector are the oracle's
        src, dst = edge_index[0], edge_index[1]
        D = pos[src] - pos[dst]
        if cell is not None and edge_shift is not None:
            sgn = 1.0 if pbc_shift == "reference" else -1.0
            D = D + sgn * torch.einsum("ni,nij->nj", edge_shift.to(pos.dtype), cell[batch[src]])
        keep["D"] = D = D.detach().requires_grad_(True)
        E = D.size(0)
        return orig(torch.cat([D, torch.zeros_like(D)]), torch.stack([torch.arange(E), torch.arange(E, 2 * E)]),
                    None, None, None, pbc_shift)

    monkeypatch.setattr(O, "with_edge", with_edge)
    cell = None if case["cell"] is None else case["cell"].double()
    e, x, _ = O.FORWARDS[kind](sd, cfg, case["pos"].double(), case["Z"], case["edge_index"], cell, case["edge_shift"],
                               case["batch"], pbc_shift=pbc_shift, return_features=True)
    monkeypatch.setattr(O, "with_edge", orig)
    (gD,) = torch.autograd.grad(e.sum(), keep["D"], allow_unused=True)
    D = keep["D"].detach()
    gD = torch.zeros_like(D) if gD is None else gD
    w = -0.5 * D[:, :, None] * gD[:, None, :]
    N = case["pos"].size(0)
    src, dst = case["edge_index"][0], case["edge_index"][1]
    W = torch.zeros((N, 3, 3), dtype=torch.float64).index_add_(0, src, w).index_add_(0, dst, w)
    e_atom = O._lin(O.scaled_silu(O._lin(x.detach(), sd, "out_energy.0")), sd, "out_energy.2").squeeze(1)
    if intensive:
        e_atom = e_atom / torch.bincount(case["batch"]).double()[case["batch"]]
    return e.detach(), e_atom, W


def _check_against_oracle(out, ref, batch):
    e_ref, ea_ref, W_ref = ref
    ea, W = out["energies"].cpu().double(), out["virials"].cpu().double()
    G = e_ref.numel()
    sums = torch.zeros(G, dtype=torch.float64).index_add_(0, batch, ea)
    assert util.rel_err(sums, e_ref) < 1e-5
    assert util.rel_err(out["energy"].cpu().double(), e_ref) < 1e-5
    assert float((ea - ea_ref).abs().max()) < 1e-4 * max(1.0, float(ea_ref.abs().max()))
    assert float((W - W_ref).abs().max()) < 1e-4 * max(1.0, float(W_ref.abs().max()))
    Wg = torch.zeros((G, 3, 3), dtype=torch.float64).index_add_(0, batch, W_ref)
    assert float((out["virial"].cpu().double() - Wg).abs().max()) < 1e-4 * max(1.0, float(Wg.abs().max()))


OCASES = [pytest.param(n, "reference", False, id=n) for n in util.ALL_CASES] + [
    pytest.param("triclinic_multi_image", "physical", False, id="triclinic_multi_image-physical"),
    pytest.param("water24_htnet", "physical", False, id="water24_htnet-physical"),
    pytest.param("batch3_mixed", "reference", True, id="batch3_mixed-intensive"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,pbc_shift,intensive", OCASES)
def test_energies_and_virials_match_float64_oracle(name, pbc_shift, intensive, monkeypatch):
    case = util.load_case(name)
    model, _ = util.make_model(case["kind"], case["cfg"], case["seed"], DEV, pbc_shift=pbc_shift, intensive=intensive)
    out = model.energy_forces_virial(util.make_data(case, DEV, requires_grad=False))
    assert set(out) == {"energy", "forces", "energies", "virials", "virial"}
    assert out["virials"].shape == (case["pos"].size(0), 3, 3) and out["virial"].shape == (int(case["batch"].max()) + 1, 3, 3)
    _check_against_oracle(out, _oracle(case, monkeypatch, intensive, pbc_shift), case["batch"])


# ---------------------------------------------------------------------------------------------------------------------
# model level: the existing route, bitwise identity, every path
# ---------------------------------------------------------------------------------------------------------------------
def _existing_route(model, data):
    """``energy``, ``forces`` and the per-graph ``sum_i pos_i (x) F_i - cell^T dE/dcell`` with its condition scale."""
    pos = data.pos.detach().clone().requires_grad_(True)
    d = H.Data(pos=pos, atomic_number=data.atomic_number, batch=data.get("batch"))
    cell = data.get("cell")
    for k in ("edge_index", "edge_shift", "graph"):
        if data.get(k) is not None:
            d[k] = data.get(k)
    wrt = [pos]
    if cell is not None:
        d.cell = cell.detach().clone().requires_grad_(True)
        wrt.append(d.cell)
    e = model(d)
    grads = torch.autograd.grad(e.sum(), wrt)
    F = -grads[0]
    batch = torch.zeros(pos.size(0), dtype=torch.long, device=pos.device) if d.get("batch") is None else d.batch.long()
    G = e.numel()
    p = pos.detach()
    W = torch.zeros((G, 3, 3), dtype=torch.float64, device=p.device).index_add_(
        0, batch, (p[:, :, None] * F[:, None, :]).double())
    scale = torch.zeros(G, dtype=torch.float64, device=p.device).index_add_(0, batch, (p.norm(dim=1) * F.norm(dim=1)).double())
    if cell is not None and model._cell_of(d) is not None:
        c, gc = d.cell.detach().reshape(-1, 3, 3).double(), grads[1].reshape(-1, 3, 3).double()
        W = W - c.transpose(1, 2) @ gc
        scale = scale + (c.abs() * gc.abs()).sum((1, 2))
    return e.detach(), F, W, scale


def _system(n=4, seed=9, periodic=True):
    pos, Z, cell = synthetic.water_box(n, seed=seed)
    pos, Z, cell = torch.from_numpy(pos).to(DEV), torch.from_numpy(Z).to(DEV), torch.from_numpy(cell)[None].to(DEV)
    return H.Data(pos=pos, atomic_number=Z, cell=cell) if periodic else H.Data(pos=pos, atomic_number=Z)


MCASES = [
    pytest.param(128, True, "reference", True, id="F128-tensor-core"),
    pytest.param(128, False, "physical", True, id="F128-no-layer0-basis-physical"),
    pytest.param(64, True, "reference", True, id="F64-tile-sweep"),
    pytest.param(256, False, "reference", True, id="F256-tile-sweep-no-layer0-basis"),
    pytest.param(96, True, "physical", True, id="F96-row"),
    pytest.param(128, True, "reference", False, id="F128-non-periodic"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("F,layer0_basis,pbc_shift,periodic", MCASES)
def test_virial_equals_cell_gradient_route_and_forces_are_bitwise(F, layer0_basis, pbc_shift, periodic):
    torch.manual_seed(11)
    model = H.HVNet(elems=["H", "O"], rc=4.5, num_layers=2, hidden_channels=F, num_rbf=64, pbc_shift=pbc_shift).to(DEV).eval()
    model.layer0_basis = layer0_basis
    for q in model.parameters():
        q.requires_grad_(False)
    data = _system(periodic=periodic)
    out = model.energy_forces_virial(data)
    e, f, W, scale = _existing_route(model, data)
    assert torch.equal(out["energy"], e) and torch.equal(out["forces"], f)
    assert bool(((out["virial"].double() - W).abs().amax((1, 2)) <= 1e-5 * scale).all())
    assert torch.allclose(out["virials"].sum(0), out["virial"][0], rtol=0, atol=1e-5 * float(scale.max()))
    assert util.rel_err(out["energies"].double().sum(), e.double()) < 1e-5
    again = model.energy_forces_virial(data)
    assert all(torch.equal(again[k], out[k]) for k in out)


@pytest.mark.gpu
def test_batch_of_graphs_checkpointing_and_intensive():
    torch.manual_seed(3)
    model = H.HPNet(elems=["H", "O"], rc=4.0, num_layers=2, hidden_channels=64, num_rbf=32, intensive=True).to(DEV).eval()
    for q in model.parameters():
        q.requires_grad_(False)
    parts = [synthetic.water_box(n, seed=s) for n, s in ((3, 1), (4, 2), (3, 5))]
    pos = torch.from_numpy(np.concatenate([p for p, _, _ in parts])).to(DEV)
    Z = torch.from_numpy(np.concatenate([z for _, z, _ in parts])).to(DEV)
    cell = torch.from_numpy(np.stack([c for _, _, c in parts])).to(DEV)
    batch = torch.cat([torch.full((len(p),), i) for i, (p, _, _) in enumerate(parts)]).to(DEV)
    outs = []
    for ckpt in (False, True):
        model.checkpoint_layers = ckpt
        data = H.Data(pos=pos, atomic_number=Z, cell=cell, batch=batch)
        out = model.energy_forces_virial(data)
        e, f, W, scale = _existing_route(model, data)
        assert torch.equal(out["energy"], e) and torch.equal(out["forces"], f)
        assert out["virial"].shape == (3, 3, 3)
        assert bool(((out["virial"].double() - W).abs().amax((1, 2)) <= 1e-5 * scale).all())
        sums = torch.zeros(3, dtype=torch.float64, device=DEV).index_add_(0, batch, out["energies"].double())
        assert util.rel_err(sums, e.double()) < 1e-5
        outs.append(out)
    for k in outs[0]:
        assert torch.allclose(outs[0][k], outs[1][k], rtol=0, atol=1e-5 * max(1.0, float(outs[0][k].abs().max()))), k


@pytest.mark.gpu
@pytest.mark.parametrize("F", [128, 64])
def test_fused_equals_composite(F):
    torch.manual_seed(5)
    model = H.HTNet(elems=["H", "O"], rc=4.0, num_layers=2, hidden_channels=F, num_rbf=32).to(DEV).eval()
    for q in model.parameters():
        q.requires_grad_(False)
    res = {}
    for path in ("fused", "composite"):
        model.edge_path = path
        res[path] = model.energy_forces_virial(_system(3, seed=2))
    for k in ("energies", "forces", "virials"):
        ref = res["composite"][k]
        assert float((res["fused"][k] - ref).abs().max()) < 1e-4 * max(1.0, float(ref.abs().max())), k


@pytest.mark.gpu
@pytest.mark.parametrize("F", [128, 256])
def test_verlet_skin_list_equals_fresh_list(F):
    torch.manual_seed(11)
    model = H.HVNet(elems=["H", "O"], rc=4.5, num_layers=2, hidden_channels=F, num_rbf=128).to(DEV).eval()
    for q in model.parameters():
        q.requires_grad_(False)
    data = _system(5)
    g_skin = model.build_graph(data.pos, data.atomic_number, data.cell, skin=0.8)
    assert g_skin.masked
    gen = torch.Generator().manual_seed(1)
    pos2 = data.pos + (0.38 * (2 * torch.rand(data.pos.shape, generator=gen) - 1) / 3 ** 0.5).to(DEV)
    outs = []
    for graph in (g_skin, None):
        d = H.Data(pos=pos2, atomic_number=data.atomic_number, cell=data.cell)
        if graph is not None:
            d.graph = graph
        outs.append(model.energy_forces_virial(d))
    for k in ("energies", "forces", "virials", "virial"):
        ref = outs[1][k]
        assert float((outs[0][k] - ref).abs().max()) < 3e-5 * max(1.0, float(ref.abs().max())), k


@pytest.mark.gpu
@pytest.mark.parametrize("edge_path", ["fused", "composite"])
def test_system_without_edges(edge_path):
    pos, Z, cell = lattice_system(3, [3, 8], 4, a=6.0, jitter=0.0)
    torch.manual_seed(1)
    model = H.HVNet(elems=["Li", "O"], rc=3.0, num_layers=2, hidden_channels=128, num_rbf=16).to(DEV).eval()
    for q in model.parameters():
        q.requires_grad_(False)
    model.edge_path = edge_path
    d = H.Data(pos=pos.to(DEV), atomic_number=Z.to(DEV), cell=cell.to(DEV))
    out = model.energy_forces_virial(d)
    assert d.graph.n_edges == 0
    for k in ("forces", "virials", "virial"):
        assert float(out[k].abs().max()) == 0.0, k
    assert torch.equal(out["energy"], model(d).detach())
    assert util.rel_err(out["energies"].sum(), out["energy"]) < 1e-6


# ---------------------------------------------------------------------------------------------------------------------
# calculator and device MD (GPU)
# ---------------------------------------------------------------------------------------------------------------------
def _check_calculator(device, Z, pos, cell, make_model):
    from hermnet_b200.plugin import md
    from hermnet_b200.plugin.calculator import NNCalculator
    res = {}
    for route, ensemble in (("per_atom", "NVT"), ("npt", "NPT")):
        calc = NNCalculator(make_model(), None, trn_mean=-3.25, device_=device, ensemble=ensemble)
        atoms = md.SimpleAtoms(Z, pos, cell)
        atoms.calc = calc
        if route == "per_atom":
            energies = calc.get_potential_energies(atoms)
            assert set(calc.results) == {"energy", "free_energy", "forces", "energies", "stresses", "stress"}
            stresses = calc.get_stresses(atoms)
            assert energies.shape == (len(Z),) and stresses.shape == (len(Z), 6)
            assert abs(float(energies.sum()) - calc.results["energy"]) < 1e-5 * max(1.0, abs(calc.results["energy"]))
            assert np.array_equal(stresses.sum(0), calc.results["stress"])
        else:
            calc.get_stress(atoms)
            assert set(calc.results) == {"energy", "free_energy", "forces", "stress"}
        res[route] = dict(calc.results)
    a, b = res["per_atom"], res["npt"]
    assert np.array_equal(a["forces"], b["forces"]) and a["energy"] == b["energy"]
    # bound of the model-level comparison, sum_i |pos_i| |F_i| standing in for the cell term of the same size
    scale = 1.6021765e6 * float((np.linalg.norm(pos, axis=1) * np.linalg.norm(a["forces"], axis=1)).sum())
    assert float(np.abs(a["stress"] - b["stress"]).max()) < 2e-5 * scale


@pytest.mark.gpu
def test_calculator_energies_and_stresses_on_gpu():
    pos, Z, cell = synthetic.water_box(4, seed=4)

    def make():
        torch.manual_seed(3)
        return H.HVNet(elems=["H", "O"], rc=4.5, num_layers=2, hidden_channels=128, num_rbf=64)
    _check_calculator(DEV, Z, pos, cell, make)


@pytest.mark.gpu
def test_device_md_virial_trace_eager_and_graphed():
    from hermnet_b200.plugin import md
    pos, Z, cell = synthetic.water_box(4, seed=9)
    torch.manual_seed(11)
    model = H.HVNet(elems=["H", "O"], rc=4.5, num_layers=2, hidden_channels=128, num_rbf=64).to(DEV).eval()
    for q in model.parameters():
        q.requires_grad_(False)
    v0 = 0.003 * torch.randn(pos.shape, generator=torch.Generator().manual_seed(2)).numpy()
    runs = {}
    for cg in (False, True):
        st = {}
        p, _, e = md.velocity_verlet_device(model, Z, pos, cell, v0, steps=4, device=DEV, skin=0.8, stats=st, cuda_graph=cg,
                                            virial=True)
        assert st["virial"].shape == (4, 3, 3) and st["virial"].is_cuda
        runs[cg] = (p, e, st["virial"])
    W0, W1 = runs[False][2], runs[True][2]
    assert float((W1 - W0).abs().max()) < 1e-5 * max(1.0, float(W0.abs().max()))
    # the default call keeps its trajectory
    p_plain, _, e_plain = md.velocity_verlet_device(model, Z, pos, cell, v0, steps=4, device=DEV, skin=0.8)
    assert torch.equal(p_plain, runs[False][0]) and torch.equal(e_plain, runs[False][1])
    # each step: the virial of energy_forces_virial at that step's positions
    c = torch.from_numpy(cell).reshape(1, 3, 3).to(DEV)
    for k in range(1, 4):
        st = {}
        p, _, _ = md.velocity_verlet_device(model, Z, pos, cell, v0, steps=k, device=DEV, stats=st, virial=True)
        ref = model.energy_forces_virial(H.Data(pos=p, atomic_number=torch.from_numpy(Z).to(DEV), cell=c))["virial"][0]
        assert torch.allclose(st["virial"][k - 1], ref, rtol=0, atol=1e-6 * max(1.0, float(ref.abs().max())))
        assert float((W0[k - 1] - ref).abs().max()) < 1e-4 * max(1.0, float(ref.abs().max()))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: host logic over the kernel emulator
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["c1_hvnet", "triclinic_multi_image", "water24_htnet"])
def test_emulated_energies_and_virials_match_float64_oracle(emu_virial, name, monkeypatch):
    case = util.load_case(name)
    model, _ = util.make_model(case["kind"], case["cfg"], case["seed"], "cpu")
    out = model.energy_forces_virial(util.make_data(case, "cpu", requires_grad=False))
    _check_against_oracle(out, _oracle(case, monkeypatch), case["batch"])


def test_emulated_calculator_energies_and_stresses(emu_virial):
    pos, Z, cell = lattice_system(3, [3, 8], 21)

    def make():
        torch.manual_seed(5)
        return H.HVNet(elems=["Li", "O"], rc=4.0, num_layers=2, hidden_channels=64, num_rbf=16)
    _check_calculator("cpu", Z.numpy(), pos.numpy(), cell[0].numpy(), make)


def test_emulated_system_without_edges(emu_virial):
    pos, Z, cell = lattice_system(3, [3, 8], 4, a=6.0, jitter=0.0)
    torch.manual_seed(1)
    model = H.HVNet(elems=["Li", "O"], rc=3.0, num_layers=2, hidden_channels=64, num_rbf=16).eval()
    out = model.energy_forces_virial(H.Data(pos=pos, atomic_number=Z, cell=cell))
    for k in ("forces", "virials", "virial"):
        assert float(out[k].abs().max()) == 0.0, k
    assert out["energies"].shape == (27,) and util.rel_err(out["energies"].sum(), out["energy"]) < 1e-6
