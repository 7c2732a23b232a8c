"""Host-side logic over the CPU kernel emulator (tests/emulator.py): graph layouts, autograd wiring, the model
classes, both formulations -- compared with the golden fixtures / the oracle.  No GPU needed."""
import numpy as np
import pytest
import torch

import hermnet_b200 as H
from oracle import hermnet_oracle as O
from tests import util

TOL_E, TOL_F = 1e-5, 1e-4      # BASELINE.json: fp32 energy 1e-5 relative, forces 1e-4 eV/A


@pytest.mark.parametrize("name", util.ALL_CASES)
@pytest.mark.parametrize("path", ["fused", "composite"])
@pytest.mark.parametrize("with_edges", [True, False])
def test_model_matches_golden(emu, name, path, with_edges):
    case = util.load_case(name)
    if name == "c1_hvnet" and path == "composite" and not with_edges:
        pytest.skip("covered by the other three combinations; keeps the CPU suite short")
    model, _ = util.make_model(case["kind"], case["cfg"], case["seed"])
    model.edge_path = path
    data = util.make_data(case, with_edges=with_edges)
    e, f, gc = util.energy_forces(model, data)
    assert util.rel_err(e, case["energy"]) < TOL_E
    assert float((f - case["forces"]).abs().max()) < TOL_F
    if case["cell_grad"] is not None:
        assert float((gc - case["cell_grad"]).abs().max()) < TOL_F * 10


@pytest.mark.parametrize("name", ["triclinic_multi_image", "batch3_mixed", "water24_hpnet", "water24_htnet"])
def test_parameter_gradients_fused_and_composite(emu, name):
    """dE/dtheta from the fused backward (incl. the filter-weight kernel formula) == composite == oracle."""
    case = util.load_case(name)
    grads = {}
    for path in ("fused", "composite"):
        model, sd = util.make_model(case["kind"], case["cfg"], case["seed"])
        model.edge_path = path
        e = model(util.make_data(case, requires_grad=False))
        e.sum().backward()
        grads[path] = {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}
    sd_o = {k: v.clone().requires_grad_(v.is_floating_point() and "offset" not in k) for k, v in sd.items()}
    eo = O.FORWARDS[case["kind"]](sd_o, case["cfg"], case["pos"], case["Z"], case["edge_index"], case["cell"],
                                  case["edge_shift"], case["batch"])
    eo.sum().backward()
    for k, go in ((k, v.grad) for k, v in sd_o.items() if v.requires_grad and v.grad is not None):
        scale = float(go.abs().max()) + 1e-6
        for path in grads:
            assert k in grads[path], (k, path)
            assert float((grads[path][k] - go).abs().max()) < 2e-4 * scale + 1e-6, (k, path)


@pytest.mark.parametrize("name", ["triclinic_multi_image", "water24_hpnet"])
def test_force_loss_double_backward(emu, name):
    """Training step of example/dist_train.py:89-99: loss on forces obtained with create_graph=True."""
    case = util.load_case(name)
    model, sd = util.make_model(case["kind"], case["cfg"], case["seed"])
    model.train()
    data = util.make_data(case)
    e = model(data)
    f = -torch.autograd.grad(e.sum(), data.pos, create_graph=True)[0]
    loss = 0.2 * (e ** 2).mean() + 0.8 * (f ** 2).mean()
    loss.backward()
    sd_o = {k: v.clone().requires_grad_(v.is_floating_point() and "offset" not in k) for k, v in sd.items()}
    pos = case["pos"].clone().requires_grad_(True)
    eo = O.FORWARDS[case["kind"]](sd_o, case["cfg"], pos, case["Z"], case["edge_index"], case["cell"],
                                  case["edge_shift"], case["batch"])
    fo = -torch.autograd.grad(eo.sum(), pos, create_graph=True)[0]
    (0.2 * (eo ** 2).mean() + 0.8 * (fo ** 2).mean()).backward()
    checked = 0
    for k, p in model.named_parameters():
        go = sd_o[k].grad
        if go is None:
            continue
        assert p.grad is not None, k
        assert float((p.grad - go).abs().max()) < 2e-4 * (float(go.abs().max()) + 1e-6) + 1e-6, k
        checked += 1
    assert checked > 10


def test_eval_mode_refuses_double_backward(emu):
    case = util.load_case("triclinic_multi_image")
    model, _ = util.make_model(case["kind"], case["cfg"], case["seed"])
    data = util.make_data(case)
    e = model(data)
    f = torch.autograd.grad(e.sum(), data.pos, create_graph=True)[0]
    with pytest.raises(RuntimeError):
        (f ** 2).sum().backward()


def test_in_subgraph_matches_reference_regrouping(emu):
    case = util.load_case("batch3_mixed")
    data = util.make_data(case, requires_grad=False)
    nids = torch.where(data.atomic_number == 8)[0]
    rel = H.in_subgraph(data, nids)
    want = O.in_subgraph_edges_literal(data.edge_index[1], nids)
    assert torch.equal(rel.edge_index, data.edge_index[:, want])
    assert torch.equal(rel.edge_shift, data.edge_shift[want])
    assert rel.pos is data.pos


def test_neighbor_search_contract(emu):
    case = util.load_case("triclinic_multi_image")
    ei, es = H.neighbor_search(case["pos"], 5.0, case["cell"])
    assert ei.dtype == torch.int64 and es.dtype == torch.float32
    assert torch.all(ei[0][1:] >= ei[0][:-1])          # sorted by edge_index[0] like ASE's 'ijS'
    from oracle.neighbor_oracle import canonical_edges
    assert np.array_equal(canonical_edges(ei.numpy(), es.numpy()), case["edges"])
    case = util.load_case("cluster_nonpbc_capped")
    ei = H.neighbor_search(case["pos"], 5.0)
    assert np.array_equal(canonical_edges(ei.numpy()), case["edges"])
    assert int(torch.bincount(ei[1]).max()) == 32


def test_batch_collation_and_intensive(emu):
    case = util.load_case("batch3_mixed")
    parts = []
    for g in range(3):
        sel = case["batch"] == g
        d = H.Data(pos=case["pos"][sel], atomic_number=case["Z"][sel], cell=case["cell"][g:g + 1])
        parts.append(H.transform(d, case["cfg"]["rc"]))
    b = H.Batch.from_data_list(parts)
    assert b.num_graphs == 3 and torch.equal(b.batch, case["batch"]) and b.cell.shape == (3, 3, 3)
    model, sd = util.make_model(case["kind"], case["cfg"], case["seed"])
    e = model(b)
    assert util.rel_err(e.detach(), case["energy"]) < TOL_E
    model_i, _ = util.make_model(case["kind"], case["cfg"], case["seed"], intensive=True)
    ei = model_i(b)
    counts = torch.bincount(case["batch"]).float()
    assert torch.allclose(ei.detach() * counts, e.detach(), rtol=1e-5, atol=1e-6)


def test_unknown_basis_raises():
    with pytest.raises(ValueError):
        H.HVNet(["H"], rbf={"name": "nope"})
    with pytest.raises(ValueError):
        H.HVNet(["H"], envelope={"name": "nope"})


def test_cpu_input_without_emulator_fails_loudly():
    model = H.HVNet(["H", "O"], num_layers=1, hidden_channels=32, num_rbf=16)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        model(H.Data(pos=torch.zeros(3, 3), atomic_number=torch.ones(3, dtype=torch.long)))


def test_layer_checkpointing_gives_identical_energy_and_forces(emu):
    """checkpoint_layers=True recomputes every layer in the backward pass (memory of one layer instead of all:
    BASELINE config 5, HTNet with 30 rows per atom) -- results must be bit-identical to the stored-activation path."""
    from tests.util import lattice_system
    pos, Z, cell = lattice_system(3, [1, 8], 5)
    for kind in ("HVNet", "HTNet"):
        torch.manual_seed(0)
        model = getattr(H, kind)(elems=["H", "O"], rc=5.0, num_layers=2, hidden_channels=32, num_rbf=16).eval()
        for p in model.parameters():
            p.requires_grad_(False)
        out = []
        for ck in (False, True):
            model.checkpoint_layers = ck
            d = H.Data(pos=pos.clone().requires_grad_(True), atomic_number=Z, cell=cell.clone().requires_grad_(True))
            e = model(d)
            gp, gc = torch.autograd.grad(e.sum(), [d.pos, d.cell])
            out.append((e.detach(), gp, gc))
        assert all(torch.equal(a, b) for a, b in zip(*out))
        model.checkpoint_layers = None
        assert model._want_checkpoint(model.build_graph(pos, Z, cell), pos) is False      # CPU tensors: never


def test_auto_attached_graph_follows_the_current_inputs(emu):
    """ADVICE r1: a graph that forward() attached to ``data`` itself must not outlive the tensors it was derived from
    (the reference always honours the current pos / edge_index, hermnet.py:134-139); a caller-attached graph is kept."""
    case = util.load_case("c1_hvnet")
    model, _ = util.make_model(case["kind"], case["cfg"], case["seed"])
    data = util.make_data(case, with_edges=False, requires_grad=False)
    e0 = model(data)
    g0 = data.graph
    assert model(data) is not None and data.graph is g0                      # unchanged inputs: re-used
    with torch.no_grad():
        data.pos[::3] += 0.8                                                 # in-place move: some pairs cross the cutoff
    e1 = model(data)
    assert data.graph is not g0
    fresh = util.make_data(case, with_edges=False, requires_grad=False)
    fresh.pos = data.pos.clone()
    assert util.rel_err(e1.detach(), model(fresh).detach()) < 1e-6
    assert abs(float(e1) - float(e0)) > 1e-4
    data.pos = data.pos.clone()                                              # re-assigned attribute: rebuilt, same answer
    g1 = data.graph
    e2 = model(data)
    assert data.graph is not g1 and util.rel_err(e2.detach(), e1.detach()) < 1e-6
    # explicit edge lists: keyed on edge_index / edge_shift, not on pos
    d2 = util.make_data(case, with_edges=True, requires_grad=False)
    model(d2)
    g2 = d2.graph
    keep = torch.ones(d2.edge_index.size(1), dtype=torch.bool)
    keep[::7] = False
    d2.edge_index, d2.edge_shift = d2.edge_index[:, keep], d2.edge_shift[keep]
    model(d2)
    assert d2.graph is not g2 and d2.graph.n_edges == int(keep.sum())
    # a graph the caller attached is trusted as is
    d3 = util.make_data(case, with_edges=False, requires_grad=False)
    d3.graph = model.build_graph(d3.pos, d3.atomic_number, d3.cell)
    g3 = d3.graph
    model(d3)
    assert d3.graph is g3


def test_loader_side_batched_graph_build_equals_per_sample_transform(emu):
    """SURVEY 8(f) rank 2: DataLoader(rc=...) builds the neighbour list of a collated batch in one batched search; the edge
    set equals per-sample ``transform`` (data.py:27-35, 58-67) followed by PyG-style collation."""
    from hermnet_b200 import synthetic
    from oracle import neighbor_oracle as NO
    samples = []
    for seed in (100, 101, 102):
        pos, Z, cell = synthetic.cubic_lattice(4 + seed % 2, 2.3, ("Li", "Si", "O"), (1 / 3, 1 / 6, 1 / 2), 0.10, seed)
        samples.append(H.Data(pos=torch.from_numpy(pos), atomic_number=torch.from_numpy(Z), cell=torch.from_numpy(cell)[None],
                              y=torch.tensor([float(seed)])))
    per_sample = H.Batch.from_data_list([H.transform(H.Data(**dict(iter(d))), 5.0) for d in samples])
    loader = H.DataLoader(samples, batch_size=3, rc=5.0)
    (batched,) = list(loader)
    a = NO.canonical_edges(per_sample.edge_index.numpy(), per_sample.edge_shift.numpy())
    b = NO.canonical_edges(batched.edge_index.numpy(), batched.edge_shift.numpy())
    assert a.shape[0] > 1000 and np.array_equal(a, b)
    assert torch.equal(batched.batch, per_sample.batch) and batched.cell.shape == (3, 3, 3)
    # and the model gives the same energies through either
    case = util.load_case("batch3_mixed")
    model, _ = util.make_model(case["kind"], case["cfg"], case["seed"])
    d = util.make_data(case, with_edges=False, requires_grad=False)
    d2 = H.transform_batch(util.make_data(case, with_edges=False, requires_grad=False), case["cfg"]["rc"])
    assert d2.edge_index.size(1) == case["edges"].shape[0]
    assert util.rel_err(model(d2).detach(), model(d).detach()) < 1e-6


@pytest.mark.parametrize("path,trainable", [pytest.param("fused", False, id="fused"),
                                            pytest.param("composite", False, id="composite"),
                                            pytest.param("fused", True, id="fused-trainable"),
                                            pytest.param("composite", True, id="composite-trainable")])
def test_verlet_skin_list_gives_the_energy_of_a_fresh_list(emu, path, trainable):
    """SURVEY 8(f) rank 1: a list searched with rc + skin and re-used after the atoms moved (< skin / 2) must give the
    energies / forces of a fresh list: entries at or beyond rc contribute nothing, not even the filter bias.  With trainable
    parameters (an eval-mode model nobody froze) the filter-weight backward runs too and must drop the dead entries."""
    from tests.util import lattice_system
    pos, Z, cell = lattice_system(5, [3, 8], 21)
    torch.manual_seed(5)
    model = H.HVNet(elems=["Li", "O"], rc=4.0, num_layers=2, hidden_channels=128, num_rbf=32).eval()
    for p in model.parameters():
        p.requires_grad_(trainable)
    model.edge_path = path
    g_skin = model.build_graph(pos, Z, cell, skin=0.6)
    g_plain = model.build_graph(pos, Z, cell)
    assert g_skin.masked and g_skin.n_edges > g_plain.n_edges
    gen = torch.Generator().manual_seed(1)
    pos2 = pos + 0.28 * (2 * torch.rand(pos.shape, generator=gen) - 1) / 3 ** 0.5     # every atom moved < 0.28 A < skin / 2
    out, wgrads = [], []
    for graph in (g_skin, None):
        d = H.Data(pos=pos2.clone().requires_grad_(True), atomic_number=Z, cell=cell.clone().requires_grad_(True))
        if graph is not None:
            d.graph = graph
        e = model(d)
        gp, gc = torch.autograd.grad(e.sum(), [d.pos, d.cell], retain_graph=trainable)
        out.append((e.detach(), gp, gc))
        if trainable:
            model.zero_grad()
            e.sum().backward()
            wgrads.append({k: q.grad.clone() for k, q in model.named_parameters() if "rbf_proj" in k})
    fresh = model.build_graph(pos2, Z, cell)
    assert fresh.n_edges != g_plain.n_edges or True
    assert util.rel_err(out[0][0], out[1][0]) < 2e-6
    assert float((out[0][1] - out[1][1]).abs().max()) < 2e-5 * max(1.0, float(out[1][1].abs().max()))
    assert float((out[0][2] - out[1][2]).abs().max()) < 2e-4 * max(1.0, float(out[1][2].abs().max()))
    if trainable:
        assert len(wgrads[1]) == 8          # 2 layers x 2 sub-networks x (weight, bias)
        for k, ref in wgrads[1].items():
            assert float((wgrads[0][k] - ref).abs().max()) < 2e-4 * float(ref.abs().max()), k


def test_device_md_reuses_the_verlet_list(emu):
    from hermnet_b200.plugin import md
    from tests.util import lattice_system
    pos, Z, cell = lattice_system(4, [3, 8], 22, a=2.6)
    torch.manual_seed(6)
    model = H.HVNet(elems=["Li", "O"], rc=3.5, num_layers=1, hidden_channels=128, num_rbf=24).eval()
    for p in model.parameters():
        p.requires_grad_(False)
    vel = 0.002 * torch.randn(pos.shape, generator=torch.Generator().manual_seed(2)).numpy()
    runs = {}
    for skin in (0.0, 0.5):
        st = {}
        p1, v1, e1 = md.velocity_verlet_device(model, Z.numpy(), pos.numpy(), cell.numpy(), vel, steps=6, dt_fs=0.5, device="cpu",
                                               skin=skin, stats=st)
        runs[skin] = (p1, e1, st)
    assert runs[0.0][2] == {"builds": 7, "reuses": 0}
    assert runs[0.5][2]["builds"] == 1 and runs[0.5][2]["reuses"] == 6
    assert float((runs[0.0][0] - runs[0.5][0]).abs().max()) < 1e-5
    assert util.rel_err(runs[0.5][1], runs[0.0][1]) < 1e-5


@pytest.mark.parametrize("kind,elems", [("HVNet", ["Li", "Al", "Si", "O"]), ("HTNet", ["Li", "O"])])
def test_graph_and_plans_are_released_without_the_garbage_collector(emu, kind, elems):
    """A graph built by forward() (row CSR, tile plans, cached geometry) must die with its Data object by reference counting
    alone: a cycle through an autograd node (plan -> geometry tensor -> grad_fn -> graph -> plan) would leak gigabytes per MD
    step -- the cycle collector cannot see through C++ autograd nodes."""
    import gc
    import weakref
    from tests.util import lattice_system
    pos, Z, cell = lattice_system(4, [3, 13, 14, 8], 5)
    torch.manual_seed(0)
    model = getattr(H, kind)(elems=elems, rc=5.0, num_layers=2, hidden_channels=128, num_rbf=32).eval()
    for p in model.parameters():
        p.requires_grad_(False)
    gc.collect()
    gc.disable()
    try:
        d = H.Data(pos=pos.clone().requires_grad_(True), atomic_number=Z, cell=cell)
        e = model(d)
        (g,) = torch.autograd.grad(e.sum(), d.pos)
        wg = weakref.ref(d.graph)
        wp = weakref.ref(d.graph._lazy["tc_dst"])
        del d, e, g
        assert wg() is None and wp() is None
    finally:
        gc.enable()


@pytest.mark.parametrize("fused_node,edge_path,frozen", [(True, "fused", True), (False, "fused", True), (False, "composite", True),
                                                         (False, "composite", False)])
def test_system_without_edges_gives_zero_forces(emu, fused_node, edge_path, frozen):
    """Isolated atoms (nothing within rc): like the reference, the energy stays attached to pos / cell and autograd.grad
    returns zeros (calculator.py:77-83 calls it without allow_unused) on every formulation."""
    from tests.util import lattice_system
    pos, Z, cell = lattice_system(3, [3, 8], 4, a=6.0, jitter=0.0)
    torch.manual_seed(1)
    model = H.HVNet(elems=["Li", "O"], rc=3.0, num_layers=2, hidden_channels=64, num_rbf=16).eval()
    for p in model.parameters():
        p.requires_grad_(not frozen)
    model.fused_node, model.edge_path = fused_node, edge_path
    d = H.Data(pos=pos.clone().requires_grad_(True), atomic_number=Z, cell=cell.clone().requires_grad_(True))
    e = model(d)
    assert d.graph.n_edges == 0 and torch.isfinite(e).all()
    gp, gc = torch.autograd.grad(e.sum(), [d.pos, d.cell])
    assert float(gp.abs().max()) == 0.0 and float(gc.abs().max()) == 0.0
    # the atomic energies are those of the bare embeddings pushed through the residual / update blocks: same on every path
    model.fused_node, model.edge_path = True, "fused"
    for p in model.parameters():
        p.requires_grad_(False)
    e_ref = model(H.Data(pos=pos.clone(), atomic_number=Z, cell=cell.clone()))
    assert torch.allclose(e.detach(), e_ref, rtol=1e-5, atol=1e-6)
