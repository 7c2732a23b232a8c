"""Parity of the CUDA path (through the C ABI) with the oracle / golden fixtures.  Run on a B200: ``-m gpu``.

Bars (BASELINE.json): neighbour and triplet lists bit-exact as sets; fp32 energy within 1e-5 relative; forces
within 1e-4 eV/A.  Nothing here reads /root/reference."""
import numpy as np
import pytest
import torch

import hermnet_b200 as H
from hermnet_b200 import functional as Fn
from hermnet_b200 import ops, synthetic
from hermnet_b200.graph import Segments
from oracle import build as obuild
from oracle import hermnet_oracle as O
from oracle import neighbor_oracle as NO
from tests import util

pytestmark = pytest.mark.gpu
TOL_E, TOL_F = 1e-5, 1e-4
DEV = "cuda"


def _search_batched(case):
    rows, off = [], 0
    for g in range(int(case["batch"].max()) + 1):
        sel = case["batch"] == g
        p = case["pos"][sel].to(DEV)
        if case["cell"] is None:
            ei = H.neighbor_search(p, case["cfg"]["rc"]).cpu().numpy()
            rows.append(NO.canonical_edges(ei + off))
        else:
            ei, es = H.neighbor_search(p, case["cfg"]["rc"], case["cell"][g:g + 1].to(DEV))
            rows.append(NO.canonical_edges(ei.cpu().numpy() + off, es.cpu().numpy()))
        off += int(sel.sum())
    got = np.concatenate(rows)
    return got[np.lexsort((got[:, 4], got[:, 3], got[:, 2], got[:, 1], got[:, 0]))]


@pytest.mark.parametrize("name", util.ALL_CASES)
def test_neighbor_list_bit_exact_vs_golden(name):
    case = util.load_case(name)
    assert np.array_equal(_search_batched(case), case["edges"])


def test_neighbor_search_accepts_cpu_tensors_like_the_reference():
    case = util.load_case("c1_hvnet")
    ei, es = H.neighbor_search(case["pos"], 5.0, case["cell"])       # CPU in -> CPU out
    assert not ei.is_cuda and np.array_equal(NO.canonical_edges(ei.numpy(), es.numpy()), case["edges"])
    assert torch.all(ei[0][1:] >= ei[0][:-1])


def test_neighbor_list_4096_atoms_vs_c_oracle():
    (pos, Z, cell), _ = synthetic.config("C2")
    ei, es = H.neighbor_search(torch.from_numpy(pos).to(DEV), 5.0, torch.from_numpy(cell)[None].to(DEV))
    i, j, S = obuild.nl_pbc_rows(pos, cell, 5.0)
    assert np.array_equal(NO.canonical_edges(ei.cpu().numpy(), es.cpu().numpy()), NO.canonical_edges(np.stack([i, j]), S))


@pytest.mark.parametrize("cfg_name,scale", [("C3", 1.0), ("C4", 1.0), ("C5", 0.5)])
def test_neighbor_list_large_properties(cfg_name, scale):
    """Full-size lists: sampled rows bit-exact vs the C oracle, (i,j,S) <=> (j,i,-S), no self edge, expected size."""
    (pos, Z, cell), cfg = synthetic.config(cfg_name, scale)
    n = len(Z)
    rc = cfg["rc"]
    ei, es = H.neighbor_search(torch.from_numpy(pos).to(DEV), rc, torch.from_numpy(cell)[None].to(DEV))
    E = ei.size(1)
    dens = n / float(np.linalg.det(cell.astype(np.float64)))
    assert abs(E / n - dens * 4 / 3 * np.pi * rc ** 3) / (E / n) < 0.3   # lattices are not a uniform continuum
    S = es.long()
    key = ((ei[0] * n + ei[1]) * 27 + (S[:, 0] + 1) * 9 + (S[:, 1] + 1) * 3 + (S[:, 2] + 1))
    rkey = ((ei[1] * n + ei[0]) * 27 + (1 - S[:, 0]) * 9 + (1 - S[:, 1]) * 3 + (1 - S[:, 2]))
    assert int(S.abs().max()) <= 1
    assert torch.equal(torch.sort(key).values, torch.sort(rkey).values)
    assert int(((ei[0] == ei[1]) & (S == 0).all(1)).sum()) == 0
    assert torch.unique(key).numel() == E
    rng = np.random.default_rng(0)
    centres = np.sort(rng.choice(n, 24, replace=False))
    i, j, So = obuild.nl_pbc_rows(pos, cell, rc, centres)
    sel = torch.isin(ei[0], torch.from_numpy(centres).to(DEV))
    got = NO.canonical_edges(ei[:, sel].cpu().numpy(), es[sel].cpu().numpy())
    assert np.array_equal(got, NO.canonical_edges(np.stack([i, j]), So))


@pytest.mark.parametrize("name", util.ALL_CASES)
@pytest.mark.parametrize("path", ["fused", "composite"])
@pytest.mark.parametrize("with_edges", [True, False])
def test_energy_forces_vs_golden(name, path, with_edges):
    case = util.load_case(name)
    model, _ = util.make_model(case["kind"], case["cfg"], case["seed"], DEV)
    model.edge_path = path
    data = util.make_data(case, DEV, with_edges=with_edges)
    e, f, gc = util.energy_forces(model, data)
    assert util.rel_err(e.cpu(), case["energy"]) < TOL_E
    assert float((f.cpu() - case["forces"]).abs().max()) < TOL_F
    if case["cell_grad"] is not None:
        assert float((gc.cpu() - case["cell_grad"]).abs().max()) < TOL_F * 10


def test_fused_path_is_deterministic():
    case = util.load_case("c1_hvnet")
    model, _ = util.make_model(case["kind"], case["cfg"], case["seed"], DEV)
    outs = [util.energy_forces(model, util.make_data(case, DEV, with_edges=False)) for _ in range(3)]
    for e, f, gc in outs[1:]:
        assert torch.equal(e, outs[0][0]) and torch.equal(f, outs[0][1]) and torch.equal(gc, outs[0][2])


@pytest.mark.parametrize("name", ["triclinic_multi_image", "batch3_mixed", "water24_hpnet", "water24_htnet"])
def test_parameter_gradients(name):
    case = util.load_case(name)
    sd = None
    grads = {}
    for path in ("fused", "composite"):
        model, sd = util.make_model(case["kind"], case["cfg"], case["seed"], DEV)
        model.edge_path = path
        model(util.make_data(case, DEV, requires_grad=False)).sum().backward()
        grads[path] = {k: p.grad.cpu() for k, p in model.named_parameters() if p.grad is not None}
    sd_o = {k: v.clone().requires_grad_(v.is_floating_point() and "offset" not in k) for k, v in sd.items()}
    O.FORWARDS[case["kind"]](sd_o, case["cfg"], case["pos"], case["Z"], case["edge_index"], case["cell"],
                             case["edge_shift"], case["batch"]).sum().backward()
    n = 0
    for k, v in sd_o.items():
        if v.requires_grad and v.grad is not None:
            for path in grads:
                assert float((grads[path][k] - v.grad).abs().max()) < 2e-4 * (float(v.grad.abs().max()) + 1e-6) + 1e-6, (k, path)
            n += 1
    assert n > 10


@pytest.mark.parametrize("name", ["triclinic_multi_image", "water24_hpnet", "water24_htnet"])
def test_force_loss_training_step(name):
    """example/dist_train.py:89-99 -- forces with create_graph=True enter the loss (double backward)."""
    case = util.load_case(name)
    model, sd = util.make_model(case["kind"], case["cfg"], case["seed"], DEV)
    model.train()
    data = util.make_data(case, DEV)
    e = model(data)
    f = -torch.autograd.grad(e.sum(), data.pos, create_graph=True)[0]
    (0.2 * (e ** 2).mean() + 0.8 * (f ** 2).mean()).backward()
    sd_o = {k: v.clone().requires_grad_(v.is_floating_point() and "offset" not in k) for k, v in sd.items()}
    pos = case["pos"].clone().requires_grad_(True)
    eo = O.FORWARDS[case["kind"]](sd_o, case["cfg"], pos, case["Z"], case["edge_index"], case["cell"],
                                  case["edge_shift"], case["batch"])
    fo = -torch.autograd.grad(eo.sum(), pos, create_graph=True)[0]
    (0.2 * (eo ** 2).mean() + 0.8 * (fo ** 2).mean()).backward()
    assert float((f.detach().cpu() - fo.detach()).abs().max()) < TOL_F
    n = 0
    for k, p in model.named_parameters():
        go = sd_o[k].grad
        if go is not None:
            assert float((p.grad.cpu() - go).abs().max()) < 5e-4 * (float(go.abs().max()) + 1e-6) + 1e-6, k
            n += 1
    assert n > 10


def test_gather_and_segment_sum_are_adjoint_and_exact():
    g = torch.Generator().manual_seed(0)
    idx = torch.randint(0, 50, (4000,), generator=g).to(torch.int32).to(DEV)
    seg = Segments.from_index(idx, 50)
    for C in (1, 3, 9, 96, 384):
        X = torch.randn(50, C, generator=g).to(DEV).requires_grad_(True)
        Y = torch.randn(4000, C, generator=g).to(DEV).requires_grad_(True)
        gx = Fn.gather_rows(X, seg)
        assert torch.equal(gx, X[idx.long()])
        sy = Fn.segment_sum(Y, seg)
        ref = torch.zeros(50, C, dtype=torch.float64, device=DEV).index_add_(0, idx.long(), Y.detach().double())
        assert float((sy.detach().double() - ref).abs().max()) < 1e-4
        lhs = (gx * Y).sum(); rhs = (X * sy).sum()            # <G X, Y> == <X, G^T Y>
        assert abs(float(lhs - rhs)) < 1e-2 * (1 + abs(float(lhs)))
        gX, = torch.autograd.grad(gx.sum() * 2.0, X)
        assert torch.allclose(gX, 2.0 * torch.bincount(idx.long(), minlength=50).float()[:, None].expand(-1, C))


def test_in_subgraph_matches_reference_regrouping_on_gpu():
    case = util.load_case("c1_hvnet")
    data = util.make_data(case, DEV, requires_grad=False)
    nids = torch.where(data.atomic_number == 8)[0]
    rel = H.in_subgraph(data, nids)
    want = O.in_subgraph_edges(case["edge_index"][1], nids.cpu(), len(case["Z"]))
    assert torch.equal(rel.edge_index.cpu(), case["edge_index"][:, want])
    assert torch.equal(rel.edge_shift.cpu(), case["edge_shift"][want])


def test_triplets_bit_exact_and_counts():
    case = util.load_case("water24_htnet")
    model, _ = util.make_model("HVNet", dict(case["cfg"]), case["seed"], DEV)
    g = model.build_graph(case["pos"].to(DEV), case["Z"].to(DEV), case["cell"].to(DEV), None)
    tp, e1, e2 = ops.triplets(g.rowptr, g.col)
    want = NO.triplets_bruteforce(g.rowptr.cpu().numpy(), g.col.cpu().numpy())
    assert np.array_equal(e1.cpu().numpy(), want[:, 3]) and np.array_equal(e2.cpu().numpy(), want[:, 4])
    deg = (g.rowptr[1:] - g.rowptr[:-1]).long()
    assert int(tp[-1]) == int((deg * (deg - 1)).sum())
    st = g.types
    for (a, c) in [(0, 0), (0, 1), (1, 1)]:
        tp2, f1, f2 = ops.triplets(g.rowptr, g.col, st, a, c)
        w = NO.triplets_bruteforce(g.rowptr.cpu().numpy(), g.col.cpu().numpy(), st.cpu().numpy(), a, c)
        assert np.array_equal(f1.cpu().numpy(), w[:, 3]) and np.array_equal(f2.cpu().numpy(), w[:, 4])


def test_triplet_sum_equals_factorised_inner_product():
    """sum over triplets (j,i,k) of <m_ij, m_ik> + diagonal == <sum_j m_ij, sum_k m_ik> (SURVEY.md A.3)."""
    (pos, Z, cell), _ = synthetic.water_box(3, seed=8), None
    model = H.HVNet(["H", "O"], rc=4.5, num_layers=1, hidden_channels=32, num_rbf=16).to(DEV)
    g = model.build_graph(torch.from_numpy(pos).to(DEV), torch.from_numpy(Z).to(DEV), torch.from_numpy(cell)[None].to(DEV))
    m_vec = torch.randn(g.n_edges, 3, 32, device=DEV)
    tp, e1, e2 = ops.triplets(g.rowptr, g.col)
    dots = ops.triplet_dots(m_vec, tp, e1, e2)
    Psum = Fn.segment_sum(m_vec, g.seg_dst)
    diag = Fn.segment_sum((m_vec ** 2).sum(1), g.seg_dst)
    want = (Psum * Psum).sum(1)
    assert float((dots + diag - want).abs().max()) < 1e-3 * float(want.abs().max())
    deg = (g.rowptr[1:] - g.rowptr[:-1]).long()
    assert int(tp[-1]) == int((deg * (deg - 1)).sum())


@pytest.mark.parametrize("kind,F", [("HVNet", 128), ("HPNet", 64), ("HTNet", 256)])
def test_mid_size_fused_equals_composite_and_invariances(kind, F):
    """~1.5k-atom periodic systems: fused kernels == composite formulation; translation invariance; sum F = 0."""
    (pos, Z, cell) = synthetic.cubic_lattice(8, 2.3, ("Li", "Si", "O"), (1 / 3, 1 / 6, 1 / 2), 0.1, 77)
    cfg = dict(elems=["Li", "Si", "O"], rc=5.0, num_layers=2, hidden_channels=F, num_rbf=128)
    model, _ = util.make_model(kind, cfg, 3, DEV, pbc_shift="physical")
    p = torch.from_numpy(pos).to(DEV)
    z = torch.from_numpy(Z).to(DEV)
    c = torch.from_numpy(cell)[None].to(DEV)
    out = {}
    for path in ("fused", "composite"):
        model.edge_path = path
        d = H.Data(pos=p.clone().requires_grad_(True), atomic_number=z, cell=c.clone().requires_grad_(True))
        out[path] = util.energy_forces(model, d)
    assert util.rel_err(out["fused"][0], out["composite"][0]) < TOL_E
    fscale = max(1.0, float(out["composite"][1].abs().max()))      # random weights give |F| ~ 10 eV/A: scale the bar
    assert float((out["fused"][1] - out["composite"][1]).abs().max()) < TOL_F * fscale
    assert float((out["fused"][2] - out["composite"][2]).abs().max()) < 1e-3 * float(out["composite"][2].abs().max())
    assert float(out["fused"][1].sum(0).abs().max()) < 1e-2       # physical shifts: no net force
    model.edge_path = "fused"
    d = H.Data(pos=(p + torch.tensor([0.37, -1.1, 2.9], device=DEV)).requires_grad_(True), atomic_number=z, cell=c)
    e2, f2, _ = util.energy_forces(model, d)
    # a rigid shift re-rounds every fp32 coordinate (~1e-6 A); random weights give force constants ~1e3 eV/A^2
    assert util.rel_err(e2, out["fused"][0]) < 5e-5
    assert float((f2 - out["fused"][1]).abs().max()) < 1e-3 * fscale


def test_c2_graph_vs_oracle_4096_atoms():
    """One 4096-atom Li/Si/O graph (C2) through HVNet F=128: CUDA path vs the CPU oracle."""
    (pos, Z, cell), _ = synthetic.config("C2")
    cfg = dict(elems=["Li", "Si", "O"], rc=5.0, num_layers=2, hidden_channels=128, num_rbf=128)
    model, sd = util.make_model("HVNet", cfg, 21, DEV)
    d = H.Data(pos=torch.from_numpy(pos).to(DEV).requires_grad_(True), atomic_number=torch.from_numpy(Z).to(DEV),
               cell=torch.from_numpy(cell)[None].to(DEV))
    e, f, _ = util.energy_forces(model, d)
    ei, es = H.neighbor_search(torch.from_numpy(pos), 5.0, torch.from_numpy(cell)[None])
    eo, fo = O.energy_and_forces("HVNet", sd, cfg, torch.from_numpy(pos), torch.from_numpy(Z), ei,
                                 torch.from_numpy(cell)[None], es)
    assert util.rel_err(e.cpu(), eo) < TOL_E
    assert float((f.cpu() - fo).abs().max()) < TOL_F


def test_ase_style_calculator_md_and_batched_displacements():
    """BASELINE configs[2] path: NNCalculator driven like ASE drives it, device-resident MD, batched force sets."""
    import sys, os
    from hermnet_b200.plugin import NNCalculator
    from hermnet_b200.plugin import md
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from plugin.phonopy_interface.phonon_calc import batched_force_sets
    pos, Z, cell = synthetic.water_box(3, seed=3)
    cfg = dict(elems=["H", "O"], rc=4.0, num_layers=2, hidden_channels=64, num_rbf=32)
    model, sd = util.make_model("HTNet", cfg, 31, DEV, pbc_shift="physical")
    calc = NNCalculator(model, None, trn_mean=-1.5, device_=DEV, ensemble="NPT")
    atoms = md.SimpleAtoms(Z, pos, cell)
    atoms.calc = calc
    f = atoms.get_forces()
    assert set(calc.results) == {"energy", "free_energy", "forces", "stress"} and calc.results["stress"].shape == (6,)
    ei, es = H.neighbor_search(torch.from_numpy(pos), 4.0, torch.from_numpy(cell)[None])
    eo, fo = O.energy_and_forces("HTNet", sd, cfg, torch.from_numpy(pos), torch.from_numpy(Z), ei,
                                 torch.from_numpy(cell)[None], es, pbc_shift="physical")
    assert abs(calc.results["energy"] - (float(eo) - 1.5)) < 1e-4 * abs(float(eo)) + 1e-4
    assert float(np.abs(f - fo.numpy()).max()) < TOL_F * max(1.0, float(fo.abs().max()))
    # host-driven and device-resident velocity Verlet follow the same trajectory
    md.maxwell_boltzmann(atoms, 300.0, seed=3)
    v0 = atoms.velocities.copy()
    e_host = md.velocity_verlet(atoms, steps=5, dt_fs=0.5)
    p_dev, v_dev, e_dev = md.velocity_verlet_device(model, Z, pos, cell, v0, steps=5, dt_fs=0.5, device=DEV)
    assert float(np.abs(p_dev.cpu().numpy() - atoms.positions).max()) < 1e-3
    assert abs(float(e_dev[-1]) - (e_host[-1] + 1.5)) < 1e-3 * max(1.0, abs(e_host[-1]))
    # all displaced cells in one batched forward == one at a time
    rng = np.random.default_rng(0)
    disp = [pos + rng.normal(0, 0.01, pos.shape).astype(np.float32) for _ in range(5)]
    fb = batched_force_sets(model, Z, cell, disp, device=DEV)
    for k, p in enumerate(disp):
        atoms.positions = p.astype(np.float64)
        assert float(np.abs(fb[k] - atoms.get_forces()).max()) < TOL_F * max(1.0, float(np.abs(fb[k]).max()))


@pytest.mark.gpu
@pytest.mark.parametrize("n,n_keys", [(0, 5), (1, 1), (1000, 7), (300000, 256), (300000, 8192), (300000, 8193), (500000, 400000)])
def test_sort_by_key_is_a_stable_counting_sort(n, n_keys):
    """hn_sort_by_key (shared-memory histogram for few keys, warp-aggregated atomics for many) == stable argsort."""
    from hermnet_b200 import ops
    gen = torch.Generator().manual_seed(n + n_keys)
    keys = torch.randint(0, n_keys, (n,), generator=gen, dtype=torch.int32)
    if n > 10:
        keys[: n // 3] = keys[: n // 3].sort().values        # sorted stretch: many equal keys inside a warp
    rowptr, order = ops.sort_by_key(keys.to(DEV), n_keys)
    ref_order = torch.sort(keys.long(), stable=True).indices
    ref_ptr = torch.zeros(n_keys + 1, dtype=torch.long)
    ref_ptr[1:] = torch.cumsum(torch.bincount(keys.long(), minlength=n_keys), 0)
    assert torch.equal(rowptr.cpu().long(), ref_ptr)
    assert torch.equal(order.cpu().long(), ref_order)


@pytest.mark.parametrize("kind,pbc_shift,trainable",
                         [pytest.param(k, s, t, id=f"{k}-{s}" + ("-trainable" if t else ""))
                          for t in (False, True) for k, s in (("HVNet", "reference"), ("HVNet", "physical"), ("HTNet", "reference"))])
def test_verlet_skin_list_reuse_on_gpu(kind, pbc_shift, trainable):
    """SURVEY 8(f) rank 1: a list searched with rc + skin, re-used after the atoms moved (< skin / 2), gives the energies /
    forces / cell gradient of a fresh list through the tensor-core edge kernels (dead entries stage zeros: they contribute
    nothing, not even the filter bias); the device MD loop re-uses it and follows the rebuild-every-step trajectory.
    trainable: an eval-mode model whose parameters still require grad runs the filter-weight backward on every force
    call; its rbf_proj gradients on the skin list equal those of a fresh list."""
    from hermnet_b200.plugin import md
    pos, Z, cell = synthetic.water_box(5, seed=9)
    pos, Z, cell = torch.from_numpy(pos).to(DEV), torch.from_numpy(Z).to(DEV), torch.from_numpy(cell)[None].to(DEV)
    torch.manual_seed(11)
    model = getattr(H, kind)(elems=["H", "O"], rc=4.5, num_layers=2, hidden_channels=128, num_rbf=64, pbc_shift=pbc_shift).to(DEV).eval()
    for p in model.parameters():
        p.requires_grad_(trainable)
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
        gp, gc = torch.autograd.grad(e.sum(), [d.pos, d.cell], retain_graph=trainable)
        out.append((e.detach(), gp, gc))
        if trainable:
            model.zero_grad()
            e.sum().backward()
            wgrads.append({k: q.grad.clone() for k, q in model.named_parameters() if "rbf_proj" in k})
    assert util.rel_err(out[0][0], out[1][0]) < 3e-6
    fs = max(1.0, float(out[1][1].abs().max()))
    assert float((out[0][1] - out[1][1]).abs().max()) < 3e-5 * fs
    assert float((out[0][2] - out[1][2]).abs().max()) < 3e-4 * max(1.0, float(out[1][2].abs().max()))
    if trainable:
        assert len(wgrads[1]) >= 8
        for k, ref in wgrads[1].items():
            assert float((wgrads[0][k] - ref).abs().max()) < 3e-4 * float(ref.abs().max()), k
    if kind == "HVNet":
        v0 = 0.003 * torch.randn(pos.shape, generator=torch.Generator().manual_seed(2)).numpy()
        runs = {}
        for skin in (0.0, 0.8):
            st = {}
            p1, _, e1 = md.velocity_verlet_device(model, Z.cpu().numpy(), pos.cpu().numpy(), cell.cpu().numpy(), v0, steps=8,
                                                  dt_fs=0.5, device=DEV, skin=skin, stats=st)
            runs[skin] = (p1, e1, st)
        assert runs[0.0][2] == {"builds": 9, "reuses": 0}
        assert runs[0.8][2]["builds"] == 1 and runs[0.8][2]["reuses"] == 8
        assert float((runs[0.0][0] - runs[0.8][0]).abs().max()) < 1e-4
        assert util.rel_err(runs[0.8][1], runs[0.0][1]) < 1e-5


def test_device_md_with_cuda_graph_replay_follows_the_eager_trajectory():
    """The Verlet-skin MD loop with the evaluation captured as one CUDA graph per list build (plugin/md.py, graphed.py)
    gives the trajectory of the eager loop."""
    from hermnet_b200.plugin import md
    pos, Z, cell = synthetic.water_box(5, seed=9)
    torch.manual_seed(11)
    model = H.HTNet(elems=["H", "O"], rc=4.5, num_layers=2, hidden_channels=128, num_rbf=64).to(DEV).eval()
    for p in model.parameters():
        p.requires_grad_(False)
    v0 = 0.003 * torch.randn(pos.shape, generator=torch.Generator().manual_seed(2)).numpy()
    runs = {}
    for cg in (False, True):
        st = {}
        p1, _, e1 = md.velocity_verlet_device(model, Z, pos, cell, v0, steps=8, dt_fs=0.5, device=DEV, skin=0.8, stats=st, cuda_graph=cg)
        runs[cg] = (p1, e1, st)
    assert runs[True][2] == runs[False][2] and runs[True][2]["reuses"] == 8
    assert float((runs[True][0] - runs[False][0]).abs().max()) < 1e-5
    assert util.rel_err(runs[True][1], runs[False][1]) < 1e-6


def test_halo_pack_unpack_kernels():
    """hn_halo_pack / hn_halo_unpack (csrc/hn_halo.cu) against torch indexing: rows [x | vec] scattered into two "peer" landing
    buffers by (peer, slot), then moved into ghost rows in place."""
    gen = torch.Generator().manual_seed(0)
    n, F, n_send = 500, 128, 180
    x = torch.randn(n, F, generator=gen).to(DEV)
    vec = torch.randn(n, 3, F, generator=gen).to(DEV)
    src = torch.randperm(n, generator=gen)[:n_send].to(torch.int32).to(DEV)
    peer = (torch.arange(n_send) % 2).to(torch.int32).to(DEV)
    slot = torch.cat([torch.randperm(90, generator=gen), torch.randperm(90, generator=gen)]).view(2, 90).t().reshape(-1)[:n_send].to(torch.int32).to(DEV)
    bufs = [torch.zeros(90, 4 * F, device=DEV) for _ in range(2)]
    base = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=DEV)
    ops.halo_pack(x, vec.view(n, 3 * F), src, peer, slot, base)
    want = torch.cat([x, vec.view(n, 3 * F)], 1)
    for p in range(2):
        sel = peer == p
        assert torch.equal(bufs[p][slot[sel].long()], want[src[sel].long()])
    ghost = torch.arange(300, 390, dtype=torch.int32, device=DEV)
    x2, v2 = x.clone(), vec.clone()
    ops.halo_unpack(bufs[0], ghost, x2, v2.view(n, 3 * F))
    assert torch.equal(x2[300:390], bufs[0][:, :F]) and torch.equal(v2[300:390].reshape(90, 3 * F), bufs[0][:, F:])
    assert torch.equal(x2[:300], x[:300]) and torch.equal(v2[390:], vec[390:])


@pytest.mark.gpu
@pytest.mark.parametrize("edge_path", ["fused", "composite"])
def test_system_without_edges_on_gpu(edge_path):
    """Isolated atoms (E = 0): every kernel of the path must accept empty edge arrays; energy finite, forces exactly zero."""
    from tests.util import lattice_system
    pos, Z, cell = lattice_system(3, [3, 8], 4, a=6.0, jitter=0.0)
    torch.manual_seed(1)
    model = H.HVNet(elems=["Li", "O"], rc=3.0, num_layers=2, hidden_channels=128, num_rbf=16).to("cuda:0").eval()
    for p in model.parameters():
        p.requires_grad_(False)
    model.edge_path = edge_path
    d = H.Data(pos=pos.cuda().requires_grad_(True), atomic_number=Z.cuda(), cell=cell.cuda().requires_grad_(True))
    e = model(d)
    assert d.graph.n_edges == 0 and torch.isfinite(e).all()
    gp, gc = torch.autograd.grad(e.sum(), [d.pos, d.cell])
    assert float(gp.abs().max()) == 0.0 and float(gc.abs().max()) == 0.0
