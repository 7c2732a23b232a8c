"""Constant-pressure (NPT) MD on the device: ``hn_md_scr_barostat`` / ``hn_md_affine_scale`` (``ops.md_scr_barostat`` /
``ops.md_affine_scale``), Verlet-skin re-use under a deforming cell (``VerletGraph(deforming=True)``) and
``plugin.md.langevin_npt_device``.

The oracle is the numpy Philox4x32-10 of tests/test_langevin.py with the barostat's counter (word 3 = 1) and the strain
step of include/hermnet_b200.h in float64; the same reference stands in for the two ops in the CPU cases over the kernel
emulator."""
import math

import numpy as np
import pytest
import torch

import hermnet_b200 as H
from hermnet_b200 import ops, synthetic
from hermnet_b200.plugin import md
from tests import util
from tests.test_atom_virial import _emu_edge_virial_atom
from tests.test_langevin import (MASK32, _boxes, _cpu_model, _cpu_systems, _mb, _np, _replica_tensors, _water_model,
                                 emu_md_kick, emu_md_langevin_baoa, philox4x32_10, ref_noise)

DEV = "cuda:0"


# ---------------------------------------------------------------------------------------------------------------------
# float64 reference of the barostat and of the two ops
# ---------------------------------------------------------------------------------------------------------------------
def ref_baro_xi(seeds, step):
    """Barostat normal of every replica: counter (0, lo32 step, hi32 step, 1), key = the replica seed."""
    seeds = np.asarray(seeds, dtype=np.int64).view(np.uint64)
    G = len(seeds)
    ctr = np.stack([np.zeros(G, np.uint64), np.full(G, step & 0xFFFFFFFF, np.uint64), np.full(G, step >> 32, np.uint64),
                    np.ones(G, np.uint64)], -1)
    r = philox4x32_10(ctr, np.stack([seeds & MASK32, seeds >> np.uint64(32)], -1)).astype(np.uint64)
    u = ((r >> np.uint64(9)) * np.uint64(2) + np.uint64(1)).astype(np.float64) * 2.0 ** -24
    return np.sqrt(-2.0 * np.log(u[:, 0])) * np.cos(2.0 * np.pi * u[:, 1])


def ref_barostat(cell, kinetic, virial, P0, kT, beta, seed, step, dt, tau_p):
    """``(mu, P)`` in float64 from the fp32 inputs."""
    h = _np(cell).astype(np.float64).reshape(-1, 3, 3)
    V = np.abs(np.linalg.det(h))
    w = _np(virial).astype(np.float64).reshape(-1, 3, 3)
    P = (2.0 * _np(kinetic).astype(np.float64) + np.trace(w, axis1=1, axis2=2)) / (3.0 * V)
    b = _np(beta).astype(np.float64) * (float(np.float32(dt)) / float(np.float32(tau_p)))
    xi = ref_baro_xi(_np(seed), int(step))
    de = -b * (_np(P0).astype(np.float64) - P) + np.sqrt(2.0 * _np(kT).astype(np.float64) * b / V) * xi
    return np.exp(de / 3.0), P


def emu_md_scr_barostat(cell, kinetic, virial, P0, kT, beta, seed, step, dt, tau_p, mu, pressure):
    """CPU stand-in of ``ops.md_scr_barostat`` (float64 reference, same contract)."""
    m, P = ref_barostat(cell, kinetic, virial, P0, kT, beta, seed, int(step[0]), dt, tau_p)
    mu.copy_(torch.from_numpy(m.astype(np.float32)))
    pressure.copy_(torch.from_numpy(P))
    cell.mul_(mu[:, None, None])


def emu_md_affine_scale(pos, vel, replica, mu):
    """CPU stand-in of ``ops.md_affine_scale``."""
    m = mu[replica.long()][:, None]
    pos.mul_(m)
    vel.div_(m)


@pytest.fixture
def emu_npt(emu, monkeypatch):
    monkeypatch.setattr(ops, "md_langevin_baoa", emu_md_langevin_baoa)
    monkeypatch.setattr(ops, "md_kick", emu_md_kick)
    monkeypatch.setattr(ops, "md_scr_barostat", emu_md_scr_barostat)
    monkeypatch.setattr(ops, "md_affine_scale", emu_md_affine_scale)
    monkeypatch.setattr(ops, "edge_virial_atom", _emu_edge_virial_atom)
    return emu


def _baro_inputs(G, seed=0, dev=DEV):
    gen = torch.Generator().manual_seed(seed)
    cell = (torch.diag_embed(8.0 + 10.0 * torch.rand(G, 3, generator=gen)) + 0.5 * torch.randn(G, 3, 3, generator=gen))
    kin = 0.03 * G * torch.rand(G, generator=gen) + 1.0
    vir = 5.0 * torch.randn(G, 3, 3, generator=gen)
    P0 = 1e-3 * torch.randn(G, generator=gen)                       # eV/A^3, both signs
    kT = 0.02 + 0.05 * torch.rand(G, generator=gen)
    beta = 100.0 * torch.rand(G, generator=gen)
    beta[::7] = 0.0
    return [t.float().contiguous().to(dev) for t in (cell, kin, vir, P0, kT, beta)]


# ---------------------------------------------------------------------------------------------------------------------
# kernel level (GPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 1000])
def test_barostat_matches_float64(G):
    cell, kin, vir, P0, kT, beta = _baro_inputs(G, seed=G)
    seeds = torch.tensor([(2 ** 40 + 977 * g) if g % 2 else (3 + g) for g in range(G)], dtype=torch.int64, device=DEV)
    for s, dt, tau in ((0, 0.5, 1000.0), (17, 2.0, 50.0), (2 ** 32 + 5, 1.0, 5.0)):
        step = torch.tensor([s], dtype=torch.int64, device=DEV)
        c = cell.clone()
        mu, pr = torch.empty(G, device=DEV), torch.empty(G, device=DEV)
        m_ref, P_ref = ref_barostat(cell, kin, vir, P0, kT, beta, seeds, s, dt, tau)
        ops.md_scr_barostat(c, kin, vir, P0, kT, beta, seeds, step, dt, tau, mu, pr)
        assert int(step) == s
        assert np.abs(_np(mu).astype(np.float64) / m_ref - 1.0).max() <= 1.2e-7
        assert np.abs(_np(pr).astype(np.float64) - P_ref).max() <= 1e-6 * np.abs(P_ref).max()
        assert torch.equal(c, cell * mu[:, None, None])            # fp32 mu * cell
        assert torch.equal(mu[::7], torch.ones_like(mu[::7]))       # beta = 0: the cell stays put


@pytest.mark.gpu
def test_affine_scale_is_torch_bitwise_and_empty_launches_are_no_ops():
    sizes = [40_000, 1, 60_002]
    replica, ptr = _replica_tensors(sizes, DEV)
    gen = torch.Generator().manual_seed(3)
    n = sum(sizes)
    pos, vel = (20.0 * torch.randn(n, 3, generator=gen)).to(DEV), (0.03 * torch.randn(n, 3, generator=gen)).to(DEV)
    mu = torch.tensor([0.99, 1.0123, 1.0 - 2.0 ** -20], device=DEV)
    p, v = pos.clone(), vel.clone()
    ops.md_affine_scale(p, v, replica, mu)
    m = mu[replica.long()][:, None]
    assert torch.equal(p, pos * m) and torch.equal(v, vel / m)
    # empty launches
    e = torch.zeros(0, 3, device=DEV)
    ops.md_affine_scale(e, e.clone(), torch.zeros(0, dtype=torch.int32, device=DEV), mu)
    z, z9 = torch.zeros(0, device=DEV), torch.zeros(0, 3, 3, device=DEV)
    step = torch.tensor([3], dtype=torch.int64, device=DEV)
    ops.md_scr_barostat(z9, z, z9.clone(), z, z, z, torch.zeros(0, dtype=torch.int64, device=DEV), step, 0.5, 100.0, z, z)
    assert int(step) == 3


@pytest.mark.gpu
def test_barostat_determinism_and_a_stream_disjoint_from_the_langevin_noise():
    G = 1000
    cell, kin, vir, P0, kT, beta = _baro_inputs(G, seed=9)
    seeds = torch.arange(G, dtype=torch.int64, device=DEV) * 7919 + 2 ** 33
    step = torch.tensor([12345], dtype=torch.int64, device=DEV)

    def run():
        c, mu, pr = cell.clone(), torch.empty(G, device=DEV), torch.empty(G, device=DEV)
        ops.md_scr_barostat(c, kin, vir, P0, kT, beta, seeds, step, 0.5, 100.0, mu, pr)
        return c, mu, pr
    a, b = run(), run()
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    # the barostat's normal, read back through mu: no drift (K = W = P0 = 0) and unit noise scale (2 kT b / V = 1)
    V = torch.abs(torch.linalg.det(cell.double())).float()
    zero = torch.zeros(G, device=DEV)
    c, mu, pr = cell.clone(), torch.empty(G, device=DEV), torch.empty(G, device=DEV)
    ops.md_scr_barostat(c, zero, torch.zeros(G, 3, 3, device=DEV), zero, V / 2.0, torch.ones(G, device=DEV), seeds, step,
                        1.0, 1.0, mu, pr)
    xi_baro = 3.0 * np.log(_np(mu).astype(np.float64))
    assert np.abs(xi_baro - ref_baro_xi(_np(seeds), 12345)).max() < 2e-5 * 3 * 6
    # the Langevin noise of every atom of the same replicas at the same counter value (c1 = 0, unit variance: v = xi)
    sizes = [4] * G
    replica, ptr = _replica_tensors(sizes, DEV)
    n = sum(sizes)
    v = torch.zeros(n, 3, device=DEV)
    ops.md_langevin_baoa(torch.zeros(n, 3, device=DEV), v, torch.zeros(n, 3, device=DEV), torch.ones(n, device=DEV), replica,
                         ptr, torch.ones(G, device=DEV), seeds, step, 0.0, 1.0, 0.5)
    lang = _np(v).astype(np.float64).reshape(G, 12)
    assert np.abs(lang - ref_noise(replica, ptr, seeds, 12345).reshape(G, 12)).max() <= 4e-6 * 6
    assert (np.abs(lang - xi_baro[:, None]).min(1) > 1e-4).mean() > 0.99


@pytest.mark.gpu
def test_ideal_gas_volume_distribution():
    """No forces: the NPT ideal gas has rho(V) ~ V^N exp(-P0 V / kT), so <V> = (N+1) kT/P0 and Var V = (N+1) (kT/P0)^2.
    Adding Bussi's +kT/V to the drift would give (N+2) kT/P0: 20 % off."""
    G, N = 16384, 4
    sizes = [N] * G
    replica, ptr = _replica_tensors(sizes, DEV)
    n = G * N
    kT = torch.ones(G, device=DEV)
    P0 = torch.ones(G, device=DEV)
    beta = torch.full((G,), 0.005, device=DEV)                      # beta P0 dt / tau_p = 0.005 with dt = tau_p = 1
    inv_m = torch.ones(n, device=DEV)
    seeds = torch.arange(G, dtype=torch.int64, device=DEV) + 101
    step = torch.zeros(1, dtype=torch.int64, device=DEV)
    gen = torch.Generator().manual_seed(0)
    pos = (torch.rand(n, 3, generator=gen) * 5.0 ** (1 / 3)).to(DEV)
    vel = torch.randn(n, 3, generator=gen).to(DEV)
    cell = (torch.eye(3) * 5.0 ** (1 / 3)).repeat(G, 1, 1).to(DEV).contiguous()
    zero_f, zero_w = torch.zeros(n, 3, device=DEV), torch.zeros(G, 3, 3, device=DEV)
    kinetic = torch.empty(n, device=DEV)
    mu, pr = torch.empty(G, device=DEV), torch.empty(G, device=DEV)
    gdt = 0.01
    c1, c2 = math.exp(-gdt), math.sqrt(-math.expm1(-2 * gdt))
    s1 = torch.zeros(G, dtype=torch.float64, device=DEV)
    s2 = torch.zeros(G, dtype=torch.float64, device=DEV)
    steps, burn = 20_000, 4_000
    for k in range(steps):
        ops.md_langevin_baoa(pos, vel, zero_f, inv_m, replica, ptr, kT, seeds, step, c1, c2, 1.0)
        ops.md_kick(vel, zero_f, inv_m, 0.5, kinetic, step)
        ke = ops.segment_sum(kinetic[:, None], ptr, None, G)[:, 0]
        ops.md_scr_barostat(cell, ke, zero_w, P0, kT, beta, seeds, step, 1.0, 1.0, mu, pr)
        ops.md_affine_scale(pos, vel, replica, mu)
        if k >= burn:
            V = cell[:, 0, 0].double() * cell[:, 1, 1].double() * cell[:, 2, 2].double()
            s1 += V
            s2 += V * V
    m = float(s1.sum()) / (G * (steps - burn))
    var = float(s2.sum()) / (G * (steps - burn)) - m * m
    print(f"ideal gas: <V> = {m:.4f} (want {N + 1}), Var V = {var:.4f} (want {N + 1})")
    assert abs(m / (N + 1) - 1.0) < 0.005, m
    assert abs(var / (N + 1) - 1.0) < 0.04, var


@pytest.mark.gpu
def test_cuda_graph_replay_of_the_step_equals_eager():
    G, N = 64, 50
    sizes = [N] * G
    replica, ptr = _replica_tensors(sizes, DEV)
    n = G * N
    gen = torch.Generator().manual_seed(7)
    pos0, vel0 = (10.0 * torch.rand(n, 3, generator=gen)).to(DEV), (0.02 * torch.randn(n, 3, generator=gen)).to(DEV)
    force = torch.randn(n, 3, generator=gen).to(DEV)
    inv_m = (1.0 / (103.642697 * (1.0 + 15.0 * torch.rand(n, generator=gen)))).to(DEV)
    cell0, _, vir, P0, kT, beta = _baro_inputs(G, seed=8)
    seeds = torch.arange(G, dtype=torch.int64, device=DEV) + 5
    c1, c2 = math.exp(-0.05), math.sqrt(-math.expm1(-0.1))

    def state():
        return [pos0.clone(), vel0.clone(), cell0.clone(), torch.zeros(1, dtype=torch.int64, device=DEV),
                torch.empty(n, device=DEV), torch.empty(G, device=DEV), torch.empty(G, device=DEV)]

    def one(p, v, c, s, kin, mu, pr):
        ops.md_langevin_baoa(p, v, force, inv_m, replica, ptr, kT, seeds, s, c1, c2, 0.5)
        ops.md_kick(v, force, inv_m, 0.25, kin, s)
        ke = ops.segment_sum(kin[:, None], ptr, None, G)[:, 0]
        ops.md_scr_barostat(c, ke, vir, P0, kT, beta, seeds, s, 0.5, 20.0, mu, pr)
        ops.md_affine_scale(p, v, replica, mu)
    eager_state, eager = state(), []
    for _ in range(3):
        one(*eager_state)
        eager.append([t.clone() for t in eager_state])
    gs = state()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        one(*gs)
    torch.cuda.synchronize()
    assert int(gs[3]) == 0 and torch.equal(gs[2], cell0)            # capture runs nothing
    for k in range(3):
        graph.replay()
        for a, b in zip(gs, eager[k]):
            assert torch.equal(a, b)
    assert not torch.equal(eager[0][2], eager[2][2])                # the cell moved


# ---------------------------------------------------------------------------------------------------------------------
# model level (GPU): HVNet of BASELINE config 1 on the water box, as tests/test_langevin.py
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_zero_compressibility_is_langevin_bitwise():
    model = _water_model()
    pos, Z, cell, batch = _boxes(4, (1, 2))
    v0 = _mb(Z, 300.0, 1)
    kw = dict(temperature_K=[300.0, 500.0], friction_per_fs=0.05, seed=11, batch=batch, device=DEV, skin=0.5)
    s_nvt, s_npt = {}, {}
    p, v, e = md.langevin_device(model, Z, pos, cell, v0, steps=20, stats=s_nvt, **kw)
    p2, v2, c2, e2 = md.langevin_npt_device(model, Z, pos, cell, v0, steps=20, stats=s_npt, compressibility_per_bar=0.0,
                                            pressure_bar=[1.0, 1000.0], **kw)
    assert torch.equal(p, p2) and torch.equal(v, v2) and torch.equal(e, e2)
    assert torch.equal(s_nvt["temperature"], s_npt["temperature"])
    assert (s_nvt["builds"], s_nvt["reuses"]) == (s_npt["builds"], s_npt["reuses"]) and s_npt["reuses"] > 0
    assert torch.equal(c2, torch.from_numpy(cell).to(DEV))
    assert s_npt["pressure"].shape == (20, 2) and s_npt["volume"].shape == (20, 2) and s_npt["virial"].shape == (20, 2, 3, 3)


def _fresh_energy_forces(model, pos, Z, cell):
    d = H.Data(pos=pos.detach().requires_grad_(True), atomic_number=torch.as_tensor(Z).long().to(pos.device),
               cell=cell.reshape(-1, 3, 3))
    e = model(d)
    (g,) = torch.autograd.grad(e.sum(), d.pos)
    return e.detach(), -g


@pytest.mark.gpu
def test_deforming_skin_list_reuse_and_parity():
    model = _water_model()                                          # rc 5, skin 0.5: re-use needs sigma_min > 5 / 5.5
    pos, Z, cell = synthetic.water_box(5, seed=3)
    Zt = torch.as_tensor(Z).long().to(DEV)
    p0, c0 = torch.from_numpy(pos).float().to(DEV), torch.from_numpy(cell).float().reshape(1, 3, 3).to(DEV)
    for s, reused in ((0.97, True), (0.90, False)):
        vg = md.VerletGraph(model, 0.5, deforming=True)
        vg.get(p0, Zt, c0)
        p1, c1 = p0 * s, c0 * s
        g = vg.get(p1, Zt, c1)
        assert (vg.builds, vg.reuses) == ((1, 1) if reused else (2, 0))
        d = H.Data(pos=p1.clone().requires_grad_(True), atomic_number=Zt, cell=c1)
        d.graph = g
        e = model(d)
        (gr,) = torch.autograd.grad(e.sum(), d.pos)
        e_ref, f_ref = _fresh_energy_forces(model, p1, Z, c1)
        assert util.rel_err(e.detach(), e_ref) < 1e-5
        assert float((-gr - f_ref).abs().max()) < 1e-5 * max(1.0, float(f_ref.abs().max()))
    # a whole run: deforming re-use against fresh lists every step
    v0 = _mb(Z, 300.0, 5)
    kw = dict(temperature_K=300.0, pressure_bar=20000.0, compressibility_per_bar=4.5e-5, tau_p_fs=100.0, friction_per_fs=0.02,
              seed=3, device=DEV)
    runs = {}
    for skin in (0.0, 0.5):
        st = {}
        runs[skin] = md.langevin_npt_device(model, Z, pos, cell, v0, steps=30, skin=skin, stats=st, **kw) + (st,)
    (pa, va, ca, ea, sa), (pb, vb, cb, eb, sb) = runs[0.0], runs[0.5]
    assert sb["reuses"] > 0 and sa["builds"] == 31
    assert float((cb - torch.from_numpy(cell).to(DEV)).abs().max()) > 1e-3          # the cell did change
    assert float((pb - pa).abs().max()) < 1e-4 and float((cb - ca).abs().max()) < 1e-4
    assert util.rel_err(eb, ea) < 1e-5


@pytest.mark.gpu
def test_cuda_graph_matches_eager_while_the_cell_changes():
    model = _water_model()
    pos, Z, cell, batch = _boxes(4, (5, 6))
    v0 = _mb(Z, 300.0, 3)
    kw = dict(batch=batch, temperature_K=[300.0, 600.0], pressure_bar=[5000.0, -5000.0], tau_p_fs=100.0, device=DEV, skin=0.8)
    runs = {}
    for cg in (False, True):
        st = {}
        runs[cg] = md.langevin_npt_device(model, Z, pos, cell, v0, steps=12, stats=st, cuda_graph=cg, **kw) + (st,)
    (p0, v0_, c0, e0, s0), (p1, v1, c1, e1, s1) = runs[False], runs[True]
    assert s1["builds"] == s0["builds"] and s1["reuses"] > 0
    assert not torch.equal(c1, torch.from_numpy(cell).to(DEV))
    assert torch.equal(p1, p0) and torch.equal(v1, v0_) and torch.equal(c1, c0) and torch.equal(e1, e0)
    assert torch.equal(s1["pressure"], s0["pressure"])


@pytest.mark.gpu
def test_restart_is_bitwise_and_a_lone_replica_matches_the_batch():
    model = _water_model()
    pos, Z, cell, batch = _boxes(4, (7, 8))
    v0 = _mb(Z, 300.0, 2)
    kw = dict(batch=batch, temperature_K=[350.0, 400.0], pressure_bar=[1000.0, 3000.0], tau_p_fs=200.0, friction_per_fs=0.05,
              seed=2 ** 40 + 1, device=DEV)
    st = {}
    p12, v12, c12, e12 = md.langevin_npt_device(model, Z, pos, cell, v0, steps=12, stats=st, **kw)
    st7 = {}
    p7, v7, c7, e7 = md.langevin_npt_device(model, Z, pos, cell, v0, steps=7, stats=st7, **kw)
    p5, v5, c5, e5 = md.langevin_npt_device(model, Z, p7, c7, v7, steps=5, step0=st7["step"], forces=st7["forces"], **kw)
    assert st["step"] == 12 and st7["step"] == 7
    assert torch.equal(p5, p12) and torch.equal(v5, v12) and torch.equal(c5, c12) and torch.equal(torch.cat([e7, e5]), e12)
    # replica 1 alone (seed + 1)
    n1 = len(Z) // 2
    sl = slice(n1, 2 * n1)
    p1, _, c1, e1 = md.langevin_npt_device(model, Z[sl], pos[sl], cell[1], v0[sl], steps=12, temperature_K=400.0,
                                           pressure_bar=3000.0, tau_p_fs=200.0, friction_per_fs=0.05, seed=2 ** 40 + 2, device=DEV)
    assert float((p1 - p12[sl]).abs().max()) < 1e-5
    assert float((c1[0] - c12[1]).abs().max()) < 1e-5
    assert util.rel_err(e1[:, 0], e12[:, 1]) < 1e-5


@pytest.mark.gpu
def test_pressure_drives_the_volume_and_the_trace_is_consistent():
    model = _water_model()
    pos, Z, cell, batch = _boxes(4, (9, 9))                          # two copies of the same box
    v0 = _mb(Z, 300.0, 4)
    v0 = np.concatenate([v0[: len(Z) // 2]] * 2)
    base = dict(batch=batch, temperature_K=300.0, friction_per_fs=0.05, seed=[21, 21], device=DEV)
    st = {}
    p, v, c, e = md.langevin_npt_device(model, Z, pos, cell, v0, steps=20, compressibility_per_bar=0.0, stats=st, **base)
    P = st["pressure"].double()
    P_start, spread = float(P[:, 0].mean()), float(P[:, 0].std())
    delta = max(10.0 * spread, 5000.0)
    st = {}
    p, v, c, e = md.langevin_npt_device(model, Z, pos, cell, v0, steps=40, pressure_bar=[P_start + delta, P_start - delta],
                                        tau_p_fs=100.0, stats=st, **base)
    V0 = abs(float(np.linalg.det(cell[0].astype(np.float64))))
    vol = st["volume"].double()
    assert float(vol[-1, 0]) < V0 < float(vol[-1, 1]), (V0, vol[-1])
    # P = (2K + tr W) / 3V from the traces: K from the temperature, V of the cell before the step
    n1 = len(Z) // 2
    K = st["temperature"].double() * 1.5 * n1 * md.KB_EV
    V_pre = torch.cat([torch.full((1, 2), V0, dtype=torch.float64, device=DEV), vol[:-1]])
    trW = st["virial"].double().diagonal(dim1=2, dim2=3).sum(-1)
    P_ref = (2.0 * K + trW) / (3.0 * V_pre) * md.EV_A3_TO_BAR
    assert float((st["pressure"].double() - P_ref).abs().max()) <= 1e-5 * float(P_ref.abs().max()) + 1e-3
    # and tr W against energy_forces_virial at the returned state of a one-step run without cell motion
    st1 = {}
    p1, v1, c1, _ = md.langevin_npt_device(model, Z, pos, cell, v0, steps=1, compressibility_per_bar=0.0, stats=st1, **base)
    out = model.energy_forces_virial(H.Data(pos=p1, atomic_number=torch.from_numpy(Z).to(DEV), cell=c1,
                                            batch=torch.from_numpy(batch).to(DEV)))
    ke = 0.5 * (v1.double() ** 2).sum(1) / md._inv_mass(Z, DEV).double()
    K1 = ke.view(2, n1).sum(1)
    P1 = (2.0 * K1 + out["virial"].double().diagonal(dim1=1, dim2=2).sum(-1)) / (3.0 * V0) * md.EV_A3_TO_BAR
    assert float((st1["pressure"][0].double() - P1).abs().max()) <= 1e-5 * float(P1.abs().max()) + 1e-3


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the driver over the kernel emulator with the float64 stand-ins
# ---------------------------------------------------------------------------------------------------------------------
def test_emulated_stats_restart_and_zero_compressibility(emu_npt):
    model = _cpu_model()
    pos, Z, cell, batch = _cpu_systems((22, 23))
    n1 = len(Z) // 2
    vel = 0.002 * np.random.default_rng(1).standard_normal(pos.shape).astype(np.float32)
    kw = dict(temperature_K=[300.0, 900.0], pressure_bar=[2e4, -2e4], tau_p_fs=50.0, friction_per_fs=0.05, seed=5,
              batch=batch, device="cpu")
    st = {}
    p, v, c, e = md.langevin_npt_device(model, Z, pos, cell, vel, steps=6, stats=st, skin=0.5, **kw)
    assert p.shape == (2 * n1, 3) and v.shape == (2 * n1, 3) and c.shape == (2, 3, 3) and e.shape == (6, 2)
    assert st["temperature"].shape == st["pressure"].shape == st["volume"].shape == (6, 2)
    assert st["virial"].shape == (6, 2, 3, 3) and st["step"] == 6
    assert st["builds"] + st["reuses"] == 7 and st["reuses"] > 0
    assert not torch.equal(c, torch.from_numpy(cell))
    assert util.rel_err(st["volume"][-1].double(), torch.linalg.det(c.double()).abs()) < 1e-6
    # cuda_graph (which evaluates eagerly on CPU tensors): the same run, bitwise
    st_g = {}
    out_g = md.langevin_npt_device(model, Z, pos, cell, vel, steps=6, stats=st_g, skin=0.5, cuda_graph=True, **kw)
    assert all(torch.equal(a, b) for a, b in zip(out_g, (p, v, c, e)))
    assert st_g.keys() == st.keys()
    assert all(torch.equal(st_g[k], st[k]) if isinstance(st[k], torch.Tensor) else st_g[k] == st[k] for k in st)
    # restart: 4 + 2 steps equal 6 steps (fresh lists every step)
    p6, v6, c6, e6 = md.langevin_npt_device(model, Z, pos, cell, vel, steps=6, **kw)
    st4 = {}
    p4, v4, c4, e4 = md.langevin_npt_device(model, Z, pos, cell, vel, steps=4, stats=st4, **kw)
    p2, v2, c2, e2 = md.langevin_npt_device(model, Z, p4, c4, v4, steps=2, step0=st4["step"], forces=st4["forces"], **kw)
    assert torch.equal(p2, p6) and torch.equal(v2, v6) and torch.equal(c2, c6) and torch.equal(torch.cat([e4, e2]), e6)
    # zero compressibility: langevin_device's trajectory and list counts, the cell untouched
    kw_nvt = dict(temperature_K=kw["temperature_K"], friction_per_fs=0.05, seed=5, batch=batch, device="cpu", skin=0.5)
    s_nvt, s_npt = {}, {}
    pa, va, ea = md.langevin_device(model, Z, pos, cell, vel, steps=5, stats=s_nvt, **kw_nvt)
    pb, vb, cb, eb = md.langevin_npt_device(model, Z, pos, cell, vel, steps=5, stats=s_npt, compressibility_per_bar=0.0,
                                            pressure_bar=[1.0, 5e3], **kw_nvt)
    assert torch.equal(pa, pb) and torch.equal(va, vb) and torch.equal(ea, eb) and torch.equal(cb, torch.from_numpy(cell))
    assert (s_nvt["builds"], s_nvt["reuses"]) == (s_npt["builds"], s_npt["reuses"])
    assert torch.equal(s_nvt["temperature"], s_npt["temperature"])


def test_emulated_deforming_skin_criterion(emu):
    model = _cpu_model()                                            # rc 3.5, skin 0.5: re-use needs sigma_min > 3.5 / 4
    pos, Z, cell, _ = _cpu_systems((24,))
    Zt = torch.from_numpy(Z).long()
    p0, c0 = torch.from_numpy(pos), torch.from_numpy(cell).reshape(1, 3, 3)

    def counts(p1, c1, deforming=True):
        vg = md.VerletGraph(model, 0.5, deforming=deforming)
        vg.get(p0, Zt, c0)
        g = vg.get(p1, Zt, c1)
        return (vg.builds, vg.reuses), g
    assert counts(p0 * 0.97, c0 * 0.97)[0] == (1, 1)
    assert counts(p0 * 0.85, c0 * 0.85)[0] == (2, 0)
    assert counts(p0 * 0.97, c0 * 0.97, deforming=False)[0] == (2, 0)   # the default still rebuilds on any cell change
    # anisotropic strain: sigma_min = 0.99 -> 4 * 0.99 - 2 max|u| > 3.5 while max|u| < 0.23
    M = torch.diag(torch.tensor([1.0, 0.99, 1.0]))
    for du, reused in ((0.2, True), (0.25, False)):
        p1 = p0 @ M
        p1[3, 0] += du
        assert counts(p1, c0 @ M)[0] == ((1, 1) if reused else (2, 0))
    # a shear and a re-used list give the fresh list's energy
    S = torch.tensor([[1.0, 0.02, 0.0], [0.0, 1.0, 0.0], [0.0, -0.01, 1.0]])
    (nb, g) = counts(p0 @ S, c0 @ S)
    assert nb == (1, 1)
    d = H.Data(pos=(p0 @ S).clone(), atomic_number=Zt, cell=c0 @ S)
    d.graph = g
    d2 = H.Data(pos=(p0 @ S).clone(), atomic_number=Zt, cell=c0 @ S)
    assert util.rel_err(model(d), model(d2)) < 1e-6


def test_sigma_min_closed_form():
    rng = np.random.default_rng(0)
    M = rng.normal(size=(500, 3, 3))
    M[:3] = 0.97 * np.eye(3)
    M[3] = np.diag([1.0, 1.0, 0.9])
    got = md._sigma_min3(torch.from_numpy(M)).numpy()
    assert np.abs(got - np.linalg.svd(M, compute_uv=False)[:, -1]).max() < 1e-9
    assert np.array_equal(got[:3], np.full(3, 0.97))


@pytest.mark.parametrize("bad", [
    dict(cell=None), dict(cell=np.diag([10.0, 10.0, 0.0])), dict(cell=np.full((3, 3), np.nan)),
    dict(compressibility_per_bar=-1e-5), dict(compressibility_per_bar=[1e-5, 1e-5]), dict(tau_p_fs=0.0), dict(tau_p_fs=-5.0),
    dict(pressure_bar=float("inf")), dict(pressure_bar=float("nan")), dict(pressure_bar=[1.0, 2.0]),
    dict(batch=[0, 0, 1, 0]), dict(temperature_K=-1.0), dict(friction_per_fs=-0.1), dict(dt_fs=0.0), dict(seed=-1),
    dict(step0=-1), dict(forces=np.zeros((3, 3)))])
def test_validation_errors(bad):
    args = dict(cell=10.0 * np.eye(3), temperature_K=300.0, pressure_bar=1.0, compressibility_per_bar=4.5e-5, tau_p_fs=1000.0,
                friction_per_fs=0.01, dt_fs=0.5, seed=0, step0=0, batch=None)
    args.update(bad)
    cell = args.pop("cell")
    with pytest.raises(ValueError):
        md.langevin_npt_device(None, [8, 1, 1, 8], np.zeros((4, 3)), cell, np.zeros((4, 3)), steps=1, device="cpu", **args)
