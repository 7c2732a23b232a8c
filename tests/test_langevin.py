"""Langevin (NVT) MD on the device: ``hn_md_langevin_baoa`` / ``hn_md_kick`` (``ops.md_langevin_baoa`` / ``ops.md_kick``)
and ``plugin.md.langevin_device``.

The oracle is a numpy Philox4x32-10 and Box-Muller in float64 that follows the noise recipe of include/hermnet_b200.h; the
same reference, applied in float64, stands in for the two ops in the CPU cases over the kernel emulator."""
import math

import numpy as np
import pytest
import torch

import hermnet_b200 as H
from hermnet_b200 import ops, synthetic
from hermnet_b200.plugin import md
from tests import util
from tests.test_atom_virial import _emu_edge_virial_atom
from tests.util import lattice_system

DEV = "cuda:0"
MASK32 = np.uint64(0xFFFFFFFF)


# ---------------------------------------------------------------------------------------------------------------------
# numpy reference of the noise and of the two ops
# ---------------------------------------------------------------------------------------------------------------------
def philox4x32_10(ctr, key):
    """Philox4x32-10 (Random123) on uint32 ``ctr [...,4]``, ``key [...,2]`` -> uint32 ``[...,4]``."""
    c = [np.asarray(ctr[..., k], dtype=np.uint64) for k in range(4)]
    k0, k1 = np.asarray(key[..., 0], dtype=np.uint64), np.asarray(key[..., 1], dtype=np.uint64)
    for r in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & MASK32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & MASK32]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & MASK32, (k1 + np.uint64(0xBB67AE85)) & MASK32
    return np.stack(c, -1).astype(np.uint32)


def ref_uniforms(seeds, local, step):
    """``u [n,4]`` (float64, exact fp32 values) of atoms with replica seeds ``seeds [n]`` and local indices ``local [n]``."""
    seeds = np.asarray(seeds, dtype=np.int64).view(np.uint64)
    n = len(local)
    ctr = np.stack([np.asarray(local, dtype=np.uint64), np.full(n, step & 0xFFFFFFFF, np.uint64),
                    np.full(n, step >> 32, np.uint64), np.zeros(n, np.uint64)], -1)
    key = np.stack([seeds & MASK32, seeds >> np.uint64(32)], -1)
    r = philox4x32_10(ctr, key).astype(np.uint64)
    return ((r >> np.uint64(9)) * np.uint64(2) + np.uint64(1)).astype(np.float64) * 2.0 ** -24


def ref_xi(u):
    """float64 Box-Muller ``[n,3]`` of the uniforms."""
    a, b = np.sqrt(-2.0 * np.log(u[:, 0])), np.sqrt(-2.0 * np.log(u[:, 2]))
    return np.stack([a * np.cos(2 * np.pi * u[:, 1]), a * np.sin(2 * np.pi * u[:, 1]), b * np.cos(2 * np.pi * u[:, 3])], -1)


def _np(t):
    return t.detach().cpu().numpy()


def ref_noise(replica, replica_ptr, seed, step):
    rep, ptr = _np(replica).astype(np.int64), _np(replica_ptr).astype(np.int64)
    local = np.arange(len(rep)) - ptr[rep]
    return ref_xi(ref_uniforms(_np(seed)[rep], local, int(step)))


def ref_baoa(pos, vel, force, inv_mass, replica, kT, xi, c1, c2, dt):
    """float64 B-A-O-A of the same formulas."""
    x, v, f = (_np(t).astype(np.float64) for t in (pos, vel, force))
    im = _np(inv_mass).astype(np.float64).reshape(-1, 1)
    sig = c2 * np.sqrt(_np(kT).astype(np.float64)[_np(replica).astype(np.int64)][:, None] * im)
    v = v + 0.5 * dt * f * im
    x = x + 0.5 * dt * v
    v = c1 * v + sig * xi
    return x + 0.5 * dt * v, v


def emu_md_langevin_baoa(pos, vel, force, inv_mass, replica, replica_ptr, kT, seed, step, c1, c2, dt):
    """CPU stand-in of ``ops.md_langevin_baoa`` (float64 reference, same contract)."""
    xi = ref_noise(replica, replica_ptr, seed, int(step[0]))
    x, v = ref_baoa(pos, vel, force, inv_mass, replica, kT, xi, c1, c2, dt)
    pos.copy_(torch.from_numpy(x))
    vel.copy_(torch.from_numpy(v))


def emu_md_kick(vel, force, inv_mass, half_dt, kinetic, step):
    """CPU stand-in of ``ops.md_kick``."""
    im = inv_mass.double().reshape(-1, 1)
    vel.copy_(vel.double() + half_dt * force.double() * im)
    if kinetic is not None:
        kinetic.copy_(0.5 * (vel.double() ** 2).sum(1) / im[:, 0])
    step += 1


@pytest.fixture
def emu_md(emu, monkeypatch):
    monkeypatch.setattr(ops, "md_langevin_baoa", emu_md_langevin_baoa)
    monkeypatch.setattr(ops, "md_kick", emu_md_kick)
    monkeypatch.setattr(ops, "edge_virial_atom", _emu_edge_virial_atom)
    return emu


def _replica_tensors(sizes, dev):
    ptr = np.concatenate([[0], np.cumsum(sizes)])
    rep = np.repeat(np.arange(len(sizes)), sizes)
    return torch.from_numpy(rep).to(dev, torch.int32), torch.from_numpy(ptr).to(dev, torch.int32)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference itself
# ---------------------------------------------------------------------------------------------------------------------
def test_numpy_philox_reproduces_random123_known_answers():
    cases = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
             ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
             ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
              (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in cases:
        got = philox4x32_10(np.array([ctr], np.uint64), np.array([key], np.uint64))[0]
        assert tuple(int(x) for x in got) == want


def test_reference_uniforms_are_exact_and_open():
    u = ref_uniforms(np.full(4096, 2 ** 40 + 3), np.arange(4096), 2 ** 33 + 1)
    assert np.array_equal(u.astype(np.float32).astype(np.float64), u)
    assert u.min() >= 2.0 ** -24 and u.max() <= 1.0 - 2.0 ** -24
    assert np.abs(ref_xi(u)).max() <= math.sqrt(-2 * math.log(2.0 ** -24))


# ---------------------------------------------------------------------------------------------------------------------
# kernel level (GPU)
# ---------------------------------------------------------------------------------------------------------------------
def _kernel_inputs(sizes, seed=0, kTs=None):
    gen = torch.Generator().manual_seed(seed)
    n = int(sum(sizes))
    rn = lambda *s: torch.randn(*s, generator=gen)
    pos = (10.0 * rn(n, 3)).to(DEV)
    vel = (0.02 * rn(n, 3)).to(DEV)
    force = rn(n, 3).to(DEV)
    inv_m = (1.0 / (103.642697 * (1.0 + 30.0 * torch.rand(n, generator=gen)))).to(DEV)
    replica, ptr = _replica_tensors(sizes, DEV)
    kT = torch.tensor(kTs if kTs is not None else [0.0258 * (1 + g) for g in range(len(sizes))], device=DEV)
    return pos, vel, force, inv_m, replica, ptr, kT


@pytest.mark.gpu
def test_noise_matches_the_recipe():
    sizes = [40_000, 1, 60_002]                               # N = 100 003: not a block multiple
    n = sum(sizes)
    replica, ptr = _replica_tensors(sizes, DEV)
    seed = torch.tensor([7, 2 ** 32 + 12345, 2 ** 62 + 99], dtype=torch.int64, device=DEV)
    for s in (0, 3, 2 ** 32 + 5):
        step = torch.tensor([s], dtype=torch.int64, device=DEV)
        pos, vel = torch.zeros(n, 3, device=DEV), torch.full((n, 3), 3.0, device=DEV)
        ops.md_langevin_baoa(pos, vel, torch.zeros(n, 3, device=DEV), torch.ones(n, device=DEV), replica, ptr,
                             torch.ones(3, device=DEV), seed, step, 0.0, 1.0, 0.5)
        ref = ref_noise(replica, ptr, seed, s)
        assert np.abs(_np(vel).astype(np.float64) - ref).max() <= 4e-6
        assert int(step) == s


@pytest.mark.gpu
@pytest.mark.parametrize("gdt", [0.0, 0.01, 1.0])
def test_baoa_and_kick_match_float64(gdt):
    sizes = [3000, 517, 12_000]
    pos, vel, force, inv_m, replica, ptr, kT = _kernel_inputs(sizes, seed=1)
    seed = torch.tensor([1, 2, 3], dtype=torch.int64, device=DEV)
    step = torch.tensor([41], dtype=torch.int64, device=DEV)
    dt = 0.5
    c1, c2 = math.exp(-gdt), math.sqrt(-math.expm1(-2 * gdt))
    xi = ref_noise(replica, ptr, seed, 41)
    x_ref, v_ref = ref_baoa(pos, vel, force, inv_m, replica, kT, xi, c1, c2, dt)
    bound_x = 1e-6 * (np.abs(_np(pos)).max() + dt * np.abs(v_ref).max())
    ops.md_langevin_baoa(pos, vel, force, inv_m, replica, ptr, kT, seed, step, c1, c2, dt)
    assert int(step) == 41
    assert np.abs(_np(pos) - x_ref).max() <= bound_x
    assert np.abs(_np(vel) - v_ref).max() <= 2e-6 * np.abs(v_ref).max()
    # closing kick against float64 from the same inputs
    force2 = torch.randn(pos.shape, generator=torch.Generator().manual_seed(5)).to(DEV)
    v_in = _np(vel).astype(np.float64)
    v_ref2 = v_in + 0.5 * dt * _np(force2) * _np(inv_m)[:, None]
    kinetic = torch.empty(sum(sizes), device=DEV)
    ops.md_kick(vel, force2, inv_m, 0.5 * dt, kinetic, step)
    assert int(step) == 42
    assert np.abs(_np(vel) - v_ref2).max() <= 2e-6 * np.abs(v_ref2).max()
    ke_ref = 0.5 * (_np(vel).astype(np.float64) ** 2).sum(1) / _np(inv_m).astype(np.float64)
    assert np.abs(_np(kinetic) - ke_ref).max() <= 1e-6 * ke_ref.max()
    assert (np.abs(_np(kinetic) - ke_ref) <= 1e-6 * ke_ref + 1e-30).all()
    ops.md_kick(vel, force2, inv_m, 0.5 * dt, None, step)
    assert int(step) == 43


@pytest.mark.gpu
def test_determinism_replica_independence_and_decorrelation():
    sizes = [7000, 33_001, 15_000]
    inp = _kernel_inputs(sizes, seed=2)
    seed = torch.tensor([11, 2 ** 33, 5], dtype=torch.int64, device=DEV)
    c1, c2 = math.exp(-0.3), math.sqrt(-math.expm1(-0.6))

    def run(pos, vel, force, inv_m, replica, ptr, kT, sd, s):
        pos, vel = pos.clone(), vel.clone()
        step = torch.tensor([s], dtype=torch.int64, device=DEV)
        ops.md_langevin_baoa(pos, vel, force, inv_m, replica, ptr, kT, sd, step, c1, c2, 0.5)
        return pos, vel
    a, b = run(*inp, seed, 9), run(*inp, seed, 9)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    pos, vel, force, inv_m, replica, ptr, kT = inp
    lo, hi = sizes[0], sizes[0] + sizes[1]                 # replica 1 alone
    alone = run(pos[lo:hi], vel[lo:hi], force[lo:hi], inv_m[lo:hi], torch.zeros(hi - lo, dtype=torch.int32, device=DEV),
                torch.tensor([0, hi - lo], dtype=torch.int32, device=DEV), kT[1:2], seed[1:2], 9)
    assert torch.equal(alone[0], a[0][lo:hi]) and torch.equal(alone[1], a[1][lo:hi])
    # consecutive steps draw uncorrelated noise (c1 = 0, unit variance: v_out = xi)
    n = sum(sizes)
    xs = []
    for s in (9, 10):
        v = torch.zeros(n, 3, device=DEV)
        ops.md_langevin_baoa(torch.zeros(n, 3, device=DEV), v, torch.zeros(n, 3, device=DEV), torch.ones(n, device=DEV), replica,
                             ptr, torch.ones(3, device=DEV), seed, torch.tensor([s], dtype=torch.int64, device=DEV), 0.0, 1.0, 0.5)
        xs.append(_np(v).astype(np.float64).reshape(-1))
    rho = np.corrcoef(xs[0], xs[1])[0, 1]
    assert abs(rho) < 5 / math.sqrt(3 * n)


@pytest.mark.gpu
def test_ornstein_uhlenbeck_variance_of_free_particles():
    sizes = [500_000, 500_000]
    n = sum(sizes)
    replica, ptr = _replica_tensors(sizes, DEV)
    T = np.array([300.0, 1000.0])
    kT = torch.tensor(md.KB_EV * T, dtype=torch.float32, device=DEV)
    inv_m = (1.0 / (103.642697 * (1.0 + 15.0 * torch.rand(n, generator=torch.Generator().manual_seed(3))))).to(DEV)
    pos, vel, zero = torch.zeros(n, 3, device=DEV), torch.zeros(n, 3, device=DEV), torch.zeros(n, 3, device=DEV)
    seed = torch.tensor([123, 456], dtype=torch.int64, device=DEV)
    step = torch.zeros(1, dtype=torch.int64, device=DEV)
    gdt, steps = 0.05, 40
    c1, c2 = math.exp(-gdt), math.sqrt(-math.expm1(-2 * gdt))
    for _ in range(steps):
        ops.md_langevin_baoa(pos, vel, zero, inv_m, replica, ptr, kT, seed, step, c1, c2, 0.5)
        ops.md_kick(vel, zero, inv_m, 0.25, None, step)
    assert int(step) == steps
    want = 1.0 - c1 ** (2 * steps)
    z = _np(vel).astype(np.float64) / np.sqrt(_np(kT).astype(np.float64)[_np(replica)][:, None] * _np(inv_m)[:, None])
    for g in range(2):
        zg = z[_np(ptr)[g]:_np(ptr)[g + 1]]
        var = (zg ** 2).mean(0)
        assert (np.abs(var / want - 1.0) < 5 * math.sqrt(2.0 / len(zg))).all(), (g, var, want)


@pytest.mark.gpu
def test_empty_launch_and_cuda_graph_capture():
    e = torch.zeros(0, 3, device=DEV)
    step = torch.tensor([4], dtype=torch.int64, device=DEV)
    r0, p0 = torch.zeros(0, dtype=torch.int32, device=DEV), torch.tensor([0, 0], dtype=torch.int32, device=DEV)
    ops.md_langevin_baoa(e, e.clone(), e, torch.zeros(0, device=DEV), r0, p0, torch.ones(1, device=DEV),
                         torch.zeros(1, dtype=torch.int64, device=DEV), step, 0.5, 0.5, 0.5)
    ops.md_kick(e.clone(), e, torch.zeros(0, device=DEV), 0.25, torch.zeros(0, device=DEV), step)
    assert int(step) == 4

    sizes = [3000, 2000]
    pos, vel, force, inv_m, replica, ptr, kT = _kernel_inputs(sizes, seed=4)
    seed = torch.tensor([8, 9], dtype=torch.int64, device=DEV)
    c1, c2 = math.exp(-0.1), math.sqrt(-math.expm1(-0.2))
    kin = torch.empty(sum(sizes), device=DEV)

    def one(p, v, s, k):
        ops.md_langevin_baoa(p, v, force, inv_m, replica, ptr, kT, seed, s, c1, c2, 0.5)
        ops.md_kick(v, force, inv_m, 0.25, k, s)
    pe, ve, se, ke = pos.clone(), vel.clone(), torch.zeros(1, dtype=torch.int64, device=DEV), kin.clone()
    eager = []
    for _ in range(3):
        one(pe, ve, se, ke)
        eager.append((pe.clone(), ve.clone(), ke.clone()))
    pg, vg_, sg, kg = pos.clone(), vel.clone(), torch.zeros(1, dtype=torch.int64, device=DEV), kin.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        one(pg, vg_, sg, kg)
    torch.cuda.synchronize()
    assert int(sg) == 0 and torch.equal(pg, pos)          # capture runs nothing
    for k in range(3):
        graph.replay()
        assert torch.equal(pg, eager[k][0]) and torch.equal(vg_, eager[k][1]) and torch.equal(kg, eager[k][2])
    assert int(sg) == 3
    assert not torch.equal(eager[1][1] - c1 * eager[0][1], eager[2][1] - c1 * eager[1][1])


# ---------------------------------------------------------------------------------------------------------------------
# model level (GPU): HVNet of BASELINE config 1 on the water box, readout scaled as bench.py C3 does
# ---------------------------------------------------------------------------------------------------------------------
def _water_model(dev=DEV):
    cfg = dict(synthetic.config("C1")[1])
    cfg.pop("kind")
    torch.manual_seed(1234)
    model = H.HVNet(**cfg).to(dev).eval()
    for q in model.parameters():
        q.requires_grad_(False)
    model.out_energy[2].weight.mul_(1.0e-3)
    model.out_energy[2].bias.mul_(1.0e-3)
    return model


def _boxes(n_side, seeds):
    parts = [synthetic.water_box(n_side, seed=s) for s in seeds]
    pos = np.concatenate([p for p, _, _ in parts])
    Z = np.concatenate([z for _, z, _ in parts])
    cell = np.stack([c for _, _, c in parts])
    batch = np.repeat(np.arange(len(seeds)), [len(z) for _, z, _ in parts])
    return pos, Z, cell, batch


def _mb(Z, T, seed):
    atoms = md.SimpleAtoms(Z, np.zeros((len(Z), 3)))
    md.maxwell_boltzmann(atoms, T, seed=seed)
    return atoms.velocities.astype(np.float32)


@pytest.mark.gpu
def test_zero_friction_is_velocity_verlet():
    model = _water_model()
    pos, Z, cell = synthetic.water_box(4, seed=0)
    v0 = _mb(Z, 300.0, 1)
    p_nve, v_nve, e_nve = md.velocity_verlet_device(model, Z, pos, cell, v0, steps=8, device=DEV)
    st = {}
    p, v, e = md.langevin_device(model, Z, pos, cell, v0, steps=8, friction_per_fs=0.0, device=DEV, stats=st)
    assert e.shape == (8, 1) and st["step"] == 8 and st["temperature"].shape == (8, 1)
    assert float((p - p_nve).abs().max()) < 1e-5
    assert util.rel_err(e[:, 0], e_nve) < 1e-5


THERMO = dict(temperature_K=[200.0, 300.0, 500.0, 800.0], friction_per_fs=0.1, dt_fs=0.5, seed=17, skin=0.5)


@pytest.mark.gpu
def test_batched_replicas_thermalise_and_match_a_lone_replica():
    model = _water_model()
    pos, Z, cell, batch = _boxes(6, (1, 2, 3, 4))
    n1 = len(Z) // 4
    st = {}
    p, v, e = md.langevin_device(model, Z, pos, cell, np.zeros_like(pos), steps=400, batch=batch, device=DEV, stats=st, **THERMO)
    assert e.shape == (400, 4) and st["temperature"].shape == (400, 4) and st["step"] == 400
    assert st["builds"] > 1 and st["reuses"] > st["builds"]
    T_mean = st["temperature"][100:].double().mean(0).cpu().numpy()
    assert (np.abs(T_mean / np.array(THERMO["temperature_K"]) - 1.0) < 0.04).all(), T_mean
    # the last row is 2 KE / (3 n k_B) of the returned velocities
    ke = 0.5 * (v.double() ** 2).sum(1) / md._inv_mass(Z, DEV).double()
    T_last = ke.view(4, n1).sum(1) * 2.0 / (3 * n1 * md.KB_EV)
    assert util.rel_err(st["temperature"][-1].double(), T_last) < 1e-6
    # replica 2 alone (seed 17 + 2), 10 steps, against the first 10 steps of the batch
    kw = dict(THERMO, temperature_K=THERMO["temperature_K"][2], seed=THERMO["seed"] + 2)
    sl = slice(2 * n1, 3 * n1)
    p1, _, e1 = md.langevin_device(model, Z[sl], pos[sl], cell[2], np.zeros_like(pos[sl]), steps=10, device=DEV, **kw)
    p10, _, e10 = md.langevin_device(model, Z, pos, cell, np.zeros_like(pos), steps=10, batch=batch, device=DEV, **THERMO)
    assert float((p1 - p10[sl]).abs().max()) < 1e-5
    assert util.rel_err(e1[:, 0], e10[:, 2]) < 1e-5


@pytest.mark.gpu
def test_restart_is_bitwise():
    model = _water_model()
    pos, Z, cell = synthetic.water_box(4, seed=0)
    v0 = _mb(Z, 300.0, 2)
    kw = dict(temperature_K=400.0, friction_per_fs=0.05, seed=2 ** 40 + 1, device=DEV)
    st = {}
    p12, v12, e12 = md.langevin_device(model, Z, pos, cell, v0, steps=12, stats=st, **kw)
    st7 = {}
    p7, v7, e7 = md.langevin_device(model, Z, pos, cell, v0, steps=7, stats=st7, **kw)
    assert st7["step"] == 7 and st["step"] == 12
    p5, v5, e5 = md.langevin_device(model, Z, p7, cell, v7, steps=5, step0=st7["step"], **kw)
    assert torch.equal(p5, p12) and torch.equal(v5, v12) and torch.equal(torch.cat([e7, e5]), e12)


@pytest.mark.gpu
def test_cuda_graph_matches_eager():
    model = _water_model()
    pos, Z, cell, batch = _boxes(4, (5, 6))
    v0 = _mb(Z, 300.0, 3)
    runs = {}
    for cg in (False, True):
        st = {}
        runs[cg] = md.langevin_device(model, Z, pos, cell, v0, steps=10, batch=batch, temperature_K=[300.0, 600.0],
                                      device=DEV, skin=0.8, stats=st, cuda_graph=cg) + (st,)
    (p0, v0_, e0, s0), (p1, v1, e1, s1) = runs[False], runs[True]
    assert s1["builds"] == s0["builds"] and s1["step"] == 10
    assert float((p1 - p0).abs().max()) < 1e-5
    assert float((v1 - v0_).abs().max()) < 1e-5 * max(1.0, float(v0_.abs().max()))
    assert util.rel_err(e1, e0) < 1e-5


@pytest.mark.gpu
def test_virial_trace():
    model = _water_model()
    pos, Z, cell, batch = _boxes(4, (7, 8))
    v0 = _mb(Z, 300.0, 4)
    kw = dict(batch=batch, temperature_K=[300.0, 500.0], friction_per_fs=0.02, device=DEV)
    st = {}
    p, v, e = md.langevin_device(model, Z, pos, cell, v0, steps=3, stats=st, virial=True, **kw)
    assert st["virial"].shape == (3, 2, 3, 3)
    p_plain, v_plain, e_plain = md.langevin_device(model, Z, pos, cell, v0, steps=3, **kw)
    assert torch.equal(p, p_plain) and torch.equal(v, v_plain) and torch.equal(e, e_plain)
    c = torch.from_numpy(cell).to(DEV)
    b = torch.from_numpy(batch).to(DEV)
    Zt = torch.from_numpy(Z).to(DEV)
    for k in range(1, 4):
        pk, _, _ = md.langevin_device(model, Z, pos, cell, v0, steps=k, **kw)
        ref = model.energy_forces_virial(H.Data(pos=pk, atomic_number=Zt, cell=c, batch=b))["virial"]
        assert torch.allclose(st["virial"][k - 1], ref, rtol=0, atol=1e-6 * max(1.0, float(ref.abs().max())))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the driver over the kernel emulator with the float64 stand-ins
# ---------------------------------------------------------------------------------------------------------------------
def _cpu_model():
    torch.manual_seed(6)
    model = H.HVNet(elems=["Li", "O"], rc=3.5, num_layers=1, hidden_channels=128, num_rbf=24).eval()
    for q in model.parameters():
        q.requires_grad_(False)
    return model


def _cpu_systems(seeds):
    parts = [lattice_system(4, [3, 8], s, a=2.6) for s in seeds]
    pos = torch.cat([p for p, _, _ in parts]).numpy()
    Z = torch.cat([z for _, z, _ in parts]).numpy()
    cell = torch.cat([c for _, _, c in parts]).numpy()
    batch = np.repeat(np.arange(len(seeds)), [len(z) for _, z, _ in parts])
    return pos, Z, cell, batch


def test_emulated_stats_restart_and_replica_independence(emu_md):
    model = _cpu_model()
    pos, Z, cell, batch = _cpu_systems((22, 23))
    n1 = len(Z) // 2
    vel = 0.002 * np.random.default_rng(1).standard_normal(pos.shape).astype(np.float32)
    kw = dict(temperature_K=[300.0, 900.0], friction_per_fs=0.05, seed=5, batch=batch, device="cpu", skin=0.5)
    st = {}
    p, v, e = md.langevin_device(model, Z, pos, cell, vel, steps=6, stats=st, **kw)
    assert p.shape == (2 * n1, 3) and v.shape == (2 * n1, 3) and e.shape == (6, 2)
    assert st["temperature"].shape == (6, 2) and st["step"] == 6 and "virial" not in st
    assert st["builds"] + st["reuses"] == 7 and st["reuses"] > 0
    assert np.array_equal(vel, 0.002 * np.random.default_rng(1).standard_normal(pos.shape).astype(np.float32))  # input untouched
    ke = 0.5 * (v.double() ** 2).sum(1) / md._inv_mass(Z, "cpu").double()
    assert util.rel_err(st["temperature"][-1].double(), ke.view(2, n1).sum(1) * 2.0 / (3 * n1 * md.KB_EV)) < 1e-6
    # with the virial, eager and cuda_graph (which evaluates eagerly on CPU tensors): the same run, bitwise
    virials = []
    for cg in (False, True):
        st_w = {}
        p_w, v_w, e_w = md.langevin_device(model, Z, pos, cell, vel, steps=6, stats=st_w, virial=True, cuda_graph=cg, **kw)
        assert torch.equal(p_w, p) and torch.equal(v_w, v) and torch.equal(e_w, e)
        assert torch.equal(st_w["temperature"], st["temperature"]) and st_w["virial"].shape == (6, 2, 3, 3)
        assert (st_w["builds"], st_w["reuses"], st_w["step"]) == (st["builds"], st["reuses"], st["step"])
        virials.append(st_w["virial"])
    assert torch.equal(virials[0], virials[1])
    # restart: 4 + 2 steps equal 6 steps (fresh lists every step)
    kw0 = dict(kw, skin=0.0)
    p6, v6, e6 = md.langevin_device(model, Z, pos, cell, vel, steps=6, **kw0)
    st4 = {}
    p4, v4, e4 = md.langevin_device(model, Z, pos, cell, vel, steps=4, stats=st4, **kw0)
    p2, v2, e2 = md.langevin_device(model, Z, p4, cell, v4, steps=2, step0=st4["step"], **kw0)
    assert torch.equal(p2, p6) and torch.equal(v2, v6) and torch.equal(torch.cat([e4, e2]), e6)
    # replica 1 alone with its own seed and temperature
    sl = slice(n1, 2 * n1)
    p1, _, e1 = md.langevin_device(model, Z[sl], pos[sl], cell[1], vel[sl], steps=6, temperature_K=900.0, friction_per_fs=0.05,
                                   seed=6, device="cpu", skin=0.0)
    assert float((p1 - p6[sl]).abs().max()) < 1e-5
    assert util.rel_err(e1[:, 0], e6[:, 1]) < 1e-5
    # a single replica: energies [steps, 1]
    p_s, _, e_s = md.langevin_device(model, Z[:n1], pos[:n1], cell[0], vel[:n1], steps=2, device="cpu")
    assert e_s.shape == (2, 1) and p_s.shape == (n1, 3)


def test_emulated_velocity_verlet_device_unchanged(emu_md):
    """The shared evaluation helper keeps the NVE loop's trajectory: the loop written out as before, bitwise -- also with the
    virial, eager and with ``cuda_graph``."""
    model = _cpu_model()
    pos, Z, cell, _ = _cpu_systems((22,))
    vel = 0.002 * np.random.default_rng(2).standard_normal(pos.shape).astype(np.float32)
    p, v, e = md.velocity_verlet_device(model, Z, pos, cell, vel, steps=4, device="cpu", skin=0.5)
    Zt, c = torch.from_numpy(Z).long(), torch.from_numpy(cell).reshape(1, 3, 3)
    masses = np.array([md.MASSES.get(int(z), 2.0 * int(z)) for z in Z])
    inv_m = torch.as_tensor(1.0 / (masses * md.AMU_A2_FS2_TO_EV), dtype=torch.float32)[:, None]
    vg = md.VerletGraph(model, 0.5)

    def forces(q):
        d = H.Data(pos=q.detach().requires_grad_(True), atomic_number=Zt, cell=c)
        d.graph = vg.get(d.pos, Zt, c)
        en = model(d)
        (g,) = torch.autograd.grad(en.sum(), d.pos)
        return en.detach(), -g
    q, w = torch.from_numpy(pos), torch.from_numpy(vel).clone()
    en, f = forces(q)
    es = []
    for _ in range(4):
        w.add_(f * inv_m, alpha=0.25)
        q = q + 0.5 * w
        en, f = forces(q)
        w.add_(f * inv_m, alpha=0.25)
        es.append(en)
    assert torch.equal(p, q) and torch.equal(v, w) and torch.equal(e, torch.cat(es))
    virials = []
    for cg in (False, True):
        st = {}
        p_w, v_w, e_w = md.velocity_verlet_device(model, Z, pos, cell, vel, steps=4, device="cpu", skin=0.5, stats=st,
                                                  cuda_graph=cg, virial=True)
        assert torch.equal(p_w, q) and torch.equal(v_w, w) and torch.equal(e_w, torch.cat(es))
        assert st["virial"].shape == (4, 3, 3) and (st["builds"], st["reuses"]) == (1, 4)
        virials.append(st["virial"])
    assert torch.equal(virials[0], virials[1])


@pytest.mark.parametrize("bad", [
    dict(batch=[0, 0, 1, 0]), dict(batch=[0, 0, 2, 2]), dict(batch=[1, 1, 1, 1]), dict(batch=[0, 1]),
    dict(temperature_K=[300.0, 400.0]), dict(temperature_K=-1.0), dict(batch=[0, 0, 1, 1], temperature_K=[300.0]),
    dict(friction_per_fs=-0.1), dict(dt_fs=0.0), dict(dt_fs=-0.5), dict(seed=-1), dict(seed=[1, 2]), dict(seed=2 ** 63),
    dict(step0=-1)])
def test_validation_errors(bad):
    args = dict(temperature_K=300.0, friction_per_fs=0.01, dt_fs=0.5, seed=0, step0=0, batch=None)
    args.update(bad)
    with pytest.raises(ValueError):
        md.langevin_device(None, [8, 1, 1, 8], np.zeros((4, 3)), 10.0 * np.eye(3), np.zeros((4, 3)), steps=1, device="cpu", **args)
