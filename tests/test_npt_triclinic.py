"""Constant-pressure MD with the cell shape free: ``hn_md_kinetic_tensor`` / ``hn_md_scr_barostat_tri`` /
``hn_md_affine_deform`` (``ops.md_kinetic_tensor`` / ``ops.md_scr_barostat_tri`` / ``ops.md_affine_deform``),
``plugin.md.langevin_npt_device(cell_dof="triclinic")`` and ``plugin.md.standard_cell``.

The oracle is the numpy Philox4x32-10 of tests/test_langevin.py with the triclinic barostat's counters (word 3 = 2) and the
cell step of include/hermnet_b200.h in float64, with ``scipy.linalg.expm`` for the strain; the same reference stands in for
the three ops in the CPU cases over the kernel emulator.  The stationary-distribution test pins the maths of DESIGN.md
("Triclinic constant pressure") against a float64 quadrature of the target density."""
import math
import re

import numpy as np
import pytest
import scipy.linalg
import torch

import hermnet_b200 as H
from hermnet_b200 import ops
from hermnet_b200.plugin import md
from tests import util
from tests.test_atom_virial import _emu_edge_virial_atom
from tests.test_langevin import (MASK32, _boxes, _cpu_model, _cpu_systems, _mb, _np, _replica_tensors, _water_model,
                                 emu_md_kick, emu_md_langevin_baoa, philox4x32_10, ref_noise)
from tests.test_npt import _fresh_energy_forces, ref_baro_xi

DEV = "cuda:0"
LI, LJ = np.array([0, 1, 1, 2, 2, 2]), np.array([0, 0, 1, 0, 1, 2])         # packed lower triangle (00, 10, 11, 20, 21, 22)


# ---------------------------------------------------------------------------------------------------------------------
# float64 reference of the cell step and of the three ops
# ---------------------------------------------------------------------------------------------------------------------
def ref_tri_xi(seeds, step):
    """The 6 normals ``[G,6]`` of every replica: counters (k, lo32 step, hi32 step, 2) for k = 0, 1, Box-Muller cos then sin
    of (u0, u1) and (u2, u3), the first 6 of the 8."""
    seeds = np.asarray(seeds, dtype=np.int64).view(np.uint64)
    G = len(seeds)
    key = np.stack([seeds & MASK32, seeds >> np.uint64(32)], -1)
    z = []
    for k in range(2):
        ctr = np.stack([np.full(G, k, np.uint64), np.full(G, step & 0xFFFFFFFF, np.uint64), np.full(G, step >> 32, np.uint64),
                        np.full(G, 2, np.uint64)], -1)
        r = philox4x32_10(ctr, key).astype(np.uint64)
        u = ((r >> np.uint64(9)) * np.uint64(2) + np.uint64(1)).astype(np.float64) * 2.0 ** -24
        a, b = np.sqrt(-2.0 * np.log(u[:, 0])), np.sqrt(-2.0 * np.log(u[:, 2]))
        z += [a * np.cos(2 * np.pi * u[:, 1]), a * np.sin(2 * np.pi * u[:, 1]), b * np.cos(2 * np.pi * u[:, 3]),
              b * np.sin(2 * np.pi * u[:, 3])]
    return np.stack(z[:6], -1)


def ref_delta(cell, kin6, virial, P0, kT, beta, seed, step, dt, tau_p):
    """``(delta [G,3,3], P [G,6])`` in float64 from the fp32 inputs: the lower-triangular strain and the packed pressure."""
    h = _np(cell).astype(np.float64).reshape(-1, 3, 3)
    V = h[:, 0, 0] * h[:, 1, 1] * h[:, 2, 2]
    w = _np(virial).astype(np.float64).reshape(-1, 3, 3)
    P = (_np(kin6).astype(np.float64) + w[:, LI, LJ]) / V[:, None]
    b = _np(beta).astype(np.float64) * (float(np.float32(dt)) / float(np.float32(tau_p)))
    bkT3V = b * _np(kT).astype(np.float64) / (3.0 * V)
    d = (b / 3.0)[:, None] * (P - np.where(LI == LJ, 1.0, 0.0)[None] * _np(P0).astype(np.float64)[:, None])
    d += np.sqrt(2.0 * bkT3V)[:, None] * ref_tri_xi(_np(seed), int(step))
    d[:, 0] += 2.0 * bkT3V
    d[:, 5] -= 2.0 * bkT3V
    D = np.zeros_like(h)
    D[:, LI, LJ] = d
    return D, P


def ref_barostat_tri(cell, kin6, virial, P0, kT, beta, seed, step, dt, tau_p):
    """``(mu, mu^-T, pressure tensor, new cell)`` in float64."""
    D, P = ref_delta(cell, kin6, virial, P0, kT, beta, seed, step, dt, tau_p)
    mu = scipy.linalg.expm(D)
    mu_inv_t = np.swapaxes(scipy.linalg.expm(-D), 1, 2)
    pt = np.zeros_like(D)
    pt[:, LI, LJ] = P
    pt[:, LJ, LI] = P
    h = _np(cell).astype(np.float64).reshape(-1, 3, 3)
    return mu, mu_inv_t, pt, np.tril(h @ mu)


def emu_md_kinetic_tensor(vel, inv_mass):
    """CPU stand-in of ``ops.md_kinetic_tensor``."""
    v = vel.double()
    return (v[:, LI] * v[:, LJ] / inv_mass.double()[:, None]).float()


def emu_md_scr_barostat_tri(cell, kin6, virial, P0, kT, beta, seed, step, dt, tau_p, mu, mu_inv_t, pressure):
    """CPU stand-in of ``ops.md_scr_barostat_tri`` (float64 reference, same contract)."""
    m, mit, pt, c = ref_barostat_tri(cell, kin6, virial, P0, kT, beta, seed, int(step[0]), dt, tau_p)
    for t, a in ((mu, m), (mu_inv_t, mit), (pressure, pt), (cell, c)):
        t.copy_(torch.from_numpy(a))


def emu_md_affine_deform(pos, vel, replica, mu, mu_inv_t):
    """CPU stand-in of ``ops.md_affine_deform``."""
    r = replica.long()
    pos.copy_(torch.einsum("ni,nij->nj", pos.double(), mu.double()[r]))
    vel.copy_(torch.einsum("ni,nij->nj", vel.double(), mu_inv_t.double()[r]))


@pytest.fixture
def emu_tri(emu, monkeypatch):
    for name, fn in (("md_langevin_baoa", emu_md_langevin_baoa), ("md_kick", emu_md_kick),
                     ("md_kinetic_tensor", emu_md_kinetic_tensor), ("md_scr_barostat_tri", emu_md_scr_barostat_tri),
                     ("md_affine_deform", emu_md_affine_deform), ("edge_virial_atom", _emu_edge_virial_atom)):
        monkeypatch.setattr(ops, name, fn)
    return emu


# ---------------------------------------------------------------------------------------------------------------------
# the stationary density of the cell step: float64 quadrature (CPU) and the kernels (GPU)
# ---------------------------------------------------------------------------------------------------------------------
H0 = np.array([[2.0, 0.0, 0.0], [0.3, 1.8, 0.0], [-0.2, 0.4, 1.6]])
K_CELL = 3.0


def target_diag_means(P0, N=4, kT=1.0, measure=True, n=240, hi=6.0):
    """Means of ``h00, h11, h22`` under ``h00^N h11^(N-1) h22^(N-2) exp(-(U_diag + P0 h00 h11 h22) / kT)`` (``measure``) or
    ``(h00 h11 h22)^N exp(...)`` (``measure=False``: the flat measure ``m = 1``), ``U = K_CELL/2 sum (h_aa - H0_aa)^2``:
    a float64 Riemann sum on a uniform grid (the integrand vanishes at both ends, so the sum converges spectrally)."""
    x = (np.arange(n) + 0.5) * (hi / n)
    powers = (N, N - 1, N - 2) if measure else (N, N, N)
    w = [x ** p * np.exp(-0.5 * K_CELL * (x - H0[a, a]) ** 2 / kT) for a, p in enumerate(powers)]
    joint = np.exp(-P0 * x[:, None, None] * x[None, :, None] * x[None, None, :] / kT)
    Z = np.einsum("i,j,k,ijk->", *w, joint)
    return np.array([np.einsum("i,j,k,ijk->", *[wb * (x if a == b else 1.0) for b, wb in enumerate(w)], joint) / Z
                     for a in range(3)])


def test_target_quadrature_reproduces_the_derivation_table():
    """The float64 quadrature against the numbers of DESIGN.md (target and flat-measure means of the diagonal)."""
    for P0, target, flat in ((0.0, (2.5479, 2.2682, 1.9688), (2.5479, 2.3878, 2.2325)),
                             (0.3, (2.2983, 1.9790, 1.6163), (2.2421, 2.0677, 1.8983))):
        assert np.abs(target_diag_means(P0) - target).max() < 2e-4
        assert np.abs(target_diag_means(P0, measure=False) - flat).max() < 2e-4


@pytest.mark.gpu
@pytest.mark.parametrize("P0", [0.0, 0.3])
def test_stationary_distribution_of_the_cell(P0):
    """16 384 replicas of 4 free atoms (no atom forces) in a cell with the separable energy U = k/2 sum_{i>=j} (h_ij - h0_ij)^2,
    k = 3, kT = 1, g = beta_T / (3 tau_p) = 1, dt = 0.002, Langevin friction gamma dt = 0.05, through the real baoa / kick /
    kinetic-tensor / barostat / deform kernels; the cell virial W = -h^T dU/dh is computed on the device every step.
    The target density m(h) V^N e^{-(U + P0 V)/kT} with m = 1/(h11 h22^2) gives diagonal marginals
    ~ h00^4 h11^3 h22^2 e^{-(U_diag + P0 V)} and Gaussian off-diagonals (mean h0_ij, variance kT/k = 1/3).  Diagonal means:

        P0    target (quadrature)        flat measure m = 1
        0     2.5479  2.2682  1.9688     2.5479  2.3878  2.2325
        0.3   2.2983  1.9790  1.6163     2.2421  2.0677  1.8983

    With 16 384 independent replicas the standard error of each mean is ~1e-3, so the flat measure's h11 and h22 means
    (and h00 under pressure) sit 80-350 standard errors away; the test asserts that distance as well as the agreement."""
    G, N = 16384, 4
    dt, gdt = 0.002, 0.05
    replica, ptr = _replica_tensors([N] * G, DEV)
    n = G * N
    h0 = torch.from_numpy(H0).float().to(DEV)
    cell = h0.repeat(G, 1, 1).contiguous()
    kT, P0_t = torch.ones(G, device=DEV), torch.full((G,), P0, device=DEV)
    beta = torch.full((G,), 3.0, device=DEV)                        # g = beta / (3 tau_p) = 1 with tau_p = 1
    seeds = torch.arange(G, dtype=torch.int64, device=DEV) * 7 + 1001
    step = torch.zeros(1, dtype=torch.int64, device=DEV)
    inv_m = torch.ones(n, device=DEV)
    gen = torch.Generator().manual_seed(5)
    pos = (torch.rand(n, 3, generator=gen) * 1.5).to(DEV)
    vel = torch.randn(n, 3, generator=gen).to(DEV)
    zero_f, kinetic = torch.zeros(n, 3, device=DEV), torch.empty(n, device=DEV)
    mu, mit, pt = (torch.empty(G, 3, 3, device=DEV) for _ in range(3))
    c1, c2 = math.exp(-gdt), math.sqrt(-math.expm1(-2 * gdt))
    s1 = torch.zeros(G, 3, 3, dtype=torch.float64, device=DEV)
    s2 = torch.zeros(G, 3, 3, dtype=torch.float64, device=DEV)
    steps, burn = 20_000, 4_000
    for k in range(steps):
        ops.md_langevin_baoa(pos, vel, zero_f, inv_m, replica, ptr, kT, seeds, step, c1, c2, dt)
        ops.md_kick(vel, zero_f, inv_m, 0.5 * dt, kinetic, step)
        kin6 = ops.segment_sum(ops.md_kinetic_tensor(vel, inv_m), ptr, None, G)
        W = -torch.bmm(cell.transpose(1, 2), K_CELL * (cell - h0)).contiguous()
        ops.md_scr_barostat_tri(cell, kin6, W, P0_t, kT, beta, seeds, step, dt, 1.0, mu, mit, pt)
        ops.md_affine_deform(pos, vel, replica, mu, mit)
        if k >= burn:
            c = cell.double()
            s1 += c
            s2 += c * c
    T = steps - burn
    assert torch.isfinite(cell).all() and torch.equal(cell.triu(1), torch.zeros_like(cell))
    m_rep = (s1 / T).cpu().numpy()                                  # per-replica time averages: independent samples
    mean = m_rep.mean(0)
    se = m_rep.std(0) / math.sqrt(G)
    var = (s2 / T).cpu().numpy().mean(0) - mean ** 2
    diag, se_diag = np.diagonal(mean), np.diagonal(se)
    target, flat = target_diag_means(P0), target_diag_means(P0, measure=False)
    off = [(1, 0), (2, 0), (2, 1)]
    print(f"\nP0 = {P0}: diagonal means {np.round(diag, 4)} +- {np.round(se_diag, 4)}, target {np.round(target, 4)}, "
          f"flat measure {np.round(flat, 4)}")
    print(f"         off-diagonal means {[round(float(mean[i, j]), 4) for i, j in off]} (h0 {[H0[i, j] for i, j in off]}), "
          f"variances {[round(float(var[i, j]), 4) for i, j in off]} (kT/k = {1 / K_CELL:.4f})")
    assert (np.abs(diag - target) < 4.0 * se_diag + 2e-3).all(), (diag, target)
    assert all(abs(mean[i, j] - H0[i, j]) < 4.0 * se[i, j] + 2e-3 for i, j in off)
    assert all(abs(var[i, j] * K_CELL - 1.0) < 0.03 for i, j in off)
    # the flat measure is ruled out: h11 and h22 (P0 = 0), all three (P0 > 0)
    gap = np.abs(diag - flat) / se_diag
    assert (gap[1:] > 30.0).all() and (P0 == 0.0 or gap[0] > 30.0), gap


# ---------------------------------------------------------------------------------------------------------------------
# kernel level (GPU)
# ---------------------------------------------------------------------------------------------------------------------
def _tri_inputs(G, seed=0, dev=DEV):
    gen = torch.Generator().manual_seed(seed)
    cell = torch.tril(torch.diag_embed(8.0 + 10.0 * torch.rand(G, 3, generator=gen)) + 1.5 * torch.randn(G, 3, 3, generator=gen),
                      -1) + torch.diag_embed(8.0 + 10.0 * torch.rand(G, 3, generator=gen))
    kin6 = (0.5 + 0.03 * G * torch.rand(G, 6, generator=gen)) * torch.tensor([1.0, 0.1, 1.0, 0.1, 0.1, 1.0])
    vir = 5.0 * torch.randn(G, 3, 3, generator=gen)
    P0 = 1e-3 * torch.randn(G, generator=gen)                       # eV/A^3, both signs
    kT = 0.02 + 0.05 * torch.rand(G, generator=gen)
    beta = 100.0 * torch.rand(G, generator=gen)
    beta[::7] = 0.0
    return [t.float().contiguous().to(dev) for t in (cell, kin6, vir, P0, kT, beta)]


def _out(G):
    return [torch.full((G, 3, 3), float("nan"), device=DEV) for _ in range(3)]


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 1000])
def test_barostat_tri_matches_float64(G):
    cell, kin6, vir, P0, kT, beta = _tri_inputs(G, seed=G)
    seeds = torch.tensor([(2 ** 40 + 977 * g) if g % 2 else (3 + g) for g in range(G)], dtype=torch.int64, device=DEV)
    for s, dt, tau in ((0, 0.5, 1000.0), (17, 2.0, 50.0), (2 ** 32 - 1, 1.0, 5.0), (2 ** 32 + 5, 1.0, 5.0)):
        step = torch.tensor([s], dtype=torch.int64, device=DEV)
        c = cell.clone()
        mu, mit, pr = _out(G)
        m_ref, mit_ref, pt_ref, c_ref = ref_barostat_tri(cell, kin6, vir, P0, kT, beta, seeds, s, dt, tau)
        ops.md_scr_barostat_tri(c, kin6, vir, P0, kT, beta, seeds, step, dt, tau, mu, mit, pr)
        assert int(step) == s
        for got, ref in ((mu, m_ref), (mit, mit_ref), (pr, pt_ref), (c, c_ref)):
            g64 = _np(got).astype(np.float64)
            assert (np.abs(g64 - ref) <= 1.2e-7 * np.abs(ref) + 1e-13).all(), np.abs(g64 - ref).max()
        zero = torch.zeros(G, 3, 3, device=DEV)
        assert torch.equal(c.triu(1), zero) and torch.equal(mu.triu(1), zero) and torch.equal(mit.tril(-1), zero)
        # beta = 0: mu = I exactly and the cell bitwise unchanged
        assert torch.equal(mu[::7], torch.eye(3, device=DEV).expand_as(mu[::7])) and torch.equal(c[::7], cell[::7])
        assert not torch.equal(c[1:2], cell[1:2]) or G == 1


@pytest.mark.gpu
def test_barostat_tri_noise_recipe_and_disjoint_streams():
    G = 1000
    cell = _tri_inputs(G, seed=9)[0]
    seeds = torch.arange(G, dtype=torch.int64, device=DEV) * 7919 + 2 ** 33
    s = 2 ** 32 + 12345
    step = torch.tensor([s], dtype=torch.int64, device=DEV)
    V = (cell[:, 0, 0].double() * cell[:, 1, 1].double() * cell[:, 2, 2].double()).float()
    zero, zero9 = torch.zeros(G, device=DEV), torch.zeros(G, 3, 3, device=DEV)
    # no pressure drift (K = W = P0 = 0), b = 1, kT = 0.015 V: noise scale sqrt(2 b kT / 3V) = 0.1, drift 0.01 diag(1, 0, -1)
    mu, mit, pr = _out(G)
    runs = []
    for _ in range(2):
        c = cell.clone()
        ops.md_scr_barostat_tri(c, torch.zeros(G, 6, device=DEV), zero9, zero, 0.015 * V, torch.ones(G, device=DEV), seeds,
                                step, 1.0, 1.0, mu, mit, pr)
        runs.append([t.clone() for t in (c, mu, mit, pr)])
    assert all(torch.equal(a, b) for a, b in zip(*runs))              # deterministic
    m64 = _np(mu).astype(np.float64)
    delta = np.stack([scipy.linalg.logm(m).real for m in m64])[:, LI, LJ]
    xi = (delta - np.array([0.01, 0, 0, 0, 0, -0.01])) / 0.1
    ref = ref_tri_xi(_np(seeds), s)
    assert np.abs(xi - ref).max() < 1e-4, np.abs(xi - ref).max()
    # disjoint from the Langevin noise of 4 atoms per replica (word 3 = 0) and the isotropic barostat's (word 3 = 1)
    replica, ptr = _replica_tensors([4] * G, DEV)
    lang = ref_noise(replica, ptr, seeds, s).reshape(G, 12)
    iso = ref_baro_xi(_np(seeds), s)
    assert (np.abs(ref[:, :, None] - lang[:, None, :]).min((1, 2)) > 1e-4).mean() > 0.99
    assert (np.abs(ref - iso[:, None]).min(1) > 1e-4).mean() > 0.99


@pytest.mark.gpu
def test_affine_deform_and_kinetic_tensor_match_float64_and_empty_launches_are_no_ops():
    sizes = [40_000, 1, 60_002]
    replica, ptr = _replica_tensors(sizes, DEV)
    gen = torch.Generator().manual_seed(3)
    n, G = sum(sizes), len(sizes)
    pos, vel = (20.0 * torch.randn(n, 3, generator=gen)).to(DEV), (0.03 * torch.randn(n, 3, generator=gen)).to(DEV)
    D = torch.tril(0.01 * torch.randn(G, 3, 3, generator=gen, dtype=torch.float64))
    mu = torch.linalg.matrix_exp(D).float().to(DEV)
    mit = torch.linalg.matrix_exp(-D).transpose(1, 2).contiguous().float().to(DEV)
    p, v = pos.clone(), vel.clone()
    ops.md_affine_deform(p, v, replica, mu, mit)
    r = replica.long()
    for got, x, m in ((p, pos, mu), (v, vel, mit)):
        ref = torch.einsum("ni,nij->nj", x.double(), m.double()[r])
        bound = torch.einsum("ni,nij->nj", x.double().abs(), m.double().abs()[r])
        assert bool(((got.double() - ref).abs() <= 4e-7 * bound).all())
    eye = torch.eye(3, device=DEV).repeat(G, 1, 1)
    p, v = pos.clone(), vel.clone()
    ops.md_affine_deform(p, v, replica, eye, eye.clone())
    assert torch.equal(p, pos) and torch.equal(v, vel)               # mu = I: bitwise unchanged
    inv_m = (1.0 / (103.642697 * (1.0 + 15.0 * torch.rand(n, generator=gen)))).to(DEV)
    kt = ops.md_kinetic_tensor(vel, inv_m)
    v64 = vel.double()
    ref = v64[:, LI] * v64[:, LJ] / inv_m.double()[:, None]
    assert kt.shape == (n, 6) and bool(((kt.double() - ref).abs() <= 2.5e-7 * ref.abs()).all())
    # empty launches
    e = torch.zeros(0, 3, device=DEV)
    ops.md_affine_deform(e, e.clone(), torch.zeros(0, dtype=torch.int32, device=DEV), mu, mit)
    assert ops.md_kinetic_tensor(e, torch.zeros(0, device=DEV)).shape == (0, 6)
    z, z9 = torch.zeros(0, device=DEV), torch.zeros(0, 3, 3, device=DEV)
    step = torch.tensor([3], dtype=torch.int64, device=DEV)
    ops.md_scr_barostat_tri(z9, torch.zeros(0, 6, device=DEV), z9.clone(), z, z, z, torch.zeros(0, dtype=torch.int64, device=DEV),
                            step, 0.5, 100.0, z9.clone(), z9.clone(), z9.clone())
    assert int(step) == 3


def _f(*shape, dtype=torch.float32, dev=DEV):
    return torch.zeros(shape, dtype=dtype, device=dev)


def _kinetic_tensor(bad, dev=DEV):
    n = 5
    vel = _f(n, 3, dtype=torch.float64 if bad == "dtype" else torch.float32, dev=dev)
    ops.md_kinetic_tensor(vel, _f(n + 1 if bad == "shape" else n, dev=dev))


def _barostat_tri(bad, dev=DEV):
    G = 3
    cell = _f(G, 3, 3, dtype=torch.float64 if bad == "dtype" else torch.float32, dev=dev)
    kin6 = _f(G, 3 if bad == "shape" else 6, dev=dev)
    ops.md_scr_barostat_tri(cell, kin6, _f(G, 3, 3, dev=dev), _f(G, dev=dev), _f(G, dev=dev), _f(G, dev=dev),
                            _f(G, dtype=torch.int64, dev=dev), _f(1, dtype=torch.int64, dev=dev), 1.0, 100.0,
                            _f(G, 3, 3, dev=dev), _f(G, 3, 3, dev=dev), _f(G, 3, 3, dev=dev))


def _affine_deform(bad, dev=DEV):
    n = 5
    replica = _f(n, dtype=torch.int64 if bad == "dtype" else torch.int32, dev=dev)
    mu_inv_t = _f(2, 3, 3, dev=dev) if bad == "shape" else _f(1, 3, 3, dev=dev)
    ops.md_affine_deform(_f(n, 3, dev=dev), _f(n, 3, dev=dev), replica, _f(1, 3, 3, dev=dev), mu_inv_t)


WRAPPERS = [("md_kinetic_tensor", _kinetic_tensor), ("md_scr_barostat_tri", _barostat_tri), ("md_affine_deform", _affine_deform)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,call", WRAPPERS, ids=[w[0] for w in WRAPPERS])
@pytest.mark.parametrize("bad", ["dtype", "shape"])
def test_wrapper_rejects_bad_argument_before_launch(name, call, bad):
    n0 = ops.LAUNCHES["n"]
    with pytest.raises(RuntimeError, match=re.escape(f"hermnet_b200.{name}:")):
        call(bad)
    assert ops.LAUNCHES["n"] == n0


@pytest.mark.parametrize("name,call", WRAPPERS, ids=[w[0] for w in WRAPPERS])
def test_wrapper_refuses_host_tensors_before_launch(name, call):
    n0 = ops.LAUNCHES["n"]
    with pytest.raises(RuntimeError, match=re.escape(f"hermnet_b200.{name}: expected a CUDA tensor")):
        call(None, dev="cpu")
    assert ops.LAUNCHES["n"] == n0


# ---------------------------------------------------------------------------------------------------------------------
# standard_cell (CPU)
# ---------------------------------------------------------------------------------------------------------------------
def _triclinic_cell():
    return np.array([[7.0, 1.0, -0.5], [0.8, 6.5, 1.2], [-1.1, 0.7, 7.5]])


def test_standard_cell_is_lower_triangular_and_keeps_distances():
    rng = np.random.default_rng(0)
    cells = np.stack([_triclinic_cell(), np.diag([5.0, 6.0, 7.0]) @ scipy.linalg.expm(np.array([[0, .3, -.2], [-.3, 0, .5],
                                                                                                [.2, -.5, 0]]))])
    x = rng.normal(size=(10, 3)) * 3.0
    v = rng.normal(size=(10, 3))
    batch = np.repeat([0, 1], 5)
    xs, hs, vs = md.standard_cell(x, cells, v, batch=batch)
    assert hs.shape == (2, 3, 3) and np.array_equal(np.triu(hs, 1), np.zeros_like(hs)) and (np.diagonal(hs, 0, 1, 2) > 0).all()
    for g in range(2):
        sl = slice(5 * g, 5 * g + 5)
        R = np.linalg.solve(cells[g], hs[g])                         # h R = L
        assert np.allclose(R @ R.T, np.eye(3), atol=1e-12) and abs(np.linalg.det(R) - 1.0) < 1e-12
        assert np.allclose(xs[sl], x[sl] @ R, atol=1e-12) and np.allclose(vs[sl], v[sl] @ R, atol=1e-12)
        d0 = np.linalg.norm(x[sl, None] - x[None, sl] + cells[g][1], axis=-1)     # a pair across the b face
        d1 = np.linalg.norm(xs[sl, None] - xs[None, sl] + hs[g][1], axis=-1)
        assert np.allclose(d0, d1, atol=1e-12)
        assert np.allclose(np.linalg.norm(cells[g], axis=1), np.linalg.norm(hs[g], axis=1), atol=1e-12)
    # one shared [3,3] cell, no velocities; an already standard cell is kept
    xs1, h1, v1 = md.standard_cell(x, cells[0])
    assert h1.shape == (3, 3) and v1 is None
    xs2, h2, _ = md.standard_cell(xs1, h1)
    assert np.allclose(h2, h1, atol=1e-12) and np.allclose(xs2, xs1, atol=1e-12)


def test_standard_cell_rejects_a_left_handed_cell():
    with pytest.raises(ValueError, match="right-handed"):
        md.standard_cell(np.zeros((2, 3)), np.diag([5.0, 5.0, -5.0]))
    with pytest.raises(ValueError):
        md.standard_cell(np.zeros((4, 3)), np.stack([np.eye(3), -np.eye(3)]) * 5.0, batch=[0, 0, 1, 1])


def test_standard_cell_keeps_energies_and_rotates_forces(emu):
    model = _cpu_model()
    pos, Z, cell, _ = _cpu_systems((31,))
    S = np.array([[1.0, 0.08, -0.05], [0.03, 1.0, 0.1], [-0.06, 0.04, 1.0]])         # shear + rotation: a general cell
    p0, c0 = pos.astype(np.float64) @ S, cell.reshape(3, 3).astype(np.float64) @ S
    p1, c1, _ = md.standard_cell(p0, c0)
    R = np.linalg.solve(c0, c1)
    out = []
    for p, c in ((p0, c0), (p1, c1)):
        d = H.Data(pos=torch.from_numpy(p).float().requires_grad_(True), atomic_number=torch.from_numpy(Z).long(),
                   cell=torch.from_numpy(c).float().reshape(1, 3, 3))
        out.append(util.energy_forces(model, d)[:2])
    (e0, f0), (e1, f1) = out
    assert util.rel_err(e1, e0) < 1e-5
    assert float((f1.double() - f0.double() @ torch.from_numpy(R)).abs().max()) < 1e-4 * max(1.0, float(f0.abs().max()))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the driver over the kernel emulator with the float64 stand-ins
# ---------------------------------------------------------------------------------------------------------------------
SHEAR = np.array([[1.0, 0.0, 0.0], [0.04, 1.0, 0.0], [-0.03, 0.05, 1.0]], dtype=np.float32)


def test_emulated_triclinic_stats_restart_and_zero_compressibility(emu_tri):
    model = _cpu_model()
    pos, Z, cell, batch = _cpu_systems((22, 23))
    pos, cell = pos @ SHEAR, cell @ SHEAR                           # lower-triangular, sheared
    n1 = len(Z) // 2
    vel = 0.002 * np.random.default_rng(1).standard_normal(pos.shape).astype(np.float32)
    kw = dict(temperature_K=[300.0, 900.0], pressure_bar=[2e4, -2e4], tau_p_fs=50.0, friction_per_fs=0.05, seed=5,
              batch=batch, device="cpu", cell_dof="triclinic")
    st = {}
    p, v, c, e = md.langevin_npt_device(model, Z, pos, cell, vel, steps=6, stats=st, skin=0.5, **kw)
    assert p.shape == (2 * n1, 3) and v.shape == (2 * n1, 3) and c.shape == (2, 3, 3) and e.shape == (6, 2)
    assert st["temperature"].shape == st["pressure"].shape == st["volume"].shape == (6, 2)
    assert st["virial"].shape == st["cell"].shape == st["pressure_tensor"].shape == (6, 2, 3, 3) and st["step"] == 6
    assert st["builds"] + st["reuses"] == 7 and st["reuses"] > 0
    assert torch.equal(st["cell"][-1], c) and torch.equal(c.triu(1), torch.zeros_like(c))
    assert not torch.equal(c, torch.from_numpy(cell))
    off = c[:, [1, 2, 2], [0, 0, 1]] / torch.from_numpy(cell)[:, [1, 2, 2], [0, 0, 1]]
    assert float((off - 1.0).abs().max()) > 1e-6                     # the shape changed, not only the size
    assert util.rel_err(st["volume"][-1].double(), torch.linalg.det(c.double()).abs()) < 1e-6
    pt = st["pressure_tensor"].double()
    assert torch.equal(pt, pt.transpose(2, 3))
    assert util.rel_err(st["pressure"].double(), pt.diagonal(dim1=2, dim2=3).sum(-1) / 3.0) < 1e-6
    # cuda_graph (which evaluates eagerly on CPU tensors): the same run, bitwise
    st_g = {}
    out_g = md.langevin_npt_device(model, Z, pos, cell, vel, steps=6, stats=st_g, skin=0.5, cuda_graph=True, **kw)
    assert all(torch.equal(a, b) for a, b in zip(out_g, (p, v, c, e)))
    assert st_g.keys() == st.keys()
    assert all(torch.equal(st_g[k], st[k]) if isinstance(st[k], torch.Tensor) else st_g[k] == st[k] for k in st)
    # restart from the returned state and stats: 4 + 2 steps equal 6 steps
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
                                            pressure_bar=[1.0, 5e3], cell_dof="triclinic", **kw_nvt)
    assert torch.equal(pa, pb) and torch.equal(va, vb) and torch.equal(ea, eb) and torch.equal(cb, torch.from_numpy(cell))
    assert (s_nvt["builds"], s_nvt["reuses"]) == (s_npt["builds"], s_npt["reuses"])
    assert torch.equal(s_nvt["temperature"], s_npt["temperature"])


def test_emulated_isotropic_stats_keys_are_unchanged(emu_tri, monkeypatch):
    from tests.test_npt import emu_md_affine_scale, emu_md_scr_barostat
    monkeypatch.setattr(ops, "md_scr_barostat", emu_md_scr_barostat)
    monkeypatch.setattr(ops, "md_affine_scale", emu_md_affine_scale)
    model = _cpu_model()
    pos, Z, cell, _ = _cpu_systems((22,))
    st = {}
    md.langevin_npt_device(model, Z, pos, cell, np.zeros_like(pos), steps=2, stats=st, device="cpu")
    assert sorted(st) == ["builds", "forces", "pressure", "reuses", "step", "temperature", "virial", "volume"]


@pytest.mark.parametrize("bad", [
    dict(cell=np.array([[10.0, 0.1, 0.0], [0.0, 10.0, 0.0], [0.0, 0.0, 10.0]])), dict(cell=np.diag([10.0, -10.0, -10.0])),
    dict(cell=np.array([[10.0, 0.0, 0.0], [0.0, 10.0, 1e-9], [0.0, 0.0, 10.0]])), dict(cell_dof="anisotropic"),
    dict(cell_dof=None), dict(cell=None), dict(cell=np.full((3, 3), np.nan)), dict(compressibility_per_bar=-1e-5),
    dict(tau_p_fs=0.0), dict(pressure_bar=float("nan")), dict(temperature_K=-1.0), dict(forces=np.zeros((3, 3)))])
def test_validation_errors(bad):
    args = dict(cell=10.0 * np.eye(3), temperature_K=300.0, pressure_bar=1.0, compressibility_per_bar=4.5e-5, tau_p_fs=1000.0,
                friction_per_fs=0.01, dt_fs=0.5, seed=0, step0=0, batch=None, cell_dof="triclinic")
    args.update(bad)
    cell = args.pop("cell")
    with pytest.raises(ValueError) as info:
        md.langevin_npt_device(None, [8, 1, 1, 8], np.zeros((4, 3)), cell, np.zeros((4, 3)), steps=1, device="cpu", **args)
    if "cell" in bad and bad["cell"] is not None and np.isfinite(bad["cell"]).all():
        assert "standard_cell" in str(info.value)


# ---------------------------------------------------------------------------------------------------------------------
# model level (GPU): HVNet of BASELINE config 1 on C1 water boxes, as tests/test_npt.py
# ---------------------------------------------------------------------------------------------------------------------
TRI = dict(cell_dof="triclinic")


@pytest.mark.gpu
def test_zero_compressibility_triclinic_is_langevin_bitwise():
    model = _water_model()
    pos, Z, cell, batch = _boxes(4, (1, 2))
    v0 = _mb(Z, 300.0, 1)
    kw = dict(temperature_K=[300.0, 500.0], friction_per_fs=0.05, seed=11, batch=batch, device=DEV, skin=0.5)
    s_nvt, s_npt = {}, {}
    p, v, e = md.langevin_device(model, Z, pos, cell, v0, steps=20, stats=s_nvt, **kw)
    p2, v2, c2, e2 = md.langevin_npt_device(model, Z, pos, cell, v0, steps=20, stats=s_npt, compressibility_per_bar=0.0,
                                            pressure_bar=[1.0, 1000.0], **TRI, **kw)
    assert torch.equal(p, p2) and torch.equal(v, v2) and torch.equal(e, e2)
    assert torch.equal(s_nvt["temperature"], s_npt["temperature"])
    assert (s_nvt["builds"], s_nvt["reuses"]) == (s_npt["builds"], s_npt["reuses"]) and s_npt["reuses"] > 0
    assert torch.equal(c2, torch.from_numpy(cell).to(DEV))
    assert s_npt["cell"].shape == s_npt["pressure_tensor"].shape == (20, 2, 3, 3)


@pytest.mark.gpu
def test_restart_is_bitwise_and_a_lone_replica_matches_the_batch():
    model = _water_model()
    pos, Z, cell, batch = _boxes(4, (7, 8))
    v0 = _mb(Z, 300.0, 2)
    kw = dict(batch=batch, temperature_K=[350.0, 400.0], pressure_bar=[1000.0, 3000.0], tau_p_fs=200.0, friction_per_fs=0.05,
              seed=2 ** 40 + 1, device=DEV, **TRI)
    st = {}
    p12, v12, c12, e12 = md.langevin_npt_device(model, Z, pos, cell, v0, steps=12, stats=st, **kw)
    st7 = {}
    p7, v7, c7, e7 = md.langevin_npt_device(model, Z, pos, cell, v0, steps=7, stats=st7, **kw)
    p5, v5, c5, e5 = md.langevin_npt_device(model, Z, p7, c7, v7, steps=5, step0=st7["step"], forces=st7["forces"], **kw)
    assert st["step"] == 12 and st7["step"] == 7
    assert torch.equal(p5, p12) and torch.equal(v5, v12) and torch.equal(c5, c12) and torch.equal(torch.cat([e7, e5]), e12)
    assert float(c12[:, [1, 2, 2], [0, 0, 1]].abs().max()) > 0.0     # the cells sheared
    n1 = len(Z) // 2
    sl = slice(n1, 2 * n1)
    p1, _, c1, e1 = md.langevin_npt_device(model, Z[sl], pos[sl], cell[1], v0[sl], steps=12, temperature_K=400.0,
                                           pressure_bar=3000.0, tau_p_fs=200.0, friction_per_fs=0.05, seed=2 ** 40 + 2,
                                           device=DEV, **TRI)
    assert float((p1 - p12[sl]).abs().max()) < 1e-5
    assert float((c1[0] - c12[1]).abs().max()) < 1e-5
    assert util.rel_err(e1[:, 0], e12[:, 1]) < 1e-5


@pytest.mark.gpu
def test_cuda_graph_matches_eager_while_the_cell_shears():
    model = _water_model()
    pos, Z, cell, batch = _boxes(4, (5, 6))
    v0 = _mb(Z, 300.0, 3)
    kw = dict(batch=batch, temperature_K=[300.0, 600.0], pressure_bar=[5000.0, -5000.0], tau_p_fs=100.0, device=DEV, skin=0.8,
              **TRI)
    runs = {}
    for cg in (False, True):
        st = {}
        runs[cg] = md.langevin_npt_device(model, Z, pos, cell, v0, steps=12, stats=st, cuda_graph=cg, **kw) + (st,)
    (p0, v0_, c0, e0, s0), (p1, v1, c1, e1, s1) = runs[False], runs[True]
    assert s1["builds"] == s0["builds"] and s1["reuses"] > 0
    assert float(c1[:, [1, 2, 2], [0, 0, 1]].abs().max()) > 0.0
    assert torch.equal(p1, p0) and torch.equal(v1, v0_) and torch.equal(c1, c0) and torch.equal(e1, e0)
    assert torch.equal(s1["pressure_tensor"], s0["pressure_tensor"])


@pytest.mark.gpu
def test_sheared_skin_list_reuse_and_parity():
    from hermnet_b200 import synthetic
    model = _water_model()                                          # rc 5, skin 0.5
    pos, Z, cell = synthetic.water_box(5, seed=3)
    Zt = torch.as_tensor(Z).long().to(DEV)
    p0, c0 = torch.from_numpy(pos).float().to(DEV), torch.from_numpy(cell).float().reshape(1, 3, 3).to(DEV)
    for shear, reused in ((0.03, True), (0.2, False)):              # sigma_min 0.98 and 0.87 against 5 / 5.5
        M = torch.tensor([[1.0, 0.0, 0.0], [shear, 1.0, 0.0], [-0.5 * shear, 0.5 * shear, 1.0]], device=DEV)
        vg = md.VerletGraph(model, 0.5, deforming=True)
        vg.get(p0, Zt, c0)
        p1, c1 = p0 @ M, c0 @ M
        g = vg.get(p1, Zt, c1)
        assert (vg.builds, vg.reuses) == ((1, 1) if reused else (2, 0))
        d = H.Data(pos=p1.clone().requires_grad_(True), atomic_number=Zt, cell=c1)
        d.graph = g
        e = model(d)
        (gr,) = torch.autograd.grad(e.sum(), d.pos)
        e_ref, f_ref = _fresh_energy_forces(model, p1, Z, c1)
        assert util.rel_err(e.detach(), e_ref) < 1e-5
        assert float((-gr - f_ref).abs().max()) < 1e-5 * max(1.0, float(f_ref.abs().max()))
    # a whole triclinic run: deforming re-use against fresh lists every step
    v0 = _mb(Z, 300.0, 5)
    kw = dict(temperature_K=300.0, pressure_bar=20000.0, compressibility_per_bar=4.5e-5, tau_p_fs=100.0, friction_per_fs=0.02,
              seed=3, device=DEV, **TRI)
    runs = {}
    for skin in (0.0, 0.5):
        st = {}
        runs[skin] = md.langevin_npt_device(model, Z, pos, cell, v0, steps=30, skin=skin, stats=st, **kw) + (st,)
    (pa, va, ca, ea, sa), (pb, vb, cb, eb, sb) = runs[0.0], runs[0.5]
    assert sb["reuses"] > 0 and sa["builds"] == 31
    assert float(cb[0, [1, 2, 2], [0, 0, 1]].abs().max()) > 1e-4                    # the cell sheared
    assert float((pb - pa).abs().max()) < 1e-4 and float((cb - ca).abs().max()) < 1e-4
    assert util.rel_err(eb, ea) < 1e-5


@pytest.mark.gpu
def test_pressure_drives_the_volume_and_the_stats_are_consistent():
    model = _water_model()
    pos, Z, cell, batch = _boxes(4, (9, 9))                          # two copies of the same box
    v0 = _mb(Z, 300.0, 4)
    v0 = np.concatenate([v0[: len(Z) // 2]] * 2)
    base = dict(batch=batch, temperature_K=300.0, friction_per_fs=0.05, seed=[21, 21], device=DEV, **TRI)
    st = {}
    md.langevin_npt_device(model, Z, pos, cell, v0, steps=20, compressibility_per_bar=0.0, stats=st, **base)
    P = st["pressure"].double()
    P_start, spread = float(P[:, 0].mean()), float(P[:, 0].std())
    delta = max(10.0 * spread, 5000.0)
    st = {}
    p, v, c, e = md.langevin_npt_device(model, Z, pos, cell, v0, steps=40, pressure_bar=[P_start + delta, P_start - delta],
                                        tau_p_fs=100.0, stats=st, **base)
    V0 = abs(float(np.linalg.det(cell[0].astype(np.float64))))
    vol = st["volume"].double()
    assert float(vol[-1, 0]) < V0 < float(vol[-1, 1]), (V0, vol[-1])
    # the traces: pressure = tr / 3 of the pressure tensor, volume = det of the cell trace, the last cell is the returned one
    pt = st["pressure_tensor"].double()
    assert float((st["pressure"].double() - pt.diagonal(dim1=2, dim2=3).sum(-1) / 3.0).abs().max()) <= 1e-6 * float(pt.abs().max())
    assert util.rel_err(vol, torch.linalg.det(st["cell"].double()).abs()) < 1e-6 and torch.equal(st["cell"][-1], c)
    # the pressure tensor (Kt + W)/V from the traces: Kt of the post-kick velocities is not traced, so check its trace part
    n1 = len(Z) // 2
    K = st["temperature"].double() * 1.5 * n1 * md.KB_EV
    V_pre = torch.cat([torch.full((1, 2), V0, dtype=torch.float64, device=DEV), vol[:-1]])
    trW = st["virial"].double().diagonal(dim1=2, dim2=3).sum(-1)
    P_ref = (2.0 * K + trW) / (3.0 * V_pre) * md.EV_A3_TO_BAR
    assert float((st["pressure"].double() - P_ref).abs().max()) <= 1e-5 * float(P_ref.abs().max()) + 1e-2
