"""ASE-free MD driver for BASELINE.json configs[2] ("MD inference via the ASE calculator plugin"): ASE is not
installed in this image, so this module supplies the two pieces of ASE the plugin path needs -- an ``Atoms``-like
container and a velocity-Verlet loop -- with ASE's attribute names, so ``NNCalculator`` is exercised exactly as ASE
would drive it (``atoms.get_forces()`` -> ``calc.calculate(atoms)``).  ``device_resident=True`` is SURVEY 8(f) rank 1:
positions stay on the GPU and only the graph is rebuilt per step."""
from __future__ import annotations

import numpy as np
import torch

from ..data import Data
from ..symbols import atomic_numbers, chemical_symbols

KB_EV = 8.617333262e-5
AMU_A2_FS2_TO_EV = 103.642697      # 1 amu*A^2/fs^2 in eV
MASSES = {1: 1.008, 3: 6.94, 6: 12.011, 8: 15.999, 13: 26.982, 14: 28.085, 24: 51.996, 25: 54.938, 26: 55.845,
          27: 58.933, 28: 58.693}


class SimpleAtoms:
    """The subset of ``ase.Atoms`` the calculator touches."""

    def __init__(self, numbers, positions, cell=None, pbc=True):
        self.numbers = np.asarray(numbers)
        self.positions = np.asarray(positions, dtype=np.float64)
        self.cell = None if cell is None else np.asarray(cell, dtype=np.float64).reshape(3, 3)
        self.pbc = np.array([bool(pbc)] * 3)
        self.calc = None
        self.velocities = np.zeros_like(self.positions)

    def get_chemical_symbols(self):
        return [chemical_symbols[z] for z in self.numbers]

    def todict(self):
        return {"cell": self.cell, "positions": self.positions, "numbers": self.numbers, "pbc": self.pbc}

    def get_masses(self):
        return np.array([MASSES.get(int(z), 2.0 * int(z)) for z in self.numbers])

    def get_forces(self):
        self.calc.calculate(self, ["forces"])
        return self.calc.results["forces"]

    def get_potential_energy(self):
        self.calc.calculate(self, ["energy"])
        return self.calc.results["energy"]

    def __len__(self):
        return len(self.numbers)


def maxwell_boltzmann(atoms: SimpleAtoms, temperature_K: float, seed: int = 0):
    rng = np.random.default_rng(seed)
    m = atoms.get_masses()[:, None] * AMU_A2_FS2_TO_EV
    atoms.velocities = rng.normal(size=atoms.positions.shape) * np.sqrt(KB_EV * temperature_K / m)
    atoms.velocities -= atoms.velocities.mean(0, keepdims=True)


def velocity_verlet(atoms: SimpleAtoms, steps: int, dt_fs: float = 0.5):
    """Host-driven loop, one ``calculate`` per step (what ASE's ``VelocityVerlet`` does)."""
    m = atoms.get_masses()[:, None] * AMU_A2_FS2_TO_EV
    f = atoms.get_forces()
    energies = []
    for _ in range(steps):
        atoms.velocities += 0.5 * dt_fs * f / m
        atoms.positions = atoms.positions + dt_fs * atoms.velocities
        f = atoms.get_forces()
        atoms.velocities += 0.5 * dt_fs * f / m
        energies.append(atoms.calc.results["energy"])
    return energies


@torch.no_grad()
def _kick(v, f, inv_m, dt):
    v.add_(f * inv_m, alpha=0.5 * dt)


class VerletGraph:
    """Verlet-skin re-use of a model's device graph (neighbour list + row CSR + tile plans) across MD steps -- what the
    reference rebuilds on the CPU on every call (plugin/ase_interface/calculator.py:42-57 -> build_graph).  The list is
    searched with ``rc + skin`` and stays valid while no atom has moved by more than ``skin / 2`` since it was built; the
    edge kernels drop the entries that are at or beyond ``rc`` at evaluation time, so energies / forces equal those of a
    fresh list.  ``skin = 0``: rebuild every step (the reference's behaviour).  ``builds`` / ``reuses`` count what happened.
    (Sub-networks are treated as active when the SUPERSET list has an edge for them -- hermnet.py:56-57 can only differ
    for a sub-network whose every edge sits in the skin shell.)"""

    def __init__(self, model, skin: float = 0.0, cuda_graph: bool = False, virial: bool = False):
        self.model, self.skin = model, float(skin)
        self.virial = bool(virial)    # captured evaluation also returns the per-graph virial (energy_forces_virial)
        self.graph, self.ref_pos, self.ref_cell, self.ref_Z = None, None, None, None
        self.builds = self.reuses = 0
        # cuda_graph: while a list is re-used, replay the whole evaluation (forward + backward, ~200 launches + torch glue) as
        # ONE captured CUDA graph -- small systems are bound by host launch latency, not by the kernels
        self.cuda_graph = bool(cuda_graph) and self.skin > 0.0
        self._captured, self._captured_for = None, None

    def energy_and_gradient(self, pos, Z, cell):
        """``(E [num_graphs], dE/dpos)`` at ``pos`` through the re-used (or rebuilt) list; with ``cuda_graph`` the evaluation is
        captured once per list build and replayed afterwards (the returned tensors are then the capture's static outputs;
        with ``virial`` the capture returns the virial ``[num_graphs,3,3]`` as a third one)."""
        g = self.get(pos, Z, cell)
        if self.cuda_graph and pos.is_cuda:
            if self._captured_for is not g:
                from ..graphed import graphed_forces
                self._captured = graphed_forces(self.model, pos, Z, cell, g, warmup=1, virial=self.virial)
                self._captured_for = g
            return self._captured(pos)
        p = pos.detach().requires_grad_(True)
        e, _, _ = self.model.forward_graph(p, Z, None if cell is None else cell.reshape(-1, 3, 3), g)
        (grad,) = torch.autograd.grad(e.sum(), p)
        return e.detach(), grad

    def get(self, pos, Z, cell):
        p = pos.detach()
        if (self.graph is not None and self.skin > 0.0 and p.shape == self.ref_pos.shape and (Z is self.ref_Z or torch.equal(Z, self.ref_Z))
                and ((cell is None) == (self.ref_cell is None)) and (cell is None or torch.equal(cell.detach(), self.ref_cell))):
            moved = float((p - self.ref_pos).norm(dim=1).max())          # one scalar read-back per step
            if moved < 0.5 * self.skin:
                self.reuses += 1
                return self.graph
        self.graph = self.model.build_graph(p, Z, cell, None, skin=self.skin) if self.skin > 0.0 else \
            self.model.build_graph(p, Z, cell, None)
        self.ref_pos, self.ref_Z = p.clone(), Z
        self.ref_cell = None if cell is None else cell.detach().clone()
        self.builds += 1
        return self.graph


def velocity_verlet_device(model, numbers, positions, cell, velocities, steps: int, dt_fs: float = 0.5, device="cuda",
                           skin: float = 0.0, stats: dict = None, cuda_graph: bool = False, virial: bool = False):
    """Device-resident MD (SURVEY 8(f) rank 1): positions, velocities and forces never leave the GPU; with ``skin > 0`` the
    neighbour list / row CSR / tile plans are re-used across steps (``VerletGraph``), otherwise rebuilt per step (device
    cell list).  ``stats`` (optional dict) receives the build / re-use counts and, with ``virial``, ``stats["virial"]``: the
    global virial after each step's force evaluation, ``[steps, 3, 3]`` on the device (``model.energy_forces_virial``: the
    same single backward pass plus one per-atom virial kernel and its sum)."""
    dev = torch.device(device)
    Z = torch.as_tensor(np.asarray(numbers)).long().to(dev)
    pos = torch.as_tensor(np.asarray(positions), dtype=torch.float32).to(dev)
    vel = torch.as_tensor(np.asarray(velocities), dtype=torch.float32).to(dev).clone()      # (never the caller's buffer)
    c = torch.as_tensor(np.asarray(cell), dtype=torch.float32).reshape(1, 3, 3).to(dev)
    masses = np.array([MASSES.get(int(z), 2.0 * int(z)) for z in np.asarray(numbers)])
    inv_m = torch.as_tensor(1.0 / (masses * AMU_A2_FS2_TO_EV), dtype=torch.float32).to(dev)[:, None]
    vg = VerletGraph(model, skin, cuda_graph, virial)

    def forces(p):
        if vg.cuda_graph:
            out = vg.energy_and_gradient(p, Z, c)
            # (static outputs of the capture: copy what outlives the next call)
            return (out[0].clone(), -out[1]) + ((out[2].clone(),) if virial else ())
        d = Data(pos=p.detach().requires_grad_(True), atomic_number=Z, cell=c)
        d.graph = vg.get(d.pos, Z, c)
        if virial:
            out = model.energy_forces_virial(d)
            return out["energy"], out["forces"], out["virial"]
        e = model(d)
        (g,) = torch.autograd.grad(e.sum(), d.pos)
        return e.detach(), -g

    e, f = forces(pos)[:2]
    energies, virials = [], []
    for _ in range(steps):
        _kick(vel, f, inv_m, dt_fs)
        pos = pos + dt_fs * vel
        e, f, *w = forces(pos)
        _kick(vel, f, inv_m, dt_fs)
        energies.append(e)
        virials += w
    if stats is not None:
        stats.update(builds=vg.builds, reuses=vg.reuses)
        if virial:
            stats["virial"] = torch.cat(virials) if virials else c.new_zeros((0, 3, 3))
    return pos, vel, torch.cat(energies)
