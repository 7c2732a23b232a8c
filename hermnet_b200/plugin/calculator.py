"""ASE-style calculator on the B200 hot path -- functional counterpart of
``/root/reference/plugin/ase_interface/calculator.py`` (same names, constructor arguments, result keys).

The shipped reference calculator cannot run (SURVEY F6: ``model.rc`` missing, ``cell [3,3]`` vs ``[1,3,3]``,
``torch.from_numpy`` on a tensor, missing ``batch``, stress built from ``virial[0,1]``).  Here the same entry points
work; ``compat_stress=True`` keeps the reference's stress-vector ordering (calculator.py:93-95), the default is
proper Voigt order ``[xx, yy, zz, yz, xz, xy]``.  ASE itself is not installed in this image: when it is importable
``NNCalculator`` derives from ``ase.calculators.calculator.Calculator``, otherwise from a small stand-in with the same
``calculate`` / ``results`` / ``get_*`` surface, so MD drivers (``md.velocity_verlet``) can run either way.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch
from torch import nn

from ..data import Data
from ..symbols import atomic_numbers
from ..utils import NKTV2P, virial_calc

try:  # pragma: no cover - ASE is absent from the build image
    from ase.calculators.calculator import Calculator, all_changes
except Exception:  # noqa: BLE001
    all_changes = ["positions", "numbers", "cell", "pbc", "initial_charges", "initial_magmoms"]

    class Calculator:  # minimal stand-in for ase.calculators.calculator.Calculator
        implemented_properties = []

        def __init__(self, *args, **kwargs):
            self.results, self.atoms = {}, None

        def calculate(self, atoms=None, properties=None, system_changes=all_changes):
            self.atoms = atoms

        def get_potential_energy(self, atoms=None):
            self.calculate(atoms or self.atoms, ["energy"])
            return self.results["energy"]

        def get_forces(self, atoms=None):
            self.calculate(atoms or self.atoms, ["forces"])
            return self.results["forces"]

        def get_stress(self, atoms=None):
            self.calculate(atoms or self.atoms, ["stress"])
            return self.results["stress"]

        def get_potential_energies(self, atoms=None):
            self.calculate(atoms or self.atoms, ["energies"])
            return self.results["energies"]

        def get_stresses(self, atoms=None):
            self.calculate(atoms or self.atoms, ["stresses"])
            return self.results["stresses"]


def build_graph(cell, elements, pos, rc, device="cuda"):
    """calculator.py:10-27 made functional: numpy in, device-resident ``Data`` out.  The neighbour list is NOT built
    here on the CPU: the model builds its row CSR on the GPU from ``pos`` / ``cell`` (``RowGraph``)."""
    pos = torch.as_tensor(np.asarray(pos), dtype=torch.float32)
    data = Data(atomic_number=torch.as_tensor(np.asarray(elements)).long(), pos=pos)
    if cell is not None and np.abs(np.asarray(cell)).sum() > 0:
        data.cell = torch.as_tensor(np.asarray(cell), dtype=torch.float32).reshape(1, 3, 3)
    data.batch = torch.zeros(pos.size(0), dtype=torch.long)
    return data.to(device)


class NNCalculator(Calculator):
    implemented_properties = ['energy', 'free_energy', 'forces', 'stress', 'energies', 'stresses']

    def __init__(self, model: nn.Module, model_path: Optional[str], trn_mean: float, device_: str = 'cuda',
                 ensemble: str = 'NVT', compat_stress: bool = False, skin: float = 0.0):
        super().__init__()
        self.device_ = device_
        device = torch.device(device_)
        self.model = model.to(device)
        if model_path is not None:
            self.model.load_state_dict(torch.load(model_path, map_location=device))
        self.model.eval()
        for p in self.model.parameters():      # inference: frozen parameters -> no filter-weight gradient pass
            p.requires_grad_(False)
        self.trn_mean = trn_mean
        self.ensemble = ensemble
        self.compat_stress = compat_stress
        # skin > 0: Verlet list re-used across calculate() calls while no atom moved more than skin / 2 (md.VerletGraph);
        # 0 = a fresh neighbour list per call, as the reference does (calculator.py:42-57)
        from .md import VerletGraph
        self.verlet = VerletGraph(self.model, skin)

    def calculate(self, atoms, properties=None, system_changes=all_changes):
        super().calculate(atoms=atoms, properties=properties, system_changes=system_changes)
        cell = np.asarray(atoms.cell) if hasattr(atoms, "cell") else atoms.todict()['cell']
        elems = np.array([atomic_numbers[s] for s in atoms.get_chemical_symbols()])
        pbc = bool(np.any(atoms.pbc))
        data = build_graph(cell=cell if pbc else None, elements=elems, pos=atoms.positions, rc=self.model.rc,
                           device=self.device_)
        if properties is not None and ('energies' in properties or 'stresses' in properties):
            self.results.update(self.model_calc_per_atom(data, self.device_, pbc))
            return
        energy, forces, virial = self.model_calc(data=data, device=self.device_, pbc=pbc, ensemble=self.ensemble)
        self.results['energy'] = energy
        self.results['free_energy'] = energy
        self.results['forces'] = forces
        self.results['stress'] = virial

    def model_calc(self, data, device, pbc, ensemble='NVT'):
        """calculator.py:59-99: ``(float energy, ndarray[N,3] forces, ndarray[6] virial)``."""
        data = self._prepare(data, device, pbc)
        data.pos.requires_grad_(True)
        npt = ensemble.lower() == 'npt'
        if npt and pbc:
            data.cell.requires_grad_(True)
        energy = self.model(data) + self.trn_mean
        forces = -torch.autograd.grad(energy.sum(), data.pos, retain_graph=npt and pbc)[0]
        if npt:
            cell = data.cell if pbc else None
            v = virial_calc(cell=cell, pos=data.pos.detach(), forces=forces, energy=energy, units='metal',
                            pbc=pbc).detach().cpu().numpy()
            virial = self._stress_vector(v)
        else:
            virial = np.array([0., 0., 0., 0., 0., 0.], dtype=np.float32)
        return energy.detach().cpu().item(), forces.detach().cpu().view(-1).numpy().reshape(-1, 3), virial

    def model_calc_per_atom(self, data, device, pbc):
        """Every result of ``calculate`` from ONE backward pass (``model.energy_forces_virial``), for any ensemble:
        ``energy`` / ``free_energy``, ``forces``, ``energies [N]`` (``trn_mean`` spread evenly, so they sum to ``energy``),
        ``stresses [N,6]`` (symmetrised per-atom virials in ``stress``'s units and ordering) and ``stress`` (their sum)."""
        data = self._prepare(data, device, pbc)
        out = self.model.energy_forces_virial(data)
        n = out["energies"].numel()
        W = out["virials"].detach().cpu().double().numpy()
        W = 0.5 * (W + W.transpose(0, 2, 1)) * NKTV2P['metal']
        stresses = self._stress_vector(W.transpose(1, 2, 0)).T
        energy = (out["energy"] + self.trn_mean).cpu().item()
        return {'energy': energy, 'free_energy': energy, 'forces': out["forces"].cpu().numpy().reshape(-1, 3),
                'energies': out["energies"].cpu().double().numpy() + self.trn_mean / max(n, 1),
                'stresses': stresses, 'stress': stresses.sum(0)}

    def _prepare(self, data, device, pbc):
        data = data.to(torch.device(device))
        if pbc and self.verlet.skin > 0.0 and data.get("edge_index") is None:
            data.graph = self.verlet.get(data.pos, data.atomic_number, data.get("cell"))
        return data

    def _stress_vector(self, v):
        """6-vector of a symmetric 3x3 virial ``v[a, b, ...]``."""
        if self.compat_stress:   # the reference's ordering, kept for bit-compatibility with its consumers
            return np.array([v[0, 1], v[1, 1], v[2, 2], v[0, 1], v[0, 2], v[1, 2]])
        return np.array([v[0, 0], v[1, 1], v[2, 2], v[1, 2], v[0, 2], v[0, 1]])
