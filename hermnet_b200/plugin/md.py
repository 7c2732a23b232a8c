"""MD without ASE, on the host and on the device.

Host: ASE is not installed in this image, so this module supplies the two pieces of ASE the calculator plugin path needs
(BASELINE.json configs[2]) -- ``SimpleAtoms``, an ``Atoms``-like container, and ``velocity_verlet``, a host velocity-Verlet
loop -- with ASE's attribute names, so ``NNCalculator`` is exercised exactly as ASE would drive it (``atoms.get_forces()``
-> ``calc.calculate(atoms)``).

Device (SURVEY 8(f) rank 1): positions, velocities and forces stay on the GPU.  ``velocity_verlet_device`` (NVE),
``langevin_device`` (NVT), ``langevin_npt_device`` (NPT), ``relax.fire_relax_device`` (FIRE) and ``neb.neb_device`` (NEB)
share the input set-up (``_setup``: atoms, replicas of a PyG-style batch, cell) and one evaluation,
``VerletGraph.evaluate``: a Verlet-skin list re-used across steps, eager or replayed as a captured CUDA graph."""
from __future__ import annotations

import math
from types import SimpleNamespace

import numpy as np
import torch

from .. import ops
from ..graphed import GraphedForces
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

    def __init__(self, model, skin: float = 0.0, cuda_graph: bool = False, virial: bool = False, batch=None,
                 deforming: bool = False):
        self.model, self.skin = model, float(skin)
        self.batch = batch            # [N] replica of each atom (contiguous), passed to build_graph; None: one system
        # deforming: the cell may change between calls (constant-pressure MD); a list is then re-used under the
        # affine criterion of ``_fits_deformed`` instead of being rebuilt whenever the cell differs
        self.deforming = bool(deforming)
        self.virial = bool(virial)    # evaluate also returns the per-graph virial (energy_forces_virial)
        self.graph, self.ref_pos, self.ref_cell, self.ref_Z = None, None, None, None
        self.builds = self.reuses = 0
        # cuda_graph: while a list is re-used, replay the whole evaluation (forward + backward, ~200 launches + torch glue) as
        # ONE captured CUDA graph -- small systems are bound by host launch latency, not by the kernels
        self.cuda_graph = bool(cuda_graph) and self.skin > 0.0
        self._captured, self._captured_for = None, None

    def counts(self) -> dict:
        """The ``builds`` / ``reuses`` entries of a driver's ``stats``."""
        return dict(builds=self.builds, reuses=self.reuses)

    def evaluate(self, pos, Z, cell):
        """``(energy [num_graphs], forces [N,3])`` at ``pos`` (cell ``[num_graphs,3,3]`` or None) through the re-used (or
        rebuilt) list, plus the virial ``[num_graphs,3,3]`` with ``virial``.  With ``cuda_graph`` and a CUDA ``pos``, the same
        evaluation is captured once per list build and replayed afterwards (the parameters must be frozen); the returned
        tensors are then copies of the capture's static outputs, so they outlive the next call.  Elsewhere it runs eagerly."""
        g = self.get(pos, Z, cell)
        if self.cuda_graph and pos.is_cuda:
            if self._captured_for is not g:
                if any(p.requires_grad for p in self.model.parameters()):
                    raise RuntimeError("hermnet_b200.VerletGraph: freeze the parameters first (cuda_graph is inference only)")
                # (a Verlet-skin superset list works: its per-call live mask is computed by device kernels inside the capture)
                self._captured = GraphedForces(lambda p: self._evaluate_on(p, Z, cell, g), pos, warmup=1)
                self._captured_for = g
            out = self._captured(pos)
            out = tuple(t.clone() for t in out) if self.virial else (out[0].clone(), out[1])
        else:
            out = self._evaluate_on(pos, Z, cell, g)
        return out if self.virial else (out[0], -out[1])     # (on a replay the negation is also the copy of dE/dpos)

    def _evaluate_on(self, pos, Z, cell, g):
        """``(energy, forces, virial)`` of ``model.energy_forces_virial_graph`` with ``virial``, else ``(energy, dE/dpos)`` of
        ``model.forward_graph``: what ``model(data)`` / ``model.energy_forces_virial(data)`` compute on an attached graph."""
        if self.virial:
            out = self.model.energy_forces_virial_graph(pos, Z, cell, g)
            return out["energy"], out["forces"], out["virial"]
        p = pos.detach().requires_grad_(True)
        e, _, _ = self.model.forward_graph(p, Z, cell, g)
        (grad,) = torch.autograd.grad(e.sum(), p)
        return e.detach(), grad

    def get(self, pos, Z, cell):
        p = pos.detach()
        if (self.graph is not None and self.skin > 0.0 and p.shape == self.ref_pos.shape and (Z is self.ref_Z or torch.equal(Z, self.ref_Z))
                and ((cell is None) == (self.ref_cell is None))):
            if cell is None or torch.equal(cell.detach(), self.ref_cell):
                moved = float((p - self.ref_pos).norm(dim=1).max())          # one scalar read-back per step
                if moved < 0.5 * self.skin:
                    self.reuses += 1
                    return self.graph
            elif self.deforming and cell.shape == self.ref_cell.shape and self._fits_deformed(p, cell.detach()):
                self.reuses += 1
                return self.graph
        self.graph = self.model.build_graph(p, Z, cell, self.batch, skin=self.skin) if self.skin > 0.0 else \
            self.model.build_graph(p, Z, cell, self.batch)
        self.ref_pos, self.ref_Z = p.clone(), Z
        self.ref_cell = None if cell is None else cell.detach().clone()
        self.builds += 1
        return self.graph

    def _fits_deformed(self, p, cell) -> bool:
        """Whether the list built at ``(ref_pos, ref_cell)`` still holds every pair closer than ``rc`` at ``(p, cell)``.
        Per replica ``M = ref_cell^-1 cell`` (row vectors) and ``u_i = p_i - ref_pos_i M``; for fixed integer shifts every
        edge vector is then exactly ``D = D_ref M + u_src - u_dst``, so a pair left out of the list (``|D_ref| >= rc +
        skin``) has ``|D| >= (rc + skin) sigma_min(M) - 2 max|u|``, and the list is complete while that bound exceeds
        ``rc`` in every replica.  float64; one scalar read-back."""
        c0, c1 = self.ref_cell.reshape(-1, 3, 3).double(), cell.reshape(-1, 3, 3).double()
        inv0 = torch.stack([torch.linalg.cross(c0[:, 1], c0[:, 2]), torch.linalg.cross(c0[:, 2], c0[:, 0]),
                            torch.linalg.cross(c0[:, 0], c0[:, 1])], -1) / _det3(c0)[:, None, None]
        M = (inv0[:, :, :, None] * c1[:, None, :, :]).sum(2)
        s_min = _sigma_min3(M)
        rep = self.batch if self.batch is not None else torch.zeros(p.size(0), dtype=torch.long, device=p.device)
        u = p.double() - (self.ref_pos.double()[:, :, None] * M[rep]).sum(1)
        u_max = torch.zeros(M.size(0), dtype=torch.float64, device=p.device).scatter_reduce(
            0, rep, u.norm(dim=1), "amax", include_self=True)
        rc = self.graph.list_rc - self.skin
        return float(((rc + self.skin) * s_min - 2.0 * u_max - rc).min()) > 0.0


def _sigma_min3(M):
    """Smallest singular value of ``[..., 3, 3]``: square root of the smallest eigenvalue of ``M^T M`` in closed form
    (trigonometric solution of the symmetric 3x3 eigenproblem; exact for ``M ~ I`` too, where it reduces to ``tr / 3``)."""
    A = (M[..., :, :, None] * M[..., :, None, :]).sum(-3)
    q = A.diagonal(dim1=-2, dim2=-1).sum(-1) / 3.0
    B = A - q[..., None, None] * torch.eye(3, dtype=A.dtype, device=A.device)
    sd = torch.sqrt((B * B).sum((-2, -1)) / 6.0)
    r = (_det3(B / torch.where(sd > 0, sd, 1.0)[..., None, None]) / 2.0).clamp(-1.0, 1.0)
    return torch.sqrt((q + 2.0 * sd * torch.cos(torch.acos(r) / 3.0 + 2.0 * math.pi / 3.0)).clamp(min=0.0))


def _det3(a):
    """Determinant of ``[..., 3, 3]`` (element-wise; row or column convention alike)."""
    return (a[..., 0, 0] * (a[..., 1, 1] * a[..., 2, 2] - a[..., 1, 2] * a[..., 2, 1])
            - a[..., 0, 1] * (a[..., 1, 0] * a[..., 2, 2] - a[..., 1, 2] * a[..., 2, 0])
            + a[..., 0, 2] * (a[..., 1, 0] * a[..., 2, 1] - a[..., 1, 1] * a[..., 2, 0]))


def _inv_mass(numbers, dev):
    masses = np.array([MASSES.get(int(z), 2.0 * int(z)) for z in np.asarray(numbers)])
    return torch.as_tensor(1.0 / (masses * AMU_A2_FS2_TO_EV), dtype=torch.float32).to(dev)


def velocity_verlet_device(model, numbers, positions, cell, velocities, steps: int, dt_fs: float = 0.5, device="cuda",
                           skin: float = 0.0, stats: dict = None, cuda_graph: bool = False, virial: bool = False):
    """Device-resident MD (SURVEY 8(f) rank 1): positions, velocities and forces never leave the GPU; with ``skin > 0`` the
    neighbour list / row CSR / tile plans are re-used across steps (``VerletGraph``), otherwise rebuilt per step (device
    cell list).  ``stats`` (optional dict) receives the build / re-use counts and, with ``virial``, ``stats["virial"]``: the
    global virial after each step's force evaluation, ``[steps, 3, 3]`` on the device (``model.energy_forces_virial``: the
    same single backward pass plus one per-atom virial kernel and its sum)."""
    st = _setup("velocity_verlet_device", numbers, positions, cell, None, device)
    pos = st.pos
    vel = torch.as_tensor(velocities, dtype=torch.float32, device=pos.device).clone()      # (never the caller's buffer)
    inv_m = _inv_mass(st.numbers, pos.device)[:, None]
    vg = VerletGraph(model, skin, cuda_graph, virial)

    e, f = vg.evaluate(pos, st.Z, st.c)[:2]
    energies, virials = [], []
    for _ in range(steps):
        _kick(vel, f, inv_m, dt_fs)
        pos = pos + dt_fs * vel
        e, f, *w = vg.evaluate(pos, st.Z, st.c)
        _kick(vel, f, inv_m, dt_fs)
        energies.append(e)
        virials += w
    if stats is not None:
        stats.update(vg.counts())
        if virial:
            stats["virial"] = torch.cat(virials) if virials else st.c.new_zeros((0, 3, 3))
    return pos, vel, torch.cat(energies)


def _host(x) -> np.ndarray:
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def _replicas(batch, n: int, name: str):
    """``(G, replica_ptr int64 [G+1])`` of a PyG-style batch vector: non-decreasing, every replica 0..G-1 non-empty."""
    if batch is None:
        return 1, np.array([0, n], dtype=np.int64)
    b = _host(batch).astype(np.int64).reshape(-1)
    if b.size != n or n == 0:
        raise ValueError(f"{name}: batch must have one entry per atom ({n}), got {b.size}")
    step = np.diff(b)
    if b[0] != 0 or (step < 0).any() or (step > 1).any():
        raise ValueError(f"{name}: batch must be sorted with replicas 0..G-1 all non-empty (a PyG batch vector)")
    G = int(b[-1]) + 1
    return G, np.concatenate([[0], np.cumsum(np.bincount(b, minlength=G))]).astype(np.int64)


def _per_replica(value, G: int, what: str, name: str) -> np.ndarray:
    """``value`` (one value or ``G`` values) as ``G`` values, as given."""
    v = _host(value)
    v = np.full(G, v) if v.ndim == 0 else v.reshape(-1)
    if v.size != G:
        raise ValueError(f"{name}: {what} has {v.size} values for {G} replicas")
    return v


def _replica_floats(value, G: int, what: str, name: str, ok, must: str) -> np.ndarray:
    """``value`` (a float or ``G`` values) as ``G`` float64 values; ``ValueError`` with ``must`` unless ``ok`` holds for all."""
    v = _per_replica(value, G, what, name).astype(np.float64)
    if not ok(v).all():
        raise ValueError(f"{name}: {must}")
    return v


def _setup(name, numbers, positions, cell, batch, device, cell_error=None):
    """Validated inputs of a device driver: ``n``, ``G``, ``sizes [G]`` and ``numbers`` on the host, ``replica_ptr [G+1]`` /
    ``replica [N]`` (int32), ``batch`` for ``VerletGraph`` (None for one replica), ``Z``, a private float32 copy of ``pos`` and
    the float32 cell ``c [G,3,3]`` (a ``[3,3]`` cell is shared) or None.  With ``cell_error``, a missing, non-finite or
    singular cell raises ``ValueError`` with that message."""
    numbers = _host(numbers)
    n = len(numbers)
    G, rptr = _replicas(batch, n, name)
    c_np = None if cell is None else _host(cell).astype(np.float64).reshape(-1, 3, 3)
    if c_np is not None and c_np.shape[0] not in (1, G):
        raise ValueError(f"{name}: cell must be [3,3] or [{G},3,3]")
    if cell_error and (c_np is None or not np.isfinite(c_np).all() or not (np.abs(np.linalg.det(c_np)) > 0.0).all()):
        raise ValueError(f"{name}: {cell_error}")

    dev = torch.device(device)
    sizes = np.diff(rptr)
    replica = torch.repeat_interleave(torch.arange(G, dtype=torch.int32), torch.from_numpy(sizes)).to(dev)
    return SimpleNamespace(
        n=n, G=G, sizes=sizes, numbers=numbers, replica_ptr=torch.from_numpy(rptr).to(dev, torch.int32), replica=replica,
        batch=None if batch is None else replica.long(), Z=torch.as_tensor(numbers).long().to(dev),
        # (never the caller's buffers; device tensors are accepted, e.g. the pos of a previous call to continue from)
        pos=torch.as_tensor(positions, dtype=torch.float32, device=dev).reshape(n, 3).clone(),
        c=None if c_np is None else torch.from_numpy(np.repeat(c_np.astype(np.float32), G // c_np.shape[0], axis=0)).to(dev))


def _stack(trace, like, *shape):
    """The per-step ``trace`` as one ``[steps, *shape]`` tensor (``like``'s dtype and device when there are no steps)."""
    return torch.stack(trace) if trace else like.new_zeros((0, *shape))


def _langevin_state(name, numbers, positions, cell, velocities, dt_fs, temperature_K, friction_per_fs, seed, batch, step0,
                    device, cell_error=None):
    """``_setup`` plus the Langevin state shared by ``langevin_device`` and ``langevin_npt_device``: velocities, inverse
    masses, ``kT``, seeds, the step counter, the per-atom kinetic energies, ``c1`` / ``c2`` and ``t_scale``."""
    if not dt_fs > 0.0:
        raise ValueError(f"{name}: dt_fs must be > 0 (got {dt_fs})")
    if not friction_per_fs >= 0.0:
        raise ValueError(f"{name}: friction_per_fs must be >= 0 (got {friction_per_fs})")
    st = _setup(name, numbers, positions, cell, batch, device, cell_error)
    G = st.G
    T = _replica_floats(temperature_K, G, "temperature_K", name, lambda t: t >= 0.0, "temperatures must be >= 0")
    seeds = [int(seed) + g for g in range(G)] if np.ndim(seed) == 0 else [int(s) for s in _per_replica(seed, G, "seed", name)]
    if not all(0 <= s < 2 ** 63 for s in seeds):
        raise ValueError(f"{name}: seeds must be in [0, 2^63)")
    if not 0 <= int(step0) < 2 ** 63:
        raise ValueError(f"{name}: step0 must be in [0, 2^63)")

    dev = st.pos.device
    st.vel = torch.as_tensor(velocities, dtype=torch.float32, device=dev).clone()
    st.inv_m = _inv_mass(st.numbers, dev)
    st.kT = torch.from_numpy(KB_EV * T).to(dev, torch.float32)
    st.seed = torch.tensor(seeds, dtype=torch.int64, device=dev)
    st.step = torch.tensor([int(step0)], dtype=torch.int64, device=dev)
    st.kinetic = torch.empty(st.n, dtype=torch.float32, device=dev)
    st.t_scale = torch.from_numpy(2.0 / (3.0 * st.sizes * KB_EV)).to(dev, torch.float32)
    gdt = float(friction_per_fs) * float(dt_fs)
    st.c1, st.c2 = math.exp(-gdt), math.sqrt(-math.expm1(-2.0 * gdt))
    return st


def langevin_device(model, numbers, positions, cell, velocities, steps: int, dt_fs: float = 0.5, temperature_K=300.0,
                    friction_per_fs: float = 0.01, seed=0, batch=None, step0: int = 0, device="cuda", skin: float = 0.0,
                    stats: dict = None, cuda_graph: bool = False, virial: bool = False):
    """Device-resident Langevin (NVT) MD: BAOAB (Leimkuhler-Matthews) with friction ``gamma = friction_per_fs`` (1/fs) over
    ``G`` independent replicas integrated together, each at its own temperature.  Returns ``(pos [N,3], vel [N,3],
    energies [steps, G])``; positions, velocities and forces never leave the GPU.

    ``batch``: ``None`` (one replica) or ``[N]`` replica of each atom, non-decreasing with every replica ``0..G-1``
    non-empty (a PyG batch vector).  ``cell``: ``[3,3]`` (shared) or ``[G,3,3]``.  ``temperature_K``: a float or ``G``
    values.  ``seed``: an int (replica ``g`` gets ``seed + g``) or ``G`` ints in ``[0, 2^63)``.  ``step0``: the first value
    of the noise counter -- a run continued from returned ``pos`` / ``vel`` with ``step0 = stats["step"]`` reproduces the
    uninterrupted trajectory bitwise (same skin / evaluation mode).

    Noise is Philox4x32-10 keyed on (replica seed, replica-local atom index, step) (``hn_md_langevin_baoa``): trajectories
    are bitwise reproducible, identical eager and with ``cuda_graph``, and a replica's noise does not depend on the batch it
    is run in.  The step is two fused kernels (``ops.md_langevin_baoa`` before the force evaluation, ``ops.md_kick`` after
    it) around the same evaluation as ``velocity_verlet_device``: ``skin`` list re-use, ``cuda_graph`` replay of the
    evaluation (the two integrator kernels stay eager around it) and ``virial``.  The counter and the temperatures live in
    device memory, so the loop adds no host synchronisation beyond the skin check.

    ``stats`` (optional dict) receives ``builds`` / ``reuses``, ``temperature [steps, G]`` (``2 KE_g / (3 n_g k_B)`` after
    each step, no centre-of-mass correction: Langevin dynamics does not conserve momentum), ``virial [steps, G, 3, 3]``
    with ``virial=True`` and ``step``, the final counter value."""
    st = _langevin_state("langevin_device", numbers, positions, cell, velocities, dt_fs, temperature_K, friction_per_fs, seed,
                         batch, step0, device)
    G, pos, vel, inv_m, replica_ptr, kT, step, kinetic = st.G, st.pos, st.vel, st.inv_m, st.replica_ptr, st.kT, st.step, st.kinetic
    vg = VerletGraph(model, skin, cuda_graph, virial, batch=st.batch)
    e, f = vg.evaluate(pos, st.Z, st.c)[:2]
    energies, temps, virials = [], [], []
    for _ in range(steps):
        ops.md_langevin_baoa(pos, vel, f, inv_m, st.replica, replica_ptr, kT, st.seed, step, st.c1, st.c2, dt_fs)
        e, f, *w = vg.evaluate(pos, st.Z, st.c)
        ops.md_kick(vel, f, inv_m, 0.5 * dt_fs, kinetic, step)
        energies.append(e)
        temps.append(ops.segment_sum(kinetic[:, None], replica_ptr, None, G)[:, 0] * st.t_scale)
        virials += w
    if stats is not None:
        stats.update(vg.counts(), step=int(step.item()), temperature=_stack(temps, kT, G))
        if virial:
            stats["virial"] = _stack(virials, kT, G, 3, 3)
    return pos, vel, _stack(energies, kT, G)


EV_A3_TO_BAR = 1.602176634e6       # 1 eV/A^3 in bar


def langevin_npt_device(model, numbers, positions, cell, velocities, steps: int, dt_fs: float = 0.5, temperature_K=300.0,
                        pressure_bar=1.0, compressibility_per_bar=4.5e-5, tau_p_fs: float = 1000.0,
                        friction_per_fs: float = 0.01, seed=0, batch=None, step0: int = 0, device="cuda", skin: float = 0.0,
                        stats: dict = None, cuda_graph: bool = False, forces=None, cell_dof: str = "isotropic"):
    """Device-resident constant-pressure (NPT) MD: the ``langevin_device`` step followed by isotropic stochastic cell
    rescaling (Bernetti & Bussi 2020) of every replica towards its own pressure.  Returns ``(pos [N,3], vel [N,3],
    cell [G,3,3], energies [steps, G])``; positions, velocities, cells and forces never leave the GPU.

    ``batch``, ``cell`` (required, non-singular), ``temperature_K``, ``friction_per_fs``, ``seed`` and ``step0`` as in
    ``langevin_device``.  ``pressure_bar`` (any finite value; negative is tension) and ``compressibility_per_bar`` (the
    isothermal compressibility ``beta_T >= 0``; 0 keeps the cell fixed and reproduces ``langevin_device`` bitwise) are a
    float or ``G`` values; ``tau_p_fs > 0`` is the barostat relaxation time.  Each step is BAOAB's B-A-O-A
    (``ops.md_langevin_baoa``), the evaluation with the virial, the closing B (``ops.md_kick``), then per replica the
    internal pressure ``(2 K + tr W) / 3V`` and the strain step (``ops.md_scr_barostat``, noise on counter word 3 = 1) and
    the affine scaling of positions and velocities (``ops.md_affine_scale``).  The next step's first B uses the forces of
    the unscaled positions (first order in the strain per step, as GROMACS's C-rescale).  Pressures, compressibilities,
    temperatures, seeds, the step counter and the cells live in device memory: a captured evaluation keeps reading the
    cell tensor the barostat scales in place.  ``skin`` lists are re-used across cell changes while the affine criterion of
    ``VerletGraph(deforming=True)`` holds.  Because the first B of a step uses the forces of the previous step's unscaled
    positions, the state of a run is ``pos`` / ``vel`` / ``cell`` plus those forces: a run continued from the returned
    ``pos`` / ``vel`` / ``cell`` with ``step0 = stats["step"]`` and ``forces = stats["forces"]`` reproduces the
    uninterrupted trajectory bitwise (same skin / evaluation mode).  ``forces=None`` evaluates them at ``positions``.

    ``cell_dof="triclinic"`` frees the cell's shape under the hydrostatic target pressure: every replica's cell must then be
    lower-triangular with a positive diagonal (``a`` along x, ``b`` in the xy plane; ``standard_cell`` rotates a system into
    that form).  The cell step is then the triclinic stochastic cell rescaling of DESIGN.md: the per-replica kinetic tensor
    (``ops.md_kinetic_tensor`` and a segment sum), a lower-triangular strain ``mu`` from the pressure tensor
    (``ops.md_scr_barostat_tri``, noise on counter word 3 = 2) and ``x <- x mu``, ``v <- v mu^-T``
    (``ops.md_affine_deform``).  Zero compressibility again reproduces ``langevin_device`` bitwise, and restarts, ``skin``
    and ``cuda_graph`` work as in the isotropic mode.

    ``stats`` (optional dict) receives ``builds`` / ``reuses``, ``step``, ``temperature [steps, G]`` (K),
    ``pressure [steps, G]`` (bar: the internal pressure of the post-kick state, before the cell step), ``volume
    [steps, G]`` (A^3, after the cell step) and ``virial [steps, G, 3, 3]`` (eV); with ``cell_dof="triclinic"`` also
    ``cell [steps, G, 3, 3]`` (after the cell step) and ``pressure_tensor [steps, G, 3, 3]`` (bar, of the post-kick state;
    ``pressure`` is a third of its trace)."""
    name = "langevin_npt_device"
    if not tau_p_fs > 0.0:
        raise ValueError(f"{name}: tau_p_fs must be > 0 (got {tau_p_fs})")
    if cell_dof not in ("isotropic", "triclinic"):
        raise ValueError(f"{name}: cell_dof must be 'isotropic' or 'triclinic' (got {cell_dof!r})")
    st = _langevin_state(name, numbers, positions, cell, velocities, dt_fs, temperature_K, friction_per_fs, seed, batch, step0,
                         device, cell_error="a finite, non-singular periodic cell is required")
    G = st.G
    if cell_dof == "triclinic":
        h = st.c.detach().cpu().double()
        if not (torch.equal(h.triu(1), torch.zeros_like(h)) and bool((h.diagonal(dim1=1, dim2=2) > 0.0).all())):
            raise ValueError(f"{name}: cell_dof='triclinic' needs every cell lower-triangular with a positive diagonal "
                             "(rotate the system with plugin.md.standard_cell)")
    P0 = _replica_floats(pressure_bar, G, "pressure_bar", name, np.isfinite, "pressures must be finite")
    beta = _replica_floats(compressibility_per_bar, G, "compressibility_per_bar", name, lambda b: np.isfinite(b) & (b >= 0.0),
                           "compressibilities must be finite and >= 0")

    pos, vel, c, inv_m, replica_ptr, kT, step, kinetic = st.pos, st.vel, st.c, st.inv_m, st.replica_ptr, st.kT, st.step, st.kinetic
    dev = pos.device
    P0_t = torch.from_numpy(P0 / EV_A3_TO_BAR).to(dev, torch.float32)            # eV/A^3
    beta_t = torch.from_numpy(beta * EV_A3_TO_BAR).to(dev, torch.float32)        # A^3/eV

    vg = VerletGraph(model, skin, cuda_graph, True, batch=st.batch, deforming=True)
    if forces is None:
        f = vg.evaluate(pos, st.Z, c)[1]
    else:
        f = torch.as_tensor(forces, dtype=torch.float32, device=dev).clone()
        if tuple(f.shape) != (st.n, 3):
            raise ValueError(f"{name}: forces must be [{st.n},3]")
    if cell_dof == "triclinic":
        return _npt_triclinic(st, vg, f, steps, dt_fs, tau_p_fs, P0_t, beta_t, stats)
    mu, pressure = torch.ones(G, dtype=torch.float32, device=dev), torch.zeros(G, dtype=torch.float32, device=dev)
    energies, temps, virials, pressures, cells = [], [], [], [], []
    for _ in range(steps):
        ops.md_langevin_baoa(pos, vel, f, inv_m, st.replica, replica_ptr, kT, st.seed, step, st.c1, st.c2, dt_fs)
        e, f, w = vg.evaluate(pos, st.Z, c)
        ops.md_kick(vel, f, inv_m, 0.5 * dt_fs, kinetic, step)
        ke = ops.segment_sum(kinetic[:, None], replica_ptr, None, G)[:, 0]
        w = w.contiguous()
        ops.md_scr_barostat(c, ke, w, P0_t, kT, beta_t, st.seed, step, dt_fs, tau_p_fs, mu, pressure)
        ops.md_affine_scale(pos, vel, st.replica, mu)
        energies.append(e)
        temps.append(ke * st.t_scale)
        virials.append(w)
        pressures.append(pressure.clone())
        cells.append(c.clone())
    if stats is not None:
        stats.update(vg.counts(), step=int(step.item()), temperature=_stack(temps, kT, G),
                     pressure=_stack(pressures, kT, G) * EV_A3_TO_BAR,
                     volume=_det3(_stack(cells, c, G, 3, 3).double()).abs().float(), virial=_stack(virials, kT, G, 3, 3), forces=f)
    return pos, vel, c, _stack(energies, kT, G)


def _npt_triclinic(st, vg, f, steps, dt_fs, tau_p_fs, P0_t, beta_t, stats):
    """The step loop of ``langevin_npt_device(cell_dof="triclinic")`` from its validated state ``st``, evaluation ``vg`` and
    first forces ``f``."""
    G, pos, vel, c, inv_m, replica_ptr, kT, step, kinetic = st.G, st.pos, st.vel, st.c, st.inv_m, st.replica_ptr, st.kT, st.step, \
        st.kinetic
    mu, mu_inv_t, ptensor = (torch.zeros(G, 3, 3, dtype=torch.float32, device=pos.device) for _ in range(3))
    energies, temps, virials, ptensors, cells = [], [], [], [], []
    for _ in range(steps):
        ops.md_langevin_baoa(pos, vel, f, inv_m, st.replica, replica_ptr, kT, st.seed, step, st.c1, st.c2, dt_fs)
        e, f, w = vg.evaluate(pos, st.Z, c)
        ops.md_kick(vel, f, inv_m, 0.5 * dt_fs, kinetic, step)
        ke = ops.segment_sum(kinetic[:, None], replica_ptr, None, G)[:, 0]
        kin6 = ops.segment_sum(ops.md_kinetic_tensor(vel, inv_m), replica_ptr, None, G)
        w = w.contiguous()
        ops.md_scr_barostat_tri(c, kin6, w, P0_t, kT, beta_t, st.seed, step, dt_fs, tau_p_fs, mu, mu_inv_t, ptensor)
        ops.md_affine_deform(pos, vel, st.replica, mu, mu_inv_t)
        energies.append(e)
        temps.append(ke * st.t_scale)
        virials.append(w)
        ptensors.append(ptensor.clone())
        cells.append(c.clone())
    if stats is not None:
        pt = _stack(ptensors, kT, G, 3, 3) * EV_A3_TO_BAR
        cs = _stack(cells, c, G, 3, 3)
        stats.update(vg.counts(), step=int(step.item()), temperature=_stack(temps, kT, G),
                     pressure=pt.diagonal(dim1=2, dim2=3).sum(-1) / 3.0, volume=_det3(cs.double()).abs().float(),
                     virial=_stack(virials, kT, G, 3, 3), forces=f, cell=cs, pressure_tensor=pt)
    return pos, vel, c, _stack(energies, kT, G)


def standard_cell(positions, cell, velocities=None, batch=None):
    """Rotate each replica into the lower-triangular cell form ``langevin_npt_device(cell_dof="triclinic")`` needs: lattice
    vector ``a`` along x, ``b`` in the xy plane, positive diagonal (ASE's and LAMMPS's standard orientation).  Per replica
    ``g`` the LQ factorisation ``h = L Q`` (lattice vectors = rows of ``h``, ``diag L > 0``) gives the rotation ``R = Q^T``,
    and ``x R``, ``v R``, ``L`` are returned as float64 numpy ``(positions [N,3], cell, velocities [N,3] or None)``; the cell
    keeps the input's ``[3,3]`` or ``[G,3,3]`` shape, with its upper triangle exactly 0.  ``batch`` as in the drivers (None:
    one system).  Distances, energies and the model's forces (rotated by ``R``) are unchanged.  A left-handed cell
    (``det h < 0``) raises ``ValueError``: no rotation makes it lower-triangular with a positive diagonal."""
    x = _host(positions).astype(np.float64).reshape(-1, 3)
    n = len(x)
    G, rptr = _replicas(batch, n, "standard_cell")
    h = _host(cell).astype(np.float64)
    hs = h.reshape(-1, 3, 3)
    if hs.shape[0] not in (1, G):
        raise ValueError(f"standard_cell: cell must be [3,3] or [{G},3,3]")
    if not np.isfinite(hs).all() or not (np.linalg.det(hs) > 0.0).all():
        raise ValueError("standard_cell: every cell must be finite and right-handed (det h > 0)")
    q, r = np.linalg.qr(np.swapaxes(hs, 1, 2))          # h^T = q r  ->  h = r^T q^T, L = r^T
    sgn = np.sign(np.diagonal(r, axis1=1, axis2=2))
    L = np.tril(np.swapaxes(r, 1, 2) * sgn[:, None, :])
    R = q * sgn[:, None, :]                              # h R = L with R = q diag(sgn), a rotation since det h > 0
    rep = np.repeat(np.arange(G) if hs.shape[0] == G else np.zeros(G, dtype=np.int64), np.diff(rptr))
    rot = lambda a: np.einsum("ni,nij->nj", a, R[rep])  # noqa: E731
    v = None if velocities is None else rot(_host(velocities).astype(np.float64).reshape(n, 3))
    return rot(x), L.reshape(h.shape), v
