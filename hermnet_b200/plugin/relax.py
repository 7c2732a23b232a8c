"""Device-resident structure relaxation: FIRE over batched replicas, with the unit cell relaxed under a target pressure
if asked for.  The optimizer is ASE's ``FIRE`` (its rules and defaults) applied per replica, over the generalized
coordinates of ASE's ``UnitCellFilter`` -- the route ``FIRE(UnitCellFilter(atoms))`` over ``NNCalculator`` takes one
structure at a time on the host; here every replica of a PyG-style batch relaxes at once and only one integer (the number
of replicas still moving) comes back to the host per step."""
from __future__ import annotations

import numpy as np
import torch

from .. import ops
from .md import EV_A3_TO_BAR, VerletGraph, _det3, _replica_floats, _setup


def fire_relax_device(model, numbers, positions, cell, fmax=0.05, max_steps=1000, batch=None, relax_cell=False,
                      pressure_bar=0.0, cell_factor=None, dt=0.1, dt_max=1.0, max_step=0.2, skin=0.0, cuda_graph=False,
                      stats=None, device="cuda"):
    """Relax ``G`` replicas to ``max_i |F_i| < fmax`` (eV/A) with FIRE, each on its own: own ``dt`` / ``alpha`` / ``n_pos``,
    own convergence (sticky: a converged replica never moves again and keeps its coordinates bitwise), at most
    ``max_steps`` steps.  Returns ``(pos [N,3], cell [G,3,3] or None, energy [G])``, the energy at the returned geometry.

    ``batch``: ``None`` (one replica) or ``[N]`` replica of each atom, non-decreasing with every replica ``0..G-1``
    non-empty.  ``cell``: ``None`` (clusters; not with ``relax_cell``), ``[3,3]`` (shared) or ``[G,3,3]``, rows are the
    lattice vectors.  ``dt``, ``dt_max`` (>= dt), ``max_step`` (A, the cap on a replica's whole step) are ASE's parameters;
    masses are ignored as in ASE.

    ``relax_cell``: ASE's ``UnitCellFilter``.  With ``A = h0^-1 h`` (``h0`` the starting cell) the coordinates are the atom
    rows ``x A^-1`` (forces ``f A^T``) and three cell rows ``c_f A^T`` whose force is ``(W_sym - P0 V I) A^-1 / c_f``:
    ``W_sym`` the symmetrised virial of the force pass (``model.energy_forces_virial``; it is ASE's ``-V sigma``), ``P0`` the
    target pressure (``pressure_bar``, a float or ``G`` values), ``V = |det h|`` and ``c_f`` = ``cell_factor`` (a float or
    ``G`` values; default the replica's atom count, as ASE).  The cell rows count in the norms, in ``F.v`` and in the
    convergence test like atom rows; the stationary point minimises the enthalpy ``E + P0 V``.

    Each iteration is one evaluation (``skin`` lists re-used across steps and, with the cell relaxed, across cell changes;
    ``cuda_graph`` replays the evaluation while a list is re-used), then ``ops.opt_fire_reduce`` (per-replica sums over the
    atoms), ``ops.opt_fire_step`` (per replica in float64: convergence, mixing, ``dt`` / ``alpha``, the ``max_step`` cap in
    closed form, the cell rows) and ``ops.opt_fire_update`` (the atom rows).

    ``stats`` (optional dict) receives ``converged [G]`` (bool), ``steps [G]`` (steps taken), per-evaluation traces
    ``energy``, ``fmax`` (the generalized max force) and, with ``relax_cell``, ``volume`` (A^3), all ``[iters, G]``; the
    optimizer state after each iteration's step, ``dt``, ``alpha`` and ``n_pos [iters, G]``; and ``builds`` / ``reuses``."""
    name = "fire_relax_device"
    max_steps = _fire_params(name, fmax, dt, dt_max, max_step, max_steps)
    st = _setup(name, numbers, positions, cell, batch, device,
                cell_error="relax_cell needs a finite, non-singular cell" if relax_cell else None)
    G, Z, pos, c, replica, replica_ptr = st.G, st.Z, st.pos, st.c, st.replica, st.replica_ptr
    P0 = _replica_floats(pressure_bar, G, "pressure_bar", name, np.isfinite, "pressures must be finite")
    cf = _replica_floats(st.sizes if cell_factor is None else cell_factor, G, "cell_factor", name,
                         lambda v: np.isfinite(v) & (v > 0.0), "cell_factor must be finite and > 0")
    vg = VerletGraph(model, skin, cuda_graph, relax_cell, batch=st.batch, deforming=relax_cell)

    dev = pos.device
    f64 = dict(dtype=torch.float64, device=dev)
    if relax_cell:
        rp = pos.clone()                                        # r' = x A^-1 with A = I at the start
        A = torch.eye(3, **f64).repeat(G, 1, 1)
        A_prev, vcell, h0 = A.clone(), torch.zeros((G, 3, 3), **f64), c.double()
        P0_t, cf_t = torch.from_numpy(P0 / EV_A3_TO_BAR).to(dev), torch.from_numpy(cf).to(dev)
    else:
        rp, A, A_prev = pos, None, None                         # positions only: x is r'
    fire = _Fire(rp, replica, replica_ptr, G, fmax, dt, dt_max, max_step)

    energy, volume = [], []
    for it in range(max_steps + 1):
        e, f, *w = vg.evaluate(pos, Z, c)
        if relax_cell:
            volume.append(_det3(c.double()).abs())                # of the evaluated cell, before the step moves it
        rows = (A, w[0].contiguous(), c, h0, A_prev, vcell, P0_t, cf_t) if relax_cell else ()
        energy.append(e)
        if fire.step(f, it < max_steps, *rows):
            break
        fire.update(f, pos if relax_cell else None, A_prev, A)
    if stats is not None:
        trace = fire.trace
        stats.update(vg.counts(), converged=fire.converged.bool(), steps=fire.steps.clone(), energy=torch.stack(energy),
                     fmax=torch.stack(trace["fmax"]), **({"volume": torch.stack(volume)} if relax_cell else {}),
                     **{k: torch.stack(trace[k]) for k in ("dt", "alpha", "n_pos")})
    return pos, c, e


def _fire_params(name, fmax, dt, dt_max, max_step, max_steps) -> int:
    """``max_steps`` as an int, after the checks of FIRE's parameters (``ValueError``)."""
    if not fmax > 0.0:
        raise ValueError(f"{name}: fmax must be > 0 (got {fmax})")
    if not dt > 0.0:
        raise ValueError(f"{name}: dt must be > 0 (got {dt})")
    if not dt_max >= dt:
        raise ValueError(f"{name}: dt_max must be >= dt (got {dt_max} < {dt})")
    if not max_step > 0.0:
        raise ValueError(f"{name}: max_step must be > 0 (got {max_step})")
    if not int(max_steps) >= 0:
        raise ValueError(f"{name}: max_steps must be >= 0 (got {max_steps})")
    return int(max_steps)


class _Fire:
    """ASE's FIRE over ``G`` contiguous replicas of the rows ``rp [n,3]`` (updated in place), on the device: the per-replica
    state (``dt``, ``alpha``, ``n_pos``, ``steps``, sticky ``converged``, the step's ``coef``, ``fmax``, ``n_active``), the
    row velocities and the per-iteration sequence ``ops.opt_fire_reduce`` -> ``ops.opt_fire_step`` -> ``ops.opt_fire_update``.
    ``trace`` keeps ``fmax`` and the state after each step (``dt``, ``alpha``, ``n_pos``).  The cell rows of
    ``fire_relax_device`` are passed in by the caller, which owns that state."""

    def __init__(self, rp, replica, replica_ptr, G, fmax, dt, dt_max, max_step):
        dev = rp.device
        f64 = dict(dtype=torch.float64, device=dev)
        self.rp, self.replica, self.replica_ptr = rp, replica, replica_ptr
        self.fmax_limit, self.dt_max, self.max_step = fmax, dt_max, max_step
        self.dt, self.alpha = torch.full((G,), float(dt), **f64), torch.full((G,), 0.1, **f64)
        self.n_pos, self.steps, self.converged = (torch.zeros(G, dtype=torch.int32, device=dev) for _ in range(3))
        self.coef, self.fmax = torch.zeros((G, 3), **f64), torch.zeros(G, **f64)
        self.n_active = torch.zeros(1, dtype=torch.int32, device=dev)
        self.vel = torch.zeros_like(rp)
        self.trace = {k: [] for k in ("fmax", "dt", "alpha", "n_pos")}

    def step(self, f, move, A=None, virial=None, cell=None, h0=None, A_prev=None, vcell=None, P0=None, cell_factor=None) -> bool:
        """Convergence test and, with ``move``, FIRE's step logic at forces ``f`` (cell rows with ``A``).  True when the run
        ends here: ``move`` is False or no replica moves any more (one int read back)."""
        sums = ops.opt_fire_reduce(f, self.vel, A, self.replica, self.replica_ptr)
        ops.opt_fire_step(sums, virial, cell, h0, A, A_prev, vcell, P0, cell_factor, self.dt, self.alpha, self.n_pos, self.steps,
                          self.converged, self.fmax_limit, self.dt_max, self.max_step, move, self.coef, self.fmax, self.n_active)
        for k in self.trace:
            self.trace[k].append(getattr(self, k).clone())
        return not move or int(self.n_active.item()) == 0

    def update(self, f, x=None, A_prev=None, A=None):
        """The rows of the replicas still moving (and ``x = rp A`` with ``A``)."""
        ops.opt_fire_update(x, self.rp, self.vel, f, A_prev, A, self.replica, self.converged, self.coef)
