"""Structure relaxation on the device: ``hn_opt_fire_reduce`` / ``hn_opt_fire_step`` / ``hn_opt_fire_update``
(``ops.opt_fire_*``) and ``plugin.relax.fire_relax_device``.

Two float64 references:
- the kernel reference (``ref_reduce`` / ``ref_step`` / ``ref_update``) follows the header of include/hermnet_b200.h; it is
  the oracle of the kernels on the GPU and stands in for the three ops in the CPU cases over the kernel emulator;
- ``host_fire`` is ASE's FIRE over ASE's ``UnitCellFilter`` coordinates written out on stacked ``[n + 3, 3]`` arrays, fed by
  the product's own evaluations; the driver is checked against it step by step.
The generalized cell force of the reference is pinned against central differences of ``E + P0 V`` of the float64 oracle."""
import numpy as np
import pytest
import torch

import hermnet_b200 as H
from hermnet_b200 import ops, synthetic
from hermnet_b200.plugin import md
from hermnet_b200.plugin.relax import fire_relax_device
from oracle import hermnet_oracle as O
from tests import util
from tests.test_atom_virial import _emu_edge_virial_atom
from tests.test_langevin import _cpu_model, _cpu_systems, _np, _replica_tensors, _water_model

DEV = "cuda:0"
N_MIN, F_INC, F_DEC, ALPHA_START, F_ALPHA = 5, 1.1, 0.5, 0.1, 0.99


# ---------------------------------------------------------------------------------------------------------------------
# float64 reference of the three kernels
# ---------------------------------------------------------------------------------------------------------------------
def ref_cell_force(W, h, A, P0, cf):
    """Cell-row forces ``(W_sym - P0 V I) A^-1 / c_f`` ``[G,3,3]``."""
    W, h, A = (np.asarray(t, dtype=np.float64).reshape(-1, 3, 3) for t in (W, h, A))
    V = np.abs(np.linalg.det(h))
    S = 0.5 * (W + W.transpose(0, 2, 1)) - (np.asarray(P0, dtype=np.float64) * V)[:, None, None] * np.eye(3)
    return S @ np.linalg.inv(A) / np.asarray(cf, dtype=np.float64)[:, None, None]


def ref_reduce(force, vel, A, replica, G):
    """``[G,4]``: ``(sum F'.v, sum |F'|^2, sum |v|^2, max |F'_i|^2)`` with ``F' = f A^T``."""
    rep = _np(replica).astype(np.int64)
    f, v = _np(force).astype(np.float64), _np(vel).astype(np.float64)
    if A is not None:
        f = np.einsum("nk,njk->nj", f, _np(A).reshape(-1, 3, 3)[rep])
    out = np.zeros((G, 4))
    f2 = (f * f).sum(1)
    out[:, 0] = np.bincount(rep, (f * v).sum(1), G)
    out[:, 1] = np.bincount(rep, f2, G)
    out[:, 2] = np.bincount(rep, (v * v).sum(1), G)
    np.maximum.at(out[:, 3], rep, f2)
    return out


def ref_step(sums, st, fmax, dt_max, max_step, move, cell_rows):
    """One FIRE step of every replica on the numpy state ``st`` (dict of arrays, updated in place): the header's rules
    written out per replica.  ``cell_rows``: ``(virial [G,3,3], P0 [G], cf [G])`` or ``None``."""
    G = len(st["dt"])
    st["n_active"] = 0
    for g in range(G):
        fv, ff, vv, fm = sums[g]
        if cell_rows is not None:
            W, P0, cf = cell_rows
            Fc = ref_cell_force(W[g], st["cell"][g], st["A"][g], P0[g:g + 1], cf[g:g + 1])[0]
            Vc = st["vcell"][g]
            fv, ff, vv = fv + (Fc * Vc).sum(), ff + (Fc * Fc).sum(), vv + (Vc * Vc).sum()
            fm = max(fm, (Fc * Fc).sum(1).max())
        st["fmax"][g] = np.sqrt(fm)
        if st["converged"][g]:
            continue
        if fm < fmax * fmax:
            st["converged"][g] = 1
            continue
        st["n_active"] += 1
        if not move:
            continue
        a, t, npos = st["alpha"][g], st["dt"][g], st["n_pos"][g]
        if st["steps"][g] == 0:
            cv = cm = 0.0
        elif fv > 0.0:
            cv, cm = 1.0 - a, a * np.sqrt(vv) / np.sqrt(ff)
            if npos > N_MIN:
                t, a = min(t * F_INC, dt_max), a * F_ALPHA
            npos += 1
        else:
            cv, cm, a, t, npos = 0.0, 0.0, ALPHA_START, t * F_DEC, 0
        cf_ = cm + t
        dr = t * np.sqrt(cv * cv * vv + 2 * cv * cf_ * fv + cf_ * cf_ * ff)
        s = max_step / dr if dr > max_step else 1.0
        st["coef"][g] = (cv, cf_, s * t)
        st["alpha"][g], st["dt"][g], st["n_pos"][g] = a, t, npos
        st["steps"][g] += 1
        if cell_rows is not None:
            c = cell_rows[2][g]
            st["vcell"][g] = cv * Vc + cf_ * Fc
            st["A_prev"][g] = st["A"][g]
            st["A"][g] = ((c * st["A"][g].T + s * t * st["vcell"][g]) / c).T
            st["cell"][g] = (st["h0"][g] @ st["A"][g]).astype(np.float32)


def ref_update(x, rp, vel, force, A_prev, A, replica, converged, coef):
    """float64 atom update; returns ``(x, rp, vel)`` (numpy; x is None without A)."""
    rep = _np(replica).astype(np.int64)
    live = _np(converged)[rep] == 0
    f, v, r = _np(force).astype(np.float64), _np(vel).astype(np.float64), _np(rp).astype(np.float64)
    if A is not None:
        f = np.einsum("nk,njk->nj", f, _np(A_prev).reshape(-1, 3, 3)[rep])
    c = _np(coef)[rep]
    v_new = c[:, :1] * v + c[:, 1:2] * f
    r_new = (r + c[:, 2:3] * v_new).astype(np.float32)
    vel_out = np.where(live[:, None], v_new.astype(np.float32), _np(vel))
    rp_out = np.where(live[:, None], r_new, _np(rp))
    if A is None:
        return None, rp_out, vel_out
    x_new = np.einsum("nk,nkj->nj", rp_out.astype(np.float64), _np(A).reshape(-1, 3, 3)[rep]).astype(np.float32)
    return np.where(live[:, None], x_new, _np(x)), rp_out, vel_out


# --- CPU stand-ins of the three ops (same contracts) ---
def emu_opt_fire_reduce(force, vel, A, replica, replica_ptr):
    return torch.from_numpy(ref_reduce(force, vel, A, replica, replica_ptr.numel() - 1))


def emu_opt_fire_step(sums, virial, cell, h0, A, A_prev, vcell, P0, cell_factor, dt, alpha, n_pos, steps, converged, fmax, dt_max,
                      max_step, move, coef, fmax_out, n_active):
    names = ("dt", "alpha", "n_pos", "steps", "converged", "coef")
    tens = (dt, alpha, n_pos, steps, converged, coef)
    st = {k: _np(t).copy() for k, t in zip(names, tens)}
    st["fmax"] = _np(fmax_out).copy()
    rows = None
    if A is not None:
        st.update(A=_np(A).reshape(-1, 3, 3).copy(), A_prev=_np(A_prev).reshape(-1, 3, 3).copy(),
                  vcell=_np(vcell).reshape(-1, 3, 3).copy(), cell=_np(cell).reshape(-1, 3, 3).copy(), h0=_np(h0).reshape(-1, 3, 3))
        rows = (_np(virial).reshape(-1, 3, 3).astype(np.float64), _np(P0), _np(cell_factor))
    ref_step(_np(sums), st, fmax, dt_max, max_step, move, rows)
    for k, t in zip(names, tens):
        t.copy_(torch.from_numpy(st[k]))
    fmax_out.copy_(torch.from_numpy(st["fmax"]))
    n_active.fill_(st["n_active"])
    if A is not None:
        for k, t in (("A", A), ("A_prev", A_prev), ("vcell", vcell), ("cell", cell)):
            t.copy_(torch.from_numpy(st[k]).reshape(t.shape))


def emu_opt_fire_update(x, rp, vel, force, A_prev, A, replica, converged, coef):
    x_new, rp_new, vel_new = ref_update(x, rp, vel, force, A_prev, A, replica, converged, coef)
    rp.copy_(torch.from_numpy(rp_new))
    vel.copy_(torch.from_numpy(vel_new))
    if A is not None:
        x.copy_(torch.from_numpy(x_new))


@pytest.fixture
def emu_relax(emu, monkeypatch):
    monkeypatch.setattr(ops, "opt_fire_reduce", emu_opt_fire_reduce)
    monkeypatch.setattr(ops, "opt_fire_step", emu_opt_fire_step)
    monkeypatch.setattr(ops, "opt_fire_update", emu_opt_fire_update)
    monkeypatch.setattr(ops, "edge_virial_atom", _emu_edge_virial_atom)
    return emu


# ---------------------------------------------------------------------------------------------------------------------
# host FIRE + UnitCellFilter oracle (ASE's arrays: n atom rows, then 3 cell rows)
# ---------------------------------------------------------------------------------------------------------------------
def host_fire(evaluate, x0, h0, steps, relax_cell, P0=0.0, cf=None, fmax=0.05, dt=0.1, dt_max=1.0, max_step=0.2):
    """ASE's ``FIRE(UnitCellFilter(atoms))`` (``FIRE(atoms)`` without ``relax_cell``) in float64, at most ``steps`` steps.
    ``evaluate(x, h) -> (f [n,3], W [3,3])``.  Returns ``(x, h, [(dt, alpha, n_pos) after each step])``."""
    n = len(x0)
    cf = float(n) if cf is None else cf
    r, A = np.asarray(x0, dtype=np.float64), np.eye(3)
    h0 = np.asarray(h0, dtype=np.float64)
    v, a, Ns, trace = None, ALPHA_START, 0, []
    for k in range(steps + 1):
        x, h = (r @ A, h0 @ A) if relax_cell else (r, h0)
        f, W = evaluate(x, h)
        F, q = f @ A.T, r
        if relax_cell:
            Ws = 0.5 * (W + W.T)
            F = np.vstack([F, (Ws - P0 * abs(np.linalg.det(h)) * np.eye(3)) @ np.linalg.inv(A) / cf])
            q = np.vstack([r, cf * A.T])
        if (F * F).sum(1).max() < fmax * fmax or k == steps:
            return x, h, trace
        if v is None:
            v = np.zeros_like(F)
        else:
            vf = np.vdot(F, v)
            if vf > 0.0:
                v = (1.0 - a) * v + a * F / np.sqrt(np.vdot(F, F)) * np.sqrt(np.vdot(v, v))
                if Ns > N_MIN:
                    dt, a = min(dt * F_INC, dt_max), a * F_ALPHA
                Ns += 1
            else:
                v[:] = 0.0
                a, dt, Ns = ALPHA_START, dt * F_DEC, 0
        v = v + dt * F
        dr = dt * v
        nd = np.sqrt(np.vdot(dr, dr))
        if nd > max_step:
            dr = max_step * dr / nd
        q = q + dr
        r = q[:n]
        if relax_cell:
            A = (q[n:] / cf).T
        trace.append((dt, a, Ns))


def model_evaluator(model, Z, dev):
    """``evaluate(x, h) -> (f, W)`` of one replica through ``model.energy_forces_virial`` at the fp32-rounded geometry."""
    Zt = torch.as_tensor(Z).long().to(dev)

    def evaluate(x, h):
        out = model.energy_forces_virial(H.Data(pos=torch.from_numpy(x.astype(np.float32)).to(dev), atomic_number=Zt,
                                                cell=torch.from_numpy(h.astype(np.float32)).reshape(1, 3, 3).to(dev)))
        return _np(out["forces"]).astype(np.float64), _np(out["virial"])[0].astype(np.float64)
    return evaluate


def _start_pressures_bar(model, pos, Z, cell, batch, dev):
    """Per-replica internal pressure ``tr W / 3V`` (bar) of the starting geometry."""
    out = model.energy_forces_virial(H.Data(pos=torch.from_numpy(pos).to(dev), atomic_number=torch.from_numpy(Z).to(dev),
                                            cell=torch.from_numpy(cell).to(dev), batch=torch.from_numpy(batch).to(dev)))
    W = _np(out["virial"]).astype(np.float64)
    return np.trace(W, axis1=1, axis2=2) / (3.0 * np.abs(np.linalg.det(cell.astype(np.float64)))) * md.EV_A3_TO_BAR


def check_against_host_fire(model, pos, Z, cell, batch, dev, relax_cell, pressure_bar, steps=15, **kw):
    G = int(batch.max()) + 1
    st = {}
    p, c, _ = fire_relax_device(model, Z, pos, cell, max_steps=steps, batch=batch, relax_cell=relax_cell, pressure_bar=pressure_bar,
                                stats=st, device=dev, **kw)
    assert int(st["steps"].min()) == steps, "the comparison wants every replica still moving"
    P0 = np.broadcast_to(np.asarray(pressure_bar, dtype=np.float64), (G,)) / md.EV_A3_TO_BAR
    for g in range(G):
        sl = batch == g
        ev = model_evaluator(model, Z[sl], dev)
        x, h, trace = host_fire(ev, pos[sl], cell[g], steps, relax_cell, P0[g], **kw)
        assert len(trace) == steps
        tr = np.array(trace)
        assert np.allclose(_np(st["dt"])[:steps, g], tr[:, 0], rtol=1e-12, atol=0)
        assert np.allclose(_np(st["alpha"])[:steps, g], tr[:, 1], rtol=1e-12, atol=0)
        assert np.array_equal(_np(st["n_pos"])[:steps, g], tr[:, 2].astype(np.int32))
        assert np.abs(_np(p)[sl] - x).max() < 1e-4
        if relax_cell:
            assert np.abs(_np(c)[g] - h).max() < 1e-4
    return st


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference itself
# ---------------------------------------------------------------------------------------------------------------------
def test_generalized_forces_match_central_differences_of_the_enthalpy():
    """``-dH/dr' = f A^T`` and ``-dH/dq_c = (W_sym - P0 V I) A^-1 / c_f`` for ``H = E(r' A, h0 A) + P0 |det(h0 A)|``,
    ``A = (q_c / c_f)^T``, at ``A != I`` and ``P0 != 0`` on a periodic triclinic system (float64 oracle)."""
    case = util.load_case("triclinic_multi_image")
    kind, cfg = case["kind"], case["cfg"]
    sd = {k: (v.double() if v.is_floating_point() else v) for k, v in O.make_state_dict(kind, cfg, case["seed"]).items()}
    x_ref, h_ref = case["pos"].double(), case["cell"].double()[0]
    n = x_ref.size(0)
    rng = np.random.default_rng(4)
    A0 = torch.from_numpy(np.eye(3) + 0.03 * rng.standard_normal((3, 3)))
    r0, h0 = x_ref @ torch.linalg.inv(A0), h_ref @ torch.linalg.inv(A0)   # so that x = r' A, h = h0 A at the base point
    P0, cf = 0.02, 1.7 * n

    def energy(x, h, grads=False):
        return O.energy_and_forces(kind, sd, cfg, x, case["Z"], case["edge_index"], h[None], case["edge_shift"], case["batch"],
                                   want_cell_grad=grads)

    def enthalpy(r, q):
        A = q.T / cf
        h = h0 @ A
        return float(energy(r @ A, h)[0].sum()) + P0 * abs(float(torch.linalg.det(h)))

    e, f, gc = energy(x_ref, h_ref, grads=True)
    W = (x_ref.T @ f - h_ref.T @ gc[0]).numpy()
    F_atoms = (f @ A0.T).numpy()
    F_cell = ref_cell_force(W[None], h_ref.numpy()[None], A0.numpy()[None], [P0], [cf])[0]
    q0, eps = cf * A0.T, 1e-5
    fd_atoms, fd_cell = np.zeros((n, 3)), np.zeros((3, 3))
    for i in range(n):
        for k in range(3):
            d = torch.zeros_like(r0)
            d[i, k] = eps
            fd_atoms[i, k] = -(enthalpy(r0 + d, q0) - enthalpy(r0 - d, q0)) / (2 * eps)
    for j in range(3):
        for k in range(3):
            d = torch.zeros_like(q0)
            d[j, k] = eps
            fd_cell[j, k] = -(enthalpy(r0, q0 + d) - enthalpy(r0, q0 - d)) / (2 * eps)
    assert np.abs(F_cell).max() > 1e-2 and np.abs(W - W.T).max() < 1e-8 * np.abs(W).max()
    assert np.abs(fd_atoms - F_atoms).max() < 1e-6 * max(1.0, np.abs(F_atoms).max())
    assert np.abs(fd_cell - F_cell).max() < 1e-6 * max(1.0, np.abs(F_cell).max())


def test_reference_step_branches_and_closed_form_norm():
    """The closed-form ``|v_new|`` of the step equals the norm of the explicit update, in every branch."""
    rng = np.random.default_rng(0)
    for first, sign, npos in ((True, 1, 0), (False, 1, 2), (False, 1, 9), (False, -1, 3)):
        F, v = rng.standard_normal((7, 3)), rng.standard_normal((7, 3))
        v = sign * np.abs(v) * np.sign(F)            # F.v > 0 (sign 1) or < 0 (sign -1)
        if first:
            v[:] = 0.0
        sums = np.array([[(F * v).sum(), (F * F).sum(), (v * v).sum(), (F * F).sum(1).max()]])
        st = dict(dt=np.array([0.3]), alpha=np.array([0.05]), n_pos=np.array([npos], np.int32),
                  steps=np.array([0 if first else 4], np.int32), converged=np.zeros(1, np.int32), coef=np.zeros((1, 3)),
                  fmax=np.zeros(1))
        ref_step(sums, st, 0.01, 0.32, 1e9, True, None)
        cv, cfp, sdt = st["coef"][0]
        if first:
            assert (st["dt"][0], st["alpha"][0], st["n_pos"][0]) == (0.3, 0.05, 0)
        elif sign < 0:
            assert (st["dt"][0], st["alpha"][0], st["n_pos"][0], cv) == (0.15, ALPHA_START, 0, 0.0)
        elif npos > N_MIN:
            assert (st["dt"][0], st["alpha"][0], st["n_pos"][0]) == (0.32, 0.05 * F_ALPHA, npos + 1)      # dt_max clamp
        else:
            assert (st["dt"][0], st["alpha"][0], st["n_pos"][0]) == (0.3, 0.05, npos + 1)
        v_new = cv * v + cfp * F
        if not first and sign > 0:
            mixed = (1 - 0.05) * v + 0.05 * F / np.linalg.norm(F) * np.linalg.norm(v)
            assert np.allclose(v_new, mixed + st["dt"][0] * F, rtol=1e-13, atol=1e-13)
        assert sdt == st["dt"][0]


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the driver over the kernel emulator
# ---------------------------------------------------------------------------------------------------------------------
def test_emulated_driver_matches_host_fire(emu_relax):
    model = _cpu_model()
    pos, Z, cell, batch = _cpu_systems((31, 32))
    check_against_host_fire(model, pos, Z, cell, batch, "cpu", False, 0.0, steps=8, fmax=1e-4)
    check_against_host_fire(model, pos, Z, cell, batch, "cpu", True, [2e4, -1e4], steps=8, fmax=1e-4, dt_max=0.12)
    # the cell relaxed with a skin list, eager and with cuda_graph (which evaluates eagerly on CPU tensors): bitwise equal
    runs = []
    for cg in (False, True):
        st = {}
        out = fire_relax_device(model, Z, pos, cell, fmax=1e-4, max_steps=8, batch=batch, relax_cell=True, pressure_bar=[2e4, -1e4],
                                dt_max=0.12, skin=0.5, cuda_graph=cg, stats=st, device="cpu")
        runs.append((out, st))
    (out0, st0), (out1, st1) = runs
    assert st0["steps"].tolist() == [8, 8] and st0["reuses"] > 0 and st0.keys() == st1.keys()
    assert all(torch.equal(a, b) for a, b in zip(out0, out1))
    assert all(torch.equal(st0[k], st1[k]) if isinstance(st0[k], torch.Tensor) else st0[k] == st1[k] for k in st0)


def test_emulated_stats_and_a_replica_that_starts_converged(emu_relax):
    model = _cpu_model()
    pos, Z, cell, batch = _cpu_systems((33, 34))
    st = {}
    kw = dict(batch=batch, relax_cell=True, pressure_bar=1e4, device="cpu")
    p, c, e = fire_relax_device(model, Z, pos, cell, fmax=1e-4, max_steps=5, stats=st, skin=0.5, **kw)
    assert p.shape == pos.shape and c.shape == (2, 3, 3) and e.shape == (2,)
    for k in ("energy", "fmax", "volume", "dt", "alpha", "n_pos"):
        assert st[k].shape == (6, 2), k
    assert st["steps"].tolist() == [5, 5] and not st["converged"].any() and st["builds"] + st["reuses"] == 6
    assert util.rel_err(st["volume"][-1], torch.linalg.det(c.double()).abs()) < 1e-12
    # fmax above every start force: nothing moves, one evaluation
    big = float(st["fmax"][0].max()) * 1.01
    st2 = {}
    p2, c2, _ = fire_relax_device(model, Z, pos, cell, fmax=big, stats=st2, **kw)
    assert torch.equal(p2, torch.from_numpy(pos)) and torch.equal(c2, torch.from_numpy(cell))
    assert st2["converged"].all() and st2["steps"].tolist() == [0, 0] and st2["energy"].shape == (1, 2)
    # max_steps = 0: the test only
    p3, c3, _ = fire_relax_device(model, Z, pos, cell, fmax=1e-4, max_steps=0, **kw)
    assert torch.equal(p3, torch.from_numpy(pos)) and torch.equal(c3, torch.from_numpy(cell))


def test_emulated_positions_only_cluster(emu_relax):
    model = _cpu_model()
    pos, Z, _, _ = _cpu_systems((35,))
    st = {}
    p, c, e = fire_relax_device(model, Z, pos, None, fmax=1e-4, max_steps=4, stats=st, device="cpu")
    assert c is None and e.shape == (1,) and st["steps"].tolist() == [4] and "volume" not in st
    assert float(st["energy"][-1, 0]) < float(st["energy"][0, 0])


@pytest.mark.parametrize("bad", [
    dict(fmax=0.0), dict(fmax=-1.0), dict(dt=0.0), dict(dt=0.5, dt_max=0.4), dict(max_step=0.0), dict(max_steps=-1),
    dict(relax_cell=True, cell=None), dict(relax_cell=True, cell=np.diag([10.0, 10.0, 0.0])),
    dict(relax_cell=True, cell=np.full((3, 3), np.nan)), dict(pressure_bar=float("nan")), dict(pressure_bar=float("inf")),
    dict(pressure_bar=[1.0, 2.0]), dict(cell_factor=0.0), dict(cell_factor=-2.0), dict(cell_factor=[1.0, 1.0]),
    dict(batch=[0, 0, 1, 0]), dict(batch=[0, 0, 2, 2]), dict(batch=[0, 1]), dict(cell=np.zeros((2, 3, 3)) + np.eye(3))])
def test_validation_errors(bad):
    args = dict(cell=10.0 * np.eye(3))
    args.update(bad)
    cell = args.pop("cell")
    with pytest.raises(ValueError):
        fire_relax_device(None, [8, 1, 1, 8], np.zeros((4, 3)), cell, device="cpu", **args)


# ---------------------------------------------------------------------------------------------------------------------
# kernel level (GPU)
# ---------------------------------------------------------------------------------------------------------------------
def _rand_A(G, gen, dev=DEV):
    return (torch.eye(3, dtype=torch.float64) + 0.05 * torch.randn(G, 3, 3, generator=gen, dtype=torch.float64)).to(dev)


@pytest.mark.gpu
@pytest.mark.parametrize("sizes", [[1_000_000], [1 + (37 * g) % 700 for g in range(1000)]], ids=["G1-1e6", "G1000"])
def test_reduce_matches_float64_and_is_deterministic(sizes):
    replica, ptr = _replica_tensors(sizes, DEV)
    G, n = len(sizes), sum(sizes)
    gen = torch.Generator().manual_seed(G)
    force, vel = torch.randn(n, 3, generator=gen).to(DEV), torch.randn(n, 3, generator=gen).to(DEV)
    for A in (_rand_A(G, gen), None):
        got = ops.opt_fire_reduce(force, vel, A, replica, ptr)
        ref = ref_reduce(force, vel, A, replica, G)
        g = _np(got)
        assert np.abs(g[:, :3] - ref[:, :3]).max() <= 1e-12 * np.abs(ref[:, :3]).max() * max(1.0, n / G) ** 0.5
        assert np.allclose(g[:, 3], ref[:, 3], rtol=1e-14, atol=0)
        assert torch.equal(got, ops.opt_fire_reduce(force, vel, A, replica, ptr))      # bitwise determinism


@pytest.mark.gpu
def test_empty_launches_are_no_ops():
    z3, zi = torch.zeros(0, 3, device=DEV), torch.zeros(0, dtype=torch.int32, device=DEV)
    ptr = torch.zeros(1, dtype=torch.int32, device=DEV)
    assert ops.opt_fire_reduce(z3, z3.clone(), None, zi, ptr).shape == (0, 4)
    d0, i0 = torch.zeros(0, dtype=torch.float64, device=DEV), torch.zeros(0, dtype=torch.int32, device=DEV)
    n_active = torch.full((1,), 7, dtype=torch.int32, device=DEV)
    ops.opt_fire_step(torch.zeros(0, 4, dtype=torch.float64, device=DEV), None, None, None, None, None, None, None, None, d0, d0.clone(),
                      i0, i0.clone(), i0.clone(), 0.05, 1.0, 0.2, True, torch.zeros(0, 3, dtype=torch.float64, device=DEV), d0.clone(),
                      n_active)
    assert int(n_active) == 7
    ops.opt_fire_update(None, z3, z3.clone(), z3.clone(), None, None, zi, torch.zeros(1, dtype=torch.int32, device=DEV),
                        torch.zeros(1, 3, dtype=torch.float64, device=DEV))


def _step_case(G, cell_rows, seed):
    """State covering every branch: first step, P > 0 at n_pos <= N_min and > N_min (dt_max clamp when dt is near it),
    reset, cap active (large forces) and inactive, converged now, converged before."""
    rng = np.random.default_rng(seed)
    F, V = rng.standard_normal((G, 8, 3)), rng.standard_normal((G, 8, 3))
    kind = np.arange(G) % 8
    V[kind == 2] = np.abs(V[kind == 2]) * np.sign(F[kind == 2])          # P > 0
    V[kind == 3] = np.abs(V[kind == 3]) * np.sign(F[kind == 3])
    V[kind == 4] = -np.abs(V[kind == 4]) * np.sign(F[kind == 4])         # reset
    F[kind == 5] *= 1e-6                                                  # converges now (cell rows small too: see below)
    F[kind == 6] *= 500.0                                                 # cap active: dt |v_new| >= dt^2 |F| > max_step
    F[kind == 7] *= 1e-3                                                  # cap inactive
    V[kind == 7] *= 1e-3
    sums = np.stack([(F * V).sum((1, 2)), (F * F).sum((1, 2)), (V * V).sum((1, 2)), (F * F).sum(2).max(1)], 1)
    st = dict(dt=0.05 + 0.5 * rng.random(G), alpha=0.02 + 0.08 * rng.random(G),
              n_pos=np.where(kind == 3, 6 + kind, kind % 3).astype(np.int32),
              steps=np.where(kind == 0, 0, 3 + kind).astype(np.int32),
              converged=(kind == 1).astype(np.int32), coef=np.full((G, 3), -7.0), fmax=np.zeros(G))
    st["dt"][kind == 3] = 0.95
    rows = None
    if cell_rows:
        h0 = np.diag([9.0, 10.0, 11.0]) + 0.3 * rng.standard_normal((G, 3, 3))
        A = np.eye(3) + 0.02 * rng.standard_normal((G, 3, 3))
        st.update(h0=h0, A=A, A_prev=np.zeros((G, 3, 3)), vcell=0.1 * rng.standard_normal((G, 3, 3)),
                  cell=(h0 @ A).astype(np.float32))
        W = rng.standard_normal((G, 3, 3)).astype(np.float32)
        P0 = 1e-3 * rng.standard_normal(G)
        V_ = np.abs(np.linalg.det(st["cell"].astype(np.float64)))
        W[kind == 5] = (P0[kind == 5] * V_[kind == 5])[:, None, None] * np.eye(3, dtype=np.float32)  # W_sym = P0 V I: tiny cell force
        # cap inactive: the cell rows of the step must stay small as well (|dr| is the norm over atom and cell rows)
        W[kind == 7] = (P0[kind == 7] * V_[kind == 7])[:, None, None] * np.eye(3, dtype=np.float32) + \
            1e-3 * rng.standard_normal((int((kind == 7).sum()), 3, 3)).astype(np.float32)
        st["vcell"][kind == 7] *= 1e-3
        st["vcell"][kind == 0] = 0.0
        rows = (W, P0, 5.0 + rng.random(G))
    return sums, st, rows


def _step_on_gpu(sums, st, rows, fmax, dt_max, max_step, move):
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(DEV) for k, v in st.items()}
    n_active = torch.zeros(1, dtype=torch.int32, device=DEV)
    args = [None] * 7
    if rows is not None:
        args = [torch.from_numpy(rows[0]).to(DEV), t["cell"], t["h0"], t["A"], t["A_prev"], t["vcell"],
                torch.from_numpy(rows[1]).to(DEV)]
    cf = None if rows is None else torch.from_numpy(rows[2]).to(DEV)
    ops.opt_fire_step(torch.from_numpy(sums).to(DEV), *args, cf, t["dt"], t["alpha"], t["n_pos"], t["steps"], t["converged"], fmax,
                      dt_max, max_step, move, t["coef"], t["fmax"], n_active)
    out = {k: _np(v) for k, v in t.items()}
    out["n_active"] = int(n_active)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("cell_rows", [False, True], ids=["atoms-only", "cell-rows"])
@pytest.mark.parametrize("move", [True, False], ids=["move", "test-only"])
def test_step_matches_float64_in_every_branch(cell_rows, move):
    G = 4000
    sums, st, rows = _step_case(G, cell_rows, seed=int(cell_rows))
    fmax, dt_max, max_step = 1e-3, 1.0, 0.2
    got = _step_on_gpu(sums, st, rows, fmax, dt_max, max_step, move)
    ref = {k: v.copy() for k, v in st.items()}
    ref_step(sums, ref, fmax, dt_max, max_step, move, rows)
    kind = np.arange(G) % 8
    assert got["n_active"] == ref["n_active"] > 0
    for k in ("n_pos", "steps", "converged"):
        assert np.array_equal(got[k], ref[k]), k
    for k in ("dt", "alpha", "fmax", "coef") + (("A", "A_prev", "vcell") if cell_rows else ()):
        assert np.allclose(got[k], ref[k], rtol=1e-12, atol=1e-14), k
    if cell_rows:
        assert np.abs(got["cell"].astype(np.float64) - ref["cell"]).max() <= 2e-6 * 12
    # every branch was taken, and converged replicas are untouched bitwise
    assert (ref["converged"][kind == 5] == 1).all() and (ref["converged"][kind == 6] == 0).all()
    conv = ref["converged"] == 1
    for k in st:
        if k not in ("fmax", "converged"):
            assert np.array_equal(got[k][conv], st[k][conv]), k
    if move:
        assert (ref["dt"][kind == 3] == dt_max).all()                                    # clamp
        assert (ref["alpha"][kind == 4] == ALPHA_START).all() and (ref["n_pos"][kind == 4] == 0).all()   # reset
        assert (ref["coef"][kind == 6, 2] < ref["dt"][kind == 6]).all()                  # cap active
        assert (ref["coef"][kind == 7, 2] == ref["dt"][kind == 7]).all()                 # cap inactive
        assert (ref["coef"][kind == 0, 0] == 0.0).all() and (ref["steps"][kind == 0] == 1).all()   # first step
    else:
        for k in st:
            if k not in ("fmax", "converged"):
                assert np.array_equal(got[k], st[k]), k


@pytest.mark.gpu
def test_update_matches_torch_and_identity_keeps_x_equal_to_rp():
    sizes = [5000, 1, 20_001, 333]
    replica, ptr = _replica_tensors(sizes, DEV)
    G, n = len(sizes), sum(sizes)
    gen = torch.Generator().manual_seed(5)
    rp, vel, f = (10 * torch.randn(n, 3, generator=gen)).to(DEV), torch.randn(n, 3, generator=gen).to(DEV), \
        torch.randn(n, 3, generator=gen).to(DEV)
    coef = torch.tensor([[0.9, 0.3, 0.1], [0.0, 0.1, 0.05], [0.5, 0.2, 0.01], [1.0, 1.0, 1.0]], dtype=torch.float64, device=DEV)
    converged = torch.tensor([0, 0, 0, 1], dtype=torch.int32, device=DEV)
    A, A_prev = _rand_A(G, gen), _rand_A(G, gen)
    x = torch.full((n, 3), 123.0, device=DEV)
    a, b, c = x.clone(), rp.clone(), vel.clone()
    ops.opt_fire_update(a, b, c, f, A_prev, A, replica, converged, coef)
    x_ref, rp_ref, v_ref = ref_update(x, rp, vel, f, A_prev, A, replica, converged, coef)
    assert np.abs(_np(c) - v_ref).max() <= 2.4e-7 * np.abs(v_ref).max()
    assert np.abs(_np(b) - rp_ref).max() <= 2.4e-7 * np.abs(rp_ref).max()
    assert np.abs(_np(a) - x_ref).max() <= 5e-7 * np.abs(x_ref).max()
    last = slice(n - sizes[-1], n)
    assert torch.equal(a[last], x[last]) and torch.equal(b[last], rp[last]) and torch.equal(c[last], vel[last])
    # A = I given explicitly: x == r' bitwise; A = None: the same r' and velocities
    eye = torch.eye(3, dtype=torch.float64, device=DEV).repeat(G, 1, 1)
    a1, b1, c1 = x.clone(), rp.clone(), vel.clone()
    ops.opt_fire_update(a1, b1, c1, f, eye, eye, replica, converged, coef)
    assert torch.equal(a1[: n - sizes[-1]], b1[: n - sizes[-1]])
    b2, c2 = rp.clone(), vel.clone()
    ops.opt_fire_update(None, b2, c2, f, None, None, replica, converged, coef)
    assert torch.equal(b2, b1) and torch.equal(c2, c1)


# ---------------------------------------------------------------------------------------------------------------------
# model level (GPU): HVNet of BASELINE config 1 on rattled water boxes
# ---------------------------------------------------------------------------------------------------------------------
def _rattled(seeds, n_side=3, rattle=0.1):
    parts = []
    for s in seeds:
        p, z, c = synthetic.water_box(n_side, seed=s)
        p = p + np.random.default_rng(1000 + s).normal(0, rattle, p.shape).astype(np.float32)
        parts.append((p, z, c))
    pos = np.concatenate([p for p, _, _ in parts])
    Z = np.concatenate([z for _, z, _ in parts])
    cell = np.stack([c for _, _, c in parts])
    batch = np.repeat(np.arange(len(seeds)), [len(z) for _, z, _ in parts])
    return pos, Z, cell, batch


@pytest.mark.gpu
def test_driver_matches_host_fire_and_unit_cell_filter():
    model = _water_model()
    pos, Z, cell, batch = _rattled((1, 2))
    P = _start_pressures_bar(model, pos, Z, cell, batch, DEV)
    check_against_host_fire(model, pos, Z, cell, batch, DEV, False, 0.0, fmax=1e-6)
    for shift in (-2000.0, 3000.0):
        check_against_host_fire(model, pos, Z, cell, batch, DEV, True, P + shift, fmax=1e-6, dt_max=0.12)


@pytest.mark.gpu
def test_eight_boxes_relax_to_stationary_points():
    model = _water_model()
    seeds = tuple(range(10, 18))
    pos, Z, cell, batch = _rattled(seeds)
    P = _start_pressures_bar(model, pos, Z, cell, batch, DEV) + np.linspace(100.0, 500.0, 8)   # compressed: a stationary point
    st0 = {}
    fire_relax_device(model, Z, pos, cell, max_steps=0, batch=batch, relax_cell=True, pressure_bar=P, stats=st0, device=DEV)
    fmax = 0.1 * float(st0["fmax"][0].min())
    st = {}
    p, c, e = fire_relax_device(model, Z, pos, cell, fmax=fmax, max_steps=3000, batch=batch, relax_cell=True, pressure_bar=P,
                                stats=st, device=DEV, skin=0.5)
    print(f"eight boxes: fmax {fmax:.3e}, steps {st['steps'].tolist()}, builds {st['builds']} reuses {st['reuses']}")
    assert bool(st["converged"].all())
    out = model.energy_forces_virial(H.Data(pos=p, atomic_number=torch.from_numpy(Z).to(DEV), cell=c,
                                            batch=torch.from_numpy(batch).to(DEV)))
    cf = np.bincount(batch).astype(np.float64)
    P0 = P / md.EV_A3_TO_BAR
    Fc = ref_cell_force(_np(out["virial"]), _np(c), np.linalg.solve(cell.astype(np.float64), _np(c).astype(np.float64)), P0, cf)
    f = _np(out["forces"]).astype(np.float64)
    A = np.linalg.solve(cell.astype(np.float64), _np(c).astype(np.float64))
    for g in range(8):
        sl = batch == g
        rows = np.vstack([f[sl] @ A[g].T, Fc[g]])
        assert np.sqrt((rows ** 2).sum(1).max()) < fmax * 1.01, g
    V0, V1 = np.abs(np.linalg.det(cell.astype(np.float64))), np.abs(np.linalg.det(_np(c).astype(np.float64)))
    H0 = _np(st["energy"][0]).astype(np.float64) + P0 * V0
    H1 = _np(e).astype(np.float64) + P0 * V1
    assert (H1 < H0).all(), (H0, H1)


@pytest.mark.gpu
def test_a_lone_replica_matches_the_batch_and_cuda_graph_matches_eager():
    model = _water_model()
    pos, Z, cell, batch = _rattled((21, 22, 23))
    P = _start_pressures_bar(model, pos, Z, cell, batch, DEV) + 1000.0
    kw = dict(fmax=1e-6, max_steps=10, relax_cell=True, device=DEV)
    pb, cb, _ = fire_relax_device(model, Z, pos, cell, batch=batch, pressure_bar=P, **kw)
    sl = batch == 1
    p1, c1, _ = fire_relax_device(model, Z[sl], pos[sl], cell[1], pressure_bar=P[1], **kw)
    assert float((p1 - pb[torch.from_numpy(sl).to(DEV)]).abs().max()) < 1e-5
    assert float((c1[0] - cb[1]).abs().max()) < 1e-5
    runs = {}
    for cg in (False, True):
        st = {}
        runs[cg] = fire_relax_device(model, Z, pos, cell, batch=batch, pressure_bar=P, skin=0.8, cuda_graph=cg, stats=st,
                                     **dict(kw, max_steps=40)) + (st,)
    (p0, c0, e0, s0), (p1, c1, e1, s1) = runs[False], runs[True]
    assert s1["builds"] == s0["builds"] and s1["reuses"] > 0
    assert float((p1 - p0).abs().max()) < 1e-5 and float((c1 - c0).abs().max()) < 1e-5
    assert util.rel_err(e1, e0) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("relax_cell", [False, True], ids=["positions", "cell"])
def test_a_replica_that_starts_converged_is_returned_unchanged(relax_cell):
    model = _water_model()
    pos, Z, cell, batch = _rattled((31, 32))
    kw = dict(batch=batch, relax_cell=relax_cell, pressure_bar=_start_pressures_bar(model, pos, Z, cell, batch, DEV), device=DEV)
    st0 = {}
    fire_relax_device(model, Z, pos, cell, max_steps=0, stats=st0, **kw)
    f0 = _np(st0["fmax"][0])
    k = int(np.argmin(f0))                          # replica k is converged at the start, the other one is not
    fmax = float(f0[k]) * 1.01
    assert f0[1 - k] > fmax
    st = {}
    p, c, _ = fire_relax_device(model, Z, pos, cell, fmax=fmax, max_steps=20, stats=st, **kw)
    sl = torch.from_numpy(batch == k).to(DEV)
    assert torch.equal(p[sl], torch.from_numpy(pos).to(DEV)[sl]) and torch.equal(c[k], torch.from_numpy(cell[k]).to(DEV))
    assert int(st["steps"][k]) == 0 and int(st["steps"][1 - k]) == 20 and bool(st["converged"][k])
