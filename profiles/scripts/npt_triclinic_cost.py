"""Cost of triclinic constant-pressure dynamics (``plugin.md.langevin_npt_device(cell_dof="triclinic")``, kernels of
csrc/hn_md.cu) against the isotropic mode:
  (a) per-launch time of ``hn_md_kinetic_tensor`` and ``hn_md_affine_deform`` at 10^6 and 10^7 atoms, and of
      ``hn_md_scr_barostat_tri`` (8 replicas), from CUDA events over ``--launches`` back-to-back launches, with the achieved
      bandwidth against the bytes computed from the shapes;
  (b) ms/step of the isotropic against the triclinic mode on the C3 water box (HTNet L=3 F=128, 31 944 atoms, last readout
      layer x 1e-3 as bench.py C3 does, 1 bar, tau_p 1 ps), Verlet skin 0.5 A, eager and ``cuda_graph=True``, with the list
      builds (= captures with ``cuda_graph``) and re-uses of each variant;
  (c) eight 192-atom C1 water boxes (HVNet L=3 F=128) at eight pressures in one batched run, both modes, eager and
      ``cuda_graph``: atom-steps/s and list counts.

    python profiles/scripts/npt_triclinic_cost.py [--steps 20] [--rounds 3] [--replica-steps 200] [--launches 1000] [--out DIR]

Timed calls of (b) and (c) run whole MD calls (initial evaluation, list builds and captures included) after one warm-up
call of each variant, alternating the variants across rounds; ms/step = call time / (steps + 1).  The card's name, power
limit and max SM clock are printed with the numbers; one JSON document goes to stdout and to
``DIR/npt_triclinic_cost.json`` with ``--out``.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)
from hermnet_b200 import ops, synthetic  # noqa: E402
from hermnet_b200.plugin import md  # noqa: E402
from langevin_cost import alternate, card, model_of, timed  # noqa: E402

F32, I32, I64 = 4, 4, 8
# bytes moved, from the shapes: kinetic tensor per atom -- vel [3], inv_mass read, [6] written; affine deform per atom --
# pos [3] and vel [3] read + write, replica (the per-replica mu / mu^-T are cache-resident); barostat per replica -- cell
# [9] read + write, kin6 [6], virial [9], P0, kT, beta, seed, mu / mu^-T / pressure [9] written
BYTES = {"md_kinetic_tensor": 3 * F32 + F32 + 6 * F32,
         "md_affine_deform": 2 * 3 * F32 + 2 * 3 * F32 + I32,
         "md_scr_barostat_tri": 2 * 9 * F32 + 6 * F32 + 9 * F32 + 3 * F32 + I64 + 3 * 9 * F32}


def part_a(n, launches, dev):
    G = 8
    gen = torch.Generator(device=dev).manual_seed(0)
    pos = torch.randn(n, 3, device=dev, generator=gen)
    vel = 0.01 * torch.randn(n, 3, device=dev, generator=gen)
    inv_m = torch.full((n,), 1.0 / (16.0 * md.AMU_A2_FS2_TO_EV), device=dev)
    ptr = torch.linspace(0, n, G + 1, device=dev).round().to(torch.int32)
    replica = torch.repeat_interleave(torch.arange(G, dtype=torch.int32, device=dev), (ptr[1:] - ptr[:-1]).long())
    cell = (torch.eye(3, device=dev) * 200.0).repeat(G, 1, 1).contiguous()
    kin6 = torch.tensor([1e3, 0.0, 1e3, 0.0, 0.0, 1e3], device=dev).repeat(G, 1).contiguous()
    virial = torch.zeros(G, 3, 3, device=dev)
    P0 = torch.full((G,), 1.0 / md.EV_A3_TO_BAR, device=dev)
    kT = torch.full((G,), md.KB_EV * 300.0, device=dev)
    beta = torch.full((G,), 4.5e-5 * md.EV_A3_TO_BAR, device=dev)
    seed = torch.arange(G, dtype=torch.int64, device=dev)
    step = torch.zeros(1, dtype=torch.int64, device=dev)
    mu, mu_inv_t, pressure = (torch.empty(G, 3, 3, device=dev) for _ in range(3))
    eye = torch.eye(3, device=dev).repeat(G, 1, 1).contiguous()      # (timing only: keeps pos / vel from drifting)
    calls = {"md_scr_barostat_tri": (lambda: ops.md_scr_barostat_tri(cell, kin6, virial, P0, kT, beta, seed, step, 0.5, 1000.0,
                                                                     mu, mu_inv_t, pressure), G),
             "md_kinetic_tensor": (lambda: ops.md_kinetic_tensor(vel, inv_m), n),
             "md_affine_deform": (lambda: ops.md_affine_deform(pos, vel, replica, eye, eye), n)}
    res = {}
    for k, (fn, units) in calls.items():
        for _ in range(20):
            fn()

        def run(fn=fn):
            for _ in range(launches):
                fn()
        ms, _ = timed(run)
        us = 1e3 * ms / launches
        gbs = BYTES[k] * units / (us * 1e-6) / 1e9
        res[k] = {"us_per_launch": us, "bytes_per_unit": BYTES[k], "units": units, "GB_per_s": gbs}
        print(f"(a) N={n} {k}: {us:.2f} us/launch, {BYTES[k]} B x {units} -> {gbs:.3g} GB/s", flush=True)
    return res


def _variants(run):
    return {f"{dof}_{'graph' if cg else 'eager'}": (lambda st, dof=dof, cg=cg: run(st, dof, cg))
            for cg in (False, True) for dof in ("isotropic", "triclinic")}


def part_b(steps, rounds, dev):
    (pos, Z, cell), _ = synthetic.config("C3")
    model = model_of("C3", dev)
    atoms = md.SimpleAtoms(Z, pos, cell)
    md.maxwell_boltzmann(atoms, 300.0, seed=3)
    v0 = atoms.velocities

    def run(st, dof, cg):
        return md.langevin_npt_device(model, Z, pos, cell, v0, steps, dt_fs=0.5, temperature_K=300.0, pressure_bar=1.0,
                                      friction_per_fs=0.01, device=dev, skin=0.5, cuda_graph=cg, stats=st, cell_dof=dof)
    times, lists = alternate(_variants(run), rounds)
    ms = {k: float(np.median(v)) / (steps + 1) for k, v in times.items()}
    print(f"(b) C3 N={len(Z)}: ms/step " + "  ".join(f"{k} {v:.3f} {lists[k]}" for k, v in ms.items()), flush=True)
    return {"atoms": int(len(Z)), "steps": steps, "ms_per_call": times, "ms_per_step": ms, "lists": lists}


def part_c(steps, rounds, dev):
    model = model_of("C1", dev)
    G = 8
    parts = [synthetic.water_box(4, seed=s) for s in range(G)]
    pos = np.concatenate([p for p, _, _ in parts])
    Z = np.concatenate([z for _, z, _ in parts])
    cell = np.stack([c for _, _, c in parts])
    batch = np.repeat(np.arange(G), [len(z) for _, z, _ in parts])
    pressures = [-2000.0, 1.0, 2000.0, 5000.0, 10000.0, 20000.0, 40000.0, 80000.0]

    def run(st, dof, cg):
        return md.langevin_npt_device(model, Z, pos, cell, np.zeros_like(pos), steps, dt_fs=0.5, temperature_K=300.0,
                                      pressure_bar=pressures, tau_p_fs=200.0, friction_per_fs=0.01, batch=batch, device=dev,
                                      skin=0.5, cuda_graph=cg, stats=st, cell_dof=dof)
    times, lists = alternate(_variants(run), rounds)
    rate = {k: len(Z) * (steps + 1) / (float(np.median(v)) * 1e-3) for k, v in times.items()}
    print(f"(c) {G} x 192 atoms at {pressures} bar: atom-steps/s " + "  ".join(f"{k} {v:.4g} {lists[k]}" for k, v in rate.items()),
          flush=True)
    return {"atoms": int(len(Z)), "steps": steps, "pressure_bar": pressures, "ms_per_call": times, "atom_steps_per_s": rate,
            "lists": lists}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--replica-steps", type=int, default=200)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("npt_triclinic_cost.py measures on a GPU; none is available")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"card": card(), "rounds": a.rounds}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    res["a_kernels"] = {str(n): part_a(n, a.launches, dev) for n in (10 ** 6, 10 ** 7)}
    res["b_c3"] = part_b(a.steps, a.rounds, dev)
    res["c_pressures"] = part_c(a.replica_steps, a.rounds, dev)
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "npt_triclinic_cost.json"), "w") as f:
            f.write(doc)


if __name__ == "__main__":
    main()
