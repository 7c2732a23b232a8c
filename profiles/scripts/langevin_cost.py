"""Cost of Langevin dynamics on the device (``plugin.md.langevin_device``, kernels of csrc/hn_md.cu):
  (a) ms/step of ``velocity_verlet_device`` against ``langevin_device`` on the C3 water box (HTNet L=3 F=128, 31 944 atoms,
      last readout layer x 1e-3 as bench.py C3 does), Verlet skin 0.5 A, eager and ``cuda_graph=True``;
  (b) atom-steps/s of 1, 8 and 64 batched replicas of the 192-atom C1 water box (HVNet L=3 F=128), skin 0.5 A, eager and
      ``cuda_graph=True``;
  (c) per-launch time of ``hn_md_langevin_baoa`` and ``hn_md_kick`` from CUDA events over ``--launches`` back-to-back launches,
      with the achieved bandwidth against the bytes per atom computed from the shapes.  At 10^6 atoms (what an MD user runs
      at the C4 size) the 68 MB working set fits in the 126 MB L2; at 10^7 atoms it does not, which gives the HBM figure.

    python profiles/scripts/langevin_cost.py [--steps 20] [--rounds 3] [--replica-steps 50] [--launches 1000] [--out DIR]

Timed calls of (a) and (b) run whole MD calls (initial evaluation, list builds and, with ``cuda_graph``, captures included),
after one warm-up call of each variant, alternating the variants across rounds; ms/step = call time / (steps + 1).  The card's
name, power limit and max SM clock are printed with the numbers; one JSON document goes to stdout and to
``DIR/langevin_cost.json`` with ``--out``.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import hermnet_b200 as H  # noqa: E402
from hermnet_b200 import ops, synthetic  # noqa: E402
from hermnet_b200.plugin import md  # noqa: E402

F32, I32 = 4, 4
# bytes moved per atom, from the shapes: pos [3] read + write, vel [3] read + write, force [3], inv_mass, replica (baoa);
# vel [3] read + write, force [3], inv_mass, kinetic (kick).  Per-replica arrays (kT, seed, replica_ptr) and the step
# counter are a few bytes shared by every atom.
BYTES_PER_ATOM = {"md_langevin_baoa": 2 * 3 * F32 + 2 * 3 * F32 + 3 * F32 + F32 + I32,
                  "md_kick": 2 * 3 * F32 + 3 * F32 + F32 + F32}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def model_of(name, dev):
    cfg = dict(synthetic.config(name)[1])
    kind = cfg.pop("kind")
    torch.manual_seed(1234)
    model = getattr(H, kind)(**cfg).to(dev).eval()
    for q in model.parameters():
        q.requires_grad_(False)
    model.out_energy[2].weight.mul_(1.0e-3)      # a trajectory that moves like a real one (bench.py C3)
    model.out_energy[2].bias.mul_(1.0e-3)
    return model


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def alternate(variants, rounds):
    """``{name: fn(stats)}`` -> ``({name: [ms per call]}, {name: list builds / re-uses of the last call})``: one warm-up call
    each, then ``rounds`` rounds in turn."""
    for fn in variants.values():
        fn({})
    torch.cuda.synchronize()
    times, lists = {k: [] for k in variants}, {}
    for _ in range(rounds):
        for k, fn in variants.items():
            st = {}
            times[k].append(timed(lambda: fn(st))[0])
            lists[k] = {"builds": st["builds"], "reuses": st["reuses"]}
    return times, lists


def part_a(steps, rounds, dev):
    (pos, Z, cell), _ = synthetic.config("C3")
    model = model_of("C3", dev)
    atoms = md.SimpleAtoms(Z, pos, cell)
    md.maxwell_boltzmann(atoms, 300.0, seed=3)
    v0 = atoms.velocities
    variants = {}
    for cg in (False, True):
        tag = "graph" if cg else "eager"
        variants[f"verlet_{tag}"] = lambda st, cg=cg: md.velocity_verlet_device(
            model, Z, pos, cell, v0, steps, dt_fs=0.5, device=dev, skin=0.5, cuda_graph=cg, stats=st)
        variants[f"langevin_{tag}"] = lambda st, cg=cg: md.langevin_device(
            model, Z, pos, cell, v0, steps, dt_fs=0.5, temperature_K=300.0, friction_per_fs=0.01, device=dev, skin=0.5,
            cuda_graph=cg, stats=st)
    times, lists = alternate(variants, rounds)
    ms = {k: float(np.median(v)) / (steps + 1) for k, v in times.items()}
    print(f"(a) C3 N={len(Z)}: ms/step " + "  ".join(f"{k} {v:.3f} {lists[k]}" for k, v in ms.items()), flush=True)
    return {"atoms": int(len(Z)), "steps": steps, "ms_per_call": times, "ms_per_step": ms, "lists": lists}


def part_b(steps, rounds, dev):
    model = model_of("C1", dev)
    res = {}
    for G in (1, 8, 64):
        parts = [synthetic.water_box(4, seed=s) for s in range(G)]
        pos = np.concatenate([p for p, _, _ in parts])
        Z = np.concatenate([z for _, z, _ in parts])
        cell = np.stack([c for _, _, c in parts])
        batch = np.repeat(np.arange(G), [len(z) for _, z, _ in parts])
        v0 = np.zeros_like(pos)
        variants = {("graph" if cg else "eager"): (lambda st, cg=cg: md.langevin_device(
            model, Z, pos, cell, v0, steps, dt_fs=0.5, temperature_K=300.0, friction_per_fs=0.01, batch=batch, device=dev,
            skin=0.5, cuda_graph=cg, stats=st)) for cg in (False, True)}
        times, lists = alternate(variants, rounds)
        rate = {k: len(Z) * (steps + 1) / (float(np.median(v)) * 1e-3) for k, v in times.items()}
        res[G] = {"atoms": int(len(Z)), "steps": steps, "ms_per_call": times, "atom_steps_per_s": rate, "lists": lists}
        print(f"(b) {G} x 192 atoms: atom-steps/s " + "  ".join(f"{k} {v:.4g} {lists[k]}" for k, v in rate.items()), flush=True)
    return res


def part_c(n, launches, dev):
    gen = torch.Generator(device=dev).manual_seed(0)
    pos = torch.randn(n, 3, device=dev, generator=gen)
    vel = 0.01 * torch.randn(n, 3, device=dev, generator=gen)
    force = torch.randn(n, 3, device=dev, generator=gen)
    inv_m = torch.full((n,), 1.0 / (16.0 * md.AMU_A2_FS2_TO_EV), device=dev)
    G = 8
    ptr = torch.linspace(0, n, G + 1, device=dev).round().to(torch.int32)
    replica = torch.repeat_interleave(torch.arange(G, dtype=torch.int32, device=dev), (ptr[1:] - ptr[:-1]).long())
    kT = torch.full((G,), md.KB_EV * 300.0, device=dev)
    seed = torch.arange(G, dtype=torch.int64, device=dev)
    step = torch.zeros(1, dtype=torch.int64, device=dev)
    kinetic = torch.empty(n, device=dev)
    c1, c2 = float(np.exp(-0.005)), float(np.sqrt(-np.expm1(-0.01)))
    calls = {"md_langevin_baoa": lambda: ops.md_langevin_baoa(pos, vel, force, inv_m, replica, ptr, kT, seed, step, c1, c2, 0.5),
             "md_kick": lambda: ops.md_kick(vel, force, inv_m, 0.25, kinetic, step)}
    res = {}
    for k, fn in calls.items():
        for _ in range(20):
            fn()

        def run(fn=fn):
            for _ in range(launches):
                fn()
        ms, _ = timed(run)
        us = 1e3 * ms / launches
        gbs = BYTES_PER_ATOM[k] * n / (us * 1e-6) / 1e9
        res[k] = {"us_per_launch": us, "bytes_per_atom": BYTES_PER_ATOM[k], "GB_per_s": gbs}
        print(f"(c) N={n} {k}: {us:.2f} us/launch, {BYTES_PER_ATOM[k]} B/atom -> {gbs:.0f} GB/s", flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--replica-steps", type=int, default=50)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("langevin_cost.py measures on a GPU; none is available")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"card": card(), "rounds": a.rounds}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    res["c_kernels"] = {str(n): part_c(n, a.launches, dev) for n in (10 ** 6, 10 ** 7)}
    res["a_c3"] = part_a(a.steps, a.rounds, dev)
    res["b_replicas"] = part_b(a.replica_steps, a.rounds, dev)
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "langevin_cost.json"), "w") as f:
            f.write(doc)


if __name__ == "__main__":
    main()
