"""Cost of structure relaxation on the device (``plugin.relax.fire_relax_device``, kernels of csrc/hn_opt.cu):
  (a) per-launch time of ``hn_opt_fire_reduce``, ``hn_opt_fire_step`` and ``hn_opt_fire_update`` (8 replicas, cell rows on)
      from CUDA events over ``--launches`` back-to-back launches at 10^6 and 10^7 atoms, with the achieved bandwidth against
      the bytes computed from the shapes;
  (b) ``--boxes`` rattled copies of the 192-atom C1 water box (HVNet L=3 F=128, last readout layer x 1e-3 as bench.py C3
      does) relaxed (positions only) to the same fmax: all at once with ``fire_relax_device``, eager and with ``cuda_graph``,
      Verlet skin 0.5 A; against ``--host-boxes`` of them one at a time through a host FIRE loop over ``NNCalculator`` (the
      route of ASE's ``FIRE``: one structure per optimizer, a host round trip per step).  Structures per second, steps to
      converge and list builds of each run; plus the batched run with ``relax_cell``, each box at its own starting pressure
      ``tr W / 3V`` (where the compressed side of this random-weight model has its stationary points).

    python profiles/scripts/relax_cost.py [--boxes 64] [--host-boxes 4] [--launches 1000] [--out DIR]

fmax is a fixed fraction (``--fmax-frac``) of the smallest starting max force of the boxes: the random-weight model's forces
have no physical scale.  Each device variant runs once to warm up, then once timed; the host loop is timed per box.  The
card's name, power limit and max SM clock are printed with the numbers; one JSON document goes to stdout and to
``DIR/relax_cost.json`` with ``--out``.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)
from hermnet_b200 import Data, ops, synthetic  # noqa: E402
from hermnet_b200.plugin import md  # noqa: E402
from hermnet_b200.plugin.calculator import NNCalculator  # noqa: E402
from hermnet_b200.plugin.relax import fire_relax_device  # noqa: E402
from langevin_cost import card, model_of, timed  # noqa: E402

F32, F64, I32 = 4, 8, 4
# bytes moved, from the shapes.  reduce per atom: force [3] and vel [3] read, replica (A and the chunk partials are per
# replica / per 256 atoms); update per atom: force [3] read, vel [3] and r' [3] read + write, x [3] written, replica;
# step per replica: sums [4], virial [9], cell [9] read + write, h0 / A / A_prev / vcell [9] each, state and outputs
BYTES = {"opt_fire_reduce": 6 * F32 + I32,
         "opt_fire_update": 3 * F32 + 4 * 3 * F32 + 3 * F32 + I32,
         "opt_fire_step": 4 * F64 + 9 * F32 + 18 * F32 + (9 + 9 + 18 + 18) * F64 + 2 * F64 + 6 * F64 + 3 * 2 * I32 + 4 * F64}


def part_a(n, launches, dev):
    G = 8
    gen = torch.Generator(device=dev).manual_seed(0)
    force, vel = torch.randn(n, 3, device=dev, generator=gen), torch.randn(n, 3, device=dev, generator=gen)
    x, rp = torch.randn(n, 3, device=dev, generator=gen), torch.randn(n, 3, device=dev, generator=gen)
    ptr = torch.linspace(0, n, G + 1, device=dev).round().to(torch.int32)
    replica = torch.repeat_interleave(torch.arange(G, dtype=torch.int32, device=dev), (ptr[1:] - ptr[:-1]).long())
    f64 = dict(dtype=torch.float64, device=dev)
    A = torch.eye(3, **f64).repeat(G, 1, 1) + 0.01 * torch.randn(G, 3, 3, **f64, generator=gen)
    A_prev, vcell = A.clone(), torch.zeros(G, 3, 3, **f64)
    cell = (torch.eye(3, device=dev) * 200.0).repeat(G, 1, 1).contiguous()
    h0, virial = cell.double(), torch.randn(G, 3, 3, device=dev, generator=gen)
    P0, cf = torch.zeros(G, **f64), torch.full((G,), n / G, **f64)
    dt, alpha = torch.full((G,), 0.1, **f64), torch.full((G,), 0.1, **f64)
    n_pos, steps, converged = (torch.zeros(G, dtype=torch.int32, device=dev) for _ in range(3))
    coef = torch.tensor([[1.0, 0.0, 0.0]] * G, **f64)      # (timing only: keeps r' / x / vel from drifting over the launches)
    fmax_out, n_active = torch.zeros(G, **f64), torch.zeros(1, dtype=torch.int32, device=dev)
    sums = ops.opt_fire_reduce(force, vel, A, replica, ptr)
    calls = {"opt_fire_reduce": (lambda: ops.opt_fire_reduce(force, vel, A, replica, ptr), n),
             # move=False: the convergence test and the cell rows' forces without changing the state
             "opt_fire_step": (lambda: ops.opt_fire_step(sums, virial, cell, h0, A, A_prev, vcell, P0, cf, dt, alpha, n_pos, steps,
                                                         converged, 1e-30, 1.0, 0.2, False, coef, fmax_out, n_active), G),
             "opt_fire_update": (lambda: ops.opt_fire_update(x, rp, vel, force, A_prev, A, replica, converged, coef), n)}
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


def boxes(n):
    parts = []
    for s in range(n):
        p, z, c = synthetic.water_box(4, seed=s)
        parts.append((p + np.random.default_rng(500 + s).normal(0, 0.1, p.shape).astype(np.float32), z, c))
    pos = np.concatenate([p for p, _, _ in parts])
    Z = np.concatenate([z for _, z, _ in parts])
    cell = np.stack([c for _, _, c in parts])
    return parts, pos, Z, cell, np.repeat(np.arange(n), [len(z) for _, z, _ in parts])


def host_fire(calc, pos, Z, cell, fmax, max_steps, dt=0.1, dt_max=1.0, max_step=0.2):
    """ASE's FIRE over ``NNCalculator`` on the host: one ``calculate`` per step.  Returns ``(steps, converged)``."""
    atoms = md.SimpleAtoms(Z, pos, cell)
    atoms.calc = calc
    v, a, n_pos = None, 0.1, 0
    for k in range(max_steps + 1):
        f = atoms.get_forces().astype(np.float64)
        if (f * f).sum(1).max() < fmax * fmax:
            return k, True
        if k == max_steps:
            return k, False
        if v is None:
            v = np.zeros_like(f)
        elif np.vdot(f, v) > 0.0:
            v = (1.0 - a) * v + a * f / np.sqrt(np.vdot(f, f)) * np.sqrt(np.vdot(v, v))
            if n_pos > 5:
                dt, a = min(dt * 1.1, dt_max), a * 0.99
            n_pos += 1
        else:
            v[:] = 0.0
            a, dt, n_pos = 0.1, dt * 0.5, 0
        v = v + dt * f
        dr = dt * v
        nd = np.sqrt(np.vdot(dr, dr))
        if nd > max_step:
            dr *= max_step / nd
        atoms.positions = atoms.positions + dr


def part_b(n_boxes, n_host, fmax_frac, max_steps, dev):
    model = model_of("C1", dev)
    parts, pos, Z, cell, batch = boxes(n_boxes)
    st0 = {}
    fire_relax_device(model, Z, pos, cell, max_steps=0, batch=batch, stats=st0, device=str(dev))
    fmax = fmax_frac * float(st0["fmax"][0].min())
    print(f"(b) {n_boxes} x 192 atoms, fmax {fmax:.4g} eV/A ({fmax_frac} x the smallest starting max force)", flush=True)
    res = {"boxes": n_boxes, "atoms_per_box": 192, "fmax_eV_A": fmax, "max_steps": max_steps}
    out = model.energy_forces_virial(Data(pos=torch.from_numpy(pos).to(dev), atomic_number=torch.from_numpy(Z).to(dev),
                                          cell=torch.from_numpy(cell).to(dev), batch=torch.from_numpy(batch).to(dev)))
    W = out["virial"].double().cpu().numpy()
    P_start = np.trace(W, axis1=1, axis2=2) / (3 * np.abs(np.linalg.det(cell.astype(np.float64)))) * md.EV_A3_TO_BAR
    for name, kw in (("device_eager", dict(skin=0.5)), ("device_graph", dict(skin=0.5, cuda_graph=True)),
                     ("device_cell_eager", dict(skin=0.5, relax_cell=True, pressure_bar=P_start))):
        fire_relax_device(model, Z, pos, cell, fmax=fmax, max_steps=max_steps, batch=batch, device=str(dev), **kw)
        st = {}
        ms, _ = timed(lambda: fire_relax_device(model, Z, pos, cell, fmax=fmax, max_steps=max_steps, batch=batch, device=str(dev),
                                                stats=st, **kw))
        steps = st["steps"].cpu().numpy()
        r = {"ms": ms, "structures_per_s": n_boxes / (ms * 1e-3), "iterations": int(st["energy"].shape[0]),
             "steps_mean": float(steps.mean()), "steps_max": int(steps.max()), "converged": int(st["converged"].sum()),
             "builds": st["builds"], "reuses": st["reuses"]}
        res[name] = r
        print(f"(b) {name}: {ms:.1f} ms, {r['structures_per_s']:.3g} structures/s, {r['iterations']} iterations, steps mean "
              f"{r['steps_mean']:.1f} max {r['steps_max']}, converged {r['converged']}/{n_boxes}, builds {r['builds']} "
              f"reuses {r['reuses']}", flush=True)
    calc = NNCalculator(model, None, 0.0, device_=str(dev))
    p, z, c = parts[0]
    host_fire(calc, p, z, c, fmax, 5)                      # warm-up
    torch.cuda.synchronize()
    host = []
    for k in range(n_host):
        p, z, c = parts[k]
        t0 = time.perf_counter()
        steps, conv = host_fire(calc, p, z, c, fmax, max_steps)
        torch.cuda.synchronize()
        host.append({"s": time.perf_counter() - t0, "steps": steps, "converged": conv})
    total = sum(h["s"] for h in host)
    res["host_fire_calculator"] = {"boxes": n_host, "per_box": host, "structures_per_s": n_host / total,
                                   "steps_mean": float(np.mean([h["steps"] for h in host]))}
    print(f"(b) host FIRE over NNCalculator, {n_host} boxes one at a time: {n_host / total:.3g} structures/s, steps "
          f"{[h['steps'] for h in host]}, converged {[h['converged'] for h in host]}", flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--boxes", type=int, default=64)
    ap.add_argument("--host-boxes", type=int, default=4)
    ap.add_argument("--fmax-frac", type=float, default=0.1)
    ap.add_argument("--max-steps", type=int, default=2000)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("relax_cost.py measures on a GPU; none is available")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"card": card()}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    res["a_kernels"] = {str(n): part_a(n, a.launches, dev) for n in (10 ** 6, 10 ** 7)}
    res["b_boxes"] = part_b(a.boxes, a.host_boxes, a.fmax_frac, a.max_steps, dev)
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "relax_cost.json"), "w") as f:
            f.write(doc)


if __name__ == "__main__":
    main()
