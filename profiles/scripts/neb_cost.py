"""Cost of nudged elastic band runs on the device (``plugin.neb.neb_device``, kernels of csrc/hn_neb.cu):
  (a) per-launch time of ``hn_neb_reduce``, ``hn_neb_step`` and ``hn_neb_project`` (8 bands of 7 images) from CUDA events
      over ``--launches`` back-to-back launches at 10^6 and 10^7 image atoms, with the achieved bandwidth against the bytes
      computed from the shapes;
  (b) the per-iteration NEB overhead (the three kernels) against the evaluation, for 8 bands x 7 images of the 192-atom C1
      water box (HVNet L=3 F=128, last readout layer x 1e-3 as bench.py C3 does): eager with a fresh list per call, and
      replayed with ``cuda_graph`` on a re-used skin list; plus ``neb_device`` itself per iteration in both modes;
  (c) end to end: ``--bands`` bands (two rattled copies of the C1 box as endpoints, 7 images) relaxed together with
      ``neb_device`` against one band through a host NEB + FIRE loop over ``NNCalculator``, one ``calculate`` per image per
      iteration (the route of ASE's ``NEB`` + ``FIRE``): bands converged per second.

    python profiles/scripts/neb_cost.py [--bands 8] [--fmax-frac 0.1] [--host-max-steps 600] [--launches 500] [--out DIR]

fmax is a fixed fraction of the smallest starting band fmax: the random-weight model's forces have no physical scale.  The
host loop stops after ``--host-max-steps`` steps; its bands per second then count only the steps it took.

The card's name, power limit and max SM clock are read in the same run and printed with the numbers; one JSON document goes
to stdout and to ``DIR/neb_cost.json`` with ``--out``.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import hermnet_b200 as H  # noqa: E402
from hermnet_b200 import ops, synthetic  # noqa: E402
from hermnet_b200.plugin import md  # noqa: E402
from hermnet_b200.plugin.calculator import NNCalculator  # noqa: E402
from hermnet_b200.plugin.md import VerletGraph  # noqa: E402
from hermnet_b200.plugin.neb import neb_device  # noqa: E402

F32, F64, I32 = 4, 8, 4
B_BANDS, K_IMAGES = 8, 7


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
    model.out_energy[2].weight.mul_(1.0e-3)
    model.out_energy[2].bias.mul_(1.0e-3)
    return model


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def layout(n_per_band, dev, seed=0):
    """Band-major layout of ``B_BANDS`` bands of ``K_IMAGES`` images with ``n_per_band`` atoms each."""
    B, K = B_BANDS, K_IMAGES
    gen = torch.Generator(device=dev).manual_seed(seed)
    N, M = B * n_per_band, B * K * n_per_band
    pos = 20.0 * torch.rand(M, 3, device=dev, generator=gen)
    initial, final = 20.0 * torch.rand(N, 3, device=dev, generator=gen), 20.0 * torch.rand(N, 3, device=dev, generator=gen)
    image = torch.arange(B * K, dtype=torch.int32, device=dev).repeat_interleave(n_per_band)
    image_ptr = (torch.arange(B * K + 1, device=dev) * n_per_band).to(torch.int32)
    band_ptr = (torch.arange(B + 1, device=dev) * n_per_band).to(torch.int32)
    return pos, initial, final, image, image_ptr, band_ptr


# bytes each kernel must move, per image atom: reduce reads the image's position and force and its image index, project
# reads the position and the image index and reads + writes the force; the neighbours are other images' positions (each
# position is read by three atoms: itself and its two neighbours, counted once here), the endpoints add 2 x 12 B per band
# atom, i.e. 24 / K per image atom; step: per image the five sums and the energy read, coef written.
def kernel_bytes(M):
    ends = 2 * 3 * F32 * M / K_IMAGES
    return {"neb_reduce": (3 + 3) * F32 * M + I32 * M + ends,
            "neb_project": 3 * F32 * M + 2 * 3 * F32 * M + I32 * M + ends,
            "neb_step": B_BANDS * K_IMAGES * (5 * F64 + F32 + 2 * F64)}


def part_a(M, launches, dev):
    pos, initial, final, image, image_ptr, band_ptr = layout(M // (B_BANDS * K_IMAGES), dev)
    M = pos.size(0)
    force = torch.randn(M, 3, device=dev)
    energy = torch.randn(B_BANDS * K_IMAGES, device=dev)
    end_energy = torch.randn(B_BANDS, 2, device=dev)
    spring = torch.full((B_BANDS,), 0.1, dtype=torch.float64, device=dev)
    coef = torch.zeros(B_BANDS * K_IMAGES, 2, dtype=torch.float64, device=dev)
    imax = torch.zeros(B_BANDS, dtype=torch.int32, device=dev)
    sums = ops.neb_reduce(pos, force, initial, final, image, image_ptr, band_ptr, K_IMAGES)
    zero = torch.zeros_like(coef)                 # (timing only: project with zero coefficients keeps the forces fixed)
    calls = {"neb_reduce": lambda: ops.neb_reduce(pos, force, initial, final, image, image_ptr, band_ptr, K_IMAGES),
             "neb_step": lambda: ops.neb_step(sums, energy, end_energy, spring, True, coef, imax),
             "neb_project": lambda: ops.neb_project(force, pos, initial, final, image, image_ptr, band_ptr, K_IMAGES, zero)}
    nbytes = kernel_bytes(M)
    res = {"image_atoms": M, "working_set_MB": (nbytes["neb_project"]) / 1e6, "L2_MB": 126}
    for k, fn in calls.items():
        for _ in range(20):
            fn()

        def run(fn=fn):
            for _ in range(launches):
                fn()
        ms, _ = timed(run)
        us = 1e3 * ms / launches
        gbs = nbytes[k] / (us * 1e-6) / 1e9
        res[k] = {"us_per_launch": us, "bytes": nbytes[k], "GB_per_s": gbs}
        print(f"(a) M={M} {k}: {us:.2f} us/launch, {nbytes[k] / 1e6:.3g} MB -> {gbs:.4g} GB/s", flush=True)
    return res


def water_bands(n_bands, rattle=0.05):
    p, z, c = synthetic.water_box(4, seed=0)
    x0 = np.concatenate([p + np.random.default_rng(100 + b).normal(0, rattle, p.shape).astype(np.float32) for b in range(n_bands)])
    x1 = np.concatenate([p + np.random.default_rng(200 + b).normal(0, rattle, p.shape).astype(np.float32) for b in range(n_bands)])
    Z = np.tile(z, n_bands)
    return x0, x1, Z, np.stack([c] * n_bands), np.repeat(np.arange(n_bands), len(z))


def part_b(model, dev, calls=20, launches=200):
    B, K = B_BANDS, K_IMAGES
    x0, x1, Z, cell, batch = water_bands(B)
    n = len(Z) // B
    lin = [x0 + (k + 1) / (K + 1) * (x1 - x0) for k in range(K)]
    # band-major images of the evaluation
    pos = torch.from_numpy(np.concatenate([np.stack([lin[k][batch == b] for k in range(K)]).reshape(-1, 3) for b in range(B)])).to(dev)
    Zi = torch.from_numpy(np.tile(Z[:n], B * K)).long().to(dev)
    ci = torch.from_numpy(np.repeat(cell, K, axis=0)).to(dev)
    img = torch.arange(B * K, device=dev).repeat_interleave(n)
    res = {"bands": B, "images": K, "atoms_per_image": n}
    for name, kw in (("eval_eager", dict(skin=0.0)), ("eval_graph_skin", dict(skin=0.5, cuda_graph=True))):
        vg = VerletGraph(model, batch=img, **kw)
        for _ in range(3):
            vg.evaluate(pos, Zi, ci)
        ms, _ = timed(lambda: [vg.evaluate(pos, Zi, ci) for _ in range(calls)])
        res[name] = {"ms_per_call": ms / calls, "builds": vg.builds, "reuses": vg.reuses}
        print(f"(b) {name}: {ms / calls:.3f} ms per evaluation", flush=True)
    # the three NEB kernels on this layout
    initial, final = torch.from_numpy(x0).to(dev), torch.from_numpy(x1).to(dev)
    image, image_ptr = img.to(torch.int32), (torch.arange(B * K + 1, device=dev) * n).to(torch.int32)
    band_ptr = (torch.arange(B + 1, device=dev) * n).to(torch.int32)
    force = torch.randn_like(pos)
    e, e_end = torch.randn(B * K, device=dev), torch.randn(B, 2, device=dev)
    spring = torch.full((B,), 0.1, dtype=torch.float64, device=dev)
    coef, imax = torch.zeros(B * K, 2, dtype=torch.float64, device=dev), torch.zeros(B, dtype=torch.int32, device=dev)

    def neb_kernels():
        sums = ops.neb_reduce(pos, force, initial, final, image, image_ptr, band_ptr, K)
        ops.neb_step(sums, e, e_end, spring, True, coef, imax)
        ops.neb_project(force.clone(), pos, initial, final, image, image_ptr, band_ptr, K, coef)
    for _ in range(10):
        neb_kernels()
    ms, _ = timed(lambda: [neb_kernels() for _ in range(launches)])
    res["neb_kernels_ms_per_iteration"] = ms / launches
    print(f"(b) three NEB kernels (+ one force copy): {ms / launches * 1e3:.1f} us per iteration", flush=True)
    # neb_device per iteration in steady state: the difference of a 60- and a 20-step run (set-up, endpoint evaluation and
    # graph capture cancel)
    for name, kw in (("neb_device_eager", dict(skin=0.0)), ("neb_device_graph_skin", dict(skin=0.5, cuda_graph=True))):
        def run(steps, kw=kw):
            st = {}
            ms, _ = timed(lambda: neb_device(model, Z, x0, x1, cell, n_images=K, batch=batch, climb=True, fmax=1e-9,
                                             max_steps=steps, device=str(dev), stats=st, **kw))
            return ms, st
        run(20)
        (ms0, _), (ms1, st) = run(20), run(60)
        res[name] = {"ms_per_iteration": (ms1 - ms0) / 40, "ms_20_steps": ms0, "ms_60_steps": ms1, "builds_60": st["builds"],
                     "reuses_60": st["reuses"]}
        print(f"(b) {name}: {(ms1 - ms0) / 40:.3f} ms per iteration (60- and 20-step runs: {ms1:.1f} / {ms0:.1f} ms), "
              f"builds {st['builds']} in 60 steps", flush=True)
    return res


def host_neb(calc, x0, x1, Z, cell, K, fmax, max_steps, k=0.1, dt=0.1, dt_max=1.0, max_step=0.2):
    """ASE's NEB (improved tangent, climbing image) + FIRE over ``NNCalculator`` on the host: one ``calculate`` per image per
    iteration.  Returns ``(steps, converged)``."""
    atoms = [md.SimpleAtoms(Z, x, cell) for x in [x0] + [x0 + (i + 1) / (K + 1) * (x1 - x0) for i in range(K)] + [x1]]
    for a in atoms:
        a.calc = calc
    E_ends = [atoms[0].get_potential_energy(), atoms[-1].get_potential_energy()]
    v, a_, n_pos = None, 0.1, 0
    for step in range(max_steps + 1):
        F, E = [], [E_ends[0]]
        for at in atoms[1:-1]:
            F.append(at.get_forces().astype(np.float64))
            E.append(at.calc.results["energy"])
        E.append(E_ends[1])
        imax = 1 + int(np.argmax(E[1:-1]))
        out = []
        for i in range(1, K + 1):
            tp, tm = atoms[i + 1].positions - atoms[i].positions, atoms[i].positions - atoms[i - 1].positions
            ep, e0, em = E[i + 1], E[i], E[i - 1]
            if ep > e0 > em:
                tau = tp
            elif ep < e0 < em:
                tau = tm
            else:
                vmax, vmin = max(abs(ep - e0), abs(em - e0)), min(abs(ep - e0), abs(em - e0))
                tau = tp + tm if vmax == 0 else (tp * vmax + tm * vmin if ep > em else tp * vmin + tm * vmax)
            tau = tau / np.linalg.norm(tau)
            f = F[i - 1]
            if i == imax:
                out.append(f - 2 * np.vdot(f, tau) * tau)
            else:
                out.append(f - np.vdot(f, tau) * tau + tau * k * (np.linalg.norm(tp) - np.linalg.norm(tm)))
        f = np.concatenate(out)
        if (f * f).sum(1).max() < fmax * fmax:
            return step, True
        if step == max_steps:
            return step, False
        if v is None:
            v = np.zeros_like(f)
        elif np.vdot(f, v) > 0.0:
            v = (1.0 - a_) * v + a_ * f / np.sqrt(np.vdot(f, f)) * np.sqrt(np.vdot(v, v))
            if n_pos > 5:
                dt, a_ = min(dt * 1.1, dt_max), a_ * 0.99
            n_pos += 1
        else:
            v[:] = 0.0
            a_, dt, n_pos = 0.1, dt * 0.5, 0
        v = v + dt * f
        dr = dt * v
        nd = np.sqrt(np.vdot(dr, dr))
        if nd > max_step:
            dr *= max_step / nd
        n = len(Z)
        for i in range(K):
            atoms[i + 1].positions = atoms[i + 1].positions + dr[i * n:(i + 1) * n]


def part_c(model, n_bands, fmax_frac, max_steps, host_max_steps, dev):
    K = K_IMAGES
    x0, x1, Z, cell, batch = water_bands(n_bands)
    st0 = {}
    neb_device(model, Z, x0, x1, cell, n_images=K, batch=batch, climb=True, max_steps=0, stats=st0, device=str(dev))
    fmax = fmax_frac * float(st0["fmax"][0].min())
    print(f"(c) {n_bands} bands x {K} images x 192 atoms, fmax {fmax:.4g} eV/A ({fmax_frac} x the smallest starting band fmax)",
          flush=True)
    res = {"bands": n_bands, "images": K, "fmax_eV_A": fmax}
    for name, kw in (("device_eager", dict(skin=0.5)), ("device_graph", dict(skin=0.5, cuda_graph=True))):
        run = lambda: neb_device(model, Z, x0, x1, cell, n_images=K, batch=batch, climb=True, fmax=fmax,  # noqa: E731
                                 max_steps=max_steps, device=str(dev), stats=st, **kw)
        st = {}
        run()
        st = {}
        ms, _ = timed(run)
        steps = st["steps"].cpu().numpy()
        r = {"ms": ms, "bands_per_s": n_bands / (ms * 1e-3), "iterations": int(st["energy"].shape[0]),
             "steps_mean": float(steps.mean()), "steps_max": int(steps.max()), "converged": int(st["converged"].sum()),
             "builds": st["builds"], "reuses": st["reuses"]}
        res[name] = r
        print(f"(c) {name}: {ms:.1f} ms, {r['bands_per_s']:.3g} bands/s, {r['iterations']} iterations, steps mean "
              f"{r['steps_mean']:.1f} max {r['steps_max']}, converged {r['converged']}/{n_bands}, builds {r['builds']} "
              f"reuses {r['reuses']}", flush=True)
    calc = NNCalculator(model, None, 0.0, device_=str(dev))
    sl = batch == 0
    host_neb(calc, x0[sl], x1[sl], Z[sl], cell[0], K, fmax, 3)             # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    steps, conv = host_neb(calc, x0[sl], x1[sl], Z[sl], cell[0], K, fmax, host_max_steps)
    torch.cuda.synchronize()
    s = time.perf_counter() - t0
    res["host_neb_calculator"] = {"bands": 1, "s": s, "steps": steps, "converged": conv, "bands_per_s": 1.0 / s,
                                  "ms_per_iteration": 1e3 * s / (steps + 1)}
    print(f"(c) host NEB + FIRE over NNCalculator, band 0 alone: {s:.2f} s, {steps} steps, converged {conv}, "
          f"{1.0 / s:.3g} bands/s, {1e3 * s / (steps + 1):.1f} ms per iteration", flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bands", type=int, default=8)
    ap.add_argument("--fmax-frac", type=float, default=0.1)
    ap.add_argument("--max-steps", type=int, default=2000)
    ap.add_argument("--host-max-steps", type=int, default=600)
    ap.add_argument("--launches", type=int, default=500)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("neb_cost.py measures on a GPU; none is available")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"card": card()}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    res["a_kernels"] = {str(M): part_a(M, a.launches, dev) for M in (10 ** 6, 10 ** 7)}
    model = model_of("C1", dev)
    res["b_iteration"] = part_b(model, dev)
    res["c_end_to_end"] = part_c(model, a.bands, a.fmax_frac, a.max_steps, a.host_max_steps, dev)
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "neb_cost.json"), "w") as f:
            f.write(doc)


if __name__ == "__main__":
    main()
