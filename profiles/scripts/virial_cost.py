"""Cost of the virial: per-evaluation device time of
  (a) energy + forces                          (``model(data)`` + ``autograd.grad(E, pos)``),
  (b) the NPT route of ``NNCalculator``        ((a) with ``retain_graph`` + ``utils.virial_calc``'s second backward to the cell),
  (c) ``model.energy_forces_virial``           (one backward, ``edge_virial_atom`` and a 9-wide segment sum),
and the ``edge_virial_atom`` / ``edge_geom_bwd`` kernel times from ``ops.TIMERS`` in the same run.

    python profiles/scripts/virial_cost.py [--rounds 5] [--evals 5] [--c4-scale 1.0] [--water-side 26] [--out DIR]

Systems: the C4 workload (synthetic 1 000 000-atom Li/Al/Si/O box, HVNet L=3 F=128 K=128 rc=5) and the 52 728-atom water box
of ``skin_widths.py`` with HVNet L=3 F=256 K=128 rc=5; frozen parameters, the neighbour list built once and attached.  Per
system: two warm-up evaluations of each route, then ``rounds`` rounds alternating (a), (b), (c), each timed with CUDA
events around ``evals`` evaluations.  The virials of (b) and (c) on the same seeded inputs are compared against the bound
``1e-5 * (sum_i |pos_i||F_i| + sum |cell| |dE/dcell|)``.  The card's name and power limit are printed with the numbers; one
JSON document goes to stdout and to ``DIR/virial_cost.json`` with ``--out``.
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
from hermnet_b200.utils import NKTV2P, virial_calc  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def routes(model, pos, Z, cell, g):
    def data(cell_grad):
        d = H.Data(pos=pos.clone().requires_grad_(True), atomic_number=Z,
                   cell=cell.clone().requires_grad_(cell_grad))
        d.graph = g
        return d

    def a():
        d = data(False)
        e = model(d)
        return e.detach(), -torch.autograd.grad(e.sum(), d.pos)[0]

    def b():
        d = data(True)
        e = model(d)
        f = -torch.autograd.grad(e.sum(), d.pos, retain_graph=True)[0]
        return e.detach(), f, virial_calc(cell=d.cell, pos=d.pos.detach(), forces=f, energy=e, units='metal', pbc=True)

    def c():
        d = data(False)
        return model.energy_forces_virial(d)
    return {"a": a, "b": b, "c": c}


def time_route(fn, evals):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(evals):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / evals


def compare(model, pos, Z, cell, g, fns):
    """(b) against (c), symmetrised and in the calculator's units, with the cell-gradient route's own condition scale."""
    d = H.Data(pos=pos.clone().requires_grad_(True), atomic_number=Z, cell=cell.clone().requires_grad_(True))
    d.graph = g
    e = model(d)
    gp, gc = torch.autograd.grad(e.sum(), [d.pos, d.cell])
    scale = float((pos.norm(dim=1) * gp.norm(dim=1)).double().sum() + (cell.reshape(3, 3).abs().double() *
                                                                          gc.reshape(3, 3).abs().double()).sum())
    vb = fns["b"]()[2].double()
    W = fns["c"]()["virial"][0].double()
    vc = 0.5 * (W + W.T) * NKTV2P["metal"]
    err = float((vb - vc).abs().max())
    return {"max_abs_diff": err, "bound": 1e-5 * scale * NKTV2P["metal"], "ok": err <= 1e-5 * scale * NKTV2P["metal"]}


def kernel_times(fn):
    ops.TIMERS = {}
    try:
        fn()
        torch.cuda.synchronize()
        return {k: float(np.sum([s.elapsed_time(t) for s, t in v])) for k, v in ops.TIMERS.items()
                if k in ("edge_virial_atom", "edge_geom_bwd")}
    finally:
        ops.TIMERS = None


def measure(name, pos, Z, cell, F, elems, rounds, evals, dev):
    torch.manual_seed(0)
    model = H.HVNet(elems=elems, rc=5.0, num_layers=3, hidden_channels=F, num_rbf=128).to(dev).eval()
    for q in model.parameters():
        q.requires_grad_(False)
    pos = torch.from_numpy(pos).to(dev)
    Z = torch.from_numpy(Z).to(dev)
    cell = torch.from_numpy(cell).reshape(1, 3, 3).to(dev)
    g = model.build_graph(pos, Z, cell)
    fns = routes(model, pos, Z, cell, g)
    for k in "abc":
        for _ in range(2):
            fns[k]()
    torch.cuda.synchronize()
    times = {k: [] for k in "abc"}
    for _ in range(rounds):
        for k in "abc":
            times[k].append(time_route(fns[k], evals))
    med = {k: float(np.median(v)) for k, v in times.items()}
    res = {"atoms": int(pos.size(0)), "edges": int(g.n_edges), "F": F, "ms_per_eval": times, "median_ms": med,
           "kernels_ms_c": kernel_times(fns["c"]), "kernels_ms_a": kernel_times(fns["a"]),
           "check_b_vs_c": compare(model, pos, Z, cell, g, fns)}
    print(f"{name}: N={res['atoms']} E={res['edges']} F={F}  (a) {med['a']:.2f} ms  (b) {med['b']:.2f} ms  "
          f"(c) {med['c']:.2f} ms  kernels {res['kernels_ms_c']}  check {res['check_b_vs_c']}", flush=True)
    del model, g, fns
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--evals", type=int, default=5)
    ap.add_argument("--c4-scale", type=float, default=1.0)
    ap.add_argument("--water-side", type=int, default=26)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("virial_cost.py measures on a GPU; none is available")
    dev = "cuda:0"
    res = {"card": card(), "rounds": a.rounds, "evals_per_round": a.evals, "systems": {}}
    print("card:", res["card"], flush=True)
    (pos, Z, cell), cfg = synthetic.config("C4", a.c4_scale)
    res["systems"]["C4"] = measure("C4", pos, Z, cell, 128, cfg["elems"], a.rounds, a.evals, dev)
    pos, Z, cell = synthetic.water_box(a.water_side, seed=1)
    res["systems"]["water"] = measure("water", pos, Z, cell, 256, ["H", "O"], a.rounds, a.evals, dev)
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "virial_cost.json"), "w") as f:
            f.write(doc)
    if not all(s["check_b_vs_c"]["ok"] for s in res["systems"].values()):
        raise SystemExit("virial of energy_forces_virial differs from the cell-gradient route beyond the bound")


if __name__ == "__main__":
    main()
