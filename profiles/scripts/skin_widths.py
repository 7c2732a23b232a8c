"""Verlet-skin MD at hidden widths other than 128 (tile-sweep edge kernels): ms/step of ``velocity_verlet_device`` with a
fresh neighbour list per step (skin 0) against a re-used skin list, and the per-kernel times of the edge passes on both.

    python profiles/scripts/skin_widths.py [--n-side 26] [--steps 20] [--rounds 3] [--out DIR]

HVNet, elements H / O, rc = 5, 3 layers, K = 128, F = 256 and 512, frozen parameters, on a water box of 3 * n_side^3 atoms
(26 -> 52 728 atoms) with 300 K velocities.  Per width: one warm-up run of each skin, then ``rounds`` timed runs alternating
the two (host clock around a run that ends in a device synchronise; every run evaluates steps + 1 times), then one run of
each with ``ops.TIMERS`` on for the per-kernel CUDA-event times.  The card's name and power limit are printed with the
numbers.  Prints one JSON document and writes it to ``DIR/skin_widths.json`` when ``--out`` is given.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import hermnet_b200 as H  # noqa: E402
from hermnet_b200 import ops, synthetic  # noqa: E402
from hermnet_b200.plugin import md  # noqa: E402

KERNELS = ("painn_edge_fwd", "painn_edge_bwd_dst", "painn_edge_bwd_src", "layer0_basis_fwd", "layer0_basis_bwd", "edge_geom_fwd",
           "edge_geom_bwd")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def run(model, Z, pos, cell, v0, steps, skin, dev):
    st = {}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    p1, _, e = md.velocity_verlet_device(model, Z, pos, cell, v0, steps=steps, dt_fs=0.5, device=dev, skin=skin, stats=st)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, st, p1, e


def kernel_times(model, Z, pos, cell, v0, steps, skin, dev):
    ops.TIMERS = {}
    try:
        run(model, Z, pos, cell, v0, steps, skin, dev)
        out = {}
        for name, evs in ops.TIMERS.items():
            if name in KERNELS:
                ms = [a.elapsed_time(b) for a, b in evs]
                out[name] = {"calls": len(ms), "ms_per_call": float(np.mean(ms)), "ms_total": float(np.sum(ms))}
        return out
    finally:
        ops.TIMERS = None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-side", type=int, default=26)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--skin", type=float, default=0.5)
    ap.add_argument("--widths", default="256,512")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("skin_widths.py measures on a GPU; none is available")
    dev = "cuda:0"
    pos, Z, cell = synthetic.water_box(a.n_side, seed=1)
    masses = np.array([md.MASSES[int(z)] for z in Z])[:, None] * md.AMU_A2_FS2_TO_EV
    v0 = np.random.default_rng(2).normal(size=pos.shape) * np.sqrt(md.KB_EV * 300.0 / masses)
    v0 -= v0.mean(0, keepdims=True)
    res = {"card": card(), "atoms": int(len(Z)), "steps": a.steps, "skin": a.skin, "widths": {}}
    print("card:", res["card"], "atoms:", res["atoms"], flush=True)
    for F in [int(x) for x in a.widths.split(",")]:
        torch.manual_seed(0)
        model = H.HVNet(elems=["H", "O"], rc=5.0, num_layers=3, hidden_channels=F, num_rbf=128).to(dev).eval()
        for q in model.parameters():
            q.requires_grad_(False)
        g0 = model.build_graph(torch.from_numpy(pos).to(dev), torch.from_numpy(Z).to(dev), torch.from_numpy(cell)[None].to(dev))
        g1 = model.build_graph(torch.from_numpy(pos).to(dev), torch.from_numpy(Z).to(dev), torch.from_numpy(cell)[None].to(dev),
                               skin=a.skin)
        entry = {"edges_fresh": int(g0.n_edges), "entries_skin_list": int(g1.n_edges)}
        del g0, g1
        for skin in (0.0, a.skin):                      # warm-up: module loads, allocator, cuBLAS heuristics
            run(model, Z, pos, cell, v0, 3, skin, dev)
        times = {0.0: [], a.skin: []}
        stats, final = {}, {}
        for _ in range(a.rounds):
            for skin in (0.0, a.skin):
                t, st, p1, e = run(model, Z, pos, cell, v0, a.steps, skin, dev)
                times[skin].append(1e3 * t / (a.steps + 1))
                stats[skin], final[skin] = st, (p1, e)
        entry["ms_per_step_fresh"] = times[0.0]
        entry["ms_per_step_skin"] = times[a.skin]
        entry["stats_fresh"], entry["stats_skin"] = stats[0.0], stats[a.skin]
        entry["max_dpos_A"] = float((final[0.0][0] - final[a.skin][0]).abs().max())
        entry["max_rel_dE"] = float(((final[0.0][1] - final[a.skin][1]).abs().max() / final[0.0][1].abs().max()))
        entry["kernels_fresh"] = kernel_times(model, Z, pos, cell, v0, 5, 0.0, dev)
        entry["kernels_skin"] = kernel_times(model, Z, pos, cell, v0, 5, a.skin, dev)
        res["widths"][str(F)] = entry
        print(f"F={F}: fresh {np.median(times[0.0]):.2f} ms/step  skin {np.median(times[a.skin]):.2f} ms/step  "
              f"{stats[a.skin]}  entries {entry['entries_skin_list']} vs edges {entry['edges_fresh']}", flush=True)
        del model
        torch.cuda.empty_cache()
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "skin_widths.json"), "w") as f:
            f.write(doc)


if __name__ == "__main__":
    main()
