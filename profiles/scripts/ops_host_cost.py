"""Host cost of one ``ops`` wrapper call: argument checks, pointer conversion, the ctypes call and the launch bookkeeping.

Each case times ``--calls`` back-to-back calls with ``time.perf_counter`` and ends the window with one device
synchronise.  The inputs are small, so the kernels finish well inside the host time of a call and the number is the
host's cost, not the GPU's:
  md_kick          1 024 atoms, with the kinetic energies
  md_scr_barostat  8 replicas
  opt_fire_step    8 replicas with the cell rows (``A`` given)
  gather_rows      1 024 rows of 128 floats
  segment_sum      1 024 rows of 128 floats into 64 segments
  gemm_tf32x3_ex   [128, 128] x [128, 128]^T

    python profiles/scripts/ops_host_cost.py [--calls 10000] [--rounds 1] [--out DIR]

The card's name, power limit and max SM clock are printed with the numbers; one JSON document goes to stdout and to
``DIR/ops_host_cost.json`` with ``--out``.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from hermnet_b200 import ops  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def cases(dev):
    f32 = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)
    f64 = lambda *s: torch.zeros(s, dtype=torch.float64, device=dev)
    i32 = lambda *s: torch.zeros(s, dtype=torch.int32, device=dev)
    i64 = lambda *s: torch.zeros(s, dtype=torch.int64, device=dev)
    n, G = 1024, 8
    vel, force, inv_mass, kinetic, step = f32(n, 3), f32(n, 3), torch.ones(n, device=dev), f32(n), i64(1)
    cell = (torch.eye(3, device=dev) * 20.0).repeat(G, 1, 1).contiguous()
    kin, virial = torch.full((G,), 10.0, device=dev), f32(G, 3, 3)
    P0, kT, beta = f32(G), torch.full((G,), 0.025, device=dev), torch.full((G,), 1e-3, device=dev)
    seed, mu, pressure = torch.arange(G, dtype=torch.int64, device=dev), torch.ones(G, device=dev), f32(G)
    eye = torch.eye(3, dtype=torch.float64, device=dev).repeat(G, 1, 1).contiguous()
    fire = dict(sums=f64(G, 4), virial=f32(G, 3, 3), cell=cell.clone(), h0=eye.clone() * 20.0, A=eye.clone(), A_prev=eye.clone(),
                vcell=f64(G, 3, 3), P0=f64(G), cell_factor=torch.full((G,), float(n), dtype=torch.float64, device=dev),
                dt=torch.full((G,), 0.1, dtype=torch.float64, device=dev), alpha=torch.full((G,), 0.1, dtype=torch.float64, device=dev),
                n_pos=i32(G), steps=i32(G), converged=i32(G), fmax=0.05, dt_max=1.0, max_step=0.2, move=True, coef=f64(G, 3),
                fmax_out=f64(G), n_active=i32(1))
    X, idx = torch.randn(n, 128, device=dev), torch.randperm(n, device=dev).to(torch.int32)
    rowptr = torch.arange(0, n + 1, n // 64, dtype=torch.int32, device=dev)
    a = torch.randn(128, 128, device=dev)
    w_hi, w_lo = ops.split_tf32(torch.randn(128, 128, device=dev))
    out = f32(128, 128)
    return {
        "md_kick": lambda: ops.md_kick(vel, force, inv_mass, 0.25, kinetic, step),
        "md_scr_barostat": lambda: ops.md_scr_barostat(cell, kin, virial, P0, kT, beta, seed, step, 0.5, 1000.0, mu, pressure),
        "opt_fire_step": lambda: ops.opt_fire_step(**fire),
        "gather_rows": lambda: ops.gather_rows(X, idx),
        "segment_sum": lambda: ops.segment_sum(X, rowptr, None, 64),
        "gemm_tf32x3_ex": lambda: ops.gemm_tf32x3_ex(a, w_hi, w_lo, None, out),
    }


def host_us(fn, calls):
    for _ in range(100):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / calls * 1e6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10000)
    ap.add_argument("--rounds", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ops_host_cost.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"card": card(), "calls": args.calls, "us_per_call": {}}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    fns = cases(dev)
    for _ in range(args.rounds):
        for name, fn in fns.items():
            res["us_per_call"].setdefault(name, []).append(host_us(fn, args.calls))
    for name, us in res["us_per_call"].items():
        print(f"{name:16s} " + " ".join(f"{u:7.2f}" for u in us) + " us/call", flush=True)
    doc = json.dumps(res)
    print(doc)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "ops_host_cost.json"), "w") as f:
            f.write(doc)


if __name__ == "__main__":
    main()
