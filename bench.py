#!/usr/bin/env python
"""Headline benchmark of the HermNet hot path on B200 (contract: see the task brief / DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload C4] [--scale S] [--dump-outputs DIR]

Workload (BASELINE.json configs[3], the configuration the metric "atom-steps/s (energy+forces)" is quoted on and the
largest that fits one GPU): HVNet, 3 interactions, F=128, K=128, rc=5 A on the synthetic 1 000 000-atom Li/Al/Si/O
periodic box, evaluated as energy + forces (forward + backward to positions).  N > 1 runs the SAME system with
spatial domain decomposition (hermnet_b200/parallel.py): strong scaling.

One JSON line on stdout (rank 0).  ``value``: graph and inputs resident in HBM, timed with CUDA events.
``e2e``: the same metric through the public API from pinned HOST buffers -- H2D copy of positions / numbers / cell,
neighbour-list build, forward, backward, D2H of forces + energy all inside the timed region.
``--impl reference`` times the CPU restatement of the reference PyG path (oracle/, the reference itself cannot be
imported without PyG / torch_scatter / ASE) on a bounded sample of the same workload with all host threads.
``--dump-outputs DIR`` (C4 / C5): after the timed steps, rank 0 writes what the timed path returned in its last step as
``DIR/energy.npy`` (float32 [1]) and ``DIR/forces.npy`` (float32 [N, 3], minus dE/dpos).  Inputs and weights are seeded,
so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HBM_FALLBACK_GBS = 6650.0      # /opt/skills/guides/B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C4")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the box edge (debug only; 1.0 = BASELINE size)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--micro", type=int, default=4, help="C2: graphs per micro-batch")
    ap.add_argument("--skin", type=float, default=0.4, help="C3: Verlet skin in Angstrom")
    ap.add_argument("--graph-skin", type=float, default=1.0, help="C3: Verlet skin of the CUDA-graph variant")
    ap.add_argument("--cuda-graph", type=int, default=1, help="C4: replay the resident step as ONE captured CUDA graph (0: eager launches)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the energy and forces of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload in ("C2", "C3")):
        ap.error("--dump-outputs is supported for the energy + forces workloads (C4, C5) of --impl b200")
    return args


# --------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (profiling recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, energy, grad):
    """``energy [1]`` and ``forces = -grad [N, 3]`` as float32 ``.npy`` files of at most DUMP_LIMIT_BYTES together; a larger
    force array is cut to a fixed, seeded sample of rows (the same rows in every run with the same N)."""
    os.makedirs(out_dir, exist_ok=True)
    e = energy.detach().float().cpu().numpy().reshape(-1)
    f = (-grad.detach()).float().cpu().numpy()
    max_rows = (DUMP_LIMIT_BYTES - 4096 - e.nbytes) // (3 * f.itemsize)     # 4096: room for the two .npy headers
    if f.shape[0] > max_rows:
        f = f[np.sort(np.random.default_rng(0).choice(f.shape[0], size=max_rows, replace=False))]
    np.save(os.path.join(out_dir, "energy.npy"), e)
    np.save(os.path.join(out_dir, "forces.npy"), f)


def workload(name: str, scale: float):
    from hermnet_b200 import synthetic
    (pos, Z, cell), cfg = synthetic.config(name, scale)
    return pos, Z, cell, cfg


def alg_bytes(kernel: str, N: int, E: int, T: int, F: int) -> float:
    """Algorithmic (compulsory, each array once) bytes of one launch -- SURVEY.md 8(d), stated in DESIGN.md."""
    xh, vec, out = 4.0 * N * 3 * F * T, 4.0 * N * 3 * F, 4.0 * N * 4 * F
    if kernel == "painn_edge_fwd":          # xh + vec in, dx + dvec out, (col 4 + geom 16) per edge, rowptr
        return xh + vec + out + 20.0 * E + 4.0 * (N + 1)
    if kernel == "painn_edge_bwd_dst":      # + g_dx/g_dvec in, per-edge (dL/du, dL/dd) out
        return xh + vec + out + 20.0 * E + 16.0 * E + 4.0 * (N + 1)
    if kernel == "painn_edge_bwd_src":      # xh, vec, g_dx/g_dvec in; grad_xh, grad_vec out; t_eid + edge_row + geom per edge
        return 2 * xh + 2 * vec + out + 24.0 * E + 4.0 * (N + 1)
    return float("nan")


# --------------------------------------------------------------------------------------------------------------
def _cpu_sample(cfg, n_side):
    """A ``n_side^3``-atom sample of the C4 workload (same lattice constant, jitter, species, model) for the CPU arm:
    inputs, oracle state dict and the neighbour list (k-d tree candidates + the exact ASE distance test)."""
    from hermnet_b200 import synthetic
    from oracle import hermnet_oracle as O
    from oracle import neighbor_oracle as NO
    pos, Z, cell = synthetic.cubic_lattice(n_side, 2.3, ("Li", "Al", "Si", "O"), None, 0.10, 4)
    mcfg = {k: v for k, v in cfg.items() if k != "kind"}
    sd = O.make_state_dict("HVNet", mcfg, 1234)
    t0 = time.perf_counter()
    i, j, S = NO.neighbor_list_pbc_binned(pos, cell, mcfg["rc"])
    t_nl = time.perf_counter() - t0
    ei, es = torch.from_numpy(np.stack([i, j])), torch.from_numpy(S.astype(np.float32))
    return dict(pos=torch.from_numpy(pos), Z=torch.from_numpy(Z), cell=torch.from_numpy(cell)[None], ei=ei, es=es, sd=sd,
                cfg=mcfg, t_nl=t_nl, pos_np=pos, cell_np=cell)


def _time_oracle(sm, repeats, budget, **kw):
    from oracle import hermnet_oracle as O
    times = []
    t_start = time.perf_counter()
    while len(times) < 2 or (len(times) < repeats + 1 and time.perf_counter() - t_start < budget):
        t0 = time.perf_counter()
        O.energy_and_forces("HVNet", sm["sd"], sm["cfg"], sm["pos"], sm["Z"], sm["ei"], sm["cell"], sm["es"], **kw)
        times.append(time.perf_counter() - t0)
    return statistics.median(times[1:]), len(times) - 1


def cpu_baseline(cfg, seconds_budget=25.0):
    """The reference's CPU path as BASELINE.md section 2 plans it (oracle = CPU restatement of the PyG path, all host threads):
    one 4 096-atom graph (the size of a BASELINE configs[1] cell) of the workload's lattice / species / model with the
    vectorised sub-graph mask -- forward + backward to positions, neighbour list (k-d tree + exact ASE test)
    INCLUDED in the headline value -- plus BASELINE configs[0] (192-atom water box) with the reference's literal
    ``in_subgraph`` loop (utils.py:11-24)."""
    from hermnet_b200 import synthetic
    from oracle import hermnet_oracle as O
    from oracle import neighbor_oracle as NO
    torch.set_num_threads(os.cpu_count() or 1)
    sm = _cpu_sample(cfg, 16)
    t, reps = _time_oracle(sm, 5, seconds_budget * 0.6)
    n = int(sm["Z"].numel())
    out = {"value": n / (t + sm["t_nl"]), "unit": "atom-steps/s", "cores": torch.get_num_threads(), "kind": "port",
           "sample": f"{n}-atom Li/Al/Si/O cell (16^3 sites of the workload's lattice; HVNet L=3 F=128 K=128 rc=5), E={sm['ei'].shape[1]}: "
                     f"neighbour list {sm['t_nl'] * 1e3:.0f} ms (k-d tree + exact ASE test) + oracle forward+backward {t:.3f} s (vectorised sub-graph "
                     f"mask, median of {reps} after 1 warm-up); the 1M-atom workload itself does not fit a CPU run (BASELINE.md section 2)",
           "seconds_per_step": t + sm["t_nl"], "model_only_atom_steps_per_s": n / t}
    # BASELINE configs[0]: the reference's own CPU-runnable case, literal per-destination-node loop
    (p1, z1, c1), cfg1 = synthetic.config("C1")
    m1 = {k: v for k, v in cfg1.items() if k != "kind"}
    i, j, S = NO.neighbor_list_pbc_binned(p1, c1, m1["rc"])
    s1 = dict(pos=torch.from_numpy(p1), Z=torch.from_numpy(z1), cell=torch.from_numpy(c1)[None], ei=torch.from_numpy(np.stack([i, j])),
              es=torch.from_numpy(S.astype(np.float32)), sd=O.make_state_dict("HVNet", m1, 1234), cfg=m1)
    t_lit, r_lit = _time_oracle(s1, 3, seconds_budget * 0.2, literal_subgraph=True)
    t_vec, _ = _time_oracle(s1, 3, seconds_budget * 0.1)
    out["c1_192_atoms"] = {"literal_subgraph_atom_steps_per_s": 192 / t_lit, "vectorised_atom_steps_per_s": 192 / t_vec,
                           "repeats": r_lit}
    return out


def run_reference(args):
    """``--impl reference``: the CPU restatement of the reference path (the reference itself needs PyG / torch_scatter / ASE,
    none installable here) on the 4 096-atom sample of the workload; every step = neighbour list + forward + backward."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import hermnet_oracle as O
    from oracle import neighbor_oracle as NO
    torch.set_num_threads(os.cpu_count() or 1)
    _, _, _, cfg = workload("C4", 0.05)
    sm = _cpu_sample(cfg, 16)
    times = []
    for _ in range(max(1, args.warmup) + max(1, args.steps)):
        t0 = time.perf_counter()
        i, j, S = NO.neighbor_list_pbc_binned(sm["pos_np"], sm["cell_np"], sm["cfg"]["rc"])
        sm["ei"], sm["es"] = torch.from_numpy(np.stack([i, j])), torch.from_numpy(S.astype(np.float32))
        O.energy_and_forces("HVNet", sm["sd"], sm["cfg"], sm["pos"], sm["Z"], sm["ei"], sm["cell"], sm["es"])
        times.append(time.perf_counter() - t0)
    times = times[max(1, args.warmup):]
    t = sum(times) / len(times)
    n = int(sm["Z"].numel())
    val = n / t
    base = {"value": val, "unit": "atom-steps/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{n}-atom Li/Al/Si/O cell of the workload's lattice, E={sm['ei'].shape[1]}; each step: neighbour list (k-d tree "
                      f"candidates + exact ASE test) + oracle forward + backward (vectorised sub-graph mask)",
            "seconds_per_step": t}
    line = {"impl": "reference", "metric": "atom-steps/s (energy+forces)", "value": val, "unit": "atom-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "C4: HVNet L=3 F=128 K=128 rc=5, Li/Al/Si/O periodic box; reference CPU path timed on a "
                                   "4096-atom cell of it (the 1M-atom O(N*E) path does not finish on a CPU)"},
            "cpu_baseline": base,
            "e2e": {"value": val, "unit": "atom-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def parity_check(model, pos_d, Z_d, cell_d, graph, kind, cfg):
    """Parity of THIS run's model on THIS workload: partial energy of a 19 A region, its gradient over the 34 A cut-out and
    the true forces of the interior atoms against the oracle on the cut-out (tests/cutout.py).  Outside every timed region;
    the oracle is the checker here, never the thing measured."""
    from tests import cutout
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    out = cutout.cutout_parity(model, sd, dict(cfg), pos_d, Z_d, cell_d, r_in=4.0, graph=graph, fp64_reference=True)
    return {"rel_dE": out["rel_dE"], "rel_dE_vs_fp64_oracle": out["rel_dE_vs_fp64"], "fp32_oracle_vs_fp64_oracle": out["oracle_fp32_vs_fp64"],
            "E_region_eV": out["E_region"], "max_dF": max(out["max_dF"], out.get("max_dF_interior", 0.0)), "n_checked": out["n_cutout"],
            "n_interior_true_forces": out["n_interior"], "max_dF_interior": out.get("max_dF_interior"),
            "method": f"oracle on the {out['n_cutout']}-atom cut-out (r = {out['r_cutout']:.0f} A) of the full system; E of the "
                      f"{out['n_region']}-atom region, dE/dpos over the cut-out, true forces of the interior atoms",
            "bars": {"rel_dE": 1e-5, "max_dF_eV_per_A": 1e-4},
            "neighbour_list": "bit-exact vs the builder's restatement of the ASE contract (ASE itself is absent: upstream unpinned)"}


# --------------------------------------------------------------------------------------------------------------
def run_c2(args):
    """``--workload C2`` (BASELINE.json configs[1]): HPNet L=3 F=128 K=128 on 32 synthetic 4 096-atom Li/Si/O cells, ONE
    force-matching training step (example/dist_train.py:84-104: energy + force loss, forces with create_graph=True, double
    backward, DDP gradient all-reduce, Adam) per bench step; the GLOBAL batch of 32 graphs is split over the ranks
    (strong scaling), each rank runs its share in micro-batches with gradient accumulation."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    import hermnet_b200 as H
    from hermnet_b200 import ops, parallel, synthetic
    GLOBAL = 32
    assert GLOBAL % world == 0
    n_side = max(2, int(round(16 * args.scale)))
    (_, _, _), cfg = synthetic.config("C2", args.scale)
    kind = cfg.pop("kind")
    torch.manual_seed(1234)
    model = getattr(H, kind)(**cfg).to(dev)
    ddp = parallel.data_parallel(model, device_ids=[local], output_device=local) if world > 1 else model
    ddp.train()
    opt = torch.optim.Adam(ddp.parameters(), lr=3e-4)
    mine = list(range(rank, GLOBAL, world))
    host = []
    gen = torch.Generator().manual_seed(99)
    for gidx in mine:
        pos, Z, cell = synthetic.cubic_lattice(n_side, 2.3, ("Li", "Si", "O"), (1 / 3, 1 / 6, 1 / 2), 0.10, 100 + gidx)
        host.append(H.Data(pos=torch.from_numpy(pos).pin_memory(), atomic_number=torch.from_numpy(Z).pin_memory(),
                           cell=torch.from_numpy(cell)[None].pin_memory(), y=torch.randn(1, generator=gen).pin_memory(),
                           forces=(0.1 * torch.randn(pos.shape, generator=gen)).pin_memory()))
    n_atoms_graph = int(host[0].pos.size(0))
    micro = max(1, min(args.micro, len(host)))
    resident = [H.Batch.from_data_list([d.to(dev) for d in host[i:i + micro]]) for i in range(0, len(host), micro)]

    def step_resident():
        return parallel.force_matching_step_microbatched(ddp, resident, opt, micro)

    loss_h = torch.empty(1).pin_memory()

    def step_e2e():
        graphs = [d.to(dev, non_blocking=True) for d in host]
        loss = parallel.force_matching_step_microbatched(ddp, graphs, opt, micro)
        loss_h.copy_(loss.detach().reshape(1), non_blocking=True)
        torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step_resident()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ops.TIMERS = {}
    ops.LAUNCHES["n"] = 0
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0.record()
    for _ in range(args.steps):
        step_resident()
    t1.record()
    barrier()
    launches = ops.LAUNCHES["n"]
    timers, ops.TIMERS = ops.TIMERS, None
    ms = t0.elapsed_time(t1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    clocks = sampler.stop() if rank == 0 else None
    e2e_s = float("nan")
    if args.e2e_steps > 0:
        step_e2e()
        barrier()
        w0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            step_e2e()
        barrier()
        e2e_s = (time.perf_counter() - w0) / args.e2e_steps
        if world > 1:
            t = torch.tensor([e2e_s], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = float(t)
    n_par = sum(p.numel() for p in model.parameters())
    if rank == 0:
        kernels = {}
        for name, evs in timers.items():
            dur = [a.elapsed_time(b) for a, b in evs]
            kernels[name] = {"launches": len(dur), "avg_ms": sum(dur) / len(dur), "share_of_step": sum(dur) / ms}
        atoms = GLOBAL * n_atoms_graph
        peak, peak_src = hbm_peak()
        roof = None
        if "gather_rows" in kernels:     # the hand-written kernels of the composite (double-backward) path are row gathers /
            # segmented sums over [E, 3F] tensors: HBM-bound; algorithmic bytes = rows in + rows out, measured per launch
            roof = {"kernel": "gather_rows", "bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None,
                    "traffic": None, "peak_source": peak_src,
                    "note": "training runs the composite formulation (cuBLAS + torch elementwise + gather_rows / segment_sum); "
                            "per-launch bytes vary with the tensor, see kernels{} for the time shares"}
        bytes_in = sum(int(d[k].nbytes) for d in host for k in ("pos", "atomic_number", "cell", "y", "forces"))
        line = {"metric": "atom-steps/s (training step)", "value": atoms * args.steps / (ms * 1e-3), "unit": "atom-steps/s",
                "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"C2: {kind} L={cfg['num_layers']} F={cfg['hidden_channels']} K={cfg['num_rbf']} rc={cfg['rc']}, global "
                                       f"batch {GLOBAL} x {n_atoms_graph}-atom Li/Si/O cells, force-matching training step (fwd, "
                                       f"create_graph force grad, double backward, gradient all-reduce, Adam), {n_par} parameters"
                                       + ("" if args.scale == 1.0 else f" [scale={args.scale}: NOT the BASELINE size]"),
                           "parallelism": f"dp{world} (DDP, NCCL all-reduce), {len(mine)} graphs per rank in micro-batches of {micro}",
                           "l2_policy": "per-step tensors exceed L2; no flush needed"},
                "e2e": {"value": atoms / e2e_s, "unit": "atom-steps/s", "h2d_bytes_per_step": bytes_in, "d2h_bytes_per_step": 4,
                        "ms_per_step": 1e3 * e2e_s, "includes": "H2D of the local batch, collation, batched neighbour lists + row CSR, "
                                                                  "training step, D2H of the loss"},
                "gpu_launches": launches, "clocks": clocks, "roofline": roof, "kernels": kernels}
        _finish(world, real_stdout, line)
    _finish(world, None, None)


# --------------------------------------------------------------------------------------------------------------
def run_c3(args):
    """``--workload C3`` (BASELINE.json configs[2]): HTNet L=3 F=128 on the synthetic 31 944-atom water box, MD through the
    ASE-style calculator plugin on one B200.  A step = one velocity-Verlet step (neighbour list or Verlet-skin re-use, energy +
    forces, integration).  ``value``: the device-resident loop (``plugin.md.velocity_verlet_device``, positions / velocities /
    forces never leave the GPU); ``e2e``: the host-driven loop through ``NNCalculator.calculate`` (numpy positions in, numpy
    forces out every step -- what ASE's ``VelocityVerlet`` does, plugin/ase_interface/calculator.py:42-57)."""
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    import hermnet_b200 as H
    from hermnet_b200 import ops, synthetic
    from hermnet_b200.plugin import md
    from hermnet_b200.plugin.calculator import NNCalculator
    (pos, Z, cell), cfg = synthetic.config("C3", args.scale)
    kind = cfg.pop("kind")
    torch.manual_seed(1234)
    model = getattr(H, kind)(**cfg).to(dev).eval()
    for p_ in model.parameters():
        p_.requires_grad_(False)
    # random-init weights give forces of hundreds of eV/A: the "MD" would explode within a few steps and every list would be
    # invalid at once.  Scale the last readout layer so that the synthetic trajectory moves like a real one (~0.01 A per
    # step); the work per step does not depend on it.
    model.out_energy[2].weight.mul_(1.0e-3)
    model.out_energy[2].bias.mul_(1.0e-3)
    N = len(Z)
    atoms = md.SimpleAtoms(Z, pos, cell)
    md.maxwell_boltzmann(atoms, 300.0, seed=3)
    v0 = atoms.velocities.copy()
    skin = args.skin
    out = {}
    variants = [("rebuild", 0.0, False), ("skin", skin, False), ("skin_graph", max(skin, args.graph_skin), True)]
    for name, sk, cg in variants:
        st = {}
        try:
            md.velocity_verlet_device(model, Z, pos, cell, v0, steps=max(3, args.warmup), dt_fs=0.5, device=dev, skin=sk, cuda_graph=cg)
            torch.cuda.synchronize()
            ops.LAUNCHES["n"] = 0
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            _, _, e = md.velocity_verlet_device(model, Z, pos, cell, v0, steps=args.steps, dt_fs=0.5, device=dev, skin=sk, stats=st,
                                                cuda_graph=cg)
            b.record()
            torch.cuda.synchronize()
            out[name] = (a.elapsed_time(b) / (args.steps + 1), st, ops.LAUNCHES["n"], float(e[-1]), sk)     # (+1: the initial force call)
        except Exception as exc:  # noqa: BLE001 -- a variant that cannot run is reported, not fatal
            out[name] = (float("inf"), {"error": f"{type(exc).__name__}: {str(exc)[:160]}"}, 0, float("nan"), sk)
    calc = NNCalculator(model, None, trn_mean=0.0, device_="cuda", ensemble="NVT", skin=skin)
    atoms.calc = calc
    md.velocity_verlet(atoms, steps=2, dt_fs=0.5)
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    md.velocity_verlet(atoms, steps=max(1, args.e2e_steps), dt_fs=0.5)
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - w0) / (max(1, args.e2e_steps) + 1)
    best = min(out, key=lambda k: out[k][0])
    ms = out[best][0]
    how = {"rebuild": "rebuilt every step", "skin": f"Verlet skin {out['skin'][4]} A, list re-used while valid",
           "skin_graph": f"Verlet skin {out['skin_graph'][4]} A, list re-used while valid and the whole evaluation replayed as one CUDA "
                         f"graph per step (captured once per list build, capture time included)"}[best]
    line = {"metric": "atom-steps/s (MD step: energy+forces)", "value": N / (ms * 1e-3), "unit": "atom-steps/s", "n_gpus": 1,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"C3: {kind} L={cfg['num_layers']} F={cfg['hidden_channels']} K={cfg['num_rbf']} rc={cfg['rc']} on the {N}-atom "
                                   f"water box, velocity-Verlet MD (0.5 fs, 300 K; random-init weights, last readout layer x 1e-3 so that the trajectory "
                                   f"stays physical) through the calculator plugin; neighbour list: " + how
                                   + ("" if args.scale == 1.0 else f" [scale={args.scale}: NOT the BASELINE size]"),
                       "parallelism": "single GPU", "l2_policy": "per-step tensors exceed L2; no flush needed"},
            "variants": {k: {"ms_per_step": v[0], "skin_A": v[4], "list": v[1], "final_energy": v[3]} for k, v in out.items()},
            "e2e": {"value": N / e2e_s, "unit": "atom-steps/s", "h2d_bytes_per_step": int(N * 3 * 4 + N * 8 + 36),
                    "d2h_bytes_per_step": int(N * 3 * 4 + 4), "ms_per_step": 1e3 * e2e_s,
                    "includes": "numpy positions -> H2D, (re-used) neighbour list, energy + forces, D2H of forces, host integration"},
            "gpu_launches": out[best][2], "roofline": None}
    _finish(1, real_stdout, line)


# --------------------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "C2":
        return run_c2(args)
    if args.workload == "C3":
        return run_c3(args)
    if args.workload == "C5":      # 30 rows per atom: 20 GB tensors; avoid losing tens of GB to allocator fragmentation
        os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line: anything native libraries print (e.g. "NCCL version ...") goes to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import hermnet_b200 as H
    from hermnet_b200 import ops
    pos, Z, cell, cfg = workload(args.workload, args.scale)
    N = len(Z)
    kind = cfg.pop("kind")
    torch.manual_seed(1234)
    model = getattr(H, kind)(**cfg).to(dev).eval()
    for p_ in model.parameters():          # inference: parameters frozen (the ASE plugin does the same)
        p_.requires_grad_(False)
    T, F = len(cfg["elems"]), cfg["hidden_channels"]

    pos_h = torch.from_numpy(pos).pin_memory()
    Z_h = torch.from_numpy(Z).pin_memory()
    cell_h = torch.from_numpy(cell)[None].pin_memory()
    f_h = torch.empty((N, 3), dtype=torch.float32).pin_memory()
    e_h = torch.empty(1, dtype=torch.float32).pin_memory()

    if world > 1:
        from hermnet_b200 import parallel
        engine = parallel.DomainDecomposition(model, dev)
    else:
        engine = None

    # ---- resident setup ------------------------------------------------------------------------------------
    pos_d, Z_d, cell_d = pos_h.to(dev), Z_h.to(dev), cell_h.to(dev)
    if engine is None:
        graph = model.build_graph(pos_d, Z_d, cell_d, None)
        n_edges = graph.n_edges
    else:
        engine.build(pos_d, Z_d, cell_d)
        n_edges = engine.global_edges

    def step_resident(pos_in=None):
        src = pos_d if pos_in is None else pos_in
        if engine is None:
            p = src.detach().requires_grad_(True)
            e, _, _ = model.forward_graph(p, Z_d, cell_d, graph)
            (g,) = torch.autograd.grad(e.sum(), p)
            return e.detach(), g
        return engine.energy_forces(src)

    def step_e2e():
        p = pos_h.to(dev, non_blocking=True)
        z = Z_h.to(dev, non_blocking=True)
        c = cell_h.to(dev, non_blocking=True)
        if engine is None:
            d = H.Data(pos=p.requires_grad_(True), atomic_number=z, cell=c)
            e = model(d)
            (g,) = torch.autograd.grad(e.sum(), d.pos)
        else:
            engine.build(p, z, c)
            e, g = engine.energy_forces(p)
        if rank == 0:
            f_h.copy_(-g, non_blocking=True)
            e_h.copy_(e.detach().reshape(1), non_blocking=True)   # (detach: copy_ from a grad-requiring source would chain every step's autograd graph -- and its row CSR -- onto e_h)
        torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step_resident()
    barrier()

    def timed(step_fn, collect):
        """K steps bracketed by barrier + synchronize, CUDA events, max over ranks; ``collect``: per-kernel events.
        Also returns what the last step returned, ``(energy, dE/dpos)``."""
        if collect:
            ops.TIMERS = {}
        ops.LAUNCHES["n"] = 0
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record()
        for _ in range(args.steps):
            out = step_fn()
        b.record()
        barrier()
        n_launch = ops.LAUNCHES["n"]
        tm, ops.TIMERS = ops.TIMERS, None
        t_ms = a.elapsed_time(b)
        if world > 1:
            t = torch.tensor([t_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            t_ms = float(t)
        return t_ms, n_launch, tm, out

    # eager pass: every launch individually, CUDA events around each kernel (the per-kernel table / roofline come from here)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_eager, launches, timers, last = timed(step_resident, True)
    # graphed pass: the same step (forward_graph + autograd.grad [+ halo exchange and all-reduces]) captured ONCE and replayed
    graphed, graph_note = None, "eager launches"
    if args.cuda_graph:
        try:
            from hermnet_b200.graphed import GraphedForces
            graphed = GraphedForces(step_resident, pos_d)
            for _ in range(3):
                graphed()
            ok = torch.ones(1, device=dev)
        except Exception as exc:  # noqa: BLE001 -- capture is an optimisation: fall back to eager launches, say why
            graphed, graph_note = None, f"eager launches (capture failed: {type(exc).__name__}: {str(exc)[:120]})"
            ok = torch.zeros(1, device=dev)
        if world > 1:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if float(ok) == 0:
            graphed = None
    if graphed is not None:
        ms, _, _, last = timed(graphed, False)
        graph_note = "one captured CUDA graph per step (forward + backward [+ halo exchange, all-reduces]) replayed"
    else:
        ms = ms_eager
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    ms_per_step = ms / args.steps
    value = N * args.steps / (ms * 1e-3)

    # ---- end to end from host buffers ------------------------------------------------------------------------
    e2e_s = float("nan")
    if args.e2e_steps > 0:
        for _ in range(2):      # warm-up: the caching allocator settles on the block sizes of a freshly built graph
            step_e2e()
        barrier()
        w0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            step_e2e()
        barrier()
        e2e_s = (time.perf_counter() - w0) / args.e2e_steps
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t)

    if rank != 0:
        _finish(world, None, None)

    # ---- per-kernel device times (CUDA events recorded around every launch inside the timed region) ------------
    kernels = {}
    for name, evs in timers.items():
        dur = [a.elapsed_time(b) for a, b in evs]
        kernels[name] = {"launches": len(dur), "avg_ms": sum(dur) / len(dur), "share_of_step": sum(dur) / ms_eager}
    peak, peak_src = hbm_peak()
    n_loc = N if engine is None else engine.n_owned_max
    e_loc = n_edges if engine is None else engine.local_edges_max
    roof = None
    edge_k = {k: v for k, v in kernels.items() if k.startswith("painn_edge")}
    if edge_k:
        top = max(edge_k, key=lambda k: edge_k[k]["avg_ms"] * edge_k[k]["launches"])
        ab = alg_bytes(top, n_loc, e_loc, T, F)
        ach = ab / (edge_k[top]["avg_ms"] * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(top)
        roof = {"kernel": top, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic, "peak_source": peak_src, "alg_bytes_per_launch": ab,
                "avg_launch_ms": edge_k[top]["avg_ms"]}
        for k in edge_k:
            kb = alg_bytes(k, n_loc, e_loc, T, F)
            kernels[k]["alg_GBps"] = kb / (edge_k[k]["avg_ms"] * 1e-3) / 1e9
            kernels[k]["frac_of_hbm_peak"] = kernels[k]["alg_GBps"] / peak

    line = {
        "metric": "atom-steps/s (energy+forces)", "value": value, "unit": "atom-steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {kind} L={cfg['num_layers']} F={F} K={cfg['num_rbf']} rc={cfg['rc']} on a "
                               f"{N}-atom {'/'.join(cfg['elems'])} periodic box (E={n_edges} directed edges), energy + forces, "
                               f"parameters frozen" + ("" if args.scale == 1.0 else f" [scale={args.scale}: NOT the BASELINE size]"),
                   "parallelism": "single GPU" if world == 1 else f"spatial domain decomposition over {world} GPUs, per-layer halo exchange",
                   "l2_policy": "inputs exceed L2 (feature tensors are GBs); no flush needed",
                   "launch_mode": graph_note},
        "ms_per_step_eager": ms_eager / args.steps,
        "e2e": {"value": N / e2e_s, "unit": "atom-steps/s", "h2d_bytes_per_step": int(pos_h.nbytes + Z_h.nbytes + cell_h.nbytes),
                "d2h_bytes_per_step": int(f_h.nbytes + e_h.nbytes), "ms_per_step": 1e3 * e2e_s,
                "includes": "H2D, neighbour-list + row-CSR build, forward, backward, D2H of forces and energy"},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof, "kernels": kernels,
    }
    if world == 1 and args.workload == "C4" and not args.no_parity:
        line["parity"] = parity_check(model, pos_d, Z_d, cell_d, graph, kind, cfg)
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(dict(cfg, kind=kind))
    _finish(world, real_stdout, line)


def _finish(world, real_stdout, line):
    """Print the line (rank 0) and end the process.  A single process exits normally, so atexit handlers and library
    teardown run.  Ranks of a multi-GPU run leave WITHOUT tearing down NCCL / symmetric memory / captured graphs:
    destroying a process group whose collectives live in a CUDA graph can block, and the process is done anyway."""
    sys.stdout.flush()
    sys.stderr.flush()
    if line is not None:
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    try:
        torch.cuda.synchronize()
    except Exception:  # noqa: BLE001
        pass
    if world > 1:
        os._exit(0)
    sys.exit(0)


if __name__ == "__main__":
    main()
