"""CUDA-graph capture of one energy + forces evaluation on a FIXED graph (same atoms, same neighbour list / row CSR / tile
plans; new positions every call).  One evaluation is ~190 kernel launches plus torch glue; once the kernels of a rank take
tens of microseconds (8-GPU domain decomposition, small systems, MD with a Verlet-skin list) the host launch latency shows,
and a captured graph replays the whole forward + backward with one launch.  Everything inside is the ordinary product path
(``forward_graph`` + ``autograd.grad``); collectives of the domain-decomposed path (NCCL all-reduce, the peer-memory halo
kernels and their device barrier) are captured with it.
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import torch

Tensor = torch.Tensor


class GraphedForces:
    """``fn(pos) -> (energy, dE/dpos[, ...])`` captured once; ``__call__(pos)`` copies ``pos`` into the static input and
    replays.  The returned tensors are the graph's static outputs (valid until the next call)."""

    def __init__(self, fn: Callable[[Tensor], Tuple[Tensor, Tensor]], pos: Tensor, warmup: int = 2):
        self.pos = pos.detach().clone()
        cur = torch.cuda.current_stream(pos.device)
        side = torch.cuda.Stream(pos.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):              # warm-up off the default stream: lazy caches, allocator, cuBLAS handles
            for _ in range(max(1, warmup)):
                fn(self.pos)
        cur.wait_stream(side)
        torch.cuda.synchronize(pos.device)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.outputs = tuple(fn(self.pos))
        self.energy, self.grad = self.outputs[:2]

    def __call__(self, pos: Optional[Tensor] = None) -> Tuple[Tensor, ...]:
        if pos is not None and pos.data_ptr() != self.pos.data_ptr():
            self.pos.copy_(pos.detach())
        self.graph.replay()
        return self.outputs


def graphed_forces(model, pos: Tensor, atomic_number: Tensor, cell: Optional[Tensor], graph, warmup: int = 2,
                   virial: bool = False) -> GraphedForces:
    """Captured ``energy, dE/dpos`` of ``model`` on the prebuilt ``graph`` (``model.build_graph``); parameters must be frozen
    (inference) and the graph must stay valid for the positions passed later (same edges, or a Verlet-skin superset list).
    ``virial``: the capture is ``model.energy_forces_virial_graph`` and returns the per-graph virial ``[G,3,3]`` as a third
    output (same single backward pass, plus the per-atom virial kernel and its per-graph sum)."""
    if any(p.requires_grad for p in model.parameters()):
        raise RuntimeError("hermnet_b200.graphed_forces: freeze the parameters first (inference path)")
    # (a Verlet-skin superset list works too: its per-call live mask is computed by device kernels inside the capture)

    def fn(p):
        if virial:
            out = model.energy_forces_virial_graph(p, atomic_number, cell, graph)
            return out["energy"], -out["forces"], out["virial"]
        q = p.detach().requires_grad_(True)
        e, _, _ = model.forward_graph(q, atomic_number, cell, graph)
        (g,) = torch.autograd.grad(e.sum(), q)
        return e.detach(), g
    return GraphedForces(fn, pos, warmup)
