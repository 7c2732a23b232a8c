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

