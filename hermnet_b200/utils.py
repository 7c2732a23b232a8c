"""``in_subgraph`` / ``virial_calc`` / ``DistributedEvalSampler`` with the reference's call contract
(``/root/reference/HermNet/utils.py``)."""
from __future__ import annotations

import copy
import math
from typing import Any

import torch
import torch.distributed as dist
from torch import Tensor
from torch.utils.data import Sampler

from . import ops

__all__ = ["in_subgraph", "virial_calc", "DistributedEvalSampler", "save_checkpoint", "load_checkpoint"]


def in_subgraph(data, nids: Any):
    """utils.py:11-24: shallow copy of ``data`` restricted to the edges whose DESTINATION is in ``nids``, regrouped
    by destination ascending, original order inside a destination.  One stable device sort
    (``hn_sort_by_key``) replaces the reference's ``len(nids)`` full scans of ``edge_index`` (+ host syncs).
    The models do not call this (the ``RowGraph`` holds all sub-graphs at once); it is kept for API users."""
    rel = copy.copy(data)
    ei = data.edge_index
    n = data.num_nodes if data.num_nodes is not None else int(ei.max().item()) + 1
    nids = torch.as_tensor(nids, device=ei.device).long().reshape(-1)
    member = torch.zeros(n + 1, dtype=torch.bool, device=ei.device)
    member[nids] = True
    key = torch.where(member[ei[1]], ei[1], torch.full_like(ei[1], n)).to(torch.int32).contiguous()
    rowptr, order = ops.sort_by_key(key, n + 1)
    edge_mask = order[: int(rowptr[n].item())].long()
    for k, v in list(rel):
        if k == "edge_index":
            rel.edge_index = ei[:, edge_mask]
        elif isinstance(v, Tensor) and data.is_edge_attr(k):
            rel[k] = v[edge_mask]
    return rel


NKTV2P = {'metal': 1.6021765e6, 'real': 68568.415, 'electron': 2.94210108e13}


def virial_calc(cell, pos, forces, energy, units='metal', pbc=False):
    """utils.py:138-160 (same unit table, same symmetrisation)."""
    if units in NKTV2P:
        nktv2p = NKTV2P[units]
    elif units in ['lj', 'si', 'cgs', 'micro', 'nano']:
        nktv2p = 1.0
    else:
        raise ValueError('Illegal units command')
    if pbc:
        assert cell.requires_grad
        c = cell.reshape(3, 3)
        g_cell = torch.autograd.grad(energy.sum(), cell)[0].reshape(3, 3)
        virial = torch.einsum('ij, ik->jk', pos, forces) - c.T @ g_cell
        virial = (virial + virial.T) / 2 * nktv2p
    else:
        virial = torch.einsum('ij, ik->jk', pos, forces) * nktv2p
        virial = (virial + virial.T) / 2
    return virial


class DistributedEvalSampler(Sampler):
    """Non-padding distributed evaluation sampler (same contract as utils.py:27-135): rank r takes indices
    ``r, r+W, r+2W, ...`` of the (optionally shuffled) dataset, nothing is duplicated to even out ranks."""

    def __init__(self, dataset, num_replicas=None, rank=None, shuffle=False, seed=0):
        if num_replicas is None:
            if not dist.is_available():
                raise RuntimeError("Requires distributed package to be available")
            num_replicas = dist.get_world_size()
        if rank is None:
            if not dist.is_available():
                raise RuntimeError("Requires distributed package to be available")
            rank = dist.get_rank()
        self.dataset, self.num_replicas, self.rank = dataset, num_replicas, rank
        self.epoch, self.shuffle, self.seed = 0, shuffle, seed
        self.total_size = len(self.dataset)
        self.num_samples = len(range(self.rank, self.total_size, self.num_replicas))

    def __iter__(self):
        if self.shuffle:
            gen = torch.Generator()
            gen.manual_seed(self.seed + self.epoch)
            indices = torch.randperm(len(self.dataset), generator=gen).tolist()
        else:
            indices = list(range(len(self.dataset)))
        indices = indices[self.rank:self.total_size:self.num_replicas]
        assert len(indices) == self.num_samples
        return iter(indices)

    def __len__(self):
        return self.num_samples

    def set_epoch(self, epoch):
        self.epoch = epoch


def save_checkpoint(path, model, trn_mean, trn_e_loss=None, trn_f_loss=None, val_e_loss=None, val_f_loss=None):
    """The checkpoint of the reference's hydra trainer (example/hydra-train/train.py:172-180): an ``OrderedDict`` with the
    keys ``model`` (state_dict), ``trn_e_loss``, ``trn_f_loss``, ``val_e_loss``, ``val_f_loss``, ``trn_mean`` -- same keys, same
    order, loadable by the reference's consumers."""
    from collections import OrderedDict
    infos = OrderedDict()
    infos['model'] = model.state_dict()
    infos['trn_e_loss'] = trn_e_loss
    infos['trn_f_loss'] = trn_f_loss
    infos['val_e_loss'] = val_e_loss
    infos['val_f_loss'] = val_f_loss
    infos['trn_mean'] = trn_mean
    torch.save(infos, path)
    return infos


def load_checkpoint(path, map_location=None):
    """``(state_dict, metadata)`` from either checkpoint flavour of the reference: a bare ``state_dict``
    (example/dist_train.py:141, plugin/ase_interface/calculator.py:38) or the trainer's ``infos`` dict (train.py:172-180)."""
    obj = torch.load(path, map_location=map_location)
    if isinstance(obj, dict) and 'model' in obj and isinstance(obj['model'], dict):
        return obj['model'], {k: v for k, v in obj.items() if k != 'model'}
    return obj, {}
