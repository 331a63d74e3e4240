"""Data-parallel training of the hot path over the GPUs of one box (new functionality: the reference is single-device,
SURVEY.md §2a / §8e).

The path shards naturally: reactant groups are independent (every loss is a sum over groups, the encoder is per
molecule), so whole groups are assigned to ranks as contiguous runs balanced by atom count and the only exchange step is
one SUM all-reduce of the flat gradient (3.16 MB at h=300, 12.1 MB at h=600) over NCCL / NVLink.  Exactness w.r.t. the
single-device step is kept by two rules:

* every rank packs its shard with the GLOBAL batch's ``max_num_bonds`` (padding-row multiplicities, SURVEY.md §0 trap 1);
* every rank divides its loss by the GLOBAL normaliser (groups / items / ordered pairs) and gradients are summed.
"""
from __future__ import annotations

import os
from typing import List, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist


def shard_groups(group_atoms: Sequence[int], world: int) -> List[Tuple[int, int]]:
    """Split groups 0..G-1 into ``world`` contiguous runs ``[lo, hi)`` with balanced total atom count; never splits a
    group.  Every rank gets at least one group when G >= world; with fewer groups than ranks some ranks get none."""
    w = np.asarray(group_atoms, dtype=np.float64)
    G = len(w)
    if world <= 1:
        return [(0, G)]
    cum = np.concatenate(([0.0], np.cumsum(w)))
    total = cum[-1]
    bounds = [0]
    for r in range(1, world):
        target = total * r / world
        cut = int(np.searchsorted(cum, target, side="left"))
        if cut > 0 and abs(cum[cut - 1] - target) <= abs(cum[min(cut, G)] - target):
            cut -= 1
        cut = max(cut, bounds[-1] + (1 if G - bounds[-1] > world - r else 0))   # leave groups for the remaining ranks
        cut = min(cut, G - (world - r)) if G >= world else min(cut, G)
        cut = max(cut, bounds[-1])
        bounds.append(cut)
    bounds.append(G)
    return [(bounds[r], bounds[r + 1]) for r in range(world)]


def shard_rows(scope: Sequence[int], lo: int, hi: int) -> Tuple[int, int]:
    """Row range of groups ``[lo, hi)`` inside a batch whose group sizes are ``scope``."""
    off = np.concatenate(([0], np.cumsum(np.asarray(scope, dtype=np.int64))))
    return int(off[lo]), int(off[hi])


def flat_layout(tensors) -> Tuple[List[int], int]:
    """(element offset of each tensor, total elements) of the flat gradient buffer: the tensors in the given order, each starting on a
    16-byte boundary.  ``ReactionModel``'s backward lays its buffer out over the trainable tensors with this, and ``GradSync`` its
    staging bucket, so that the in-place and the staged all-reduce have the same element count."""
    offsets, total = [], 0
    for t in tensors:
        offsets.append(total)
        total += (t.numel() + 3) // 4 * 4
    return offsets, total


class GradSync:
    """SUM all-reduce of all gradients as ONE collective per step.

    Fast path: ``ReactionModel`` writes the gradients of a backward pass into one flat buffer and gives autograd views of it, so
    ``p.grad`` aliases ``model._grad_flat``; the buffer is all-reduced in place (3.16 MB at h = 300, 12.1 MB at h = 600) and nothing
    is copied.  Whenever that aliasing does not hold (gradients accumulated over several backward passes into older tensors, a
    hook that replaced ``p.grad``, parameters outside the model) the gradients go through a flat staging bucket instead.

    Only the tensors of ``params`` that have ``requires_grad`` take part, decided at every call: frozen tensors are neither exchanged nor
    given a gradient, and the collective carries the trainable bytes only.  Freezing or unfreezing tensors after this object was built
    is therefore exact; the first step after such a change may take the staging path."""

    def __init__(self, params, group=None, model=None):
        self.candidates = list(params)
        self.group = group
        self.model = model
        self.flat = None
        self.fast_path_steps = 0
        self.copy_path_steps = 0
        self.params = None
        self._refresh()

    def _refresh(self):
        # ONE layout for both paths (flat_layout, as ReactionModel's backward lays its flat buffer out): a rank whose shard is empty has no
        # backward pass and goes through the staging bucket while its peers all-reduce their aliased buffers in place -- the collective
        # must have the same element count on every rank
        params = [p for p in self.candidates if p.requires_grad]
        if self.params is not None and len(params) == len(self.params) and all(a is b for a, b in zip(params, self.params)):
            return
        self.params = params
        self.offsets, self.numel = flat_layout(params)
        self.flat = None

    def _aliased(self):
        m = self.model
        flat = getattr(m, "_grad_flat", None) if m is not None else None
        if flat is None or flat.numel() != self.numel:
            return None
        hot = m.hot_parameters()
        if len(hot) != len(self.params) or any(a is not b for a, b in zip(hot, self.params)) or list(m._grad_offsets) != self.offsets:
            return None
        base = flat.data_ptr()
        for p, off in zip(hot, self.offsets):
            g = p.grad
            if g is None or not g.is_contiguous() or g.data_ptr() != base + 4 * off:
                return None
        return flat

    def __call__(self):
        if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(self.group) == 1:
            return
        self._refresh()
        flat = self._aliased()
        if flat is not None:
            dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group)
            self.fast_path_steps += 1
            return
        self.copy_path_steps += 1
        for p in self.params:
            if p.grad is None:                     # a rank whose shard is empty still takes part in the collective
                p.grad = torch.zeros_like(p)
        grads = [p.grad for p in self.params]
        if not grads:
            return
        if self.flat is None or self.flat.device != grads[0].device:
            self.flat = torch.zeros(self.numel, dtype=grads[0].dtype, device=grads[0].device)      # the alignment gaps stay zero
        views = [self.flat[o:o + g.numel()].view_as(g) for o, g in zip(self.offsets, grads)]
        torch._foreach_copy_(views, grads)
        dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=self.group)
        torch._foreach_copy_(grads, views)         # copies INTO p.grad whatever its strides are (the gaps hold sums of zeros: still zero)


# ---- process-group plumbing for the entry points (train(), run_train(), main.py, main_ranknet.py, bench.py) ------------------------
def world_from_env() -> Tuple[int, int, int]:
    """(rank, world size, local rank) as torchrun exports them; (0, 1, 0) in a plain ``python main.py`` run."""
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def init_from_env(device=None, backend: str = None) -> Tuple[int, int]:
    """Join the process group torchrun describes (no-op for world size 1 or when a group already exists).  ``device``: this rank's CUDA
    device (NCCL) or None (gloo: the CPU tests).  Returns (rank, world)."""
    rank, world, _ = world_from_env()
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if backend is None:
            backend = "nccl" if device is not None and torch.cuda.is_available() else "gloo"
        kw = {"device_id": torch.device(device)} if backend == "nccl" and device is not None else {}
        dist.init_process_group(backend, rank=rank, world_size=world, **kw)
    if dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def current() -> Tuple[int, int]:
    """(rank, world) of the initialised default group, (0, 1) otherwise."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def plan_shard(scope: Sequence[int], atoms_per_row: Sequence[int], rank: int, world: int) -> Tuple[int, int, int, int]:
    """This rank's part of a global batch: ``(group_lo, group_hi, row_lo, row_hi)``.  ``scope`` = the batch's group sizes in rows,
    ``atoms_per_row`` = atoms of every candidate row (balances the shards by work, SURVEY.md 8e)."""
    scope = np.asarray(scope, dtype=np.int64)
    off = np.concatenate(([0], np.cumsum(scope)))
    atoms = np.asarray(atoms_per_row, dtype=np.float64)
    csum = np.concatenate(([0.0], np.cumsum(atoms)))
    group_atoms = csum[off[1:]] - csum[off[:-1]]
    lo, hi = shard_groups(group_atoms, world)[rank]
    return lo, hi, int(off[lo]), int(off[hi])


def broadcast_parameters(model, src: int = 0, group=None):
    """Make every rank start from rank ``src``'s weights (and frozen buffers)."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    for t in list(model.parameters()) + list(model.buffers()):
        dist.broadcast(t.data, src=src, group=group)
