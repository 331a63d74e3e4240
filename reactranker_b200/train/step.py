"""One optimiser step of the listwise / pointwise training loop (train/train_listwise.py:177-290), single-GPU or data-parallel.

``train()`` and ``bench.py`` both drive this object, so the step that is benchmarked (and whose 1 -> 8 GPU scaling the driver measures)
is the step the product trains with:

    step = TrainStep(model, optimizer, scheduler, task_type, gpu)          # joins torchrun's process group when WORLD_SIZE > 1
    for batch in data_processor.generate_batch_reactions(...):            # the GLOBAL batch plan, identical on every rank
        prepared = step.prepare(batch, smiles2graph_dic)                  # host: this rank's shard -> device graphs, targets, normalisers
        loss = step.run(prepared, epoch, epochs)                          # forward, loss, backward, gradient all-reduce, Adam, NoamLR

Data parallelism (SURVEY.md 8e; the reference is single-device): reactant groups are independent, so the global batch is cut into
contiguous runs of whole groups balanced by atom count (parallel.plan_shard).  Two rules keep the sharded step equal to the
single-device step: every shard is packed with the GLOBAL batch's ``max_num_bonds`` (the padding-row multiplicities of
featurization.py:281-286 depend on it), and every loss term divides by the GLOBAL number of groups / items (loss.dp_normalisers) while
the gradients are SUM-all-reduced -- one collective per step on the flat gradient buffer the backward pass wrote (parallel.GradSync).
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from .. import _lib, parallel
from ..models.base_model import reactant_dedup_exact
from .loss import dp_normalisers


class PreparedBatch:
    """What ``TrainStep.run`` consumes: this rank's rows of one global batch, already on their way to the device."""
    __slots__ = ("r", "p", "targets", "scope", "feats", "groups", "items", "rows", "h2d_bytes")

    def __init__(self, r, p, targets, scope, feats, groups, items, rows, h2d_bytes=0):
        self.r, self.p, self.targets, self.scope, self.feats = r, p, targets, scope, feats
        self.groups, self.items, self.rows, self.h2d_bytes = groups, items, rows, h2d_bytes


def _atoms_per_row(batch_graph) -> np.ndarray:
    sizes = getattr(batch_graph, "_a_size", None)
    if sizes is None:                                                 # a duck-typed featuriser's BatchMolGraph (reference interface)
        sizes = [n for _, n in batch_graph.a_scope]
    return np.asarray(sizes, dtype=np.int64)


class TrainStep:
    def __init__(self, model, optimizer, scheduler, task_type: str, gpu, max_coeff: float = 0.0001, group=None, batch_loss=None):
        self.dev_idx = _lib.require_device(gpu)
        self.dev = torch.device("cuda", self.dev_idx)
        self.model, self.optimizer, self.scheduler = model, optimizer, scheduler
        self.task_type, self.max_coeff, self.group = task_type, max_coeff, group
        self.rank, self.world = parallel.init_from_env(device=self.dev)
        if batch_loss is None:
            from .train_listwise import batch_loss
        self.batch_loss = batch_loss
        self.sync = None
        if self.world > 1:
            parallel.broadcast_parameters(model, 0, group)             # every rank starts from rank 0's weights
            self.sync = parallel.GradSync(model.parameters(), group, model)     # the trainable ones, decided at every step

    # ---- host side ---------------------------------------------------------------------------
    def prepare(self, batch, smiles2graph_dic, pinned: bool = True, device_graphs: bool = False) -> PreparedBatch:
        """``batch`` = one item of ``DataProcessor.generate_batch_reactions``: (reactions [N,2], targets [N,1], scope, add_features).
        ``device_graphs``: build the two DeviceGraphs now (ids / row offsets go up asynchronously, the batch is assembled on the device
        behind whatever is running) instead of inside the next ``model(...)`` call -- what a loop that reads a result every step wants."""
        from ..features.featurization import BatchMolGraph, DeviceGraph
        reactions, targets, scope, add_features = batch
        scope = [int(s) for s in scope]
        G, N = len(scope), int(sum(scope))
        r0, r1, g_lo, g_hi = 0, N, 0, G
        w_r = w_p = None
        if self.world > 1:
            r_glob, p_glob = smiles2graph_dic.parsing_reactions(reactions)      # sizes only: nothing is built or uploaded for the global batch
            g_lo, g_hi, r0, r1 = parallel.plan_shard(scope, _atoms_per_row(p_glob), self.rank, self.world)
            w_r, w_p = r_glob.max_num_bonds, p_glob.max_num_bonds
        targets_t = torch.FloatTensor(np.asarray(targets)[r0:r1]).squeeze()      # train_listwise.py:187
        feats = None if add_features is None else np.asarray(add_features)[r0:r1]
        if r1 == r0:                                                            # fewer groups than ranks: this rank only joins the all-reduce
            return PreparedBatch(None, None, targets_t, [], feats, G, N, 0)
        r_inputs, p_inputs = smiles2graph_dic.parsing_reactions(reactions[r0:r1] if self.world > 1 else reactions)
        if self.world > 1:
            # the shard is packed with the GLOBAL batch's max_num_bonds: the multiplicity of the padding rows (featurization.py:281-286)
            # is what makes a shard's rows equal the same rows of the whole batch
            r_inputs.max_num_bonds, p_inputs.max_num_bonds = w_r, w_p
        h2d = 0
        if device_graphs or self.world > 1:
            model = self.model
            store_backed = isinstance(r_inputs, BatchMolGraph) and r_inputs._ids is not None and p_inputs._ids is not None
            if store_backed and reactant_dedup_exact(model):
                r_inputs, p_inputs = DeviceGraph.from_batches_dedup([r_inputs], [p_inputs], self.dev)     # exact without dropout only
            else:
                r_inputs, p_inputs = DeviceGraph.pair_from_batches([r_inputs], [p_inputs], self.dev)
            h2d = r_inputs.h2d_bytes + p_inputs.h2d_bytes
        if pinned:                                                              # targets / extra features ride up asynchronously with the graphs
            targets_t = targets_t.pin_memory().to(self.dev, non_blocking=True)
            h2d += targets_t.numel() * 4
            if feats is not None:
                f = torch.as_tensor(np.asarray(feats, dtype=np.float32)).reshape(r1 - r0, -1)
                feats = f.pin_memory().to(self.dev, non_blocking=True)
                h2d += feats.numel() * 4
        return PreparedBatch(r_inputs, p_inputs, targets_t, scope[g_lo:g_hi], feats, G, N, r1 - r0, h2d)

    def prepare_rows(self, proc, rows, scope, smiles2graph_dic, smiles_list=None, target_name='std_targ', add_features_name=None, df=None,
                     pinned: bool = True) -> PreparedBatch:
        """The same as ``prepare`` for one item of ``DataProcessor.plan_batch_reactions`` -- row positions and scope instead of the gathered
        SMILES / target arrays.  With the package's ``Parsing_features`` the molecules of the rows are two integer fancy-indexes of the
        per-frame store-id vectors (``frame_ids``), the shard's control blocks are one C++ pass each (``rr_batch_build``) into pinned
        memory, and nothing is gathered for rows of other ranks: a rank's host work per step stays ~0.5 ms however large the GLOBAL
        batch is.  Any other featuriser (the reference's interface: ``parsing_reactions`` on SMILES) goes through ``prepare``."""
        from ..features.featurization import DeviceGraph
        df = proc.df if df is None else df
        rows = np.asarray(rows)
        scope = [int(s) for s in scope]
        cols = ['rsmi', 'psmi'] if smiles_list is None else list(smiles_list)
        fast = hasattr(smiles2graph_dic, "frame_ids")
        if fast:
            r_all, p_all = smiles2graph_dic.frame_ids(df, cols[0])[rows], smiles2graph_dic.frame_ids(df, cols[1])[rows]
            fast = rows.shape[0] == 0 or (int(r_all.min()) >= 0 and int(p_all.min()) >= 0)
        if not fast:
            smiles, targets, feats = proc._gather(df, rows, smiles_list, target_name, add_features_name)
            return self.prepare((smiles, targets.reshape(-1, 1), scope, feats), smiles2graph_dic, pinned, device_graphs=True)
        store = smiles2graph_dic.store
        G, N = len(scope), int(sum(scope))
        r0, r1, g_lo, g_hi = 0, N, 0, G
        w_r = w_p = None
        if self.world > 1:
            g_lo, g_hi, r0, r1 = parallel.plan_shard(scope, store.nA[p_all], self.rank, self.world)
            w_r = [max(1, int(store.maxdeg[r_all].max()))]           # the GLOBAL batch's max_num_bonds (featurization.py:281)
            w_p = [max(1, int(store.maxdeg[p_all].max()))]
        mine = rows[r0:r1]
        proc._index(df)
        targets_t = torch.FloatTensor(proc._col(df, target_name)[mine].reshape(-1, 1)).squeeze()      # train_listwise.py:187
        feats = None
        if add_features_name is not None:
            names = list(add_features_name) if isinstance(add_features_name, (list, tuple)) else [add_features_name]
            feats = np.stack([proc._col(df, c)[mine] for c in names], axis=1)
        if r1 == r0:
            return PreparedBatch(None, None, targets_t, [], feats, G, N, 0)
        model = self.model
        dedup = reactant_dedup_exact(model)
        rg, pg = DeviceGraph.from_id_groups(store, r_all[r0:r1], p_all[r0:r1], [r1 - r0], self.dev, dedup, w_r, w_p)
        h2d = rg.h2d_bytes + pg.h2d_bytes
        if pinned:
            targets_t = targets_t.pin_memory().to(self.dev, non_blocking=True)
            h2d += targets_t.numel() * 4
            if feats is not None:
                f = torch.as_tensor(np.asarray(feats, dtype=np.float32)).reshape(r1 - r0, -1)
                feats = f.pin_memory().to(self.dev, non_blocking=True)
                h2d += feats.numel() * 4
        return PreparedBatch(rg, pg, targets_t, scope[g_lo:g_hi], feats, G, N, r1 - r0, h2d)

    # ---- device side -------------------------------------------------------------------------
    def run(self, b: PreparedBatch, epoch: int = 0, epochs: int = 1) -> torch.Tensor:
        """forward -> loss -> zero_grad -> backward -> (all-reduce) -> optimizer.step -> scheduler.step (train_listwise.py:189-290).
        Returns this rank's loss term (already divided by the global normaliser: the terms of all ranks sum to the batch loss)."""
        model, opt = self.model, self.optimizer
        if b.rows == 0:
            opt.zero_grad(set_to_none=True)
            loss = torch.zeros(1, device=self.dev)
        else:
            output = model(b.r, b.p, gpu=self.dev_idx, add_features=b.feats)
            if self.world > 1:
                with dp_normalisers(groups=b.groups, items=b.items):
                    loss = self.batch_loss(self.task_type, output, b.scope, b.targets, self.dev_idx, self.max_coeff, epoch, epochs)
            else:
                loss = self.batch_loss(self.task_type, output, b.scope, b.targets, self.dev_idx, self.max_coeff, epoch, epochs)
            opt.zero_grad(set_to_none=True)
            loss.backward()
        if self.sync is not None:
            self.sync()
        opt.step()
        self.scheduler.step()
        return loss

    def global_loss(self, loss: torch.Tensor) -> float:
        """The batch loss as one number on every rank (a 4-byte all-reduce; used once per epoch for logging)."""
        v = loss.detach().reshape(-1)[:1].float().to(self.dev).clone()
        if self.world > 1:
            torch.distributed.all_reduce(v, op=torch.distributed.ReduceOp.SUM, group=self.group)
        return float(v)

    def is_main(self) -> bool:
        return self.rank == 0

    def broadcast_floats(self, values, src: int = 0):
        """Rank ``src``'s list of floats on every rank (validation metrics: only rank 0 evaluates)."""
        if self.world == 1:
            return [float(v) for v in values]
        t = torch.tensor([float(v) for v in values], dtype=torch.float64, device=self.dev)
        torch.distributed.broadcast(t, src=src, group=self.group)
        return t.tolist()

    def barrier(self):
        if self.world > 1:
            torch.distributed.barrier(group=self.group)
