"""RankNet training loop ``factorized_training_loop``, 'sum_session' and 'accelerate_grad' (train/train_pairwise.py:81-173).

The reference evaluates one reactant group per forward, keeps every group's autograd graph alive until the accumulated
candidate count reaches ``batch_size``, then divides the summed pairwise cost by the window's ordered-pair count and
steps.  Here a whole accumulation window is ONE forward / loss / backward: the groups are packed as separate segments
of one DeviceGraph (each keeps its own padding rows and ``max_num_bonds``, exactly as if it had been batched alone) and
the all-pairs cost of every group is evaluated by one segmented kernel.  Window boundaries, the skip of groups without
a positive pair, the normalisation by the pair count and the tail flush WITHOUT ``scheduler.step()`` follow the reference.
"""
from __future__ import annotations

import numpy as np
import torch

from .. import _lib, parallel
from ..features.featurization import DeviceGraph
from .loss import count_ordered_pairs, ranknet_window_loss


def _window_graphs(window, smiles2graph_dic, dev):
    """Reactant and product DeviceGraphs of a window, one segment per group.  With the package's Parsing_features the whole window goes
    to the device as two id vectors; any other featuriser (the reference's interface: parsing_smiles only) gets one BatchMolGraph per group."""
    if hasattr(smiles2graph_dic, "parsing_ids"):
        r_ids = smiles2graph_dic.parsing_ids([s for w in window for s in w[0]])
        p_ids = smiles2graph_dic.parsing_ids([s for w in window for s in w[1]])
        if r_ids is not None and p_ids is not None:
            return DeviceGraph.from_id_groups(smiles2graph_dic.store, r_ids, p_ids, [len(w[0]) for w in window], dev, dedup=False)
    return (DeviceGraph.from_batches([smiles2graph_dic.parsing_smiles(w[0]) for w in window], dev),
            DeviceGraph.from_batches([smiles2graph_dic.parsing_smiles(w[1]) for w in window], dev))


def _dp_shard(model, window, smiles2graph_dic):
    """Data-parallel (torchrun): this rank's contiguous run of the window's groups, balanced by atom count (parallel.shard_groups).  A
    group is its own segment with its own ``max_num_bonds`` already, and ``pairs`` is the whole window's count, so the ranks' loss terms
    sum to the window loss and the SUM all-reduce of the gradients reproduces the single-device step."""
    rank, world = parallel.current()
    if world == 1:
        return window, None
    sync = getattr(model, "_dp_sync", None)
    if sync is None:
        sync = model._dp_sync = parallel.GradSync(model.parameters(), None, model)
    atoms = [smiles2graph_dic.parsing_smiles(w[1]).n_atoms - 1 for w in window]
    lo, hi = parallel.shard_groups(atoms, world)[rank]
    return window[lo:hi], sync


def prepare_window(model, window, smiles2graph_dic, gpu):
    """Host side of one accumulation window: (data-parallel) this rank's groups, their DeviceGraphs (one segment per group; the id
    vectors go up asynchronously), targets, extra features and scope.  Returns ``(prepared | None, sync)``; None = this rank has no group."""
    dev = torch.device("cuda", gpu)
    window, sync = _dp_shard(model, window, smiles2graph_dic)
    if not window:
        return None, sync
    rg, pg = _window_graphs(window, smiles2graph_dic, dev)
    targets = np.concatenate([w[2] for w in window]).astype(np.float32)
    feats = None
    if window[0][3] is not None:
        feats = np.concatenate([np.asarray(w[3], dtype=np.float64).reshape(len(w[2]), -1) for w in window], axis=0)
    return (rg, pg, targets, feats, [len(w[2]) for w in window]), sync


def run_window(model, prepared, sync, pairs, optimizer, gpu, sigma=1.0, training_algo='sum_session'):
    """Device side: forward, window loss / ``pairs``, backward, (all-reduce,) optimizer.step, zero_grad (train_pairwise.py:146-158)."""
    if prepared is None:                                # more ranks than groups in this window: join the all-reduce with zero gradients
        sync()
        optimizer.step()
        model.zero_grad()
        return torch.zeros((), device=torch.device("cuda", gpu))
    rg, pg, targets, feats, scope = prepared
    y = model(rg, pg, gpu=gpu, add_features=feats)
    loss = ranknet_window_loss(y, scope, targets, pairs, sigma=sigma, gpu=gpu, training_algo=training_algo)
    loss.backward()
    if sync is not None:
        sync()
    optimizer.step()
    model.zero_grad()
    return loss


def _run_window(model, window, pairs, optimizer, gpu, sigma, training_algo='sum_session', smiles2graph_dic=None):
    prepared, sync = prepare_window(model, window, smiles2graph_dic, gpu)
    return run_window(model, prepared, sync, pairs, optimizer, gpu, sigma, training_algo)


def iter_windows(train_data_processor, epoch, batch_size, smiles_list=None, target_name: str = 'ea', add_features_name=None):
    """The accumulation windows of one epoch, as train_pairwise.py:81-171 forms them: groups in ``generate_batch_per_query`` order, groups
    without a positive pair skipped (103-104), a window closes once its candidate count reaches ``batch_size`` (146); the remainder is
    the tail.  Yields ``(window, ordered pairs of the window, is_tail)`` with window = [(reactant tokens, product tokens, targets, feats)]."""
    window, pairs, count = [], 0.0, 0
    for X, Y, add_features in train_data_processor.generate_batch_per_query(smiles_list=smiles_list, target_name=target_name, seed=epoch,
                                                                           add_features_name=add_features_name):
        if X is None or X.shape[0] == 0:
            continue
        Y = np.asarray(Y, dtype=np.float64).reshape(-1)
        n_pairs = count_ordered_pairs(Y)
        if n_pairs == 0:
            continue
        window.append(([s[0] for s in X], [s[1] for s in X], Y, add_features))
        pairs += n_pairs
        count += len(Y)
        if count >= batch_size:
            yield window, pairs, False
            window, pairs, count = [], 0.0, 0
    if pairs:
        yield window, pairs, True


def factorized_training_loop(epoch, model, loss_func, optimizer, scheduler, smiles2graph_dic, train_data_processor, batch_size=2, sigma=1.0,
                             training_algo='sum_session', gpu=None, smiles_list=None, target_name: str = 'ea', add_features_name=None):
    if training_algo not in ('sum_session', 'accelerate_grad'):
        raise ValueError("training algo {} not implemented".format(training_algo))
    gpu = _lib.require_device(gpu)
    minibatch_loss = []
    for window, pairs, tail in iter_windows(train_data_processor, epoch, batch_size, smiles_list, target_name, add_features_name):
        if tail:                                        # tail flush, no scheduler.step() (train_pairwise.py:162-171)
            print('+' * 10, "End of batch, remaining pairs {}".format(pairs))
        minibatch_loss.append(_run_window(model, window, pairs, optimizer, gpu, sigma, training_algo, smiles2graph_dic))
        if not tail:
            scheduler.step()
    if not minibatch_loss:
        return float('nan')
    total = torch.stack([l.detach().reshape(()).float() for l in minibatch_loss])
    if parallel.current()[1] > 1:                       # the ranks' terms of every window sum to the window loss
        torch.distributed.all_reduce(total, op=torch.distributed.ReduceOp.SUM)
    return float(total.double().mean())


def _unbuilt(name):
    def f(*a, **k):
        raise NotImplementedError(f"{name} is not reachable from main_ranknet.py's defaults (SURVEY.md §2 row 9)")
    f.__name__ = name
    return f


baseline_pairwise_training_loop = _unbuilt("baseline_pairwise_training_loop")
beta_dis_train_loop = _unbuilt("beta_dis_train_loop")
beta_evi_train_loop = _unbuilt("beta_evi_train_loop")
