"""Validation / test metrics with the reference's names and return values (train/eval.py:76-177, 475-555).

The reference runs ONE model forward per reactant group.  Here up to ``groups_per_launch`` groups share a
launch: every group is its own segment of the DeviceGraph, so it keeps its own padding rows and its own
``max_num_bonds`` and the scores equal the one-forward-per-group scores of the reference.
"""
from __future__ import annotations

import numpy as np
import torch

from .. import _lib
from ..features.featurization import DeviceGraph
from ..models.base_model import reactant_dedup_exact
from .loss import segment_offsets

GROUPS_PER_LAUNCH = 256


def _launch_graphs(chunks, smiles2graph_dic, dev, dedup):
    """chunks: list of (smiles [n,2], add_features | None); every chunk becomes ONE segment of the DeviceGraph (its own padding rows and
    ``max_num_bonds``, exactly as if it had been the reference's whole BatchMolGraph).  Yields ``(lo, hi, rg, pg, feats)`` per launch of up
    to GROUPS_PER_LAUNCH chunks: the two device graphs of chunks[lo:hi], rows in chunk order, and their extra features (host, or None)."""
    fast = hasattr(smiles2graph_dic, "parsing_ids")
    for lo in range(0, len(chunks), GROUPS_PER_LAUNCH):
        part = chunks[lo:lo + GROUPS_PER_LAUNCH]
        feats = None
        if part[0][1] is not None:
            feats = np.concatenate([np.asarray(f, dtype=np.float64).reshape(len(X), -1) for X, f in part], axis=0)
        rg = pg = None
        if fast:                       # store ids of the whole launch at once: no BatchMolGraph per group
            r_ids = smiles2graph_dic.parsing_ids([s[0] for X, _ in part for s in X])
            p_ids = smiles2graph_dic.parsing_ids([s[1] for X, _ in part for s in X])
            if r_ids is not None and p_ids is not None:
                rg, pg = DeviceGraph.from_id_groups(smiles2graph_dic.store, r_ids, p_ids, [len(X) for X, _ in part], dev, dedup)
        if rg is None:
            r_b = [smiles2graph_dic.parsing_smiles([s[0] for s in X]) for X, _ in part]
            p_b = [smiles2graph_dic.parsing_smiles([s[1] for s in X]) for X, _ in part]
            if dedup:
                rg, pg = DeviceGraph.from_batches_dedup(r_b, p_b, dev)       # a group's candidates share one reactant graph
            else:
                rg, pg = DeviceGraph.from_batches(r_b, dev), DeviceGraph.from_batches(p_b, dev)
        yield lo, lo + len(part), rg, pg, feats


def _forward_chunks(model, gpu, chunks, smiles2graph_dic):
    """Yields ``(lo, hi, preds)`` with the scores of chunks[lo:hi] on the device, rows in chunk order: one forward per launch of
    ``_launch_graphs``."""
    dev = torch.device("cuda", gpu) if isinstance(gpu, int) else torch.device(gpu)
    for lo, hi, rg, pg, feats in _launch_graphs(chunks, smiles2graph_dic, dev, reactant_dedup_exact(model)):
        yield lo, hi, model(rg, pg, gpu=gpu, add_features=feats)


def compute_NDCG(truth, pred):
    """eval.py:460-472 (exponential gain, log2 discount) for two already-ordered host lists; kept for API parity, the validation
    pass itself uses ``group_metrics``."""
    truth, pred = np.asarray(truth, dtype=np.float64), np.asarray(pred, dtype=np.float64)
    disc = np.log2(np.arange(2, len(truth) + 2))
    return float(np.sum(np.exp(pred) / disc) / np.sum(np.exp(truth) / disc))


def group_metrics(preds: torch.Tensor, scope, targets, ratio: float = 0.25) -> torch.Tensor:
    """Per-group ranking metrics ON THE DEVICE (``rr_rank_metrics``): ``preds`` [N] or [N, k] (column 0 ranks), ``scope`` the group sizes,
    ``targets`` the fp64 target column.  Returns a device tensor [G, 8]; columns as in include/rr_sm100.h.  Replaces the per-group host
    sorts of eval.py:497-553 / 112-165; nothing but 8 doubles per group ever crosses PCIe."""
    if not preds.is_cuda:
        raise _lib.RRError("group_metrics: scores must be on the GPU (no CPU fallback)")
    sc = preds.detach()
    if sc.dtype != torch.float32:
        sc = sc.float()
    if sc.dim() > 2 or (sc.dim() == 2 and sc.stride(1) != 1) or (sc.dim() == 1 and sc.stride(0) != 1):
        sc = sc.contiguous()
    ld = sc.stride(0) if sc.dim() == 2 else 1
    scope = [int(n) for n in scope]
    N, G = sum(scope), len(scope)
    if N != sc.shape[0]:
        raise _lib.RRError(f"sum(scope)={N} does not match the {sc.shape[0]} scores")
    t = np.ascontiguousarray(np.asarray(targets, dtype=np.float64).reshape(-1))
    if t.shape[0] != N:
        raise _lib.RRError(f"{t.shape[0]} targets for {N} scores")
    t_d = torch.from_numpy(t).pin_memory().to(sc.device, non_blocking=True)
    seg = segment_offsets(scope, sc.device)
    out = torch.empty(G, 8, dtype=torch.float64, device=sc.device)
    with torch.cuda.device(sc.device):
        _lib.check(_lib.lib().rr_rank_metrics(N, G, sc.data_ptr(), ld, t_d.data_ptr(), seg.data_ptr(), max(scope), float(ratio), out.data_ptr(),
                                              _lib.stream_ptr()))
    return out


def ranking_metrics(model, gpu, data_processor, smiles2graph_dic, show_info=True, smiles_list=None, target_name: str = 'ea',
                    logger=None, add_features_name=None):
    """top-1 hit, recall@25 %, top-25 % hit, [NDCG@1, NDCG@2, NDCG@25 %, NDCG@all] (eval.py:475-555).  As in the
    reference the groups come from ``generate_batch_per_query`` (so the extra feature is the target column, load_reactions.py:264).
    Up to GROUPS_PER_LAUNCH groups share a forward, the per-group metrics are computed on the device, and the host waits once."""
    was_training = model.training
    model.eval()
    groups, targets = [], []
    for X, t, feats in data_processor.generate_batch_per_query(smiles_list=smiles_list, target_name=target_name, shuffle_query=False,
                                                                shuffle_batch=False, add_features_name=add_features_name):
        groups.append((X, feats))
        targets.append(np.asarray(t, dtype=np.float64).reshape(-1))
    parts = []
    with torch.no_grad():
        for lo, hi, preds in _forward_chunks(model, gpu, groups, smiles2graph_dic):
            parts.append(group_metrics(preds, [len(t) for t in targets[lo:hi]], np.concatenate(targets[lo:hi]), 0.25))
    model.train(was_training)
    if not parts:
        return 0.0, float('nan'), 0.0, np.full(4, np.nan)
    m = torch.cat(parts).cpu().numpy()
    return float(m[:, 0].mean()), float(m[:, 1].mean()), float(m[:, 2].mean()), m[:, 4:8].mean(axis=0)


def evaluate_top_scores(model, gpu, data_processor, smiles2graph_dic, ratio=0.25, batch_size=2, show_info=False, smiles_list=None,
                        target_name: str = 'ea', add_features_name=None):
    """top-1 accuracy, mean overlap of predicted/true top-``ratio`` sets, true top-1 inside predicted top-``ratio``
    (eval.py:76-177).  Groups come from ``generate_batch_querys`` (real ``add_features_name`` column); in the reference
    ``batch_size`` groups share one BatchMolGraph and therefore one ``max_num_bonds`` -- reproduced by packing each
    ``batch_size`` chunk as one segment; many chunks share a launch and the metrics are computed on the device."""
    chunks, scopes, targets = [], [], []
    for X, t, scope, feats in data_processor.generate_batch_querys(smiles_list=smiles_list, target_name=target_name, batch_size=batch_size,
                                                                   shuffle_query=False, shuffle_batch=False, add_features_name=add_features_name):
        chunks.append((X, feats))
        scopes.append([int(n) for n in scope])
        targets.append(np.asarray(t, dtype=np.float64).reshape(-1))
    parts = []
    with torch.no_grad():
        for lo, hi, preds in _forward_chunks(model, gpu, chunks, smiles2graph_dic):
            parts.append(group_metrics(preds, [n for sc in scopes[lo:hi] for n in sc], np.concatenate(targets[lo:hi]), ratio))
    m = torch.cat(parts).cpu().numpy()
    return float(m[:, 0].mean()), float(m[:, 1].mean()), float(m[:, 3].mean())


def calculate_ndcg(model, gpu, data_processor, smiles2graph_dic, batch_size=2, NDCG_cut=0.5, show_info=False, smiles_list=None,
                   target_name: str = 'ea', logger=None, is_order=True, means=None, stds=None, add_features_name=None):
    """Rank-based NDCG@cut, KL(softmax(targets) || softmax(scores)), the per-item order table and the re-ordered SMILES of the
    test report (eval.py:329-457).  ``batch_size`` groups share one forward (one BatchMolGraph, one ``max_num_bonds``) as in the
    reference; everything after the forward is the reference's host arithmetic in fp32:
      * ``means/stds`` de-normalise scores (and scale the variance column by ``stds**2``) first (eval.py:379-387);
      * per group: items sorted by target (descending); ``pred_order`` = rank of each item's score among the group (1 = best);
        gains are ``n + 1 - order`` and NDCG uses the first ``ceil(n * NDCG_cut)`` positions with a log2 discount (eval.py:309-326, 426-430);
      * rows of ``total_order``: [target, score, (uncertainty,) true_order, pred_order]; ``smiles_and_idx``: [iteration, rsmi, psmi].
    ``is_order=False`` only collects [target, score...] rows and SMILES pairs and returns ``None`` for both means."""
    import math
    ndcg_list, kl_list, total_order, smiles_and_idx = [], [], [], []
    it = 0
    with torch.no_grad():
        for X, targets, scope, add_features in data_processor.generate_batch_querys(smiles_list=smiles_list, target_name=target_name,
                                                                                     batch_size=batch_size, shuffle_query=False, shuffle_batch=False,
                                                                                     add_features_name=add_features_name):
            rsmi, psmi = [s[0] for s in X], [s[1] for s in X]
            preds_ini = model(smiles2graph_dic.parsing_smiles(rsmi), smiles2graph_dic.parsing_smiles(psmi), gpu=gpu, add_features=add_features)
            it += 1
            preds_ini = preds_ini.detach().float().cpu()
            if means is not None:
                if preds_ini.dim() > 1:
                    preds_ini = torch.stack((preds_ini[:, 0] * stds + means, preds_ini[:, 1] * (stds ** 2)), dim=1)
                else:
                    preds_ini = preds_ini * stds + means
            with_unc = preds_ini.dim() > 1
            preds = preds_ini[:, 0] if with_unc else preds_ini
            unc = preds_ini[:, 1] if with_unc else None
            t_all = torch.FloatTensor(np.squeeze(targets).tolist())
            if not is_order:
                rows = preds_ini.numpy().tolist()
                total_order.extend([[t] + r for t, r in zip(t_all.tolist(), rows)] if with_unc else [[t, r] for t, r in zip(t_all.tolist(), rows)])
                smiles_and_idx.extend([[a, b] for a, b in zip(rsmi, psmi)])
                continue
            o = 0
            for n in scope:
                bt, bp = t_all[o:o + n], preds[o:o + n]
                P, Q = torch.softmax(bt, 0), torch.softmax(bp, 0)
                # eval.py:400-402 writes exp(x)/sum(exp(x)) without a max shift; identical in exact arithmetic, and fp32-identical to ~1e-7
                P = torch.exp(bt) / torch.sum(torch.exp(bt))
                Q = torch.exp(bp) / torch.sum(torch.exp(bp))
                kl_list.append(float(torch.sum(P * torch.log(P / Q))))
                st, idx = torch.sort(bt, descending=True)
                sp = bp[idx]
                pred_order = torch.argsort(torch.argsort(sp, descending=True)) + 1
                true_order = torch.arange(n, dtype=torch.float32) + 1
                cols = [st, sp] + ([unc[o:o + n][idx]] if with_unc else []) + [true_order, pred_order.float()]
                total_order.extend(torch.stack(cols, dim=1).tolist())
                k = math.ceil(n * NDCG_cut)
                disc = torch.log2(torch.arange(min(k, n), dtype=torch.float32) + 2)
                pred_gain, true_gain = (n + 1 - pred_order).float()[:k], (n + 1 - true_order)[:k]
                ndcg_list.append(float(torch.sum(pred_gain / disc) / torch.sum(true_gain / disc)))
                order = idx.tolist()
                smiles_and_idx.extend([[it, rsmi[o + i], psmi[o + i]] for i in order])
                o += n
    if not is_order:
        return None, None, total_order, smiles_and_idx
    return np.mean(np.array(ndcg_list), axis=0), np.mean(np.array(kl_list)), total_order, smiles_and_idx


def _not_built(name):
    def f(*a, **k):
        raise NotImplementedError(f"{name} is an inference-side metric outside the hot path (SURVEY.md §2 row 8)")
    f.__name__ = name
    return f


def calculate_mse(model, gpu, data_processor, smiles2graph_dic, batch_size=2, show_info=True, smiles_list=None, target_name: str = 'ea',
                  logger=None, add_features_name=None):
    """Validation MSE for ``save_metric='mse'`` (eval.py:558-609, called at train_listwise.py:345-352).

    The reference's function cannot run: it unpacks three values from the four ``generate_batch_querys`` yields (SURVEY.md appendix A.10),
    calls the model without its extra features, and would return the squared error of the LAST chunk only.  What it is there for is
    clear from its caller -- keep the checkpoint with the smallest validation error -- so this computes the mean squared error of the
    first output column against ``target_name`` over ALL validation rows: every reactant group is one segment of a batched forward (its own
    padding rows and ``max_num_bonds``, i.e. the scores of the reference's per-chunk forward), the squared errors are summed on the
    device and one double comes back."""
    model.eval()
    chunks, targets = [], []
    for X, t, scope, feats in data_processor.generate_batch_querys(smiles_list=smiles_list, target_name=target_name, batch_size=1,
                                                                    shuffle_query=False, shuffle_batch=False,
                                                                    add_features_name=add_features_name):
        chunks.append((X, feats))
        targets.append(np.asarray(t, dtype=np.float64).reshape(-1))
    if not chunks:
        return float('nan')
    total = None
    with torch.no_grad():
        for lo, hi, preds in _forward_chunks(model, gpu, chunks, smiles2graph_dic):
            p = preds[:, 0] if preds.dim() > 1 else preds
            t = torch.from_numpy(np.concatenate(targets[lo:hi]).astype(np.float32)).pin_memory().to(p.device, non_blocking=True)
            sq = torch.sum((t.double() - p.double()) ** 2)
            total = sq if total is None else total + sq
    n = sum(len(t) for t in targets)
    mse = float(total) / n
    if show_info:
        print('the validation MSE over {} reactions is: {}'.format(n, mse))
    if logger is not None:
        logger.info('the validation MSE is {}'.format(mse))
    return mse


pairwise_acc = _not_built("pairwise_acc")
pairwise_baseline_acc = _not_built("pairwise_baseline_acc")
eval_cross_entropy_loss = _not_built("eval_cross_entropy_loss")
