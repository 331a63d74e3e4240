"""Rank new candidate reactions with a trained model: ``predict(model, data, ...)`` scores every candidate of a frame that has no target
column and returns, per candidate, its score, its rank within its reactant group and how sure the model is of that rank.

Groups are reactant groups as ``DataProcessor`` forms them (rows sharing ``rsmi``).  Up to ``eval.GROUPS_PER_LAUNCH`` groups share a
forward, each as its own segment (its own padding rows and ``max_num_bonds``), so a candidate's score is the score of a forward over its
group alone, whichever groups share the launch.  The per-group statistics are computed on the device by ``rr_rank_predict``
(include/rr_sm100.h) and the host waits once, at the end.

``mc_samples = T > 1`` is MC dropout: the model runs in train mode (dropout active) under ``torch.no_grad()``, every launch's two device
graphs are assembled once and forwarded T times.  Forwards run chunk-major, then sample t = 0..T-1, and each draws its dropout seed from
torch's RNG (``ReactionModel._cfg``), so ``torch.manual_seed`` before the call reproduces the result.
"""
from __future__ import annotations

import numpy as np
import pandas as pd
import torch

from . import _lib
from .data.load_reactions import DataProcessor
from .models.base_model import reactant_dedup_exact
from .train import eval as E
from .train.loss import segment_offsets

COLUMNS = ("score", "score_std", "rank", "p_top1", "top1_freq", "mean_rank")     # rr_rank_predict's columns 0-5


def predict(model, data: pd.DataFrame, smiles2graph_dic, gpu, smiles_list=None, add_features_name=None, mc_samples: int = 1) -> pd.DataFrame:
    """``data``'s rows, in its order and with its index, plus the columns
      score       mean of the ranking score (output column 0) over the samples
      score_std   its standard deviation over the samples (ddof 0; 0 for mc_samples = 1)
      rank        1-based rank of ``score`` within the reactant group (stable: ties keep the earlier row)
      p_top1      mean over samples of the within-group softmax: the ListNet / Plackett-Luce probability of ranking first
      top1_freq   fraction of samples in which the candidate ranks first
      mean_rank   mean over samples of the candidate's rank
      out1 ...    for heads with task_num > 1, the sample means of the other output columns (e.g. the variance of evidential_ranking)
    ``smiles_list`` names the (reactant, product) columns (default rsmi / psmi); ``add_features_name`` the extra-feature column(s) the
    model was built with.  No target column is read.  Scores are unit-free (listwise losses are shift-invariant)."""
    T = int(mc_samples)
    if T < 1:
        raise ValueError(f"mc_samples must be >= 1 (got {mc_samples})")
    if T > 1 and not model.any_dropout():
        raise ValueError("mc_samples > 1 samples dropout masks, but every dropout of this model is 0")
    dev_idx = _lib.require_device(gpu)
    dev = torch.device("cuda", dev_idx)
    proc = DataProcessor(data)
    groups = list(proc.plan_batch_per_query(data, shuffle_query=False, shuffle_batch=False))
    max_group = _lib.lib().rr_loss_max_group()
    if groups and max(len(r) for r in groups) > max_group:
        raise _lib.RRError(f"a reactant group of {max(len(r) for r in groups)} candidates exceeds the limit of {max_group}")
    cols = ['rsmi', 'psmi'] if smiles_list is None else list(smiles_list)
    smiles = np.stack([data[c].values for c in cols], axis=1) if len(data) else np.empty((0, 2), object)
    feats = None
    if add_features_name is not None:
        names = list(add_features_name) if isinstance(add_features_name, (list, tuple)) else [add_features_name]
        feats = np.stack([data[c].values for c in names], axis=1)
    chunks = [(smiles[r], None if feats is None else feats[r]) for r in groups]

    was_training = model.training
    parts = []
    try:
        model.train(T > 1)
        with torch.no_grad(), torch.cuda.device(dev):
            for lo, hi, rg, pg, f in E._launch_graphs(chunks, smiles2graph_dic, dev, reactant_dedup_exact(model)):
                scope = [len(r) for r in groups[lo:hi]]
                n = sum(scope)
                if f is not None:              # uploaded once, read by all T forwards
                    f = torch.as_tensor(np.asarray(f, dtype=np.float32)).reshape(n, -1).pin_memory().to(dev, non_blocking=True)
                samples = torch.stack([model(rg, pg, gpu=dev_idx, add_features=f).reshape(n, -1) for _ in range(T)])   # [T, n, task_num]
                task_num = samples.shape[2]
                table = torch.empty(n, len(COLUMNS), dtype=torch.float32, device=dev)
                _lib.check(_lib.lib().rr_rank_predict(n, len(scope), T, samples.data_ptr(), n * task_num, task_num,
                                                      segment_offsets(scope, dev).data_ptr(), max(scope), table.data_ptr(), _lib.stream_ptr()))
                parts.append((table, samples[:, :, 1:].mean(dim=0) if task_num > 1 else None))
    finally:
        model.train(was_training)

    out = data.copy()
    if not parts:
        for c in COLUMNS:
            out[c] = pd.Series(dtype=np.int64 if c == "rank" else np.float64)
        return out
    table = torch.cat([p[0] for p in parts]).cpu().numpy()                 # the one host wait
    rows = np.concatenate(groups)                                           # frame positions in the order of the table
    for k, c in enumerate(COLUMNS):
        v = np.empty(len(data), np.int64 if c == "rank" else np.float64)
        v[rows] = table[:, k]
        out[c] = v
    if parts[0][1] is not None:
        extra = torch.cat([p[1] for p in parts]).cpu().numpy()
        for k in range(extra.shape[1]):
            v = np.empty(len(data), np.float64)
            v[rows] = extra[:, k]
            out[f"out{k + 1}"] = v
    return out
