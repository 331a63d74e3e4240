"""LTR loss layer with the reference's module names and call signatures
(train/loss.py:64-99, 144-162, 317-352, 477-556; RankNet: train/train_pairwise.py:98-147).

Each loss is ONE segmented sm_100a kernel (csrc/rr_loss.cu) that returns the normalised
loss and dL/dscore together; the Python loop over groups of the reference is gone.
Normalisation follows the reference exactly: ListMLE / UC-Listwise average per group then
over groups, ListNet averages over all items of the batch, RankNet divides by the ordered
pair count of the accumulation window.  ``mle`` and ``evidential_ranking`` return shape [1]
like the reference, the others a 0-d tensor.

Every task key the reference can run is dispatched by ``train()`` (train_listwise.batch_loss): the five north-star keys, the composite
keys that are sums of their terms, the distribution-valued ``MLEDisLoss`` / ``Listnet_For_Gauss``, ``Listnet_with_uq``, ``Dirichlet_uq``,
``Lognorm`` and the NIG ``evidential_loss_new``.  Only the two losses no task key constructs (``Listnetlognorm``,
``Listnet_For_evidential``) raise.  ``LambdaRankLoss`` (keys ``lambdarank`` / ``lambdarank_top``) is this project's own, not the
reference's: it trains for the validation's NDCG.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from .. import _lib


def _device_of(gpu, like: torch.Tensor) -> torch.device:
    if not like.is_cuda:
        raise _lib.RRError("scores live on the CPU: reactranker_b200 losses run on a B200 only (no CPU fallback)")
    if gpu is not None:
        _lib.require_device(gpu)
    return like.device


def _to_dev(x, dev, dtype=torch.float32) -> torch.Tensor:
    if isinstance(x, torch.Tensor):
        if x.device == dev and x.dtype == dtype:
            return x.contiguous()
        return x.to(dtype).pin_memory().to(dev, non_blocking=True) if not x.is_cuda else x.to(dev, dtype)
    return torch.as_tensor(np.asarray(x), dtype=dtype).pin_memory().to(dev, non_blocking=True)


_SEG_CACHE: dict = {}


def segment_offsets(scope: Sequence[int], dev) -> torch.Tensor:
    """``scope`` (python list of group sizes, as the reference passes it) -> device prefix sums.
    A few recent scopes are kept on the device so a repeated batch shape costs no copy."""
    key = (tuple(scope), str(dev))
    hit = _SEG_CACHE.get(key)
    if hit is not None:
        return hit
    off = np.zeros(len(scope) + 1, np.int32)
    np.cumsum(np.asarray(scope, np.int64), out=off[1:])
    t = torch.from_numpy(off).pin_memory().to(dev, non_blocking=True)
    if len(_SEG_CACHE) >= 64:
        _SEG_CACHE.pop(next(iter(_SEG_CACHE)))
    _SEG_CACHE[key] = t
    return t


class _LossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, scores, targets, seg_off, kind: int, n_items: int, n_groups: int, norm: float, sigma: float, out_shape, max_group: int = 0):
        L = _lib.lib()
        scores_c = scores.contiguous()
        loss = torch.empty(1, dtype=torch.float32, device=scores.device)
        dscore = torch.empty_like(scores_c)
        _lib.set_deterministic(_lib.deterministic_requested())
        with torch.cuda.device(scores.device):
            _lib.check(L.rr_loss_fwdbwd_ex(kind, n_items, n_groups, scores_c.data_ptr(), targets.data_ptr(), _lib.ptr(seg_off), int(max_group),
                                           float(norm), float(sigma), loss.data_ptr(), dscore.data_ptr(), _lib.stream_ptr()))
        ctx.save_for_backward(dscore)
        return loss.reshape(out_shape)

    @staticmethod
    def backward(ctx, g):
        (dscore,) = ctx.saved_tensors
        return dscore * g.reshape(()), None, None, None, None, None, None, None, None, None


def _segmented(kind, scores, scope, targets, gpu, norm, out_shape, sigma=1.0, check_max=False):
    dev = _device_of(gpu, scores)
    scope = [int(s) for s in scope]
    n_items = int(sum(scope))
    if n_items != scores.shape[0]:
        raise _lib.RRError(f"sum(scope)={n_items} does not match the {scores.shape[0]} scores")
    if check_max and max(scope) > _lib.lib().rr_loss_max_group():
        raise _lib.RRError(f"group of {max(scope)} candidates exceeds the segmented kernel's limit {_lib.lib().rr_loss_max_group()}")
    t = _to_dev(targets, dev).reshape(-1)
    if t.numel() != n_items:
        raise _lib.RRError(f"{t.numel()} targets for {n_items} scores")
    seg = segment_offsets(scope, dev)
    return _LossFn.apply(scores.float(), t, seg, kind, n_items, len(scope), norm, sigma, out_shape, max(scope) if scope else 0)


# ---- data-parallel normalisers -------------------------------------------------------------------------------------------------
# When reaction groups are sharded over ranks (reactranker_b200/parallel.py), every rank divides by the GLOBAL batch's normaliser and the
# gradients are SUM-all-reduced, which reproduces the single-device loss exactly (SURVEY.md 8e).  The reference's losses normalise in one
# of two ways: a mean over the batch's groups (ListMLE, UC-Listwise, the distribution-valued and uncertainty ListNet / ListMLE variants,
# Dirichlet) or a mean over the batch's items (ListNet, Gaussian / log-normal NLL, MSE).  ``dp_normalisers(groups=G, items=N)`` sets both
# for every loss evaluated inside the ``with`` block (train.step.TrainStep does, from the global batch plan); outside it, and for
# world size 1, the local counts are used.  ``global_norm=`` on a loss object overrides the context for that object.
import contextlib
import threading

_DP = threading.local()


@contextlib.contextmanager
def dp_normalisers(groups=None, items=None):
    prev = getattr(_DP, "norms", None)
    _DP.norms = (groups, items)
    try:
        yield
    finally:
        _DP.norms = prev


def _global(kind: int):
    n = getattr(_DP, "norms", None)
    return None if n is None else n[kind]


def _items_norm(local_items: int) -> float:
    g = _global(1)
    return float(local_items if g is None else g)


class _DPNorm(nn.Module):
    """Base of the segmented losses: ``_norm(local)`` is the divisor of a mean over GROUPS, ``_norm(local, items=True)`` of a mean over
    ITEMS; ``global_norm`` (constructor) > ``dp_normalisers`` context > the local count."""

    def __init__(self, global_norm=None):
        super().__init__()
        self.global_norm = global_norm

    def _norm(self, local, items: bool = False):
        if self.global_norm is not None:
            return self.global_norm
        g = _global(1 if items else 0)
        return local if g is None else g


class MLEloss(_DPNorm):
    """ListMLE (loss.py:64-99 with LogCumsumExp 9-61): per group, sort by target descending,
    ``mean(logcumsumexp_tail(x) - x)``; then the mean over groups.  Returns shape [1]."""

    def forward(self, score, scope, targets_train, gpu: int):
        return _segmented(_lib.LOSS_LISTMLE, score, scope, targets_train, gpu, norm=self._norm(len(scope)), out_shape=(1,), check_max=True)


class LambdaRankLoss(_DPNorm):
    """LambdaRank (Burges et al.), this project's own key: RankNet over each group's pairs ``t_i > t_j`` (each once), every pair weighted
    by ``|dNDCG@K|``, the change of the validation's NDCG (gain ``exp(t)``, discount ``1 / log2(1 + rank)``) if the two items swapped
    places at the current scores; the sum over groups divided by the number of groups.  ``top=False``: ``K = n``; ``top=True``: the
    ``K = max(1, round(n / 4))`` of NDCG@25%.  The weights are constants of the scores, so the gradient is RankNet's pair gradient times
    the weight.  Returns shape [1]."""

    def __init__(self, sigma: float = 1.0, top: bool = False, global_norm=None):
        super().__init__(global_norm)
        self.sigma, self.top = float(sigma), bool(top)

    def forward(self, score, scope, targets, gpu: int):
        kind = _lib.LOSS_LAMBDARANK_TOP if self.top else _lib.LOSS_LAMBDARANK
        return _segmented(kind, score, scope, targets, gpu, norm=self._norm(len(scope)), out_shape=(1,), sigma=self.sigma, check_max=True)


class ListnetLoss(_DPNorm):
    """ListNet top-1 (loss.py:317-352): ``mean over all items`` of ``-softmax(t) * log softmax(s)``."""

    def forward(self, score, scope, targets, gpu: int):
        return _segmented(_lib.LOSS_LISTNET, score, scope, targets, gpu, norm=self._norm(int(sum(scope)), items=True), out_shape=())


class evidential_ranking(_DPNorm):
    """UC-Listwise (loss.py:477-556, live branch 526-554).  ``max_coeff, epoch, epochs`` are
    accepted and unused, as in the reference.  Returns shape [1]."""

    def forward(self, possibilities, scope, targets, max_coeff, epoch, epochs, gpu: int):
        if possibilities.dim() != 2 or possibilities.shape[1] != 2:
            raise _lib.RRError("evidential_ranking expects model outputs of shape [N, 2] (score, variance)")
        return _segmented(_lib.LOSS_EVIDENTIAL, possibilities, scope, targets, gpu, norm=self._norm(len(scope)), out_shape=(1,))


def _mean_variance(mean, variance) -> torch.Tensor:
    """(mean [N] or [N,1], variance [N] or [N,1]) -> contiguous [N,2], the layout of the distribution-valued kernels."""
    m, v = mean.reshape(-1), variance.reshape(-1)
    if m.shape != v.shape:
        raise _lib.RRError(f"mean has {m.numel()} entries, variance {v.numel()}")
    return torch.stack((m, v), dim=1)


class MLEDisLoss(_DPNorm):
    """ListMLE over Gaussian scores (loss.py:102-141).  The reference builds an n x n lower-triangular matrix per group; it equals
    ``mean_j(logcumsumexp_tail(z)_j - z_j + v_j)`` with ``z = mean + variance / 2`` in target-descending order, averaged over groups.
    Returns shape [1]."""

    def forward(self, mean, variance, scope, targets, gpu: int):
        return _segmented(_lib.LOSS_LISTMLE_DIS, _mean_variance(mean, variance), scope, targets, gpu, norm=self._norm(len(scope)), out_shape=(1,),
                          check_max=True)


class Listnet_For_Gauss(_DPNorm):
    """ListNet top-1 over log-normal scores (loss.py:233-272): per group ``mean_i softmax(t)_i (lse(u) - u_i + v_i)`` with
    ``u = mean + variance / 2``, then the mean over groups.  Returns shape [1]."""

    def forward(self, mean, variance, scope, targets, gpu: int):
        return _segmented(_lib.LOSS_LISTNET_DIS, _mean_variance(mean, variance), scope, targets, gpu, norm=self._norm(len(scope)), out_shape=(1,))


class Listnet_with_uq(_DPNorm):
    """ListNet on normalised positive scores with an uncertainty penalty (loss.py:355-399): ``pred = s / sum(s)``, ``p = softmax(t)``,
    per group ``KL(p || pred) / n + coef * mean_i |log(p_i / pred_i) (s_i - 1)|`` with the reference's annealing
    ``coef = max_coeff * (epoch / (epochs - 1)) ** 3`` (a ZeroDivisionError at ``epochs == 1``, as there).  Returns shape [1]."""

    def forward(self, score, scope, targets, max_coeff, epoch, epochs, gpu: int):
        coef = max_coeff * (epoch / (epochs - 1)) ** 3
        return _segmented(_lib.LOSS_LISTNET_UQ, score, scope, targets, gpu, norm=self._norm(len(scope)), out_shape=(1,), sigma=coef)


class Dirichlet_uq(_DPNorm):
    """Dirichlet mean / variance loss on 1-D positive concentrations (loss.py:440-474): per group
    ``mean_i((pred_i - p_i)^2 + pred_i (1 - pred_i) / (S + 1) + coef |log(p_i / pred_i) (a_i - 1)|)``, ``pred = a / S``.  Returns shape [1]."""

    def forward(self, concentration, scope, targets, max_coeff, epoch, epochs, gpu: int):
        if concentration.dim() != 1:
            raise _lib.RRError("Dirichlet_uq is built for the 1-D output of a task_num = 1 model (the only shape train_listwise.py:269-270 passes)")
        coef = max_coeff * (epoch / (epochs - 1)) ** 3
        return _segmented(_lib.LOSS_DIRICHLET_UQ, concentration, scope, targets, gpu, norm=self._norm(len(scope)), out_shape=(1,), sigma=coef)


def evidential_loss_new(mu, v, alpha, beta, targets, gpu, lam=1, epsilon=1e-4):
    """Deep-evidential-regression loss (loss.py:402-437) with the shapes its four call sites pass (train_listwise.py:229-260):
    ``mu, v, alpha, beta`` are ``[N, 1]`` column slices and ``targets`` is ``[N]``, so ``targets - mu`` broadcasts to ``[N, N]`` and
    the value is the mean over ALL (reaction i, target j) pairs of the batch.  That is what the reference trains on, so that is what
    one all-pairs launch computes here; 1-D / mismatched shapes (element-wise in torch) are rejected rather than guessed."""
    if epsilon != 1e-4:
        raise _lib.RRError("evidential_loss_new: epsilon is fixed at the reference default 1e-4")
    if _global(1) is not None and int(_global(1)) != int(mu.shape[0]):
        raise _lib.RRError("the NIG task keys pair every reaction with EVERY target of the batch (the reference's [N,1] x [N] broadcast): "
                           "the loss does not shard over ranks; train these keys on one GPU")
    cols = [mu, v, alpha, beta]
    n = mu.shape[0]
    if any(c.dim() != 2 or c.shape != (n, 1) for c in cols):
        raise _lib.RRError("evidential_loss_new expects the [N, 1] column slices of a task_num = 4 model (train_listwise.py:230-233)")
    dev = _device_of(gpu, mu)
    t = _to_dev(targets, dev).reshape(-1)
    if t.numel() != n:
        raise _lib.RRError(f"{t.numel()} targets for {n} rows")
    scores = torch.cat(cols, dim=1).float()
    return _LossFn.apply(scores, t, None, _lib.LOSS_NIG, n, 0, float(n) * float(n), float(lam), ())


class Lognorm(nn.Module):
    """Log-normal NLL (loss.py:165-184): ``mean(0.5 log 2pi + 0.5 log(v m^2) + (log m - t)^2 / (2 v))`` (without its ``print``)."""

    def forward(self, scores, std_scores, targets, gpu: int):
        dev = _device_of(gpu, scores)
        both = _mean_variance(scores, std_scores).float()
        n = both.shape[0]
        return _LossFn.apply(both, _to_dev(targets, dev).reshape(-1), None, _lib.LOSS_LOGNORM, n, 0, _items_norm(n), 1.0, ())


class _GaussFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mean, var, targets):
        both = torch.stack((mean, var), dim=1).contiguous()
        L = _lib.lib()
        n = both.shape[0]
        loss = torch.empty(1, dtype=torch.float32, device=both.device)
        d = torch.empty_like(both)
        _lib.set_deterministic(_lib.deterministic_requested())
        with torch.cuda.device(both.device):
            _lib.check(L.rr_loss_fwdbwd(_lib.LOSS_GAUSS, n, 0, both.data_ptr(), targets.data_ptr(), None, _items_norm(n), 1.0,
                                        loss.data_ptr(), d.data_ptr(), _lib.stream_ptr()))
        ctx.save_for_backward(d)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        (d,) = ctx.saved_tensors
        d = d * g
        return d[:, 0], d[:, 1], None


class GaussDisLoss(nn.Module):
    """Gaussian NLL (loss.py:144-162): ``mean(0.5 log 2pi + 0.5 log v + (mu - t)^2 / (2 v))``."""

    def forward(self, mean_scores, std_scores, targets, gpu: int):
        dev = _device_of(gpu, mean_scores)
        return _GaussFn.apply(mean_scores.float(), std_scores.float(), _to_dev(targets, dev).reshape(-1))


class MSELoss(nn.Module):
    """The default 'regression' criterion (``nn.MSELoss``, train_listwise.py:166-167, 282-285)."""

    def forward(self, output, targets):
        dev = _device_of(None, output)
        n = output.shape[0]
        return _LossFn.apply(output.float().reshape(-1), _to_dev(targets, dev).reshape(-1), None, _lib.LOSS_MSE, n, 0, _items_norm(n), 1.0, ())


class ExpMSELoss(nn.Module):
    """``mean((exp(targets) - exp(output))**2)``: the 'regression_exploss' key, written inline in the reference (train_listwise.py:276-281)."""

    def forward(self, output, targets):
        dev = _device_of(None, output)
        n = output.shape[0]
        return _LossFn.apply(output.float().reshape(-1), _to_dev(targets, dev).reshape(-1), None, _lib.LOSS_EXPMSE, n, 0, _items_norm(n), 1.0, ())


def ranknet_window_loss(scores, scope, targets, num_pairs: float, sigma: float = 1.0, gpu: Optional[int] = None,
                        training_algo: str = 'sum_session'):
    """RankNet cost of one accumulation window (train_pairwise.py:98-137, 141-152):
    ``sum over groups and ordered pairs of the pairwise logistic cost / num_pairs``; groups of the
    window are evaluated by one launch.  ``num_pairs`` is the window's ordered-pair count.
    'accelerate_grad' reports the same cost but back-propagates the hand-written lambda of lines 125-133,
    ``sum_j (-sigma pos_ij / (1 + e^{sigma (s_i - s_j)}) + sigma neg_ij / (1 + e^{-sigma (s_i - s_j)})) / pairs``: the row sums only,
    i.e. exactly half of what autograd gives 'sum_session' (the column sums are equal by symmetry)."""
    if training_algo not in ('sum_session', 'accelerate_grad'):
        raise ValueError("training algo {} not implemented".format(training_algo))
    if scores.dim() > 1:
        scores = scores[:, 0]                        # train_pairwise.py:115-116
    kind = _lib.LOSS_RANKNET if training_algo == 'sum_session' else _lib.LOSS_RANKNET_ACC
    return _segmented(kind, scores, scope, targets, gpu, norm=float(num_pairs), out_shape=(), sigma=sigma, check_max=True)


def count_ordered_pairs(targets: np.ndarray) -> float:
    """``2 * #{(i, j): t_i > t_j}`` of one group (train_pairwise.py:98-106)."""
    t = np.asarray(targets, np.float64).reshape(-1)
    _, counts = np.unique(t, return_counts=True)
    n = t.shape[0]
    return float(n * n - np.sum(counts.astype(np.float64) ** 2))


def _unbuilt(name):
    class _Missing(nn.Module):
        def __init__(self, *a, **k):
            raise NotImplementedError(f"{name} is one of the reference's experimental losses (SURVEY.md §2 row 6), not on the "
                                      "north-star path; only mle / listnet / evidential_ranking / gauss_regression / regression are built")
    _Missing.__name__ = name
    return _Missing


# constructed by no task key (Listnetlognorm's only call is commented out at train_listwise.py:219; Listnet_For_evidential is imported only)
Listnet_For_evidential = _unbuilt("Listnet_For_evidential")
Listnetlognorm = _unbuilt("Listnetlognorm")
