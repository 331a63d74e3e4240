"""LambdaRank without a GPU: the float64 restatement of rr_loss_fwdbwd's RR_LOSS_LAMBDARANK(_TOP) (the GPU tests in
test_gpu_lambdarank.py check the kernel against it), its pair weights against a brute-force swap of two items, its NDCG against the
validation's (oracle.group_metrics), and the Python wiring: enum values, the loss module's arguments and the task-key dispatch."""
import os
import re

import numpy as np
import pytest
import torch

from oracle import reactranker_oracle as O
from reactranker_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def cutoff(n, top):
    """K of the NDCG: n, or for the top variant the K of the validation's NDCG@25% (Python's round: half to even)."""
    return max(1, round(0.25 * n)) if top else n


def ndcg_at(order, t, K):
    """NDCG@K of the items listed in `order` (best first) with gain exp(t) and discount 1 / log2(1 + position)."""
    t = np.asarray(t, np.float64)
    disc = 1.0 / np.log2(2.0 + np.arange(K))
    return float(np.sum(np.exp(t[order[:K]]) * disc) / np.sum(np.sort(np.exp(t))[::-1][:K] * disc))


def pair_weights(s, t, top=False):
    """float64 tensors s, t [n] -> [n, n]: w[i, j] = |G_i - G_j| |D(r_i) - D(r_j)| / IDCG_K where t_i > t_j, else 0 (G_i = exp(t_i - max t),
    D(r) = 1 / log2(1 + r) for r <= K, else 0, r the stable rank of s).  Runs on the tensors' device."""
    n = t.shape[0]
    K = cutoff(n, top)
    g = torch.exp(t - t.max())
    order = torch.sort(s, descending=True, stable=True).indices
    r = torch.empty_like(order)
    r[order] = torch.arange(1, n + 1, device=s.device)
    D = torch.where(r <= K, 1.0 / torch.log2(1.0 + r.double()), 0.0)
    idcg = (torch.sort(g, descending=True).values[:K] / torch.log2(2.0 + torch.arange(K, dtype=torch.float64, device=s.device))).sum()
    w = (g[:, None] - g[None, :]).abs() * (D[:, None] - D[None, :]).abs() / idcg
    return torch.where(t[:, None] > t[None, :], w, 0.0)


def lambdarank_loss(s, scope, t, sigma=1.0, top=False, norm=None):
    """The loss in float64: sum over groups and pairs t_i > t_j of w_ij softplus(-sigma (s_i - s_j)), over `norm` (default: the number of
    groups).  `s` is a float64 tensor (it may require grad); the weights are computed from its values without a gradient, as the kernel's
    are constants of the scores."""
    t = torch.as_tensor(np.asarray(t, np.float64), device=s.device)
    total = s.new_zeros(())
    o = 0
    for n in scope:
        if n == 0:                                                # an empty group counts in the normaliser only
            continue
        x = s[o:o + n]
        w = pair_weights(x.detach(), t[o:o + n], top)
        total = total + (w * torch.nn.functional.softplus(-sigma * (x[:, None] - x[None, :]))).sum()
        o += n
    return total / (len(scope) if norm is None else norm)


def _weights(s, t, top=False):
    return pair_weights(torch.tensor(s, dtype=torch.float64), torch.tensor(t, dtype=torch.float64), top).numpy()


def _random_group(rng, n):
    """Scores and targets with ties in both: targets on a coarse grid, some scores copied."""
    t = rng.integers(-3, 4, n) * 0.5 + (rng.random(n) < 0.5) * rng.standard_normal(n)
    s = rng.standard_normal(n).astype(np.float32)
    if n > 2:
        s[rng.integers(0, n, n // 3)] = s[0]
    return s, t


@pytest.mark.parametrize("top", [False, True])
def test_pair_weight_is_the_ndcg_change_of_swapping_the_pair(top):
    rng = np.random.default_rng(11)
    for trial in range(300):
        n = 1 + trial % 12
        s, t = _random_group(rng, n)
        K = cutoff(n, top)
        order = np.argsort(-s.astype(np.float64), kind="stable")
        now = ndcg_at(order, t, K)
        w = _weights(s, t, top)
        pos = np.empty(n, np.int64)
        pos[order] = np.arange(n)
        for i in range(n):
            for j in range(n):
                swapped = order.copy()
                swapped[pos[i]], swapped[pos[j]] = j, i
                delta = abs(ndcg_at(swapped, t, K) - now)
                if t[i] > t[j]:
                    assert w[i, j] == pytest.approx(delta, rel=1e-12, abs=1e-15), (n, i, j)
                else:
                    assert w[i, j] == 0.0
                    if t[i] == t[j]:
                        assert delta < 1e-15              # tied targets: swapping them changes nothing, the pair is left out
        assert np.all(w >= 0.0)


def test_ndcg_of_the_restatement_is_the_validation_ndcg():
    """The NDCG that LambdaRank's weights differentiate is the validation's: group_metrics column 7 (NDCG@all) for the full list and
    column 6 (NDCG@25%) for the top variant, at the same scores and targets."""
    rng = np.random.default_rng(5)
    for trial in range(200):
        n = 1 + trial % 12
        s, t = _random_group(rng, n)
        order = np.argsort(-s.astype(np.float64), kind="stable")
        cols = O.group_metrics(s.astype(np.float64), t, 0.25)
        assert ndcg_at(order, t, cutoff(n, False)) == pytest.approx(cols[7], rel=1e-12)
        assert ndcg_at(order, t, cutoff(n, True)) == pytest.approx(cols[6], rel=1e-12)


def test_loss_gradient_is_the_weighted_ranknet_gradient():
    """dL/ds_k = (sigma / norm) [sum_{t_j < t_k} -w_kj sigmoid(-sigma (s_k - s_j)) + sum_{t_j > t_k} w_jk sigmoid(sigma (s_k - s_j))],
    and a group without an ordered pair adds nothing but counts in the normaliser."""
    rng = np.random.default_rng(3)
    scope, sigma = [7, 1, 4, 9], 0.8
    N = sum(scope)
    t = rng.standard_normal(N)
    t[8:12] = 0.25                                                         # the third group: all targets tied
    s = torch.tensor(rng.standard_normal(N), dtype=torch.float64, requires_grad=True)
    loss = lambdarank_loss(s, scope, t, sigma=sigma, top=False)
    loss.backward()
    want = np.zeros(N)
    o = 0
    x = s.detach().numpy()
    for n in scope:
        w = _weights(x[o:o + n], t[o:o + n])
        d = sigma * (x[o:o + n, None] - x[None, o:o + n])
        sig = lambda z: 1.0 / (1.0 + np.exp(-z))  # noqa: E731
        want[o:o + n] = sigma / len(scope) * ((-w * sig(-d)).sum(axis=1) + (w.T * sig(d)).sum(axis=1))
        o += n
    assert np.allclose(s.grad.numpy(), want, rtol=1e-12, atol=1e-15)
    assert not s.grad[8:12].any() and not s.grad[7]
    assert float(lambdarank_loss(s.detach()[7:12], [1, 4], t[7:12])) == 0.0


def test_loss_kinds_match_the_header():
    header = open(os.path.join(ROOT, "include", "rr_sm100.h")).read()
    enum = {name: int(v) for name, v in re.findall(r"\bRR_LOSS_([A-Z_]+)\s*=\s*(\d+)", header)}
    assert enum["LAMBDARANK"] == _lib.LOSS_LAMBDARANK == 14
    assert enum["LAMBDARANK_TOP"] == _lib.LOSS_LAMBDARANK_TOP == 15
    assert sorted(enum.values()) == list(range(16))
    assert re.search(r"#define RR_ABI_VERSION 3\b", header)


def test_loss_module_passes_kind_norm_and_sigma(monkeypatch):
    """LambdaRankLoss divides by the number of groups (the global one under data parallelism), keeps a group limit check and returns [1]."""
    from reactranker_b200.train import loss as L
    calls = []
    monkeypatch.setattr(L, "_segmented", lambda kind, score, scope, targets, gpu, norm, out_shape, sigma=1.0, check_max=False:
                        calls.append((kind, norm, out_shape, sigma, check_max)))
    scope = [3, 4, 5]
    L.LambdaRankLoss()(None, scope, None, 0)
    L.LambdaRankLoss(sigma=2.5, top=True)(None, scope, None, 0)
    with L.dp_normalisers(groups=9, items=40):
        L.LambdaRankLoss()(None, scope, None, 0)
        L.LambdaRankLoss(global_norm=4)(None, scope, None, 0)
    assert calls == [(_lib.LOSS_LAMBDARANK, 3, (1,), 1.0, True), (_lib.LOSS_LAMBDARANK_TOP, 3, (1,), 2.5, True),
                     (_lib.LOSS_LAMBDARANK, 9, (1,), 1.0, True), (_lib.LOSS_LAMBDARANK, 4, (1,), 1.0, True)]


def test_batch_loss_routes_the_two_keys(monkeypatch):
    from reactranker_b200.train import train_listwise as T
    seen = []

    class Rec:
        def __init__(self, name, **kw):
            self.name, self.kw = name, kw

        def __call__(self, *args):
            seen.append((self.name, self.kw))
            return 0.0
    monkeypatch.setattr(T, "LambdaRankLoss", lambda **kw: Rec("lambdarank", **kw))
    monkeypatch.setattr(T, "MSELoss", lambda **kw: Rec("mse", **kw))
    for key in ("lambdarank", "lambdarank_top", "lambdarank_at_1"):
        T.batch_loss(key, None, [2], None, 0)
    assert seen == [("lambdarank", {"top": False}), ("lambdarank", {"top": True}), ("mse", {})]
    assert {"lambdarank", "lambdarank_top"} <= set(T.BUILT_TASKS)
