"""LambdaRank on the B200: the RR_LOSS_LAMBDARANK(_TOP) kernel against the float64 restatement of test_lambdarank_cpu.py through both
C entry points, its capacity and deterministic-mode behaviour, the LambdaRankLoss module under autograd, and the task keys end to end
(train(), main.py, torchrun)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from reactranker_b200 import _lib
from test_lambdarank_cpu import lambdarank_loss, ndcg_at

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = [(_lib.LOSS_LAMBDARANK, False), (_lib.LOSS_LAMBDARANK_TOP, True)]
SIGMA = 0.7


def S():
    return torch.cuda.current_stream().cuda_stream


def close(got, want, tol):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    scale = max(float(want.abs().max()), 1e-30)
    err = float((got - want).abs().max()) / scale
    assert err < tol, err


def run(cmd, timeout=900):
    res = subprocess.run([sys.executable] + cmd, cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    return res.stdout


def inputs(scope, seed):
    """Scores and targets with tied targets (a fifth of them on a coarse grid, one group entirely tied when there are several) and
    duplicated scores."""
    N = sum(scope)
    g = torch.Generator().manual_seed(seed)
    s, t = torch.randn(N, generator=g), torch.randn(N, generator=g)
    t[::5] = torch.round(t[::5] * 2) / 2
    s[1::7] = s[0::7][:s[1::7].numel()]
    if len(scope) > 2:
        t[scope[0]:scope[0] + scope[1]] = 0.5
    return s, t


def launch(kind, scope, s, t, max_group=None, sigma=SIGMA):
    """loss [1] and dscore [N] of one rr_loss_fwdbwd (max_group None) or rr_loss_fwdbwd_ex launch; norm = the number of groups."""
    L = _lib.lib()
    N, G = sum(scope), len(scope)
    seg = torch.tensor(np.concatenate([[0], np.cumsum(scope)]), dtype=torch.int32, device=DEV)
    sd, td = s.to(DEV), t.to(DEV)
    loss, ds = torch.full((1,), float("nan"), device=DEV), torch.full_like(sd, float("nan"))
    if max_group is None:
        st = L.rr_loss_fwdbwd(kind, N, G, sd.data_ptr(), td.data_ptr(), seg.data_ptr(), float(G), sigma, loss.data_ptr(), ds.data_ptr(), S())
    else:
        st = L.rr_loss_fwdbwd_ex(kind, N, G, sd.data_ptr(), td.data_ptr(), seg.data_ptr(), max_group, float(G), sigma, loss.data_ptr(),
                                 ds.data_ptr(), S())
    torch.cuda.synchronize()
    return st, loss, ds


def restated(scope, s, t, top, sigma=SIGMA):
    sx = s.double().to(DEV).requires_grad_(True)
    want = lambdarank_loss(sx, scope, t.double().numpy(), sigma=sigma, top=top)
    want.backward()
    return want.detach().reshape(1), sx.grad


@pytest.mark.parametrize("kind,top", KINDS)
@pytest.mark.parametrize("scope", [[5, 3, 6], [1, 2, 1], [32] * 8, [50, 100, 200, 500], [2048], [3000, 5], [8192]])
def test_kernel_matches_the_fp64_restatement(kind, top, scope):
    s, t = inputs(scope, sum(scope) + kind)
    want, grad = restated(scope, s, t, top)
    big = max(scope) > 2048
    entries = [max(scope)] if big else [None, max(scope)]
    for max_group in entries:
        st, loss, ds = launch(kind, scope, s, t, max_group)
        assert st == 0, _lib.lib().rr_last_error()
        close(loss, want, 5e-6 if big else 2e-6)
        close(ds, grad, 5e-5 if big else 2e-5)


@pytest.mark.parametrize("kind,top", KINDS)
def test_groups_beyond_the_capacity_are_nan_and_max_group_beyond_8192_is_refused(kind, top):
    scope = [3000, 5]
    s, t = inputs(scope, 3)
    st, loss, ds = launch(kind, scope, s, t)                      # the plain entry holds groups of up to 2048
    assert st == 0
    assert bool(torch.isnan(loss).all()) and bool(torch.isnan(ds[:3000]).all())
    _, grad = restated(scope, s, t, top)
    close(ds[3000:], grad[3000:], 2e-5)                           # the small group is still computed
    st, _, _ = launch(kind, scope, s, t, max_group=8193)
    assert st != 0


@pytest.mark.parametrize("kind,top", KINDS)
def test_deterministic_mode_repeats_bit_for_bit(kind, top):
    L = _lib.lib()
    scope = [50] * 82 + [500] * 8 + [1, 0, 7]
    s, t = inputs(scope, 17)
    want, grad = restated(scope, s, t, top)
    _lib.check(L.rr_set_deterministic(1))
    try:
        runs = [launch(kind, scope, s, t, max(scope)) for _ in range(3)]
    finally:
        _lib.check(L.rr_set_deterministic(0))
    for st, loss, ds in runs:
        assert st == 0
        assert torch.equal(loss, runs[0][1]) and torch.equal(ds, runs[0][2])
    close(runs[0][1], want, 2e-6)
    close(runs[0][2], grad, 2e-5)


def test_loss_module_under_autograd():
    from reactranker_b200.train.loss import LambdaRankLoss
    scope = [3000, 40, 7, 1]
    s, t = inputs(scope, 23)
    for top in (False, True):
        want, grad = restated(scope, s, t, top, sigma=1.5)
        sd = s.to(DEV).requires_grad_(True)
        loss = LambdaRankLoss(sigma=1.5, top=top)(sd, scope, t, 0)
        assert loss.shape == (1,)
        (3.0 * loss).sum().backward()
        close(loss, want, 5e-6)
        close(sd.grad, 3.0 * grad, 5e-5)
    with pytest.raises(_lib.RRError):
        LambdaRankLoss()(torch.zeros(9000, device=DEV), [9000], torch.zeros(9000), 0)


@pytest.fixture
def _deterministic_off_afterwards():
    yield
    torch.use_deterministic_algorithms(False)
    _lib.check(_lib.lib().rr_set_deterministic(0))


def test_train_lambdarank_raises_the_validation_ndcg(tmp_path, _deterministic_off_afterwards):
    """train(task_type='lambdarank') on reactions ranked by a teacher: a separately seeded ReactionModel of the same shape, whose
    eval-mode scores (standardised within each group) replace lgk.  The student can represent the teacher exactly, so training must
    lower the LambdaRank loss over the training frame and raise the validation NDCG@all of ranking_metrics.

    The margin is fixed before training from the validation targets alone: a scorer that has learnt nothing ranks each group in an order
    unrelated to its targets, and the mean NDCG@all over the V validation groups of such a random order has a standard deviation of
    sqrt(sum_g var_g) / V (var_g: the variance of group g's NDCG@all over uniformly random orders, estimated from 2000 of them).  The
    trained model must beat the untrained one by four of those standard deviations."""
    from reactranker_b200 import synthetic
    from reactranker_b200.data.load_reactions import DataProcessor, Parsing_features
    from reactranker_b200.models.base_model import build_model
    from reactranker_b200.predict import predict
    from reactranker_b200.train.eval import ranking_metrics
    from reactranker_b200.train.loss import LambdaRankLoss
    from reactranker_b200.train.train_listwise import normalized_targets, train
    from reactranker_b200.train.utils import build_lr_scheduler, build_optimizer
    torch.use_deterministic_algorithms(True)
    n_train, n_val, n, epochs, batch = 240, 60, 10, 12, 100
    ds = synthetic.make_dataset(41, [n] * (n_train + n_val))
    fz = Parsing_features(ds.mols)
    cols = ["rsmi", "psmi"]
    df = ds.to_dataframe()

    def model(seed):
        torch.manual_seed(seed)
        return build_model(hidden_size=64, task_num=1, ffn_last_layer="with_softplus", dropout=0.0).cuda(0)
    teacher = model(1001).eval()
    z = predict(teacher, df, fz, 0, smiles_list=cols)["score"].to_numpy().reshape(-1, n)
    df["lgk"] = ((z - z.mean(axis=1, keepdims=True)) / z.std(axis=1, keepdims=True)).reshape(-1)
    train_df = df[df.flag < n_train].reset_index(drop=True)
    val_df = df[df.flag >= n_train].reset_index(drop=True)

    rng = np.random.default_rng(0)
    var = [np.var([ndcg_at(rng.permutation(n), tv, n) for _ in range(2000)]) for tv in val_df.lgk.to_numpy().reshape(-1, n)]
    margin = 4.0 * np.sqrt(np.sum(var)) / n_val

    student = model(7)
    targets = torch.tensor(normalized_targets(train_df.lgk, val_df.lgk, "lgk", True)[0].to_numpy())

    def measure():
        scores = torch.tensor(predict(student, train_df, fz, 0, smiles_list=cols)["score"].to_numpy(), device=DEV)
        loss = float(LambdaRankLoss()(scores, [n] * n_train, targets, 0))
        ndcg_all = ranking_metrics(student, 0, DataProcessor(val_df), fz, show_info=False, smiles_list=cols, target_name="lgk")[3][3]
        return loss, ndcg_all
    loss0, ndcg0 = measure()
    opt = build_optimizer(student)
    sched = build_lr_scheduler(opt, warmup_epochs=2, total_epochs=epochs, train_data_size=len(train_df), batch_size=batch, init_lr=1e-4,
                               max_lr=3e-3, final_lr=1e-4)
    train(student, sched, train_df, val_df, str(tmp_path / "ck.pt"), opt, epochs, fz, batch_size=batch, seed=0, gpu=0, task_type="lambdarank", writer=None,
          target_name="lgk", smiles_list=cols, save_metric="NDCG@all")
    loss1, ndcg1 = measure()
    assert loss1 < loss0, (loss0, loss1)
    assert ndcg1 > ndcg0 + margin, (ndcg0, ndcg1, margin)


def test_main_trains_lambdarank_top_and_writes_a_checkpoint(tmp_path):
    out = run(["main.py", "--synthetic", "40,10", "--path", str(tmp_path), "--gpu", "0", "--task_type", "lambdarank_top", "--batch_size", "100",
               "--total_epochs", "3", "--hidden_size", "64", "--max_lr", "3e-3"])
    losses = [float(l.rsplit(":", 1)[1]) for l in out.splitlines() if "train loss" in l]
    assert len(losses) == 3 and all(np.isfinite(losses)) and losses[0] > 0
    assert os.path.exists(os.path.join(str(tmp_path), "T1", "0.pt"))
    assert "test score for k_fold vailidation" in out


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_torchrun_lambdarank_reproduces_the_one_gpu_loss_curve(tmp_path):
    """Under torchrun every rank divides by the global group count (TrainStep's dp_normalisers), so the two-rank loss curve is the
    one-GPU curve to rounding."""
    def curve(out):
        return [float(l.rsplit("=", 1)[1]) for l in out.splitlines() if "full precision" in l]
    args = ["main.py", "--synthetic", "40,10", "--task_type", "lambdarank", "--batch_size", "100", "--total_epochs", "4", "--hidden_size", "64",
            "--max_lr", "3e-3", "--dropout", "0.0"]
    one = run(args + ["--gpu", "0", "--path", str(tmp_path / "one")])
    two = run(["-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29641"]
              + args + ["--path", str(tmp_path / "two")])
    want, got = curve(one), curve(two)
    assert len(want) == 4 and len(got) == 4, (one[-2000:], two[-2000:])
    assert np.allclose(got, want, rtol=1e-4), (got, want)
    assert os.path.exists(os.path.join(str(tmp_path / "two"), "T1", "0.pt"))
