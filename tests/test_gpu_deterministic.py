"""Deterministic mode (torch.use_deterministic_algorithms / rr_set_deterministic): the same inputs give the same bits, run after run.

Every test compares three runs with torch.equal.  The default mode sums weight-gradient slabs, segment padding rows and loss parts with
float atomics, whose order changes from run to run; the deterministic mode stores those partials and adds them in a fixed order."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from reactranker_b200 import _lib, synthetic
from reactranker_b200.features.featurization import BatchMolGraph, DeviceGraph
from reactranker_b200.models.base_model import build_model
from reactranker_b200.train import loss as RL
from reactranker_b200.train.train_listwise import batch_loss
from reactranker_b200.train.utils import build_optimizer
from helpers import add_features

pytestmark = pytest.mark.gpu
GPU = 0
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(autouse=True)
def _deterministic_off_afterwards():
    yield
    torch.use_deterministic_algorithms(False)
    _lib.check(_lib.lib().rr_set_deterministic(0))


def _disturb():
    """Queue a large matmul loop on a second stream: it occupies SMs while the step runs, so the step's CTAs are scheduled differently."""
    s2 = torch.cuda.Stream()
    a = torch.randn(8192, 8192, device="cuda")
    with torch.cuda.stream(s2):
        for _ in range(30):
            a = a @ a * 1e-4
    return a


def _step(make_model, mols, feats, loss_fn, seed=5, disturb=False):
    """One training step (forward, loss, backward, Adam) from the weights make_model() builds: (loss, scores, flat gradient, weights)."""
    torch.manual_seed(0)
    model = make_model().cuda(GPU).train()
    opt = build_optimizer(model)
    keep = _disturb() if disturb else None
    torch.manual_seed(seed)
    out = model(mols[0], mols[1], gpu=GPU, add_features=feats)
    loss = loss_fn(out)
    opt.zero_grad()
    loss.backward()
    grad = model._grad_flat.clone()
    opt.step()
    torch.cuda.synchronize()
    del keep
    return (loss.detach().clone(), out.detach().clone(), grad, torch.cat([p.detach().reshape(-1) for p in model.parameters()]))


def _three_equal(runs):
    for other in runs[1:]:
        for a, b, what in zip(runs[0], other, ("loss", "scores", "gradient", "weights")):
            assert torch.equal(a, b), f"{what} differs between two deterministic runs"


def _listwise(seed, sizes, task="mle"):
    ds = synthetic.make_dataset(seed, sizes)
    targets = torch.tensor(ds.lgk.astype(np.float32))
    mols = (BatchMolGraph([ds.mols[t] for t in ds.rsmi]), BatchMolGraph([ds.mols[t] for t in ds.psmi]))
    return mols, add_features(ds, 1), (lambda out: batch_loss(task, out, sizes, targets, GPU))


def _model(hidden=300, depth=3, dropout=0.1, task_num=1, last="with_softplus", task_type=None):
    return lambda: build_model(hidden_size=hidden, mpnn_depth=depth, mpnn_diff_depth=depth, ffn_depth=3, use_bias=True, dropout=dropout,
                               task_num=task_num, ffn_last_layer=last, task_type=task_type, add_features_dim=1)


def test_c5_step_is_bit_identical(gemm_mode):
    """The c5 batch (82 groups x 50 candidates, ListMLE h300 d3, dropout 0.1): loss, scores, gradient and Adam-updated weights of three
    steps from the same weights and seed are equal bit for bit, one of them with a second stream competing for the SMs."""
    torch.use_deterministic_algorithms(True)
    mols, feats, loss_fn = _listwise(4100, [50] * 82)
    runs = [_step(_model(), mols, feats, loss_fn, disturb=(i == 1)) for i in range(3)]
    _three_equal(runs)


@pytest.mark.parametrize("case", ["h1040_first_generation", "mp_v1", "backward_tf32", "evidential_ranking_h600"])
def test_other_paths_are_bit_identical(case, monkeypatch):
    """Hidden 1040 (the row pipeline refuses it: first-generation gathers), RR_MP_V1=1, the 3 x tf32 backward split (k_tc_wgrad2), and
    evidential_ranking at hidden 600."""
    torch.use_deterministic_algorithms(True)
    L = _lib.lib()
    make, task, hidden = _model(), "mle", 300
    if case == "h1040_first_generation":
        make = _model(hidden=1040, depth=2)
    elif case == "mp_v1":
        monkeypatch.setenv("RR_MP_V1", "1")
        L.rr_reload_switches()
    elif case == "backward_tf32":
        L.rr_set_backward_bf16(0)
    else:
        make, task = _model(hidden=600, task_num=2, task_type="evidential_ranking"), "evidential_ranking"
    mols, feats, loss_fn = _listwise(77, [40, 30, 50, 25], task)
    _three_equal([_step(make, mols, feats, loss_fn) for _ in range(3)])


def test_ranknet_window_of_64_segments_is_bit_identical():
    """A RankNet window of 64 groups as 64 segments of one launch: 128 padding rows in the joint encoder graph."""
    torch.use_deterministic_algorithms(True)
    sizes = [6, 9, 4, 7] * 16
    ds = synthetic.make_dataset(91, sizes)
    cuts = np.cumsum([0] + sizes)
    dev = torch.device("cuda", GPU)
    rg = DeviceGraph.from_batches([BatchMolGraph([ds.mols[t] for t in ds.rsmi[a:b]]) for a, b in zip(cuts[:-1], cuts[1:])], dev)
    pg = DeviceGraph.from_batches([BatchMolGraph([ds.mols[t] for t in ds.psmi[a:b]]) for a, b in zip(cuts[:-1], cuts[1:])], dev)
    targets = ds.lgk.astype(np.float32)
    pairs = sum(RL.count_ordered_pairs(targets[a:b]) for a, b in zip(cuts[:-1], cuts[1:]))
    loss_fn = lambda y: RL.ranknet_window_loss(y, sizes, targets, pairs, sigma=1.0, gpu=GPU)    # noqa: E731
    make = _model(dropout=0.2, last="no_softplus")
    _three_equal([_step(make, (rg, pg), ds.temp.reshape(-1, 1), loss_fn) for _ in range(3)])


def test_dropout_zero_training_encodes_every_reactant_copy():
    """At dropout 0 the default mode encodes each distinct reactant once and sums the gradient of its copies with atomics; deterministic
    training encodes every copy instead (same scores), and its steps repeat bit for bit."""
    from reactranker_b200.data.load_reactions import DataProcessor, Parsing_features
    ds = synthetic.make_dataset(3, [12] * 20)
    fz = Parsing_features(ds.mols)
    dp = DataProcessor(ds.to_dataframe())
    reactions, targets, scope, feats = next(iter(dp.generate_batch_reactions(smiles_list=["rsmi_mapped", "psmi_mapped"], target_name="lgk",
                                                                             batch_size=240, seed=0, add_features_name="temp")))
    r, p = fz.parsing_reactions(reactions)
    loss_fn = lambda out: RL.MLEloss()(out, scope, torch.FloatTensor(targets).squeeze(), GPU)     # noqa: E731
    make = _model(hidden=64, dropout=0.0)
    default = _step(make, (r, p), feats, loss_fn)
    torch.use_deterministic_algorithms(True)
    runs = [_step(make, (r, p), feats, loss_fn) for _ in range(3)]
    _three_equal(runs)
    assert torch.allclose(default[1], runs[0][1], rtol=1e-6, atol=0)     # de-duplication changes the work, not the scores


def test_eval_mode_backward_under_the_flag_encodes_every_reactant_copy():
    """In eval mode with autograd enabled a backward pass may follow, so under the flag the model does not de-duplicate reactants there
    either; under torch.no_grad() it still does (no backward can follow)."""
    from reactranker_b200.data.load_reactions import DataProcessor, Parsing_features
    ds = synthetic.make_dataset(3, [12] * 4)
    fz = Parsing_features(ds.mols)
    reactions, _, _, feats = next(iter(DataProcessor(ds.to_dataframe()).generate_batch_reactions(
        smiles_list=["rsmi_mapped", "psmi_mapped"], target_name="lgk", batch_size=48, seed=0, add_features_name="temp")))
    r, p = fz.parsing_reactions(reactions)
    model = _model(hidden=64, dropout=0.0)().cuda(GPU).eval()
    torch.use_deterministic_algorithms(True)
    out = model(r, p, gpu=GPU, add_features=feats)
    assert getattr(out.grad_fn.rg, "atom_map", None) is None
    out.sum().backward()
    with torch.no_grad():
        model(r, p, gpu=GPU, add_features=feats)


def _train_step_run(prepare_kind):
    """Two TrainStep steps (prepare_rows / prepare + run: forward, loss, backward, Adam) at dropout 0 from the same weights, the way
    train() drives them: (prepared reactant graph, loss, flat gradient, weights)."""
    from reactranker_b200.data.load_reactions import DataProcessor, Parsing_features
    from reactranker_b200.train.step import TrainStep
    from reactranker_b200.train.utils import build_lr_scheduler
    ds = synthetic.make_dataset(11, [12] * 20)
    fz = Parsing_features()
    for tok, m in ds.mols.items():
        fz.add(tok, m)
    dp = DataProcessor(ds.to_dataframe())
    torch.manual_seed(0)
    model = _model(hidden=64, dropout=0.0)().cuda(GPU).train()
    opt = build_optimizer(model)
    sched = build_lr_scheduler(opt, warmup_epochs=2, total_epochs=30, train_data_size=2400, batch_size=240, init_lr=1e-4, max_lr=1e-3,
                               final_lr=1e-4)
    step = TrainStep(model, opt, sched, "mle", GPU)
    cols = ["rsmi_mapped", "psmi_mapped"]
    if prepare_kind == "rows":
        rows, scope = next(iter(dp.plan_batch_reactions(batch_size=240, seed=0)))
        b = step.prepare_rows(dp, rows, scope, fz, cols, "lgk", "temp")
    else:
        batch = next(iter(dp.generate_batch_reactions(smiles_list=cols, target_name="lgk", batch_size=240, seed=0, add_features_name="temp")))
        b = step.prepare(batch, fz, device_graphs=True)
    loss = step.run(b).detach().clone()
    torch.cuda.synchronize()
    return b.r, loss, model._grad_flat.clone(), torch.cat([p.detach().reshape(-1) for p in model.parameters()])


@pytest.mark.parametrize("prepare_kind", ["rows", "batch"])
def test_train_step_at_dropout_zero_is_bit_identical(prepare_kind):
    """train()'s own step (TrainStep.prepare_rows, and TrainStep.prepare with device graphs) at dropout 0: the default mode encodes each
    distinct reactant once, deterministic mode every copy, and three deterministic steps give the same loss, gradient and weights."""
    r_default = _train_step_run(prepare_kind)[0]
    assert getattr(r_default, "atom_map", None) is not None          # the batch does repeat reactants: the default de-duplicates
    torch.use_deterministic_algorithms(True)
    runs = [_train_step_run(prepare_kind) for _ in range(3)]
    assert all(getattr(r[0], "atom_map", None) is None for r in runs)
    for other in runs[1:]:
        for a, b, what in zip(runs[0][1:], other[1:], ("loss", "gradient", "weights")):
            assert torch.equal(a, b), f"{what} differs between two deterministic steps"


def _wgrad(M, n, k, dZ, X):
    dW = torch.zeros(n, k, device="cuda")
    db = torch.zeros(n, device="cuda")
    _lib.check(_lib.lib().rr_linear_wgrad(M, n, k, dZ.data_ptr(), n, X.data_ptr(), k, dW.data_ptr(), k, db.data_ptr(), _lib.stream_ptr()))
    torch.cuda.synchronize()
    return dW, db


@pytest.mark.parametrize("mode", [0, 1], ids=["simt", "tc"])
def test_wgrad_kernel_is_bit_identical(mode):
    """rr_linear_wgrad at M = 160 000, n = k = 304 with a bias: three deterministic runs equal bit for bit, and within the kernel tests'
    fp64 tolerance (3e-6 on the exact-fp32 SIMT kernels, 2e-5 on the tensor cores' 3 x bf16 split)."""
    L = _lib.lib()
    L.rr_set_gemm_mode(mode)
    M, n, k = 160000, 304, 304
    g = torch.Generator(device="cuda").manual_seed(1)
    dZ = torch.randn(M, n, device="cuda", generator=g)
    X = torch.randn(M, k, device="cuda", generator=g)
    _lib.check(L.rr_set_deterministic(1))
    runs = [_wgrad(M, n, k, dZ, X) for _ in range(3)]
    for dW, db in runs[1:]:
        assert torch.equal(dW, runs[0][0]) and torch.equal(db, runs[0][1])
    want = dZ.double().t() @ X.double()
    err = float((runs[0][0].double() - want).abs().max() / want.abs().max())
    assert err < (3e-6 if mode == 0 else 2e-5), err
    want_b = dZ.double().sum(0)
    err_b = float((runs[0][1].double() - want_b).abs().max() / want_b.abs().max())
    assert err_b < (3e-6 if mode == 0 else 2e-5), err_b


def test_losses_are_bit_identical():
    """rr_loss_fwdbwd_ex of every kind at G = 4096 groups (NIG at N = 2048, all pairs): three deterministic runs equal bit for bit.  The
    kinds the fp64 oracle implements (ListMLE, ListNet, UC-Listwise, Gaussian NLL, MSE) match it within test_gpu_kernels.py's tolerances
    (loss 2e-6, dL/dscore 2e-5 of the largest value); the others agree with the default mode to 1e-4."""
    from oracle import reactranker_oracle as O
    oracle_task = {_lib.LOSS_LISTMLE: "mle", _lib.LOSS_LISTNET: "listnet", _lib.LOSS_EVIDENTIAL: "evidential_ranking",
                   _lib.LOSS_GAUSS: "gauss_regression", _lib.LOSS_MSE: "regression"}
    L = _lib.lib()
    G, n = 4096, 6
    N = G * n
    g = torch.Generator(device="cuda").manual_seed(2)
    seg = torch.arange(0, N + 1, n, dtype=torch.int32, device="cuda")
    targets = torch.randn(N, device="cuda", generator=g)
    pos = lambda *s: torch.rand(*s, device="cuda", generator=g) + 0.5    # noqa: E731
    cases = {
        _lib.LOSS_LISTMLE: (torch.randn(N, device="cuda", generator=g), G), _lib.LOSS_LISTNET: (torch.randn(N, device="cuda", generator=g), N),
        _lib.LOSS_EVIDENTIAL: (torch.stack([torch.randn(N, device="cuda", generator=g), pos(N)], 1), G),
        _lib.LOSS_RANKNET: (torch.randn(N, device="cuda", generator=g), 1000.0), _lib.LOSS_RANKNET_ACC: (torch.randn(N, device="cuda", generator=g), 1000.0),
        _lib.LOSS_GAUSS: (torch.stack([torch.randn(N, device="cuda", generator=g), pos(N)], 1), N), _lib.LOSS_MSE: (torch.randn(N, device="cuda", generator=g), N),
        _lib.LOSS_EXPMSE: (torch.randn(N, device="cuda", generator=g), N),
        _lib.LOSS_LISTMLE_DIS: (torch.stack([torch.randn(N, device="cuda", generator=g), pos(N)], 1), G),
        _lib.LOSS_LISTNET_DIS: (torch.stack([torch.randn(N, device="cuda", generator=g), pos(N)], 1), G),
        _lib.LOSS_LISTNET_UQ: (pos(N), G), _lib.LOSS_LOGNORM: (torch.stack([pos(N), pos(N)], 1), N), _lib.LOSS_DIRICHLET_UQ: (pos(N), G),
    }
    nig_n = 2048
    cases[_lib.LOSS_NIG] = (torch.stack([torch.randn(nig_n, device="cuda", generator=g), pos(nig_n), pos(nig_n) + 1.0, pos(nig_n)], 1), nig_n * nig_n)

    def run(kind, scores, norm):
        n_items = scores.shape[0]
        loss = torch.empty(1, device="cuda")
        d = torch.empty_like(scores)
        groups, seg_ptr = (0, None) if kind == _lib.LOSS_NIG else (G, seg.data_ptr())
        _lib.check(L.rr_loss_fwdbwd_ex(kind, n_items, groups, scores.data_ptr(), targets[:n_items].contiguous().data_ptr(), seg_ptr, n,
                                       float(norm), 0.5, loss.data_ptr(), d.data_ptr(), _lib.stream_ptr()))
        torch.cuda.synchronize()
        return loss.clone(), d.clone()

    for kind, (scores, norm) in cases.items():
        scores = scores.contiguous()
        L.rr_set_deterministic(0)
        ref = run(kind, scores, norm)
        _lib.check(L.rr_set_deterministic(1))
        runs = [run(kind, scores, norm) for _ in range(3)]
        for loss, d in runs[1:]:
            assert torch.equal(loss, runs[0][0]) and torch.equal(d, runs[0][1]), kind
        if kind in oracle_task:
            sx = scores.double().cpu().requires_grad_(True)
            want = O.loss_for_task(oracle_task[kind], sx, [n] * G, targets.double().cpu())
            want.backward(torch.ones_like(want))
            _close(runs[0][0], want.detach().reshape(1), 2e-6)
            _close(runs[0][1], sx.grad, 2e-5)
        else:
            assert torch.allclose(runs[0][0], ref[0], rtol=1e-4, atol=1e-6), (kind, runs[0][0], ref[0])
            assert torch.allclose(runs[0][1], ref[1], rtol=1e-4, atol=1e-7), kind


def _close(got, want, tol):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    err = float((got - want).abs().max()) / max(float(want.abs().max()), 1e-30)
    assert err < tol, err


@pytest.mark.parametrize("name", ["nobias", "depth2_diff4", "h1040", "tiny_mols"])
def test_configuration_parity_holds_in_deterministic_mode(name, gemm_mode):
    """The fp64-oracle parity of test_gpu_model.test_configuration_vs_fp64_oracle, with the same tolerances, in deterministic mode."""
    from test_gpu_model import test_configuration_vs_fp64_oracle as parity
    torch.use_deterministic_algorithms(True, warn_only=True)
    parity(name, gemm_mode)


def test_backward_refuses_a_workspace_sized_without_the_scratch():
    """A workspace sized with the switch off is too small for a deterministic backward: RR_ERR_WORKSPACE, and nothing is written."""
    L = _lib.lib()
    ds = synthetic.make_dataset(5, [8, 6, 7])
    model = _model(hidden=64, dropout=0.0)().cuda(GPU)
    r_g, p_g = BatchMolGraph([ds.mols[t] for t in ds.rsmi]), BatchMolGraph([ds.mols[t] for t in ds.psmi])
    out = model(r_g, p_g, gpu=GPU, add_features=ds.temp.reshape(-1, 1))
    node = out.grad_fn
    need = L.rr_model_workspace_bytes(ctypes.byref(node.cfg), ctypes.byref(node.rg.c), ctypes.byref(node.pg.c))
    ws = node.ws[:need]
    _lib.check(L.rr_set_deterministic(1))
    assert L.rr_model_workspace_bytes(ctypes.byref(node.cfg), ctypes.byref(node.rg.c), ctypes.byref(node.pg.c)) > need
    params = [p for _, p in model._named_slots()]
    w = model._param_struct(params)
    grads = [torch.full_like(p, 7.0) for p in params]
    gw = model._param_struct(grads)
    before = ws.clone()
    dscores = torch.ones_like(out)
    st = L.rr_model_backward(ctypes.byref(node.cfg), ctypes.byref(w), ctypes.byref(node.rg.c), ctypes.byref(node.pg.c), dscores.data_ptr(),
                             ctypes.byref(gw), ws.data_ptr(), need, _lib.stream_ptr())
    torch.cuda.synchronize()
    assert st == -5                                      # RR_ERR_WORKSPACE
    assert torch.equal(ws, before) and all(bool((t == 7.0).all()) for t in grads)


def _run(args):
    res = subprocess.run([sys.executable] + args, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    return [l for l in res.stdout.splitlines() if "full precision" in l or "train loss" in l]


def _state_dict(path):
    from reactranker_b200.utils import load_checkpoint
    return load_checkpoint(path)["state_dict"]


@pytest.mark.parametrize("script", ["main.py", "main.py-dropout0", "main_ranknet.py"])
def test_training_script_repeats_bit_for_bit(tmp_path, script):
    """`--deterministic`: two runs of three epochs (the Noam schedule warms up for two) log the same per-epoch losses and save
    bit-identical checkpoints; with dropout, and for main.py also at dropout 0, where the default mode would de-duplicate reactants."""
    if script.startswith("main.py"):
        args = ["main.py", "--synthetic", "40,10", "--gpu", "0", "--task_type", "mle", "--batch_size", "100", "--total_epochs", "3",
                "--hidden_size", "64", "--dropout", "0.0" if script.endswith("dropout0") else "0.1", "--deterministic"]
    else:
        args = ["main_ranknet.py", "--synthetic", "40,8", "--gpu", "0", "--batch_size", "64", "--total_epochs", "3", "--deterministic"]
    logs = [_run(args + ["--path", str(tmp_path / k)]) for k in "ab"]
    assert len(logs[0]) >= 3 and logs[0] == logs[1]
    ck = [os.path.join(root, f) for root, _, files in os.walk(str(tmp_path / "a")) for f in files if f.endswith(".pt")]
    assert ck
    for f in ck:
        a, b = _state_dict(f), _state_dict(f.replace(str(tmp_path / "a"), str(tmp_path / "b")))
        assert a.keys() == b.keys() and all(torch.equal(a[k], b[k]) for k in a)
