"""Parity against the LIVE reference, the original ReactRanker source (imported with rdkit stubbed, oracle/ref_loader.py; point
RR_REFERENCE_ROOT at a checkout of it), on freshly seeded inputs that the committed goldens do not contain.  Without that source the
whole module is skipped; the goldens under tests/golden/, generated from the reference by tests/golden/make_golden.py, carry the parity.

  * host logic of the PRODUCT (batch planners, BatchMolGraph tensors): bit-exact against the reference's own classes;
  * the ORACLE (model forward + every runnable task key's loss + gradients): against the reference's modules in fp64, so that the
    checker the GPU tests rely on is held to the reference on more than the golden cases.
"""
import contextlib
import io
import os
import sys

import numpy as np
import pytest
import torch

from oracle import ref_loader
from oracle import reactranker_oracle as O
from reactranker_b200 import synthetic

pytestmark = pytest.mark.skipif(not ref_loader.available(), reason="needs the original ReactRanker source (set RR_REFERENCE_ROOT)")
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
COLS = ["rsmi_mapped", "psmi_mapped"]


def _quiet():
    return contextlib.redirect_stdout(io.StringIO())


@pytest.mark.parametrize("seed", [101, 102, 103, 104])
def test_planners_bit_exact_on_fresh_frames(seed):
    """generate_batch_reactions (incl. truncation and tail yields), generate_batch_per_query, generate_batch_querys
    (load_reactions.py:235-421): same rows, same order, same scope, same targets / extra features, for random group sizes and seeds."""
    from reactranker_b200.data.load_reactions import DataProcessor
    lr = ref_loader.ref("data.load_reactions")
    rng = np.random.default_rng(seed)
    sizes = [int(x) for x in rng.integers(1, 28, size=int(rng.integers(5, 14)))]
    ds = synthetic.make_dataset(seed, sizes, atoms_lo=3, atoms_hi=4)
    df = ds.to_dataframe()
    ours, ref = DataProcessor(df), lr.DataProcessor(df)
    for batch_size in (int(rng.integers(2, 12)), int(rng.integers(12, 40)), 200):
        for epoch in (0, int(rng.integers(1, 50))):
            kw = dict(smiles_list=COLS, target_name="lgk", batch_size=batch_size, seed=epoch, add_features_name="temp")
            a, b = list(ours.generate_batch_reactions(**kw)), list(ref.generate_batch_reactions(**kw))
            assert len(a) == len(b)
            for (s1, t1, c1, f1), (s2, t2, c2, f2) in zip(a, b):
                assert np.array_equal(np.asarray(s1, dtype=object), np.asarray(s2, dtype=object)) and list(c1) == list(c2)
                assert np.array_equal(np.asarray(t1, np.float64), np.asarray(t2, np.float64))
                assert np.array_equal(np.asarray(f1, np.float64), np.asarray(f2, np.float64))
    for epoch in (0, 7):
        kw = dict(smiles_list=COLS, target_name="lgk", seed=epoch, add_features_name="temp")
        for (s1, t1, f1), (s2, t2, f2) in zip(ours.generate_batch_per_query(**kw), ref.generate_batch_per_query(**kw)):
            assert np.array_equal(np.asarray(s1, dtype=object), np.asarray(s2, dtype=object))
            assert np.array_equal(np.asarray(t1, np.float64).reshape(-1), np.asarray(t2, np.float64).reshape(-1))
            assert np.array_equal(np.asarray(f1, np.float64).reshape(-1), np.asarray(f2, np.float64).reshape(-1))
        kw = dict(smiles_list=COLS, target_name="lgk", batch_size=3, seed=epoch, add_features_name="temp", shuffle_query=False, shuffle_batch=False)
        a, b = list(ours.generate_batch_querys(**kw)), list(ref.generate_batch_querys(**kw))
        assert len(a) == len(b)
        for (s1, t1, c1, f1), (s2, t2, c2, f2) in zip(a, b):
            assert np.array_equal(np.asarray(s1, dtype=object), np.asarray(s2, dtype=object)) and list(c1) == list(c2)
            assert np.array_equal(np.asarray(t1, np.float64).reshape(-1), np.asarray(t2, np.float64).reshape(-1))


@pytest.mark.parametrize("seed,sizes,star", [(201, [4, 1, 6], None), (202, [3, 5], {1: 9}), (203, [1], None), (204, [2, 2, 2, 7], {3: 5})])
def test_batchmolgraph_bit_exact_on_fresh_batches(seed, sizes, star):
    """BatchMolGraph (featurization.py:246-329) of the product, host-packed and store-backed, against the reference's class."""
    from reactranker_b200.data.load_reactions import Parsing_features
    from reactranker_b200.features.featurization import BatchMolGraph
    ds = synthetic.make_dataset(seed, sizes, star_leaves_in_group=star)
    ref_fz = ref_loader.RefFeaturizer(ds.mols)
    fz = Parsing_features(ds.mols)
    for col in (ds.rsmi, ds.psmi):
        want = ref_fz.parsing_smiles(list(col))
        for got in (BatchMolGraph([ds.mols[t] for t in col]), fz.parsing_smiles(list(col))):
            fa, fb, a2b, b2a, b2revb, a_scope, b_scope = got.get_components()
            wa, wb, w2b, wb2a, wrev, wa_scope, wb_scope = want.get_components()
            assert torch.equal(fa, wa) and torch.equal(fb, wb)
            assert torch.equal(a2b.long(), w2b.long()) and torch.equal(b2a.long(), wb2a.long()) and torch.equal(b2revb.long(), wrev.long())
            assert list(a_scope) == list(wa_scope) and list(b_scope) == list(wb_scope)
            assert torch.equal(got.get_a2a().long(), want.get_a2a().long())
            assert (got.n_atoms, got.n_bonds, got.max_num_bonds) == (want.n_atoms, want.n_bonds, want.max_num_bonds)


def _tasks():
    import make_golden as MG
    return MG.TASKS_ALL


@pytest.mark.parametrize("task", ["mle", "listnet", "evidential_ranking", "gauss_regression", "regression", "mle_gaussian", "listnet_gauss",
                                  "mle_regression", "listnet_regression", "regression_exploss", "mledis_gaussian", "listnetdis_gauss",
                                  "listnet_uq", "listnetdis_lognorm", "dirichlet_uq", "evidential", "mle_evidential", "mledis_evidential",
                                  "listnet_evidential"])
def test_oracle_equals_live_reference_on_fresh_inputs(task):
    """Every runnable task key (train_listwise.py:196-285): the oracle's scores, loss and all gradients against the reference's own modules
    in fp64, on a model / batch the goldens do not hold (hidden 32, depth 4 / 2, ragged groups with a single-candidate group and a star)."""
    _oracle_vs_live_reference(task, 300 + len(task), 32, 4, 2)


@pytest.mark.parametrize("ffn_depth,use_bias,add", [(1, True, 1), (4, True, 3), (3, False, 0)], ids=["ffn1", "ffn4_add3", "nobias_add0"])
def test_oracle_equals_live_reference_at_other_configurations(ffn_depth, use_bias, add):
    """The same at FFN depth 1 and 4, without the W_i / W_h / FFN biases, and with 0 or 3 add features: the model configurations the GPU
    parity sweep (tests/test_gpu_model.py::test_configuration_vs_fp64_oracle) holds the kernels to the oracle at."""
    _oracle_vs_live_reference("mle", 350 + ffn_depth, 32, 3, 2, ffn_depth=ffn_depth, use_bias=use_bias, add=add)


def _oracle_vs_live_reference(task, seed, hidden, depth, ddepth, ffn_depth=3, use_bias=True, add=1):
    import make_golden as MG
    from helpers import add_features
    tn, last, tt = MG.TASKS_ALL[task]
    sizes, star = [4, 1, 7, 3], {2: 6}
    with _quiet():
        ds, model, scores, loss, grads = MG.run_case(task, hidden, seed, sizes, star, torch.float64, depth, ddepth, ffn_depth, use_bias, add)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items() if "cached_zero" not in k}
    full = dict(sd)
    full.update(params)
    r_g = O.OracleBatch([ds.mols[t] for t in ds.rsmi])
    p_g = O.OracleBatch([ds.mols[t] for t in ds.psmi])
    out = O.model_forward(full, r_g, p_g, add_features(ds, add), mpnn_depth=depth, mpnn_diff_depth=ddepth, ffn_depth=ffn_depth,
                          head=O.resolve_task_type(tn, last, tt))
    targets = torch.tensor(ds.lgk.astype(np.float32)).double()
    got_loss = O.loss_for_task(task, out, sizes, targets)
    got_loss.backward()
    assert tuple(out.shape) == tuple(scores.shape) and np.abs(out.detach().numpy() - scores).max() <= 1e-10 * max(1.0, np.abs(scores).max())
    # mle / evidential_ranking accumulate into an fp32 ``torch.Tensor([0])`` (loss.py:79, 493) even in an fp64 run
    tol = 2e-7 if np.asarray(loss).dtype == np.float32 else 1e-10
    assert tuple(got_loss.shape) == tuple(np.asarray(loss).shape)
    assert abs(float(got_loss.detach().reshape(-1)[0]) - float(np.asarray(loss).reshape(-1)[0])) <= tol * max(1.0, abs(float(np.asarray(loss).reshape(-1)[0])))
    gscale = max(float(np.abs(g).max()) for g in grads.values())
    for k, g in grads.items():
        assert np.abs(params[k].grad.numpy() - g).max() <= 1e-6 * gscale, k


@pytest.mark.parametrize("seed,quant", [(401, None), (402, 0.5), (403, 0.25), (404, None)])
def test_group_metrics_restatement_equals_live_reference(seed, quant):
    """oracle.group_metrics (the checker of the rr_rank_metrics kernel) against the reference's ranking_metrics and evaluate_top_scores
    (eval.py:475-555, 76-177) on fresh frames; ``quant`` coarsens the scorer so that groups contain exactly tied scores (stable order)."""
    import make_golden as MG
    lr = ref_loader.ref("data.load_reactions")
    ev = ref_loader.ref("train.eval")
    rng = np.random.default_rng(seed)
    sizes = [int(x) for x in rng.integers(1, 24, size=int(rng.integers(4, 12)))]
    ds = synthetic.make_dataset(seed, sizes, atoms_lo=3, atoms_hi=4)
    df = ds.to_dataframe()

    class Scorer(MG.StubScorer):
        def forward(self, r_inputs, p_inputs, gpu=None, add_features=None):
            s = super().forward(r_inputs, p_inputs, gpu, add_features)
            return torch.round(s / quant) * quant if quant else s

    class Feat:
        class B:
            def __init__(self, toks):
                self.smiles_batch = list(toks)

        def parsing_smiles(self, toks):
            return Feat.B(toks)

    m = Scorer(False).eval()
    dp = lr.DataProcessor(df)
    with _quiet():
        a, b, c = ev.evaluate_top_scores(m, gpu=None, data_processor=dp, smiles2graph_dic=Feat(), ratio=0.25, batch_size=3, smiles_list=COLS,
                                         target_name="lgk", add_features_name="temp")
        r = ev.ranking_metrics(m, gpu=None, data_processor=dp, smiles2graph_dic=Feat(), show_info=False, smiles_list=COLS, target_name="lgk",
                               add_features_name="temp")

    def score(X, feats):
        return m(None, Feat.B([s[1] for s in X]), add_features=feats).numpy()
    rows = []
    for X, t, scope, feats in dp.generate_batch_querys(smiles_list=COLS, target_name="lgk", batch_size=3, shuffle_query=False, shuffle_batch=False,
                                                       add_features_name="temp"):
        p, t, o = score(X, feats), np.asarray(t, np.float64).reshape(-1), 0
        for n in scope:
            rows.append(O.group_metrics(p[o:o + n], t[o:o + n], 0.25))
            o += n
    rows = np.asarray(rows)
    assert np.allclose([rows[:, 0].mean(), rows[:, 1].mean(), rows[:, 3].mean()], [a, b, c], rtol=0, atol=1e-12)
    rows = np.asarray([O.group_metrics(score(X, feats), np.asarray(t, np.float64).reshape(-1), 0.25)
                       for X, t, feats in dp.generate_batch_per_query(smiles_list=COLS, target_name="lgk", shuffle_query=False, shuffle_batch=False,
                                                                      add_features_name="temp")])
    got = [rows[:, 0].mean(), rows[:, 1].mean(), rows[:, 2].mean()] + list(rows[:, 4:8].mean(axis=0))
    assert np.allclose(got, [r[0], r[1], r[2]] + list(np.asarray(r[3], np.float64)), rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("algo", ["sum_session", "accelerate_grad"])
def test_oracle_ranknet_window_equals_live_reference_arithmetic(algo):
    """Both training_algo branches of factorized_training_loop (train_pairwise.py:98-152) on a fresh window: the reference's lines, run with
    the reference's model class, against the oracle's ranknet_group_cost / ranknet_group_lambda, in fp64."""
    import make_golden as MG
    sizes, star, seed = [3, 6, 2, 5], {1: 5}, 505
    ds, fz = MG.dataset_case(seed, sizes, star)
    model = MG.build_ref_model(32, 1, "no_softplus", None, seed=seed, depth=3, diff_depth=2, dtype=torch.float64).train()
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items() if "cached_zero" not in k}
    full = dict(sd)
    full.update(params)
    orig = torch.FloatTensor
    torch.FloatTensor = lambda x: torch.tensor(np.asarray(x, np.float32), dtype=torch.float64)  # type: ignore   (mpn.py:183 casts the extra feature)
    try:
        start, loss, pairs, ys, grads = 0, 0, 0, [], []
        for n in sizes:
            rows = slice(start, start + n)
            start += n
            r_g, p_g = fz.parsing_smiles(list(ds.rsmi[rows])), fz.parsing_smiles(list(ds.psmi[rows]))
            for g in (r_g, p_g):
                g.f_atoms, g.f_bonds = g.f_atoms.double(), g.f_bonds.double()
            Y = ds.lgk[rows].reshape(-1, 1)
            rel = Y - Y.T
            pos, neg = torch.tensor((rel > 0).astype(np.float64)), torch.tensor((rel < 0).astype(np.float64))
            y = model(r_g, p_g, gpu=None, add_features=ds.lgk[rows].reshape(-1, 1)).unsqueeze(1)
            if algo == "sum_session":                           # lines 119-122
                loss = loss + torch.sum(pos * torch.log(1 + torch.exp(-(y - y.t()))) + neg * torch.log(1 + torch.exp(y - y.t())), (0, 1))
            else:                                               # lines 123-137
                ys.append(y)
                with torch.no_grad():
                    l_pos, l_neg = 1 + torch.exp(y - y.t()), 1 + torch.exp(-(y - y.t()))
                    loss = loss + torch.sum(torch.log(l_neg) * pos + torch.log(l_pos) * neg, (0, 1))
                    grads.append(torch.sum(-pos / l_pos + neg / l_neg, dim=1, keepdim=True))
            pairs += 2 * float(pos.sum())
    finally:
        torch.FloatTensor = orig  # type: ignore
    model.zero_grad()
    if algo == "sum_session":
        (loss / pairs).backward()
    else:
        for g, y in zip(grads, ys):
            y.backward(g / pairs, retain_graph=True)
    want = {k: p.grad.numpy() for k, p in model.named_parameters() if p.grad is not None}
    start, total, opairs, lam, oys = 0, 0, 0.0, [], []
    for n in sizes:
        rows = slice(start, start + n)
        start += n
        y = O.model_forward(full, O.OracleBatch([ds.mols[t] for t in ds.rsmi[rows]]), O.OracleBatch([ds.mols[t] for t in ds.psmi[rows]]),
                            ds.lgk[rows].reshape(-1, 1), mpnn_depth=3, mpnn_diff_depth=2, head="no_softplus")
        if algo == "sum_session":
            c, npairs = O.ranknet_group_cost(y, ds.lgk[rows])
        else:
            c, l, npairs = O.ranknet_group_lambda(y, ds.lgk[rows])
            lam.append(l)
            oys.append(y)
        if c is not None:
            total, opairs = total + c, opairs + npairs
    assert opairs == pairs
    if algo == "sum_session":
        (total / opairs).backward()
    else:
        for l, y in zip(lam, oys):
            if l is not None:
                y.reshape(-1, 1).backward(l / opairs, retain_graph=True)
    assert abs(float((total / opairs).detach()) - float((loss / pairs).detach())) <= 1e-12
    gscale = max(float(np.abs(g).max()) for g in want.values())
    for k, g in want.items():
        assert np.abs(params[k].grad.numpy() - g).max() <= 1e-10 * gscale, k


@pytest.mark.parametrize("seed,two", [(601, False), (602, True), (603, True)])
def test_calculate_ndcg_equals_live_reference(seed, two):
    """The test-report routine calculate_ndcg (eval.py:329-457; host arithmetic in the product too): NDCG / KL means, the per-item order
    table and the re-ordered tokens against the reference's function on fresh frames, raw and de-normalised, ordered and unordered."""
    import make_golden as MG
    from reactranker_b200.data.load_reactions import DataProcessor, Parsing_features
    from reactranker_b200.train import eval as E
    lr = ref_loader.ref("data.load_reactions")
    ev = ref_loader.ref("train.eval")
    rng = np.random.default_rng(seed)
    sizes = [int(x) for x in rng.integers(2, 15, size=int(rng.integers(3, 9)))]
    ds = synthetic.make_dataset(seed, sizes, atoms_lo=3, atoms_hi=4)
    df = ds.to_dataframe()

    class Feat:
        class B:
            def __init__(self, toks):
                self.smiles_batch = list(toks)

        def parsing_smiles(self, toks):
            return Feat.B(toks)

    m = MG.StubScorer(two).eval()
    fz = Parsing_features(ds.mols)
    for means, stds, cut in ((None, None, 0.5), (0.3, 2.5, 0.25)):
        kw = dict(batch_size=int(rng.integers(1, 5)), NDCG_cut=cut, smiles_list=COLS, target_name="lgk", means=means, stds=stds, add_features_name="temp")
        with _quiet():
            want = ev.calculate_ndcg(m, gpu=None, data_processor=lr.DataProcessor(df), smiles2graph_dic=Feat(), **kw)
            got = E.calculate_ndcg(m, gpu=None, data_processor=DataProcessor(df), smiles2graph_dic=fz, **kw)
        assert np.allclose([got[0], got[1]], [want[0], want[1]], rtol=1e-6)
        assert np.allclose(np.asarray(got[2], np.float64), np.asarray(want[2], np.float64), rtol=1e-6, atol=1e-6)
        assert [list(x) for x in got[3]] == [list(x) for x in want[3]]
    with _quiet():
        want = ev.calculate_ndcg(m, gpu=None, data_processor=lr.DataProcessor(df), smiles2graph_dic=Feat(), batch_size=2, smiles_list=COLS, target_name="lgk",
                                 is_order=False, add_features_name="temp")
        got = E.calculate_ndcg(m, gpu=None, data_processor=DataProcessor(df), smiles2graph_dic=fz, batch_size=2, smiles_list=COLS, target_name="lgk",
                               is_order=False, add_features_name="temp")
    assert got[0] is None and got[1] is None and want[0] is None
    assert np.allclose(np.asarray(got[2], np.float64), np.asarray(want[2], np.float64), rtol=1e-6, atol=1e-6) and [list(x) for x in got[3]] == [list(x) for x in want[3]]


@pytest.mark.parametrize("target_name", ["lgk", "ea", "lgk_bi"])
@pytest.mark.parametrize("normalize_target", [True, False, 2.5, "1,7"])
@pytest.mark.parametrize("save_metric", ["all", "NDCG@2"])
def test_target_normalisation_equals_live_reference_train(monkeypatch, target_name, normalize_target, save_metric):
    """The target transform at the top of train() (train_listwise.py:66-124: sign flip for everything but lgk / lgk_bi, z-score / float
    scale / "lo,hi" range, raw validation targets for the NDCG save metrics) against the reference's own train(), stopped where it hands
    the two frames to its DataProcessor."""
    import logging
    from reactranker_b200.train.train_listwise import NDCG_METRICS, normalized_targets
    tl = ref_loader.ref("train.train_listwise")
    ds = synthetic.make_dataset(701, [4, 3, 5, 2], atoms_lo=3, atoms_hi=4)
    df = ds.to_dataframe()
    df["ea"] = df["lgk"] * 3.0 + 11.0
    df["lgk_bi"] = (df["lgk"] > 0).astype(np.float64)
    train_df, val_df = df.iloc[:9].reset_index(drop=True), df.iloc[9:].reset_index(drop=True)
    frames = []

    class Stop(Exception):
        pass

    class Capture:
        def __init__(self, frame):
            frames.append(frame.copy())
            if len(frames) == 2:
                raise Stop()

    monkeypatch.setattr(tl, "DataProcessor", Capture)
    with _quiet(), pytest.raises(Stop):
        tl.train(torch.nn.Linear(1, 1), None, train_df, val_df, "unused", None, 1, None, 4, 0, None, task_type="mle", writer=None,
                 logger=logging.getLogger("live"), target_name=target_name, smiles_list=COLS, save_metric=save_metric,
                 normalize_target=normalize_target)
    t_std, v_std, mean, std = normalized_targets(train_df[target_name], val_df[target_name], target_name, normalize_target)
    assert np.allclose(np.asarray(t_std, np.float64), frames[0]["std" + target_name].to_numpy(np.float64), rtol=0, atol=1e-15)
    want_val = val_df[target_name] if save_metric in NDCG_METRICS else v_std
    assert np.allclose(np.asarray(want_val, np.float64), frames[1]["std" + target_name].to_numpy(np.float64), rtol=0, atol=1e-15)
    assert mean == train_df[target_name].mean() and std == train_df[target_name].std(ddof=0)


@pytest.mark.parametrize("cfg", [dict(warmup_epochs=2, total_epochs=30, train_data_size=4100, batch_size=410, init_lr=1e-4, max_lr=1e-3, final_lr=1e-4),
                                 dict(warmup_epochs=1, total_epochs=3, train_data_size=57, batch_size=10, init_lr=3e-5, max_lr=2e-3, final_lr=5e-6),
                                 dict(warmup_epochs=2.5, total_epochs=8, train_data_size=1000, batch_size=64, init_lr=1e-4, max_lr=1e-3, final_lr=1e-4)])
def test_noam_schedule_and_optimizer_equal_live_reference(cfg):
    """build_optimizer / build_lr_scheduler / NoamLR (train/utils.py:7-133): the learning rate written into the optimizer at every step of
    a whole run, past total_steps too, and Adam's hyper-parameters."""
    from reactranker_b200.train.utils import build_lr_scheduler, build_optimizer
    ru = ref_loader.ref("train.utils")
    m1, m2 = torch.nn.Linear(3, 2), torch.nn.Linear(3, 2)
    o1, o2 = build_optimizer(m1), ru.build_optimizer(m2)
    g1, g2 = o1.param_groups[0], o2.param_groups[0]
    assert (g1["lr"], g1["betas"], g1["eps"], g1["weight_decay"], g1["amsgrad"]) == (g2["lr"], g2["betas"], g2["eps"], g2["weight_decay"], g2["amsgrad"])
    s1, s2 = build_lr_scheduler(o1, **cfg), ru.build_lr_scheduler(o2, **cfg)
    steps = int(cfg["total_epochs"] * (cfg["train_data_size"] // cfg["batch_size"])) + 5
    for _ in range(steps):
        assert o1.param_groups[0]["lr"] == o2.param_groups[0]["lr"]
        s1.step()
        s2.step()
    assert o1.param_groups[0]["lr"] == o2.param_groups[0]["lr"] == cfg["final_lr"]


def test_checkpoints_cross_load_with_the_reference(tmp_path):
    """save_checkpoint (utils.py:152-173): a file written here is read by the reference's loader lines (test_listwise.py:27-38:
    ``torch.load(path, map_location=...)`` then ``['state_dict']`` / ``['data_scaler']``), and a file written by the reference's function
    (numpy-scalar means / stds) is read by load_checkpoint.  A resumable state file reads like a plain checkpoint on the reference's side."""
    from reactranker_b200.utils import load_checkpoint, save_checkpoint, save_train_state
    from reactranker_b200.train.utils import build_lr_scheduler, build_optimizer
    ref_utils = ref_loader.ref("utils")
    torch.manual_seed(1)
    model = torch.nn.Linear(4, 3)
    mean, std = np.float64(1.25), np.float64(0.5)
    ours, theirs, state = str(tmp_path / "ours.pt"), str(tmp_path / "theirs.pt"), str(tmp_path / "state.pt")
    save_checkpoint(ours, model, mean, std)
    ref_utils.save_checkpoint(theirs, model, mean, std)
    opt = build_optimizer(model)
    save_train_state(state, model, opt, build_lr_scheduler(opt, 1, 2, 20, 5, 1e-4, 1e-3, 1e-4), epoch=0, means=mean, stds=std, best=0.5)
    for path in (ours, state):
        got = torch.load(path, map_location=lambda storage, loc: storage)          # the reference's loader line, torch >= 2.6 defaults
        assert got["data_scaler"] == {"means": 1.25, "stds": 0.5}
        assert all(torch.equal(v, model.state_dict()[k]) for k, v in got["state_dict"].items())
    got = load_checkpoint(theirs)
    assert float(got["data_scaler"]["means"]) == 1.25 and float(got["data_scaler"]["stds"]) == 0.5
    assert all(torch.equal(v, model.state_dict()[k]) for k, v in got["state_dict"].items())


# ---- the drop-in boundary (SURVEY.md 8b): same public callables, same signatures ------------------------------------------------------
# (reference module, attribute path); compared against the same path under this repo's ``reactranker`` import names
_PUBLIC = [
    ("models.base_model", "build_model"), ("models.base_model", "ReactionModel.__init__"), ("models.base_model", "ReactionModel.forward"),
    ("models.base_model", "FFN.__init__"), ("models.mpn", "MPN.__init__"), ("models.mpn", "MPNDiff.__init__"),
    ("train.train_listwise", "train"), ("train.run_train_pairwise", "run_train"), ("train.train_pairwise", "factorized_training_loop"),
    ("train.test_listwise", "test"), ("train.test_ranknet", "test"),
    ("train.utils", "build_optimizer"), ("train.utils", "build_lr_scheduler"), ("train.utils", "NoamLR.__init__"), ("train.utils", "NoamLR.step"),
    ("utils", "save_checkpoint"), ("utils", "index_select_ND"),
    ("train.loss", "MLEloss.forward"), ("train.loss", "ListnetLoss.forward"), ("train.loss", "evidential_ranking.forward"),
    ("train.loss", "GaussDisLoss.forward"), ("train.loss", "MLEDisLoss.forward"), ("train.loss", "Listnet_For_Gauss.forward"),
    ("train.loss", "Listnet_with_uq.forward"), ("train.loss", "Dirichlet_uq.forward"), ("train.loss", "Lognorm.forward"),
    ("train.loss", "evidential_loss_new"),
    ("train.eval", "evaluate_top_scores"), ("train.eval", "ranking_metrics"), ("train.eval", "calculate_ndcg"), ("train.eval", "calculate_mse"),
    ("data.load_reactions", "get_data.__init__"), ("data.load_reactions", "get_data.filter_bacth"), ("data.load_reactions", "get_data.split_data"),
    ("data.load_reactions", "DataProcessor.__init__"), ("data.load_reactions", "DataProcessor.generate_batch_reactions"),
    ("data.load_reactions", "DataProcessor.generate_batch_per_query"), ("data.load_reactions", "DataProcessor.generate_batch_querys"),
    ("data.load_reactions", "Parsing_features.parsing_smiles"), ("data.load_reactions", "Parsing_features.parsing_reactions"),
    ("features.featurization", "MolGraph.__init__"), ("features.featurization", "BatchMolGraph.__init__"),
    ("features.featurization", "BatchMolGraph.get_components"), ("features.featurization", "BatchMolGraph.get_a2a"),
    ("features.featurization", "mol2graph"),
]
# Deliberate, documented extensions: extra TRAILING keyword parameters with defaults that keep every reference call valid.
_EXTENSIONS = {
    ("train.train_listwise", "train"): ["resume_path"],                      # DESIGN.md 7.2: full-state resume (the reference saves weights only)
    ("train.run_train_pairwise", "run_train"): ["resume_path"],
    ("train.eval", "calculate_mse"): ["add_features_name"],                  # the reference's version cannot run (SURVEY.md appendix A.10)
}


def _resolve(mod, path):
    obj = mod
    for part in path.split("."):
        obj = getattr(obj, part)
    return obj


@pytest.mark.parametrize("module,path", _PUBLIC, ids=[f"{m}:{p}" for m, p in _PUBLIC])
def test_public_signatures_equal_the_reference(module, path):
    """inspect.signature of every public callable on the path: same parameter names, order, kinds and defaults as the live reference
    (type annotations are not part of the contract); the only differences allowed are the trailing defaulted parameters of _EXTENSIONS."""
    import importlib
    import inspect
    ref_obj = _resolve(ref_loader.ref(module), path)
    our_obj = _resolve(importlib.import_module("reactranker." + module), path)
    rp = list(inspect.signature(ref_obj).parameters.values())
    op = list(inspect.signature(our_obj).parameters.values())
    extra = _EXTENSIONS.get((module, path), [])
    assert [p.name for p in op[len(rp):]] == extra, ([p.name for p in op], [p.name for p in rp])
    assert all(p.default is not inspect.Parameter.empty for p in op[len(rp):])

    def same_default(a, b):
        if a is inspect.Parameter.empty or b is inspect.Parameter.empty:
            return a is b
        if inspect.isclass(a) or inspect.isclass(b):               # e.g. writer=SummaryWriter: the class object of whichever tensorboard is installed
            return getattr(a, "__name__", a) == getattr(b, "__name__", b)
        return a == b
    for a, b in zip(op, rp):
        assert a.name == b.name and a.kind == b.kind and same_default(a.default, b.default), (path, str(a), str(b))
