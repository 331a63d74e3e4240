#!/usr/bin/env python
"""Generate ``tests/golden/*.npz`` by EXECUTING THE REAL REFERENCE (``/root/reference``,
rdkit stubbed) on synthetic MolGraphs.  Run in the build container only:

    python tests/golden/make_golden.py

The GPU box has no ``/root/reference``; the parity tests there read these files.
Nothing here is product code.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import ref_loader  # noqa: E402
from reactranker_b200 import synthetic  # noqa: E402
from helpers import add_features  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
os.makedirs(OUT, exist_ok=True)


def np_sd(sd):
    return {k: v.detach().cpu().numpy().copy() for k, v in sd.items()}   # copy: Adam updates in place


def build_ref_model(hidden, task_num, ffn_last_layer, task_type, seed, depth=3, diff_depth=3, dropout=0.0, dtype=torch.float32,
                    ffn_depth=3, use_bias=True, add_features_dim=1):
    bm = ref_loader.ref("models.base_model")
    torch.manual_seed(seed)
    model = bm.build_model(hidden_size=hidden, mpnn_depth=depth, mpnn_diff_depth=diff_depth, ffn_depth=ffn_depth,
                           use_bias=use_bias, dropout=dropout, task_num=task_num, ffn_last_layer=ffn_last_layer,
                           task_type=task_type, add_features_dim=add_features_dim)
    return model.to(dtype)


TASKS = {
    # key: (task_num, ffn_last_layer, build_model task_type)
    "mle": (1, "with_softplus", None),
    "listnet": (1, "with_softplus", None),
    "evidential_ranking": (2, "with_softplus", "evidential_ranking"),
    "gauss_regression": (2, "with_softplus", None),
    "regression": (1, "with_softplus", None),
}
# composite keys of train_listwise.py:196-285 whose terms are the losses above (golden_composite)
COMPOSITE = {
    "mle_gaussian": (2, "with_softplus", None),
    "listnet_gauss": (2, "with_softplus", None),
    "mle_regression": (1, "with_softplus", None),
    "listnet_regression": (1, "with_softplus", None),
    "regression_exploss": (1, "with_softplus", None),
    "mledis_gaussian": (2, "with_softplus", None),
    "listnetdis_gauss": (2, "with_softplus", None),
    "listnet_uq": (1, "with_softplus", "listnet"),          # positive scores: build_model -> 'listnet_with_softplus' head
    "listnetdis_lognorm": (2, "with_softplus", "listnetdis_lognorm"),
    "dirichlet_uq": (1, "with_uncertainty", "listnet"),     # -> 'listnet_with_uncertainty' head: softplus + 1
    "evidential": (4, "with_softplus", None),               # -> 'evidential_with_softplus': the NIG head
    "mle_evidential": (4, "with_softplus", None),
    "mledis_evidential": (4, "with_softplus", None),
    "listnet_evidential": (4, "with_softplus", None),
}
TASKS_ALL = dict(TASKS, **COMPOSITE)


def ref_loss(task, out, scope, targets):
    L = ref_loader.ref("train.loss")
    if task == "mle":
        return L.MLEloss()(out, scope, targets, None)
    if task == "listnet":
        return L.ListnetLoss()(out, scope, targets, None)
    if task == "evidential_ranking":
        return L.evidential_ranking()(out, scope, targets, 0.0001, 0, 1, None)
    if task == "gauss_regression":
        return L.GaussDisLoss()(out[:, 0], out[:, 1], targets, None)
    if task == "mle_gaussian":            # train_listwise.py:204-207
        return L.MLEloss()(out[:, 0], scope, targets, None) + L.GaussDisLoss()(out[:, 0], out[:, 1], targets, None)
    if task == "listnet_gauss":           # 208-210
        return L.ListnetLoss()(out[:, 0], scope, targets, None) + L.GaussDisLoss()(out[:, 0], out[:, 1], targets, None)
    if task == "mle_regression":          # 263-266
        return torch.nn.MSELoss()(out, targets) + L.MLEloss()(out, scope, targets, None)
    if task == "listnet_regression":      # 224-227
        return L.ListnetLoss()(out, scope, targets, None) + torch.nn.MSELoss()(out, targets)
    if task == "regression_exploss":      # 276-281
        return torch.mean((torch.exp(targets) - torch.exp(out)) ** 2)
    if task == "mledis_gaussian":         # 196-203
        mu = out[:, [j for j in range(len(out[0])) if j % 2 == 0]]
        variance = torch.exp(out[:, [j for j in range(len(out[0])) if j % 2 == 1]])
        return L.MLEDisLoss()(mu, variance, scope, targets, None) + L.GaussDisLoss()(out[:, 0], out[:, 1], targets, None)
    if task == "listnet_uq":              # 228-229, in the middle of the annealing schedule
        return L.Listnet_with_uq()(out, scope, targets, 0.05, 3, 5, None)
    if task == "listnetdis_lognorm":      # 215-219 (Lognorm prints its value; silenced by the caller)
        return L.Lognorm()(out[:, 0], out[:, 1], targets, None)
    if task == "dirichlet_uq":            # 269-270
        return L.Dirichlet_uq()(out, scope, targets, 0.05, 3, 5, None)
    if task in ("evidential", "mle_evidential", "mledis_evidential", "listnet_evidential"):     # 229-260, slices exactly as written there
        mu = out[:, [j for j in range(len(out[0])) if j % 4 == 0]]
        lambdas = out[:, [j for j in range(len(out[0])) if j % 4 == 1]]
        alphas = out[:, [j for j in range(len(out[0])) if j % 4 == 2]]
        betas = out[:, [j for j in range(len(out[0])) if j % 4 == 3]]
        if task == "evidential":
            return L.evidential_loss_new(mu, lambdas, alphas, betas, targets, None, lam=0.1)
        if task == "mle_evidential":
            return L.MLEloss()(out[:, 0], scope, targets, None) + L.evidential_loss_new(mu, lambdas, alphas, betas, targets, None, lam=0.2)
        variance = betas / (lambdas * (alphas - 1))
        rank = L.MLEDisLoss() if task == "mledis_evidential" else L.Listnet_For_Gauss()     # 138-139, 144-145
        return rank(mu, variance, scope, targets, None) + L.evidential_loss_new(mu, lambdas, alphas, betas, targets, None, lam=0.1)
    if task == "listnetdis_gauss":        # 211-215
        mu = out[:, [j for j in range(len(out[0])) if j % 2 == 0]]
        variance = out[:, [j for j in range(len(out[0])) if j % 2 == 1]]
        return L.Listnet_For_Gauss()(mu, variance, scope, targets, None) + L.GaussDisLoss()(out[:, 0], out[:, 1], targets, None)
    return torch.nn.MSELoss()(out, targets)


def dataset_case(seed, group_sizes, star=None):
    ds = synthetic.make_dataset(seed, group_sizes, star_leaves_in_group=star)
    return ds, ref_loader.RefFeaturizer(ds.mols)


def golden_batching():
    """BatchMolGraph tensors (featurization.py:246-329) for two small batches."""
    out = {}
    for name, seed, sizes, star in (("plain", 11, [3, 2], None), ("star", 12, [2, 3], {1: 7})):
        ds, fz = dataset_case(seed, sizes, star)
        for side, col in (("r", ds.rsmi), ("p", ds.psmi)):
            g = fz.parsing_smiles(list(col))
            fa, fb, a2b, b2a, b2revb, a_scope, b_scope = g.get_components()
            pre = f"{name}.{side}."
            out[pre + "f_atoms"] = fa.numpy()
            out[pre + "f_bonds"] = fb.numpy()
            out[pre + "a2b"] = a2b.numpy()
            out[pre + "b2a"] = b2a.numpy()
            out[pre + "b2revb"] = b2revb.numpy()
            out[pre + "a2a"] = g.get_a2a().numpy()
            out[pre + "a_scope"] = np.asarray(a_scope, np.int64)
            out[pre + "b_scope"] = np.asarray(b_scope, np.int64)
            out[pre + "max_num_bonds"] = np.int64(g.max_num_bonds)
        out[f"{name}.seed"] = np.int64(seed)
        out[f"{name}.sizes"] = np.asarray(sizes, np.int64)
        out[f"{name}.star"] = np.asarray([[k, v] for k, v in (star or {}).items()], np.int64).reshape(-1, 2)
    np.savez_compressed(os.path.join(OUT, "batching.npz"), **out)
    print("batching.npz", len(out))


def golden_planner():
    """Row ids + scope per step of generate_batch_reactions / generate_batch_per_query
    (load_reactions.py:235-273, 336-421) for several seeds, incl. the truncation branch."""
    lr = ref_loader.ref("data.load_reactions")
    sizes = [20, 7, 13, 20, 5, 31, 20, 9, 20, 16, 2, 20]
    ds = synthetic.make_dataset(21, sizes, atoms_lo=3, atoms_hi=4)
    df = ds.to_dataframe()
    row_of = {p: i for i, p in enumerate(ds.psmi)}
    out = {"sizes": np.asarray(sizes, np.int64), "seed": np.int64(21)}
    dp = lr.DataProcessor(df)
    for batch_size in (50, 24, 64):
        for seed in (0, 1, 5):
            rows, scopes, steps = [], [], []
            for smiles, targets, scope, feats in dp.generate_batch_reactions(
                    smiles_list=["rsmi_mapped", "psmi_mapped"], target_name="lgk", batch_size=batch_size,
                    seed=seed, add_features_name="temp"):
                ids = [row_of[s[1]] for s in smiles]
                assert np.allclose(targets[:, 0], ds.lgk[ids]) and np.allclose(feats[:, 0], ds.temp[ids])
                rows += ids
                scopes += list(scope)
                steps.append((len(ids), len(scope)))
            key = f"reactions.bs{batch_size}.seed{seed}."
            out[key + "rows"] = np.asarray(rows, np.int64)
            out[key + "scope"] = np.asarray(scopes, np.int64)
            out[key + "steps"] = np.asarray(steps, np.int64)
    for seed in (0, 3):
        rows, lens, featcheck = [], [], []
        for smiles, targets, feats in dp.generate_batch_per_query(
                smiles_list=["rsmi_mapped", "psmi_mapped"], target_name="lgk", seed=seed, add_features_name="temp"):
            ids = [row_of[s[1]] for s in smiles]
            rows += ids
            lens.append(len(ids))
            featcheck.append(np.allclose(feats[:, 0], ds.lgk[ids]))     # the target-column leak (line 264-267)
        assert all(featcheck)
        out[f"per_query.seed{seed}.rows"] = np.asarray(rows, np.int64)
        out[f"per_query.seed{seed}.lens"] = np.asarray(lens, np.int64)
    np.savez_compressed(os.path.join(OUT, "planner.npz"), **out)
    print("planner.npz", len(out))


def run_case(task, hidden, seed, sizes, star, dtype, depth=3, diff_depth=3, ffn_depth=3, use_bias=True, add_features_dim=1):
    """The reference's forward, loss and backward on a synthetic batch.  The add features are the temperature column and, beyond the
    first, seeded normal columns (helpers.add_features); none for add_features_dim = 0."""
    ds, fz = dataset_case(seed, sizes, star)
    tn, last, tt = TASKS_ALL[task]
    model = build_ref_model(hidden, tn, last, tt, seed=seed, depth=depth, diff_depth=diff_depth, dtype=dtype, ffn_depth=ffn_depth,
                            use_bias=use_bias, add_features_dim=add_features_dim)
    model.train()
    reactions = np.stack([ds.rsmi, ds.psmi], axis=1)
    r_g, p_g = fz.parsing_reactions(reactions)
    for g in (r_g, p_g):                     # let the reference run in fp64 too
        g.f_atoms, g.f_bonds = g.f_atoms.to(dtype), g.f_bonds.to(dtype)
    feats = add_features(ds, add_features_dim)
    if dtype == torch.float64:
        # mpn.py:183 casts add_features with FloatTensor (fp32); lift the result to fp64
        orig = torch.FloatTensor
        torch.FloatTensor = lambda x: torch.tensor(np.asarray(x, np.float32), dtype=torch.float64)  # type: ignore
    import contextlib
    import io
    try:
        with contextlib.redirect_stdout(io.StringIO()):            # base_model.py:90 prints the whole output of the lognorm head
            out = model(r_g, p_g, gpu=None, add_features=feats)
    finally:
        if dtype == torch.float64:
            torch.FloatTensor = orig  # type: ignore
    targets = torch.tensor(ds.lgk.astype(np.float32)).to(dtype)     # train_listwise.py:187 FloatTensor(...).squeeze()
    with contextlib.redirect_stdout(io.StringIO()):
        loss = ref_loss(task, out, list(sizes), targets)
    model.zero_grad()
    loss.backward()
    grads = {k: p.grad.detach().numpy() for k, p in model.named_parameters() if p.grad is not None}
    return ds, model, out.detach().numpy(), loss.detach().numpy(), grads


def golden_model():
    cases = []
    for task in TASKS:
        cases.append((f"{task}.h40", task, 40, 31, [5, 3, 6], None, 3, 3))
    cases.append(("mle.star.h40", "mle", 40, 32, [4, 4], {0: 7}, 3, 3))          # padding-row trap
    cases.append(("evidential_ranking.h24d5", "evidential_ranking", 24, 33, [6, 4], None, 5, 5))
    cases.append(("mle.h300", "mle", 300, 34, [4, 3], None, 3, 3))
    out = {}
    for name, task, hidden, seed, sizes, star, depth, ddepth in cases:
        for dtype, tag in ((torch.float32, "f32"), (torch.float64, "f64")):
            ds, model, scores, loss, grads = run_case(task, hidden, seed, sizes, star, dtype, depth, ddepth)
            pre = f"{name}.{tag}."
            out[pre + "scores"] = scores
            out[pre + "loss"] = loss
            big = hidden >= 128
            for k, v in grads.items():
                if big and v.size > 4096:
                    out[pre + "gradsum." + k] = np.asarray([v.sum(dtype=np.float64), np.abs(v).sum(dtype=np.float64),
                                                            (v.astype(np.float64) ** 2).sum()])
                else:
                    out[pre + "grad." + k] = v
            if tag == "f32" and not big:
                for k, v in np_sd(model.state_dict()).items():
                    out[f"{name}.sd.{k}"] = v
        out[name + ".meta"] = np.asarray([hidden, seed, depth, ddepth], np.int64)
        out[name + ".sizes"] = np.asarray(sizes, np.int64)
        out[name + ".star"] = np.asarray([[k, v] for k, v in (star or {}).items()], np.int64).reshape(-1, 2)
        out[name + ".task"] = np.asarray(task)
        print(name, "loss", out[name + ".f32.loss"], out[name + ".f64.loss"])
    np.savez_compressed(os.path.join(OUT, "model.npz"), **out)
    print("model.npz", len(out))


def golden_composite():
    """The composite task keys (sums of the built losses, train_listwise.py:196-285) at hidden 40: scores, loss, all gradients."""
    out = {}
    for task in COMPOSITE:
        name = f"{task}.h40"
        for dtype, tag in ((torch.float32, "f32"), (torch.float64, "f64")):
            ds, model, scores, loss, grads = run_case(task, 40, 41, [5, 3, 6], None, dtype, 3, 3)
            pre = f"{name}.{tag}."
            out[pre + "scores"] = scores
            out[pre + "loss"] = loss
            for k, v in grads.items():
                out[pre + "grad." + k] = v
            if tag == "f32":
                for k, v in np_sd(model.state_dict()).items():
                    out[f"{name}.sd.{k}"] = v
        out[name + ".meta"] = np.asarray([40, 41, 3, 3], np.int64)
        out[name + ".sizes"] = np.asarray([5, 3, 6], np.int64)
        out[name + ".star"] = np.zeros((0, 2), np.int64)
        out[name + ".task"] = np.asarray(task)
        print(name, "loss", out[name + ".f32.loss"], out[name + ".f64.loss"])
    np.savez_compressed(os.path.join(OUT, "model_composite.npz"), **out)
    print("model_composite.npz", len(out))


def golden_ranknet():
    """factorized_training_loop 'sum_session' (train_pairwise.py:81-173): accumulated loss /
    pairs over a window of groups, each group its OWN forward (own max_num_bonds), grads."""
    out = {}
    sizes, star = [5, 4, 6], {1: 6}
    for dtype, tag in ((torch.float32, "f32"), (torch.float64, "f64")):
        ds, fz = dataset_case(41, sizes, star)
        torch.manual_seed(41)
        bm = ref_loader.ref("models.base_model")
        model = bm.build_model(hidden_size=40, mpnn_depth=3, mpnn_diff_depth=3, ffn_depth=3, use_bias=True, dropout=0.0,
                               task_num=1, ffn_last_layer="no_softplus", add_features_dim=1).to(dtype)
        model.train()
        start, loss, pairs = 0, 0, 0
        scores = []
        acc_loss, grad_batch, y_pred_batch = 0, [], []       # 'accelerate_grad' state of the same window (train_pairwise.py:86, 123-137)
        for n in sizes:
            rows = slice(start, start + n)
            start += n
            r_g = fz.parsing_smiles(list(ds.rsmi[rows]))
            p_g = fz.parsing_smiles(list(ds.psmi[rows]))
            for g in (r_g, p_g):
                g.f_atoms, g.f_bonds = g.f_atoms.to(dtype), g.f_bonds.to(dtype)
            Y = ds.lgk[rows].reshape(-1, 1)
            rel = Y - Y.T
            pos = torch.tensor((rel > 0).astype(np.float32)).to(dtype)
            neg = torch.tensor((rel < 0).astype(np.float32)).to(dtype)
            feats = ds.lgk[rows].reshape(-1, 1)       # the leak: add_features = target column
            orig = torch.FloatTensor
            if dtype == torch.float64:
                torch.FloatTensor = lambda x: torch.tensor(np.asarray(x, np.float32), dtype=torch.float64)  # type: ignore
            try:
                y = model(r_g, p_g, gpu=None, add_features=feats)
            finally:
                torch.FloatTensor = orig  # type: ignore
            scores.append(y.detach().numpy())
            y = y.unsqueeze(1)
            C = pos * torch.log(1 + torch.exp(-(y - y.t()))) + neg * torch.log(1 + torch.exp(y - y.t()))
            loss = loss + torch.sum(C, (0, 1))
            pairs += 2 * float(pos.sum())
            y_pred_batch.append(y)
            with torch.no_grad():                     # lines 125-137 with sigma = 1
                l_pos = 1 + torch.exp(y - y.t())
                l_neg = 1 + torch.exp(-(y - y.t()))
                lam = -pos / l_pos + neg / l_neg
                acc_loss = acc_loss + torch.sum(torch.log(l_neg) * pos + torch.log(l_pos) * neg, (0, 1))
                grad_batch.append(torch.sum(lam, dim=1, keepdim=True))
        model.zero_grad()
        for grad, y_pred in zip(grad_batch, y_pred_batch):   # line 151-152
            y_pred.backward(grad / pairs, retain_graph=True)
        out[f"acc.{tag}.loss"] = (acc_loss / pairs).numpy()
        for k, p in model.named_parameters():
            if p.grad is not None:
                out[f"acc.{tag}.grad.{k}"] = p.grad.numpy().copy()
        loss = loss / pairs
        model.zero_grad()
        loss.backward()
        out[f"{tag}.loss"] = loss.detach().numpy()
        out[f"{tag}.pairs"] = np.float64(pairs)
        out[f"{tag}.scores"] = np.concatenate(scores)
        for k, p in model.named_parameters():
            if p.grad is not None:
                out[f"{tag}.grad.{k}"] = p.grad.numpy()
        if tag == "f32":
            for k, v in np_sd(model.state_dict()).items():
                out[f"sd.{k}"] = v
    out["sizes"] = np.asarray(sizes, np.int64)
    out["star"] = np.asarray([[k, v] for k, v in star.items()], np.int64)
    out["seed"] = np.int64(41)
    np.savez_compressed(os.path.join(OUT, "ranknet.npz"), **out)
    print("ranknet.npz loss", out["f32.loss"], out["f64.loss"])


def golden_steps():
    """Three optimiser steps of the train() body (train_listwise.py:177-290) with Adam
    (train/utils.py:93-106) + NoamLR (train/utils.py:7-81), dropout 0, 'mle'."""
    tu = ref_loader.ref("train.utils")
    ds, fz = dataset_case(51, [6, 5, 4, 6, 3, 6], None)
    model = build_ref_model(40, 1, "with_softplus", None, seed=51)
    opt = tu.build_optimizer(model)
    sched = tu.build_lr_scheduler(opt, warmup_epochs=2, total_epochs=4, train_data_size=30, batch_size=10,
                                  init_lr=1e-4, max_lr=1e-3, final_lr=1e-4)
    out = {}
    for k, v in np_sd(model.state_dict()).items():
        out["sd0." + k] = v
    windows = [(0, 11, [6, 5]), (11, 21, [4, 6]), (21, 30, [3, 6])]
    losses, lrs = [], []
    model.train()
    for lo, hi, scope in windows:
        reactions = np.stack([ds.rsmi[lo:hi], ds.psmi[lo:hi]], axis=1)
        r_g, p_g = fz.parsing_reactions(reactions)
        o = model(r_g, p_g, gpu=None, add_features=ds.temp[lo:hi].reshape(-1, 1))
        loss = ref_loss("mle", o, scope, torch.tensor(ds.lgk[lo:hi].astype(np.float32)))
        lrs.append(opt.param_groups[0]["lr"])
        opt.zero_grad()
        loss.backward()
        opt.step()
        sched.step()
        losses.append(float(loss))
    out["losses"] = np.asarray(losses)
    out["lrs"] = np.asarray(lrs + [opt.param_groups[0]["lr"]])
    for k, v in np_sd(model.state_dict()).items():
        out["sd3." + k] = v
    np.savez_compressed(os.path.join(OUT, "steps.npz"), **out)
    print("steps.npz losses", losses, "lrs", out["lrs"])


class StubScorer(torch.nn.Module):
    """Deterministic 'model' for the metric goldens: scores depend only on the product token and the extra feature, so the
    reference's metric code and ours can be fed identical predictions without a GPU (tests/test_host_cpu.py re-creates it)."""

    def __init__(self, two_columns):
        super().__init__()
        self.two = two_columns

    @staticmethod
    def token_value(tok):
        h = 0
        for ch in tok:
            h = (h * 131 + ord(ch)) % 1000003
        return (h % 2001) / 1000.0 - 1.0

    def forward(self, r_inputs, p_inputs, gpu=None, add_features=None):
        base = torch.tensor([self.token_value(t) for t in p_inputs.smiles_batch], dtype=torch.float32)
        if add_features is not None:
            base = base + 0.25 * torch.tensor(np.asarray(add_features, dtype=np.float32).reshape(-1))
        if self.two:
            return torch.stack((base, 0.5 + base.abs()), dim=1)
        return base


def golden_metrics():
    """evaluate_top_scores / ranking_metrics / calculate_ndcg of the reference (eval.py:76-177, 329-457, 475-555) on a fixed
    synthetic frame with the stub scorer: return values, the order table and the re-ordered tokens."""
    lr = ref_loader.ref("data.load_reactions")
    ev = ref_loader.ref("train.eval")
    sizes = [6, 3, 9, 4, 7, 2, 5]
    ds = synthetic.make_dataset(33, sizes, atoms_lo=3, atoms_hi=4)
    df = ds.to_dataframe()

    class Feat:                                   # duck-typed Parsing_features: only .smiles_batch is read by the stub
        class B:
            def __init__(self, toks):
                self.smiles_batch = list(toks)

        def parsing_smiles(self, toks):
            return Feat.B(toks)

    cols = ["rsmi_mapped", "psmi_mapped"]
    out = {"sizes": np.asarray(sizes, np.int64), "seed": np.int64(33)}
    for two in (False, True):
        m = StubScorer(two).eval()
        tag = "two." if two else "one."
        dp = lr.DataProcessor(df)
        a, b, c = ev.evaluate_top_scores(m, gpu=None, data_processor=dp, smiles2graph_dic=Feat(), ratio=0.25, batch_size=3, smiles_list=cols,
                                         target_name="lgk", add_features_name="temp")
        out[tag + "top_scores"] = np.asarray([a, b, c], np.float64)
        r = ev.ranking_metrics(m, gpu=None, data_processor=dp, smiles2graph_dic=Feat(), show_info=False, smiles_list=cols, target_name="lgk",
                               add_features_name="temp")
        out[tag + "ranking"] = np.asarray([r[0], r[1], r[2]] + list(np.asarray(r[3], np.float64)), np.float64)
        for means, stds, name in ((None, None, "raw"), (0.7, 1.9, "scaled")):
            nd, kl, order, smi = ev.calculate_ndcg(m, gpu=None, data_processor=dp, smiles2graph_dic=Feat(), batch_size=3, NDCG_cut=0.25,
                                                  smiles_list=cols, target_name="lgk", means=means, stds=stds, add_features_name="temp")
            out[tag + name + ".ndcg_kl"] = np.asarray([nd, kl], np.float64)
            out[tag + name + ".order"] = np.asarray(order, np.float64)
            out[tag + name + ".smi_iter"] = np.asarray([x[0] for x in smi], np.int64)
            out[tag + name + ".smi_p"] = np.asarray([x[2] for x in smi])
        nd, kl, order, smi = ev.calculate_ndcg(m, gpu=None, data_processor=dp, smiles2graph_dic=Feat(), batch_size=3, NDCG_cut=0.25, smiles_list=cols,
                                              target_name="lgk", is_order=False, add_features_name="temp")
        assert nd is None and kl is None
        out[tag + "unordered.rows"] = np.asarray(order, np.float64)
        out[tag + "unordered.smi_p"] = np.asarray([x[1] for x in smi])
    np.savez_compressed(os.path.join(OUT, "metrics.npz"), **out)
    print("metrics.npz", len(out))


if __name__ == "__main__":
    assert ref_loader.available(), "needs /root/reference"
    only = sys.argv[1:]
    for fn in (golden_batching, golden_planner, golden_model, golden_ranknet, golden_steps, golden_metrics, golden_composite):
        if not only or fn.__name__[len("golden_"):] in only:
            fn()
