"""predict() and rr_rank_predict on the GPU: the kernel against the float64 host restatement (test_predict_cpu.host_predict), the scores
against the fp64 oracle, the segment semantics of the batched launches, MC dropout replayed in the documented seed order, and predict.py
on a checkpoint written by main.py."""
import os
import subprocess
import sys

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import reactranker_oracle as O
from reactranker_b200 import _lib, synthetic
from reactranker_b200.data.load_reactions import DataProcessor, Parsing_features
from reactranker_b200.models.base_model import build_model
from reactranker_b200.predict import COLUMNS, predict
from reactranker_b200.train import eval as E
from helpers import TOL, rel_err
from test_predict_cpu import host_predict, stable_ranks

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COLS = ["rsmi_mapped", "psmi_mapped"]


def S():
    return torch.cuda.current_stream().cuda_stream


def close(got, want, rtol=1e-6):
    """element-wise |got - want| <= rtol |want| (exact where want is 0)"""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    bad = np.abs(got - want) > rtol * np.abs(want)
    assert not bad.any(), (np.flatnonzero(bad)[:8], got[bad][:8], want[bad][:8])


def rank_predict(samples, scope, ld, max_group=None):
    """rr_rank_predict on samples [T, N, ld] (column 0 ranks), straight through the C ABI."""
    T, N = samples.shape[0], samples.shape[1]
    off = torch.tensor(np.concatenate(([0], np.cumsum(scope))), dtype=torch.int32, device=DEV)
    out = torch.full((N, 6), -7.0, device=DEV)
    s = samples.contiguous().to(DEV)
    _lib.check(_lib.lib().rr_rank_predict(N, len(scope), T, s.data_ptr(), N * ld, ld, off.data_ptr(), max_group or max(scope), out.data_ptr(), S()))
    return out.cpu().numpy()


@pytest.mark.parametrize("T", [1, 3, 16])
@pytest.mark.parametrize("ld", [1, 2, 4])
def test_kernel_matches_the_host_restatement(T, ld):
    """Quantised scores (exact ties, ranked by the stable rule), groups of 1 to 8192 candidates and an empty one, strided score columns.
    Ranks and top-1 frequencies are exact, the means, spreads and probabilities within 1e-6; a second call is bit-identical."""
    scope = [1, 2, 0, 7, 50, 500, 8192]
    g = torch.Generator().manual_seed(T * 10 + ld)
    s = torch.round(torch.randn(T, sum(scope), ld, generator=g) * 4) / 4
    got = rank_predict(s, scope, ld)
    want = host_predict(s[:, :, 0].numpy(), scope)
    assert np.array_equal(got[:, [2, 4]], want[:, [2, 4]].astype(np.float32))        # the fp32 rounding of the exact fraction (1/3 at T = 3)
    for c in (0, 1, 3, 5):
        close(got[:, c], want[:, c])
    assert np.array_equal(rank_predict(s, scope, ld), got)


def test_kernel_poisons_a_group_above_max_group_and_refuses_bad_arguments():
    scope = [8, 32, 5]
    s = torch.round(torch.randn(3, sum(scope), 1, generator=torch.Generator().manual_seed(1)) * 4) / 4
    got = rank_predict(s, scope, 1, max_group=8)
    want = host_predict(s[:, :, 0].numpy(), scope)
    assert np.isnan(got[8:40]).all() and np.isfinite(got[:8]).all() and np.isfinite(got[40:]).all()
    exact = want[:, [2, 4]].astype(np.float32)
    assert np.array_equal(got[:8, [2, 4]], exact[:8]) and np.array_equal(got[40:, [2, 4]], exact[40:])
    close(got[:8, 0], want[:8, 0])
    close(got[40:, 3], want[40:, 3])
    L = _lib.lib()
    x = torch.zeros(16, device=DEV)
    off = torch.tensor([0, 16], dtype=torch.int32, device=DEV)
    out = torch.zeros(16, 6, device=DEV)
    assert L.rr_rank_predict(16, 1, 0, x.data_ptr(), 16, 1, off.data_ptr(), 16, out.data_ptr(), S()) != 0            # T = 0
    assert L.rr_rank_predict(16, 1, 1, x.data_ptr(), 16, 1, off.data_ptr(), L.rr_loss_max_group() + 1, out.data_ptr(), S()) != 0
    with pytest.raises(_lib.RRError):
        predict(_model(0.0), synthetic.make_dataset(2, [L.rr_loss_max_group() + 1], atoms_lo=2, atoms_hi=3).to_dataframe(), None, gpu=0)


def _model(dropout, hidden=40, task_num=1, task_type=None, seed=0):
    torch.manual_seed(seed)
    return build_model(hidden_size=hidden, mpnn_depth=2, mpnn_diff_depth=2, ffn_depth=3, use_bias=True, dropout=dropout, task_num=task_num,
                       ffn_last_layer="with_softplus", task_type=task_type, add_features_dim=1).cuda(0)


def _groups(df):
    return list(DataProcessor(df).plan_batch_per_query(df, shuffle_query=False, shuffle_batch=False))


def test_scores_match_the_fp64_oracle(gemm_mode):
    """More than GROUPS_PER_LAUNCH groups (two launches), groups of one to six candidates, the temp feature: every group's scores are the
    oracle's forward over that group alone, and the ranks are the stable order of the returned scores (near-ties may order differently in
    the oracle)."""
    sizes = [1, 6, 2, 5, 3, 4] * 45                      # 270 groups
    ds = synthetic.make_dataset(41, sizes, atoms_lo=4, atoms_hi=9)
    df = ds.to_dataframe()
    model = _model(0.1).eval()
    got = predict(model, df, Parsing_features(ds.mols), 0, smiles_list=COLS, add_features_name="temp")
    sd = {k: v.double().cpu() for k, v in model.state_dict().items()}
    want, o = np.empty(len(df)), 0
    for n in sizes:
        want[o:o + n] = O.model_forward(sd, O.OracleBatch([ds.mols[t] for t in ds.rsmi[o:o + n]]), O.OracleBatch([ds.mols[t] for t in ds.psmi[o:o + n]]),
                                        ds.temp[o:o + n].reshape(-1, 1), mpnn_depth=2, mpnn_diff_depth=2, head="with_softplus").detach().numpy().reshape(-1)
        o += n
    assert rel_err(got["score"].values, want) < TOL[gemm_mode]["score"]
    for rows in _groups(df):
        assert np.array_equal(got["rank"].values[rows], stable_ranks(got["score"].values[rows].astype(np.float32)))
    assert np.array_equal(got["score_std"].values, np.zeros(len(df)))


def test_segments_are_the_per_group_forward(capsys):
    """A shuffled frame (groups interleaved, a custom index, a single-candidate group, a star molecule): the output keeps the input's
    index and row order; each group's scores are those of model(...) on that group alone; de-duplicated and per-candidate reactants agree;
    p_top1 sums to one and rank is a permutation of 1..n in every group."""
    sizes = [5, 1, 8, 3, 6]
    ds = synthetic.make_dataset(43, sizes, star_leaves_in_group={2: 7})
    fz = Parsing_features(ds.mols)
    df = ds.to_dataframe().sample(frac=1.0, random_state=3)
    df.index = [f"row{i}" for i in range(len(df))]
    model = _model(0.1, hidden=64).eval()
    got = predict(model, df, fz, 0, smiles_list=COLS, add_features_name="temp")
    assert list(got.index) == list(df.index) and got[df.columns].equals(df)
    identical = 0
    for rows in _groups(df):
        sub = df.iloc[rows]
        with torch.no_grad():
            alone = model(fz.parsing_smiles(list(sub.rsmi_mapped)), fz.parsing_smiles(list(sub.psmi_mapped)), gpu=0,
                          add_features=sub.temp.values.reshape(-1, 1)).cpu().numpy().reshape(-1)
        close(got["score"].values[rows], alone)
        identical += int(np.array_equal(got["score"].values[rows].astype(np.float32), alone))
        assert abs(got["p_top1"].values[rows].sum() - 1.0) < 1e-6
        assert sorted(got["rank"].values[rows].tolist()) == list(range(1, len(rows) + 1))
    with capsys.disabled():
        print(f"\npredict vs one forward per group: {identical} of {len(sizes)} groups bit-identical")
    model.dedup_reactants = False
    close(predict(model, df, fz, 0, smiles_list=COLS, add_features_name="temp")["score"].values, got["score"].values)
    assert not model.training


def test_mc_dropout_replays_in_the_documented_seed_order():
    """mc_samples = T: train-mode forwards, chunk-major then t = 0..T-1, each drawing its seed from torch's RNG.  Replaying them under
    the same torch.manual_seed and feeding the samples to the host restatement gives predict()'s frame, out1 included (a two-output
    head).  The same seed gives the same frame, another seed another spread; a dropout-free model is refused; model.training is restored."""
    T = 5
    sizes = [4, 1, 7] + [3] * 260                        # two launches
    ds = synthetic.make_dataset(47, sizes, atoms_lo=4, atoms_hi=9)
    fz = Parsing_features(ds.mols)
    df = ds.to_dataframe()
    model = _model(0.2, task_num=2, task_type="evidential_ranking").eval()
    torch.manual_seed(11)
    got = predict(model, df, fz, 0, smiles_list=COLS, add_features_name="temp", mc_samples=T)
    assert not model.training
    groups = _groups(df)
    chunks = [(df[COLS].values[r], df[["temp"]].values[r]) for r in groups]
    torch.manual_seed(11)
    model.train()
    want = np.empty((len(df), 6))
    out1 = np.empty(len(df))
    rows = np.concatenate(groups)
    o = 0
    with torch.no_grad():
        for lo, hi, rg, pg, f in E._launch_graphs(chunks, fz, torch.device(DEV), False):
            s = torch.stack([model(rg, pg, gpu=0, add_features=f) for _ in range(T)])      # [T, n, 2]
            n = s.shape[1]
            want[rows[o:o + n]] = host_predict(s[:, :, 0].cpu().numpy(), [len(r) for r in groups[lo:hi]])
            out1[rows[o:o + n]] = s[:, :, 1].mean(dim=0).cpu().numpy()
            o += n
    model.eval()
    for k, c in enumerate(COLUMNS):
        close(got[c].values, want[:, k])
    close(got["out1"].values, out1)
    assert (got["score_std"].values > 0).mean() > 0.9 and got["top1_freq"].values.min() >= 0
    torch.manual_seed(11)
    again = predict(model, df, fz, 0, smiles_list=COLS, add_features_name="temp", mc_samples=T)
    pd.testing.assert_frame_equal(again, got, check_exact=True)
    torch.manual_seed(12)
    other = predict(model.train(), df, fz, 0, smiles_list=COLS, add_features_name="temp", mc_samples=T)
    assert model.training
    assert not np.array_equal(other["score_std"].values, got["score_std"].values)
    with pytest.raises(ValueError):
        predict(_model(0.0), df, fz, 0, smiles_list=COLS, add_features_name="temp", mc_samples=T)


def run(cmd, timeout=900):
    res = subprocess.run([sys.executable] + cmd, cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    return res.stdout


def test_predict_script_on_a_main_py_checkpoint(tmp_path):
    """main.py --synthetic 40,10 writes a checkpoint; predict.py --synthetic 40,10 ranks the same 400 candidates with it, sorted by group
    and rank, and its rows are what predict() returns in process for the same checkpoint."""
    model_args = ["--hidden_size", "64", "--task_type", "listnet"]
    run(["main.py", "--synthetic", "40,10", "--total_epochs", "1", "--save_metric", "average_score", "--batch_size", "100", "--gpu", "0",
         "--path", str(tmp_path)] + model_args)
    ckpt = str(tmp_path / "0.pt")
    assert os.path.exists(ckpt)
    out = str(tmp_path / "ranked.csv")
    run(["predict.py", "--checkpoint", ckpt, "--synthetic", "40,10", "--out", out] + model_args)
    got = pd.read_csv(out)
    assert len(got) == 400 and set(COLUMNS) <= set(got.columns)
    import main
    from reactranker_b200.utils import load_checkpoint
    model = main.make_model("listnet", 64, 3, 0.1)
    model.load_state_dict(load_checkpoint(ckpt)["state_dict"])
    ds = synthetic.make_dataset(0, [10] * 40)
    want = predict(model.cuda(0), ds.to_dataframe(), Parsing_features(ds.mols), 0, smiles_list=COLS, add_features_name="temp")
    want = want.iloc[np.lexsort((want["rank"].values, pd.factorize(want["rsmi"])[0]))].reset_index(drop=True)
    assert got["psmi"].tolist() == want["psmi"].tolist()
    for c in COLUMNS:
        close(got[c].values, want[c].values)
