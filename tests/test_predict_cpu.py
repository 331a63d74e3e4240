"""Prediction without a GPU: the float64 host restatement of rr_rank_predict's six columns (the GPU tests in test_gpu_predict.py check the
kernel against it) on hand-worked cases, and the argument checks of predict() and predict.py that run before any device is touched."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def stable_ranks(x):
    """1-based descending ranks, ties keep the earlier item: rank(i) = 1 + #{j : x_j > x_i} + #{j < i : x_j == x_i}."""
    x = np.asarray(x)
    r = np.empty(len(x), np.int64)
    r[np.argsort(-x, kind="stable")] = np.arange(1, len(x) + 1)
    return r


def host_predict(samples, scope):
    """rr_rank_predict in float64: samples [T, N] (item i of sample t), scope the group sizes.  Returns [N, 6]: mean, standard deviation
    (ddof 0), rank of the fp32 mean, mean softmax probability, top-1 frequency, mean rank.  Empty groups have no rows."""
    s = np.asarray(samples, np.float64)
    s = s.reshape(1, -1) if s.ndim == 1 else s
    out = np.zeros((s.shape[1], 6))
    o = 0
    for n in scope:
        x = s[:, o:o + n]
        if n:
            ranks = np.stack([stable_ranks(row) for row in x])
            e = np.exp(x - x.max(axis=1, keepdims=True))
            mean = x.mean(axis=0)
            out[o:o + n, 0] = mean
            out[o:o + n, 1] = x.std(axis=0)
            out[o:o + n, 2] = stable_ranks(mean.astype(np.float32))       # the kernel ranks the fp32 score it returns
            out[o:o + n, 3] = (e / e.sum(axis=1, keepdims=True)).mean(axis=0)
            out[o:o + n, 4] = (ranks == 1).mean(axis=0)
            out[o:o + n, 5] = ranks.mean(axis=0)
        o += n
    return out


def test_exact_ties_keep_the_earlier_item():
    got = host_predict([[1.0, 3.0, 3.0, 2.0, 3.0]], [5])
    assert got[:, 2].tolist() == [5, 1, 2, 4, 3]
    assert got[:, 4].tolist() == [0, 1, 0, 0, 0]          # only the first of the tied maxima ranks first
    assert np.allclose(got[:, 3].sum(), 1.0)
    assert np.allclose(got[1, 3], got[2, 3]) and np.allclose(got[2, 3], got[4, 3])


def test_one_sample_has_no_spread_and_ranks_first_where_its_rank_is_one():
    x = np.array([0.5, -1.0, 2.0, 0.25, 2.0, 7.0, -3.0])
    got = host_predict(x[None], [3, 4])
    assert np.array_equal(got[:, 0], x) and np.array_equal(got[:, 1], np.zeros(7))
    assert got[:, 2].tolist() == [2, 3, 1, 3, 2, 1, 4]
    assert np.array_equal(got[:, 4], (got[:, 2] == 1).astype(float))
    assert np.array_equal(got[:, 5], got[:, 2])
    e = np.exp([0.5, -1.0, 2.0])
    assert np.allclose(got[:3, 3], e / e.sum(), rtol=1e-15)


def test_two_samples_by_hand():
    # item 0 scores (1, 3), item 1 scores (2, 0): means (2, 1), population std (1, 1); each ranks first once
    got = host_predict([[1.0, 2.0], [3.0, 0.0]], [2])
    assert np.allclose(got[:, 0], [2.0, 1.0]) and np.allclose(got[:, 1], [1.0, 1.0])
    assert got[:, 2].tolist() == [1, 2]
    assert got[:, 4].tolist() == [0.5, 0.5] and got[:, 5].tolist() == [1.5, 1.5]
    p0 = 0.5 * (1 / (1 + np.e) + 1 / (1 + np.exp(-3.0)))
    assert np.allclose(got[:, 3], [p0, 1 - p0], rtol=1e-15)


def test_empty_groups_have_no_rows():
    got = host_predict([[1.0, 2.0, 0.0]], [0, 2, 0, 1, 0])
    assert got[:, 2].tolist() == [2, 1, 1]


def _frame():
    from reactranker_b200 import synthetic
    return synthetic.make_dataset(3, [3, 2]).to_dataframe()


def _model(dropout):
    from reactranker_b200.models.base_model import build_model
    return build_model(hidden_size=16, task_num=1, ffn_last_layer="with_softplus", add_features_dim=1, dropout=dropout)


def test_predict_refuses_what_it_cannot_run():
    from reactranker_b200 import _lib
    from reactranker_b200.predict import predict
    with pytest.raises(_lib.RRError):                       # no CPU path
        predict(_model(0.1), _frame(), None, gpu=None)
    for bad in (0, -1):
        with pytest.raises(ValueError):
            predict(_model(0.1), _frame(), None, gpu=0, mc_samples=bad)
    with pytest.raises(ValueError):                         # nothing to sample without a dropout
        predict(_model(0.0), _frame(), None, gpu=0, mc_samples=4)


def test_predict_script_parses_and_builds_main_py_models():
    res = subprocess.run([sys.executable, "predict.py", "--help"], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr
    assert "--mc_samples" in res.stdout and "--checkpoint" in res.stdout
    import main
    import predict
    assert predict._MODEL_FOR_TASK is main._MODEL_FOR_TASK
    assert predict.make_model is main.make_model
    for task, (task_num, _, _) in list(main._MODEL_FOR_TASK.items()) + [("listnet", (1, None, None))]:
        m = predict.make_model(task, 16, 2, 0.1)
        assert m._task_num == task_num and m._add == 1 and m._depth == m._diff_depth == 2
    a = predict.parse(["--checkpoint", "c.pt", "--synthetic", "40,10", "--out", "r.csv"])
    assert (a.mc_samples, a.gpu, a.task_type) == (1, 0, "listnet")
