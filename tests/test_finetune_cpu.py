"""Fine-tuning with frozen sub-modules, the host side (no GPU): which tensors freeze() freezes, what load_pretrained copies and skips,
the flat gradient layout the backward pass and GradSync share over the trainable tensors (with a 2-rank gloo run of a frozen toy
model on the in-place path), the optimiser's parameter set, and the --freeze / --pretrained command line.
tests/test_gpu_finetune.py runs the frozen backward itself."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from reactranker_b200 import _lib, parallel
from reactranker_b200.models import base_model
from reactranker_b200.models.base_model import build_model, freeze, parse_freeze
from reactranker_b200.train.utils import build_optimizer
from reactranker_b200.utils import load_pretrained, save_checkpoint

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ENC = ["encoder.W_i.weight", "encoder.W_i.bias", "encoder.W_h.weight", "encoder.W_h.bias", "encoder.W_o.weight", "encoder.W_o.bias"]
DIF = [n.replace("encoder", "diff_encoder") for n in ENC]
FFN = [f"ffn.ffn.{i}.{k}" for i in (1, 4, 7) for k in ("weight", "bias")]


def _model(diff_depth=3, task_num=1, add=1, seed=0):
    torch.manual_seed(seed)
    return build_model(hidden_size=24, mpnn_depth=3, mpnn_diff_depth=diff_depth, ffn_depth=3, dropout=0.1, task_num=task_num,
                       add_features_dim=add)


def _pretrained(tmp_path, model, name="pre.pt"):
    path = str(tmp_path / name)
    save_checkpoint(path, model)
    return path


def _frozen(model):
    return sorted(n for n, p in model.named_parameters() if not p.requires_grad and "cached_zero" not in n)


@pytest.mark.parametrize("kw, want", [
    (dict(encoder=True), ENC),
    (dict(encoder=True, diff_encoder=True), ENC + DIF),
    (dict(encoder=True, diff_encoder=True, ffn_layers=1), ENC + DIF + FFN[:2]),
    (dict(ffn_layers=2), FFN[:4]),
    (dict(diff_encoder=True, ffn_layers=3), DIF + FFN),
    (dict(), []),
])
def test_freeze_sets_exactly_the_expected_flags(tmp_path, kw, want):
    model = _model()
    load_pretrained(model, _pretrained(tmp_path, _model(seed=1)))
    assert sorted(freeze(model, **kw)) == sorted(want)
    assert _frozen(model) == sorted(want)


def test_freeze_at_diff_depth_0():
    """Diff depth 0 has no diff_encoder.W_h / W_o: freezing the diff encoder freezes its W_i alone."""
    model = _model(diff_depth=0)
    model.pretrained_names = set(model.state_dict())
    assert sorted(freeze(model, diff_encoder=True)) == ["diff_encoder.W_i.bias", "diff_encoder.W_i.weight"]
    assert _frozen(model) == ["diff_encoder.W_i.bias", "diff_encoder.W_i.weight"]


def test_freeze_refuses_weights_that_were_not_loaded(tmp_path):
    with pytest.raises(ValueError, match="not loaded"):
        freeze(_model(), encoder=True)                                       # random weights
    with pytest.raises(ValueError, match="ffn_layers"):
        freeze(_model(), ffn_layers=4)


@pytest.mark.parametrize("src, dst, skipped", [
    (dict(task_num=1), dict(task_num=2), ["ffn.ffn.7.bias", "ffn.ffn.7.weight"]),      # pretrain with mle, fine-tune evidential_ranking
    (dict(add=1), dict(add=0), ["ffn.ffn.1.weight"]),
    (dict(add=0), dict(add=3), ["ffn.ffn.1.weight"]),
])
def test_load_pretrained_skips_exactly_the_mismatched_ffn_layer(tmp_path, src, dst, skipped):
    pre = _model(seed=1, **src)
    model = _model(seed=2, **dst)
    before = {k: v.clone() for k, v in model.state_dict().items()}
    got = load_pretrained(model, _pretrained(tmp_path, pre))
    assert sorted(n for n, _ in got) == skipped and all("shape" in why for _, why in got)
    sd, psd = model.state_dict(), pre.state_dict()
    for k in sd:
        assert torch.equal(sd[k], before[k] if k in skipped else psd[k]), k
    assert model.pretrained_names == set(sd) - set(skipped)
    # the encoder and the diff encoder are fully loaded; the FFN is not
    freeze(model, encoder=True, diff_encoder=True)
    with pytest.raises(ValueError, match="not loaded"):
        freeze(model, ffn_layers=3)


def test_load_pretrained_reports_names_missing_on_either_side(tmp_path):
    pre = _model(diff_depth=3, seed=1)
    model = _model(diff_depth=1, seed=2)                                      # no diff_encoder.W_h
    got = dict(load_pretrained(model, _pretrained(tmp_path, pre)))
    assert got == {"diff_encoder.W_h.weight": "not in the model", "diff_encoder.W_h.bias": "not in the model"}
    with pytest.raises(Exception):
        load_pretrained(model, str(tmp_path / "missing.pt"))


def test_hot_parameters_and_flat_layout_are_over_trainable_tensors(tmp_path):
    """The backward pass lays its flat gradient buffer out with parallel.flat_layout over hot_parameters(); GradSync, given every
    parameter, arrives at the same tensors and offsets."""
    assert base_model.flat_layout is parallel.flat_layout
    model = _model()
    model.pretrained_names = set(model.state_dict())
    freeze(model, encoder=True, ffn_layers=1)
    hot = model.hot_parameters()
    names = {id(p): n for n, p in model.named_parameters()}
    assert [names[id(p)] for p in hot] == DIF + FFN[2:]
    offs, total = parallel.flat_layout(hot)
    assert all(o % 4 == 0 for o in offs) and total == sum((p.numel() + 3) // 4 * 4 for p in hot)
    sync = parallel.GradSync(model.parameters(), None, model)
    assert sync.params == hot and sync.offsets == offs and sync.numel == total
    # unfreezing afterwards: the next call sees the new set
    model.encoder.W_o.bias.requires_grad_(True)
    sync._refresh()
    assert sync.params == model.hot_parameters() and sync.numel == parallel.flat_layout(model.hot_parameters())[1]


def test_build_optimizer_freeze_holds_exactly_the_trainable_tensors(tmp_path):
    model = _model()
    model.pretrained_names = set(model.state_dict())
    freeze(model, encoder=True, diff_encoder=True)
    ps = build_optimizer(model, freeze=True).param_groups[0]["params"]
    want = [p for p in model.parameters() if p.requires_grad]
    assert len(ps) == len(want) == 6 and all(a is b for a, b in zip(ps, want))


class _FrozenToy(torch.nn.Module):
    """ReactionModel's gradient plumbing on the CPU: the first layer frozen, backward() leaves the trainable gradients as views of one
    flat buffer laid out by parallel.flat_layout."""

    def __init__(self):
        super().__init__()
        self.net = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.Linear(5, 3), torch.nn.Linear(3, 1))
        self.net[0].requires_grad_(False)
        self._grad_flat, self._grad_offsets = None, None

    def hot_parameters(self):
        return [p for p in self.net.parameters() if p.requires_grad]

    def alias_grads(self):
        ps = self.hot_parameters()
        offs, total = parallel.flat_layout(ps)
        flat = torch.zeros(total)
        for p, o in zip(ps, offs):
            flat[o:o + p.numel()] = p.grad.reshape(-1)
            p.grad = flat[o:o + p.numel()].view(p.shape)
        self._grad_flat, self._grad_offsets = flat, offs


def _toy_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    parallel.init_from_env(device=None)
    try:
        torch.manual_seed(0)
        m = _FrozenToy()
        g = torch.Generator().manual_seed(7)
        X, t = torch.randn(12, 6, generator=g), torch.randn(12, generator=g)
        lo, hi = [(0, 5), (5, 12)][rank]
        sync = parallel.GradSync(m.parameters(), None, m)
        (((m.net(X[lo:hi]).squeeze(-1) - t[lo:hi]) ** 2).sum() / 12).backward()
        m.alias_grads()
        sync()
        out[rank] = (sync.fast_path_steps, sync.copy_path_steps, sync.numel, m.net[0].weight.grad is None,
                     torch.cat([p.grad.reshape(-1) for p in m.hot_parameters()]).numpy())
    finally:
        dist.destroy_process_group()


def test_gloo_world2_frozen_model_takes_the_in_place_path():
    world, port = 2, 33500 + os.getpid() % 2000
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_toy_worker, args=(world, port, out), nprocs=world, join=True)
        res = dict(out)
    torch.manual_seed(0)
    m = _FrozenToy()
    g = torch.Generator().manual_seed(7)
    X, t = torch.randn(12, 6, generator=g), torch.randn(12, generator=g)
    ((m.net(X).squeeze(-1) - t) ** 2).mean().backward()
    want = torch.cat([p.grad.reshape(-1) for p in m.hot_parameters()]).numpy()
    for r in (0, 1):
        fast, copy, numel, frozen_none, got = res[r]
        assert (fast, copy) == (1, 0) and frozen_none
        assert numel == parallel.flat_layout(m.hot_parameters())[1] == 16 + 4 + 4 + 4   # layers 2 and 3, weights and biases, each rounded up to 4
        assert np.allclose(got, want, rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("script", ["main.py", "main_ranknet.py"])
def test_entry_points_parse_freeze_and_reject_unknown_modules(script):
    base = [sys.executable, script, "--help"]
    ok = subprocess.run(base, cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert ok.returncode == 0 and "--freeze" in ok.stdout and "--pretrained" in ok.stdout
    for spec, msg in (("encoder,decoder", "unknown module 'decoder'"), ("ffn:0", "unknown module 'ffn:0'"), ("encoder", "needs --pretrained")):
        args = [sys.executable, script, "--freeze", spec] + (["--pretrained", "x.pt"] if spec != "encoder" else [])
        res = subprocess.run(args, cwd=ROOT, capture_output=True, text=True, timeout=300)
        assert res.returncode == 2 and msg in res.stderr, res.stderr[-2000:]


def test_parse_freeze():
    assert parse_freeze("encoder") == dict(encoder=True, diff_encoder=False, ffn_layers=0)
    assert parse_freeze("ffn:2,diff_encoder, encoder") == dict(encoder=True, diff_encoder=True, ffn_layers=2)
    for bad in ("", "Encoder", "ffn", "ffn:x", "ffn:-1"):
        with pytest.raises(ValueError):
            parse_freeze(bad)


def test_exports_and_header_still_agree_at_48():
    header = open(os.path.join(ROOT, "include", "rr_sm100.h")).read()
    declared = set(re.findall(r"\b(rr_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTS) and len(_lib.EXPORTS) == 48
    assert re.search(r"#define RR_ABI_VERSION 3\b", header)
