"""Shared helpers for the parity tests (test infrastructure)."""
import numpy as np
import torch

from reactranker_b200 import synthetic


def star_dict(arr):
    return {int(k): int(v) for k, v in np.asarray(arr).reshape(-1, 2)} or None


def dataset_from_golden(g, name):
    hidden, seed, depth, ddepth = (int(x) for x in g[name + ".meta"])
    sizes = [int(x) for x in g[name + ".sizes"]]
    ds = synthetic.make_dataset(seed, sizes, star_leaves_in_group=star_dict(g[name + ".star"]))
    return ds, sizes, hidden, depth, ddepth


def sd_from_golden(g, prefix, dtype=torch.float32):
    pre = prefix + "."
    return {k[len(pre):]: torch.tensor(g[k]).to(dtype) for k in g.files if k.startswith(pre)}


def add_features(ds, add):
    """The ``add_features`` of a synthetic batch for a model built with ``add_features_dim = add``: none for 0, the temperature column
    for 1 (the reference's setting), and seeded standard-normal columns after it for more."""
    if add == 0:
        return None
    rng = np.random.default_rng(add)
    return np.concatenate([ds.temp.reshape(-1, 1), rng.standard_normal((len(ds.temp), add - 1))], axis=1)


# Model configurations outside the shape the other parity tests build (ffn_depth 3, biases, one add feature, equal depths), each taking
# code that only it runs: the FFN as one Linear / with a third hidden layer; no W_i / W_h / FFN biases (W_o keeps its own); no encoder
# W_h (depth 1) / no diff-encoder W_h (diff depth 1); unequal depths; no add features; add features beyond the padded hidden width
# (hidden 302 + 3 -> vp 320); multi-column raw heads up to RR_OUT_LD; the narrowest padded width (hidden 8 -> 16); hidden > 1024, where the
# message-passing row pipeline declines; molecules of one to three atoms (no bonds, in-degree 0, a batch whose only bond row is padding);
# >= 256 reactions, where the FFN weight gradients go to the tensor cores.
CONFIG_DEFAULTS = dict(hidden=40, depth=3, ddepth=3, ffn_depth=3, use_bias=True, add=1, task_num=1, sizes=(7, 5, 9, 4), atoms=(12, 28))
CONFIGS = {
    "ffn1_raw3": dict(ffn_depth=1, task_num=3),
    "ffn4": dict(ffn_depth=4),
    "nobias": dict(use_bias=False),
    "depth1": dict(depth=1),
    "diff_depth1": dict(ddepth=1),
    "depth2_diff4": dict(depth=2, ddepth=4),
    "add0": dict(add=0),
    "raw16": dict(task_num=16),
    "h8": dict(hidden=8),
    "h1040": dict(hidden=1040, depth=2, ddepth=2, sizes=(3, 2, 4)),
    "tiny_mols": dict(atoms=(1, 3), sizes=(5, 4, 6, 3, 5)),
    "one_atom_mols": dict(atoms=(1, 1), sizes=(4, 3)),
    "h302_add3_n320": dict(hidden=302, add=3, atoms=(3, 6), sizes=(40,) * 8),
}


def config(name):
    """CONFIGS[name] with the defaults filled in."""
    return dict(CONFIG_DEFAULTS, **CONFIGS[name])


def config_model(c, dropout=0.0):
    """build_model for a filled-in configuration (head: the raw output, ffn_last_layer 'with_softplus' with task_type None)."""
    from reactranker_b200.models.base_model import build_model
    return build_model(hidden_size=c["hidden"], mpnn_depth=c["depth"], mpnn_diff_depth=c["ddepth"], ffn_depth=c["ffn_depth"],
                       use_bias=c["use_bias"], dropout=dropout, task_num=c["task_num"], ffn_last_layer="with_softplus",
                       add_features_dim=c["add"])


def config_dataset(c, seed=61):
    ds = synthetic.make_dataset(seed, list(c["sizes"]), atoms_lo=c["atoms"][0], atoms_hi=c["atoms"][1])
    return ds, add_features(ds, c["add"])


def rel_err(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def grads_close(got: dict, want: dict, rtol: float):
    """Per-tensor max-abs error <= rtol * max|want_k| + 1e-2 * rtol * (largest gradient entry
    of the whole model).  The second term absorbs tensors whose true gradient is zero (e.g. the
    last bias under a shift-invariant ranking loss).  Returns a list of offending keys."""
    gscale = max(float(np.abs(v).max()) for v in want.values())
    bad = []
    for k, w in want.items():
        a = np.asarray(got[k], np.float64)
        w = np.asarray(w, np.float64)
        err = np.abs(a - w).max()
        if not err <= rtol * np.abs(w).max() + 1e-2 * rtol * gscale:
            bad.append((k, float(err), float(np.abs(w).max())))
    return bad


# ------------------------------------------------------------------------------------------------
# per-GEMM-mode tolerances and the ReLU-kink-aware gradient check
# ------------------------------------------------------------------------------------------------
# gemm mode 0 = exact-fp32 SIMT GEMMs, 1 = the product default and the benchmarked path (tcgen05: forward 3 x TF32, backward 3 x bf16).
# North star: 1e-4 relative on losses, 1e-3 on gradients.  Mode 0 is held 5x tighter than that, mode 1 to the north star itself.
TOL = {0: dict(score=2e-5, loss=2e-5, grad=2e-4), 1: dict(score=5e-5, loss=2e-5, grad=1e-3)}
# a pre-activation this close to zero (relative to its row's largest entry) may legitimately get the other ReLU mask in mode 1: 4x the
# measured forward error of the 3 x TF32 split (2-5e-6; tests/test_gpu_kernels.py::test_tcgen05_linear_matches_fp64)
KINK = 2e-5


def gpu_relu_masks(model, out, r_rows, p_rows, hidden, depth, ddepth, ffn_depth=3):
    """The ReLU masks the GPU forward behind ``out`` used, in the order the oracle calls ``torch.relu`` (mpn_forward(r), mpn_forward(p),
    mpndiff_forward, ffn_forward), read from the activations saved in the autograd node's workspace.  Call BEFORE ``backward()`` (the
    workspace is recycled afterwards); needs dropout 0 (a dropped entry would look like a masked one).  With dropout, use
    tests/test_gpu_dropout.py::relu_masks_and_keeps, which pairs each mask with the host-regenerated keep mask of its site and passes
    both to forced_relu_masks(masks, keeps=...).
    r_rows / p_rows = (n_atoms, n_bonds) of the two batches, padding rows included."""
    from reactranker_b200 import _lib
    hp = _lib.lib().rr_padded(hidden)
    n_mols = out.shape[0]

    def act(name, rows):
        return model.saved_activation(out, name, rows, hp)[:, :hidden].detach().cpu()
    masks = []
    for k, (na, nb) in enumerate((r_rows, p_rows)):
        masks.append(act(f"enc{k}.inp", nb) > 0)
        for t in range(1, depth):
            masks.append(act(f"enc{k}.m{t}", nb) != 0)
        masks.append(act(f"enc{k}.hid", na) != 0)
    na = p_rows[0]
    masks.append(act("inp2", na) > 0)
    for t in range(1, ddepth):
        masks.append(act(f"m2_{t}", na) != 0)
    masks.append(act("hid2", na) != 0)
    for l in range(ffn_depth - 1):
        masks.append(act(f"x{l}", n_mols) != 0)
    return masks


class forced_relu_masks:
    """Context manager: while active, the i-th ``torch.relu`` call (the oracle's) multiplies by ``masks[i]`` instead of [x > 0].
    Every entry where the forced mask differs from the oracle's own must lie within ``kink`` (relative to its row's largest
    magnitude) of zero -- i.e. the GPU's forward error, not a wrong value, decided it.  ``flips`` counts them.
    ``keeps`` (optional, parallel to ``masks``; an entry may be None): where keeps[i] is False the entry was dropped by dropout, the GPU's
    activation is 0 whatever its ReLU decided, and the oracle keeps its own decision there (it is multiplied by 0 afterwards)."""

    def __init__(self, masks, kink=KINK, keeps=None):
        self.masks, self.kink, self.i, self.flips, self.worst = masks, kink, 0, 0, 0.0
        self.keeps = keeps

    def __enter__(self):
        self._orig = torch.relu

        def relu(x):
            m = self.masks[self.i].to(x.device)
            keep = self.keeps[self.i] if self.keeps is not None else None
            self.i += 1
            assert tuple(m.shape) == tuple(x.shape), (self.i - 1, tuple(m.shape), tuple(x.shape))
            own = x.detach() > 0
            if keep is not None:
                m = torch.where(keep.to(x.device), m, own)
            diff = m != own
            if bool(diff.any()):
                rel = (x.detach().abs() / x.detach().abs().amax(dim=-1, keepdim=True).clamp_min(1e-300))[diff]
                self.flips += int(diff.sum())
                self.worst = max(self.worst, float(rel.max()))
            return x * m.to(x.dtype)
        torch.relu = relu
        return self

    def __exit__(self, *exc):
        torch.relu = self._orig
        if exc[0] is None:
            assert self.i == len(self.masks), (self.i, len(self.masks))
            assert self.worst <= self.kink, f"a ReLU mask differs at a pre-activation {self.worst:.2e} (relative) away from zero (allowed: {self.kink:.0e})"
        return False


def check_grads(mode, got, want, masked_oracle=None, max_flips=8):
    """``got`` within TOL[mode]['grad'] of ``want`` for every tensor.  In mode 1, a miss is accepted only if (a) the oracle re-run with
    the GPU's own ReLU masks (``masked_oracle()`` -> (gradients, flips); see forced_relu_masks, which asserts that every differing mask
    sits on a kink) reproduces the gradients to the mode-0 tolerance, and (b) at most ``max_flips`` masks differ.  On a batch of a few
    hundred atom rows a single mask flip moves a weight gradient by ~1e-2 of its maximum (DESIGN.md section 2), which no forward
    accuracy short of fp64 can exclude; the check pins every such difference to a pre-activation within 2e-5 of zero."""
    gscale = max(float(np.abs(v).max()) for v in want.values())
    live = {k: w for k, w in want.items() if float(np.abs(w).max()) >= 1e-6 * gscale}     # drop structurally-zero gradients (e.g. the last
    bad = grads_close(got, live, TOL[mode]["grad"])                                         # bias under a shift-invariant ranking loss)
    if not bad:
        return
    assert mode == 1 and masked_oracle is not None, bad
    want2, flips = masked_oracle()
    assert 0 < flips <= max_flips, (flips, bad)
    bad2 = grads_close(got, {k: want2[k] for k in live}, TOL[0]["grad"])
    assert not bad2, (flips, bad2)
