"""GPU parity of the models ReactionModel builds beyond build_model's tied ones (tests/test_model_variants_cpu.py::VARIANTS): diff depth 0,
separate encoder / diff encoder / FFN widths and dropouts, biases off in one sub-module.  Against the fp64 oracle in both GEMM modes, with
dropout under the GPU's own Philox masks regenerated on the host (tests/test_gpu_dropout.py), padding rows on the tensor-core path,
deterministic mode, de-duplicated reactants and train() end to end.  And tied models: the _ex entry points compute bit for bit what the
ABI-3 ones do."""
import os

import numpy as np
import pytest
import torch

from oracle import reactranker_oracle as O
from reactranker_b200 import _lib, synthetic
from reactranker_b200.features.featurization import BatchMolGraph, DeviceGraph
from reactranker_b200.models.base_model import build_model
from helpers import TOL, check_grads, forced_relu_masks, grads_close, rel_err
from test_gpu_dropout import Layout, keep_mask
from test_model_variants_cpu import VARIANTS, oracle_forward, variant, variant_dataset, variant_model

pytestmark = pytest.mark.gpu
GPU = 0


# ------------------------------------------------------------------------------------------------
# dropout / ReLU sites with per-module widths
# ------------------------------------------------------------------------------------------------
def site_order(c):
    """(saved buffer, Layout row key, module, kind) of every ReLU / dropout site, in the order of the oracle's torch.relu and _drop calls
    for one group.  kind 'pre': the buffer is a pre-activation only a ReLU reads; 'act': ReLU, then that module's dropout; 'drop': dropout
    only (the readout vector).  At diff depth 0, hid2 = dropout(relu(W_i d)) is the diff encoder's only site."""
    order = []
    for k, (a, b) in enumerate((("ra", "rb"), ("pa", "pb"))):
        order += [(f"enc{k}.inp", b, "e", "pre")] + [(f"enc{k}.m{t}", b, "e", "act") for t in range(1, c["depth"])]
        order += [(f"enc{k}.hid", a, "e", "act")]
    if c["ddepth"] > 0:
        order += [("inp2", "pa", "d", "pre")] + [(f"m2_{t}", "pa", "d", "act") for t in range(1, c["ddepth"])]
    order += [("hid2", "pa", "d", "act"), ("vec", "m", "f", "drop")] + [(f"x{l}", "m", "f", "act") for l in range(c["ffn_depth"] - 1)]
    return order


def stream_ids(c):
    """rr_model.cu model_forward's Philox stream id of every dropout site: one id per dense layer in launch order from 1, then the
    readout's, then the FFN's.  At diff depth 0 the diff encoder's W_i carries hid2."""
    sid = iter(range(1, 1 << 10))
    next(sid)                                                    # encoder W_i
    ids = {f"m{t}": next(sid) for t in range(1, c["depth"])}
    ids["hid"] = next(sid)
    if c["ddepth"] > 0:
        next(sid)                                                # diff encoder W_i (ReLU applied by its consumers)
        ids.update({f"m2_{t}": next(sid) for t in range(1, c["ddepth"])})
    ids["hid2"] = next(sid)
    ids["vec"] = next(sid)
    ids.update({f"x{l}": next(sid) for l in range(c["ffn_depth"] - 1)})
    return ids


def widths(c):
    L = _lib.lib()
    w = dict(e=c["he"], d=c["hd"], f=c["hf"])
    ld = {k: L.rr_padded(v) for k, v in w.items()}
    return w, ld, c["hd"] + c["add"], L.rr_padded(c["hd"] + c["add"])


def saved_buffers(model, out, c, lay):
    """Every activation a ReLU or dropout acted on, [rows, width] (call BEFORE backward: the workspace is recycled)."""
    w, ld, vw, vp = widths(c)
    rows = dict(ra=lay.A_r, rb=lay.B_r, pa=lay.A_p, pb=lay.B_p, m=lay.N)
    buf = {}
    for name, key, mod, kind in site_order(c):
        cols, stride = (vw, vp) if name == "vec" else (w[mod], ld[mod])
        buf[name] = model.saved_activation(out, name, rows[key], stride)[:, :cols].detach().cpu()
    return buf


def site_keeps(seed, c, p, lay):
    """{buffer: host keep mask} of every site whose module has dropout > 0; the encoder draws over the joint rows [reactants | products]."""
    w, ld, vw, vp = widths(c)
    pm = dict(e=p[0], d=p[1], f=p[2])
    ids = stream_ids(c)
    keeps = {}
    for name, key, mod, kind in site_order(c):
        if kind == "pre" or pm[mod] == 0 or name.startswith("enc1"):
            continue
        if name.startswith("enc0"):
            base = name.split(".")[1]
            joint_rows = (lay.B_r + lay.B_p) if base.startswith("m") else (lay.A_r + lay.A_p)
            j = torch.from_numpy(keep_mask(seed, ids[base], joint_rows, w["e"], ld["e"], pm["e"]))
            split = lay.B_r if base.startswith("m") else lay.A_r
            keeps[name], keeps["enc1." + base] = j[:split], j[split:]
        elif name == "vec":
            keeps[name] = torch.from_numpy(keep_mask(seed, ids["vec"], lay.N, vw, vp, pm["f"]))
        else:
            rows = lay.A_p if key == "pa" else lay.N
            keeps[name] = torch.from_numpy(keep_mask(seed, ids[name], rows, w[mod], ld[mod], pm[mod]))
    return keeps


def relu_masks_and_keeps(buf, keeps, c, lay):
    """Per group, the GPU's ReLU decision of every oracle torch.relu call and the keep mask of its site (None without dropout)."""
    masks, kps = [], []
    for grp in lay.groups:
        for name, key, mod, kind in site_order(c):
            if kind == "drop":
                continue
            x = buf[name][grp[key]]
            masks.append(x > 0 if kind == "pre" else x != 0)
            kps.append(keeps[name][grp[key]] if name in keeps else None)
    return masks, kps


class oracle_drops:
    """While active, the oracle's _drop (called at every dropout site of a training forward, mpn.py / base_model.py order) takes the next
    entry of ``drops``: None leaves the site as it is (its module has no dropout), (keep, p) multiplies by the host keep mask / (1 - p).
    So each site gets its own module's p, which the oracle's single ``dropout`` argument cannot express."""

    def __init__(self, drops):
        self.it = iter(drops)

    def __enter__(self):
        self._orig = O._drop

        def drop(x, p_, training):
            if not training:
                return x
            e = next(self.it)
            if e is None:
                return x
            keep, p = e
            assert tuple(keep.shape) == tuple(x.shape), (tuple(keep.shape), tuple(x.shape))
            return x * keep.to(x.dtype) / (1 - p)
        O._drop = drop
        return self

    def __exit__(self, *exc):
        O._drop = self._orig
        if exc[0] is None:
            assert next(self.it, None) is None
        return False


def oracle_run(sd, c, groups, upstream, drops=None, relu=None):
    """fp64 oracle forward (one per group) + (scores * upstream).sum() + backward; ``drops``: one entry per dropout site and group (see
    oracle_drops), None for a forward without dropout; with ``relu`` = (masks, keeps) the ReLU decisions of the kept entries are the GPU's.
    Returns (scores, {name: gradient}, flips)."""
    sd64 = {k: v.double().cpu() for k, v in sd.items()}
    params = {k: v.clone().requires_grad_(True) for k, v in sd64.items() if "cached_zero" not in k}
    full = dict(sd64, **params)
    training = drops is not None
    flips = 0
    with oracle_drops(drops or ()):
        if relu is None:
            want = torch.cat([oracle_forward(full, c, r, q, f, training) for r, q, f in groups])
        else:
            with forced_relu_masks(relu[0], keeps=relu[1]) as fm:
                want = torch.cat([oracle_forward(full, c, r, q, f, training) for r, q, f in groups])
            flips = fm.flips
    (want * upstream.double()).sum().backward()
    return want.detach().numpy(), {k: v.grad.numpy() for k, v in params.items()}, flips


def _case(c, p, segments=1, seed=61):
    """Model (dropouts p), data, host batches of each segment and the oracle's per-group inputs."""
    ds, feats = variant_dataset(c, seed)
    sizes = list(c["sizes"])
    torch.manual_seed(3)
    model = variant_model(c, p).cuda(GPU)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    cuts = np.linspace(0, len(sizes), segments + 1).astype(int)
    off = np.cumsum([0] + sizes)
    rb, pb, groups = [], [], []
    for a, b in zip(cuts[:-1], cuts[1:]):
        lo, hi = off[a], off[b]
        rm, pm = [ds.mols[t] for t in ds.rsmi[lo:hi]], [ds.mols[t] for t in ds.psmi[lo:hi]]
        rb.append(BatchMolGraph(rm))
        pb.append(BatchMolGraph(pm))
        groups.append((O.OracleBatch(rm), O.OracleBatch(pm), None if feats is None else feats[lo:hi]))
    n = sum(sizes)
    w = torch.randn((n,) if c["task_num"] == 1 else (n, c["task_num"]), generator=torch.Generator().manual_seed(1))
    return model, sd, ds, feats, rb, pb, groups, w


def _graphs(rb, pb):
    if len(rb) == 1:
        return rb[0], pb[0]
    dev = torch.device("cuda", GPU)
    return DeviceGraph.from_batches(rb, dev), DeviceGraph.from_batches(pb, dev)


# ------------------------------------------------------------------------------------------------
# 1. every variant against the fp64 oracle at dropout 0
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(VARIANTS))
def test_variant_vs_fp64_oracle(name, gemm_mode):
    """Each variant at dropout 0 in both GEMM modes; the loss is a fixed random weighting of the outputs (a ranking loss would leave the
    last bias without a gradient).  Scores to TOL[mode], gradients by helpers.check_grads (mode 1: the oracle re-run with the GPU's ReLU
    masks when a mask flipped on a kink)."""
    c = variant(name)
    model, sd, ds, feats, rb, pb, groups, w = _case(c, (0.0, 0.0, 0.0))
    model.train()
    ws, wg, _ = oracle_run(sd, c, groups, w)
    lay = Layout(rb, pb)
    out = model(rb[0], pb[0], gpu=GPU, add_features=feats)
    masks = relu_masks_and_keeps(saved_buffers(model, out, c, lay), {}, c, lay) if gemm_mode == 1 else None
    (out * w.to(out.device)).sum().backward()
    assert tuple(out.shape) == tuple(ws.shape)
    e_s = rel_err(out.detach().cpu().numpy(), ws)
    assert e_s < TOL[gemm_mode]["score"], e_s
    got = {k: q.grad.cpu().numpy() for k, q in model.named_parameters() if q.requires_grad}
    assert set(got) == set(wg)

    def redo():
        _, g, flips = oracle_run(sd, c, groups, w, relu=masks)
        return g, flips
    check_grads(gemm_mode, got, wg, redo if masks else None)


# ------------------------------------------------------------------------------------------------
# 2. per-module dropout, one training step under the GPU's Philox masks
# ------------------------------------------------------------------------------------------------
DROPOUT_CASES = {"untied_e01_d03": ("w40_64_24", (0.1, 0.3, 0.0)), "untied_d02_f04": ("w40_64_24", (0.0, 0.2, 0.4)),
                 "ddepth0_d03": ("ddepth0", (0.1, 0.3, 0.2))}


@pytest.mark.parametrize("case", list(DROPOUT_CASES))
def test_per_module_dropout_step_vs_fp64_oracle(case, gemm_mode):
    """Each sub-module's dropout at its own p, on two segments in one launch: nothing a host mask drops survives in any saved activation,
    every site without dropout is untouched, and scores, activations and gradients equal the fp64 oracle's under the same masks and the
    GPU's ReLU decisions (the gradients to 2e-4)."""
    name, p = DROPOUT_CASES[case]
    c = variant(name)
    model, sd, ds, feats, rb, pb, groups, w = _case(c, p, segments=2)
    model.train()
    rg, pg = _graphs(rb, pb)
    lay = Layout(rb, pb)
    torch.manual_seed(17)
    out = model(rg, pg, gpu=GPU, add_features=feats)
    seed = int(out.grad_fn.cfg.seed)
    assert seed != 0 and abs(out.grad_fn.cfg.diff_dropout - p[1]) < 1e-7 and abs(out.grad_fn.cfg.ffn_dropout - p[2]) < 1e-7
    buf = saved_buffers(model, out, c, lay)
    keeps = site_keeps(seed, c, p, lay)
    for site, keep in keeps.items():
        assert not bool(((buf[site] != 0) & ~keep).any()), f"{site}: an entry the host mask drops survived"
    relu = relu_masks_and_keeps(buf, keeps, c, lay)
    (out * w.to(out.device)).sum().backward()
    got = {k: q.grad.double().cpu().numpy() for k, q in model.named_parameters() if q.requires_grad}
    pm = dict(e=p[0], d=p[1], f=p[2])
    drops = [(keeps[site][grp[key]], pm[mod]) if site in keeps else None
             for grp in lay.groups for site, key, mod, kind in site_order(c) if kind != "pre"]
    ws, wg, flips = oracle_run(sd, c, groups, w, drops, relu)
    e_s = rel_err(out.detach().cpu().numpy(), ws)
    assert e_s < TOL[gemm_mode]["score"], e_s
    n_pre = sum(int(m.numel()) for m in relu[0])
    assert flips <= max(8, 2e-4 * n_pre), (flips, n_pre)
    gscale = max(float(np.abs(v).max()) for v in wg.values())
    live = {k: wg[k] for k in got if float(np.abs(wg[k]).max()) >= 1e-6 * gscale}
    assert not grads_close(got, live, 2e-4), (flips, grads_close(got, live, 2e-4))


# ------------------------------------------------------------------------------------------------
# 3. padding rows on the tensor-core path
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["ddepth0", "w300_600_300_n320"])
def test_padding_rows_are_exact_on_the_tensor_core_path(name, tc_mode):
    """Every segment's padding rows of the encoder's messages and hiddens and of hid2 equal the fp64 oracle to fp32 rounding (5e-7 of the
    row's maximum, 1e-6 for hid2) with three segments in one launch: k_pad_rows_linear recomputes them at each sub-module's own width,
    and at diff depth 0 after the diff encoder's W_i."""
    c = variant(name, sizes=(6, 4, 5), atoms=(12, 28))
    model, sd, ds, feats, rb, pb, groups, w = _case(c, (0.0, 0.0, 0.0), segments=3, seed=31)
    model.eval()
    for q in model.parameters():
        q.requires_grad_(True)
    rg, pg = _graphs(rb, pb)
    out = model(rg, pg, gpu=GPU, add_features=feats)
    wd, ld, _, _ = widths(c)
    sd64 = {k: v.double().cpu() for k, v in sd.items()}
    a0 = b0 = 0
    for s_, (r, q, f) in enumerate(groups):
        trace = {}
        oracle_forward(sd64, c, r, q, f, trace=trace)
        for site, rows, row0, key, mod in (("enc1.m1", pg.n_bonds, b0, "encoder.msg1", "e"), ("enc1.m2", pg.n_bonds, b0, "encoder.msg2", "e"),
                                           ("enc1.hid", pg.n_atoms, a0, "p_hiddens", "e"),
                                           ("hid2", pg.n_atoms, a0, "diff_encoder.atom_hiddens", "d")):
            got = model.saved_activation(out, site, rows, ld[mod])[row0, :wd[mod]].double().cpu()
            want = trace[key][0]
            err = float((got - want).abs().max()) / max(float(want.abs().max()), 1e-30)
            assert err <= (1e-6 if site == "hid2" else 5e-7), (s_, site, err)
        a0 += pb[s_].n_atoms
        b0 += pb[s_].n_bonds


# ------------------------------------------------------------------------------------------------
# 4. tied models: the _ex entry points compute what the ABI-3 ones do
# ------------------------------------------------------------------------------------------------
def _c5_step(L):
    """The c5 step (ListMLE h300 d3, dropout 0.1, 82 x 50 reactions) in deterministic mode: scores, loss, flat gradient and the launches of
    every kernel class."""
    from reactranker_b200.train.train_listwise import batch_loss
    sizes = [50] * 82
    ds = synthetic.make_dataset(4100, sizes)
    targets = torch.tensor(ds.lgk.astype(np.float32))
    torch.manual_seed(0)
    model = build_model(hidden_size=300, mpnn_depth=3, mpnn_diff_depth=3, ffn_depth=3, use_bias=True, dropout=0.1, task_num=1,
                        ffn_last_layer="with_softplus", add_features_dim=1).cuda(GPU).train()
    r_g, p_g = BatchMolGraph([ds.mols[t] for t in ds.rsmi]), BatchMolGraph([ds.mols[t] for t in ds.psmi])
    torch.manual_seed(5)
    torch.cuda.synchronize()
    _lib.profile_begin()
    out = model(r_g, p_g, gpu=GPU, add_features=ds.temp.reshape(-1, 1))
    loss = batch_loss("mle", out, sizes, targets, GPU)
    loss.backward()
    torch.cuda.synchronize()
    counts = {k: n for k, (_, n) in _lib.profile_end().items()}
    return out.detach().cpu(), loss.detach().cpu(), model._grad_flat.cpu(), counts


@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_tied_model_ex_path_equals_abi3_path(mode, monkeypatch):
    """For the c5 model in GEMM modes 0-3 (deterministic mode, so that a difference could only come from the code path), the _ex entry points
    the package calls and the ABI-3 entry points give bit-identical scores, loss and flat gradient, and the same launches per kernel class."""
    L = _lib.lib()
    _lib.check(L.rr_set_gemm_mode(mode))
    torch.use_deterministic_algorithms(True)
    try:
        ex = _c5_step(L)
        for f in ("rr_model_workspace_bytes", "rr_model_buffer_offset", "rr_model_forward", "rr_model_backward"):
            monkeypatch.setattr(L, f + "_ex", getattr(L, f))          # the same calls, through the ABI-3 entry points
        abi3 = _c5_step(L)
    finally:
        torch.use_deterministic_algorithms(False)
        _lib.check(L.rr_set_deterministic(0))
    for a, b, what in zip(ex, abi3, ("scores", "loss", "gradient")):
        assert torch.equal(a, b), what
    assert ex[3] == abi3[3] and sum(ex[3].values()) > 0


# ------------------------------------------------------------------------------------------------
# 5. deterministic mode
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,p", [("w300_600_300_n320", (0.1, 0.2, 0.3)), ("ddepth0", (0.1, 0.2, 0.3))])
def test_variant_is_bit_identical_in_deterministic_mode(name, p):
    """Three training steps with per-module dropout from the same weights and seed are bit-identical under
    torch.use_deterministic_algorithms(True): the scratch of every weight gradient and gather backward is sized at its own module's width."""
    c = variant(name)
    ds, feats = variant_dataset(c)
    r_g, p_g = BatchMolGraph([ds.mols[t] for t in ds.rsmi]), BatchMolGraph([ds.mols[t] for t in ds.psmi])
    n = sum(c["sizes"])
    w = torch.randn(n, generator=torch.Generator().manual_seed(1)).cuda(GPU)
    torch.use_deterministic_algorithms(True)
    runs = []
    try:
        for _ in range(3):
            torch.manual_seed(3)
            model = variant_model(c, p).cuda(GPU).train()
            torch.manual_seed(9)
            out = model(r_g, p_g, gpu=GPU, add_features=feats)
            (out * w).sum().backward()
            torch.cuda.synchronize()
            runs.append((out.detach().clone(), model._grad_flat.clone()))
    finally:
        torch.use_deterministic_algorithms(False)
        _lib.check(_lib.lib().rr_set_deterministic(0))
    for other in runs[1:]:
        assert torch.equal(runs[0][0], other[0]) and torch.equal(runs[0][1], other[1])


# ------------------------------------------------------------------------------------------------
# 6. de-duplicated reactants
# ------------------------------------------------------------------------------------------------
def test_dedup_of_an_untied_model():
    """Eval mode: an untied model (and one at diff depth 0) scores bit for bit the same with each reactant encoded once as with one copy per
    candidate.  Training with dropout in the FFN only still refuses de-duplicated reactants."""
    from reactranker_b200.data.load_reactions import Parsing_features
    for name in ("w40_64_24", "ddepth0"):
        c = variant(name, sizes=(6, 5, 7))
        ds, feats = variant_dataset(c)
        torch.manual_seed(3)
        model = variant_model(c, (0.0, 0.0, 0.2)).cuda(GPU).eval()
        fz = Parsing_features(ds.mols)            # store-backed batches: the molecule ids tell which reactants repeat
        r_b, p_b = fz.parsing_smiles(list(ds.rsmi)), fz.parsing_smiles(list(ds.psmi))
        dev = torch.device("cuda", GPU)
        res = []
        for dedup in (True, False):
            rg, pg = DeviceGraph.from_batches_dedup([r_b], [p_b], dev) if dedup else DeviceGraph.pair_from_batches([r_b], [p_b], dev)
            assert (getattr(rg, "atom_map", None) is not None) == dedup
            with torch.no_grad():
                res.append(model(rg, pg, gpu=GPU, add_features=feats).cpu())
        assert torch.equal(res[0], res[1]), name
        model.train()
        rg, pg = DeviceGraph.from_batches_dedup([r_b], [p_b], dev)
        with pytest.raises(_lib.RRError, match="dropout"):
            model(rg, pg, gpu=GPU, add_features=feats)


# ------------------------------------------------------------------------------------------------
# 7. train() end to end
# ------------------------------------------------------------------------------------------------
def test_train_an_untied_diff_depth0_model_and_reload_its_checkpoint(tmp_path):
    """train() for a few epochs on a synthetic frame with ReactionModel(64 / 48 / 32 wide, diff depth 0, per-module dropout): the loss
    stays finite, the checkpoint's state_dict has the module tree's keys (no diff_encoder.W_o) and another model of the same shape loads it
    and scores as the trained one does."""
    from reactranker_b200.data.load_reactions import Parsing_features
    from reactranker_b200.train.train_listwise import train
    from reactranker_b200.train.utils import build_lr_scheduler, build_optimizer
    from reactranker_b200.utils import load_checkpoint
    ds = synthetic.make_dataset(11, [10] * 30)
    fz = Parsing_features()
    for tok, m in ds.mols.items():
        fz.add(tok, m)
    df = ds.to_dataframe()
    groups = df.rsmi.unique()
    train_df, val_df = df[df.rsmi.isin(groups[:24])], df[df.rsmi.isin(groups[24:])]
    c = variant("ddepth0", he=64, hd=48, hf=32)
    torch.manual_seed(0)
    model = variant_model(c, (0.1, 0.2, 0.1))
    keys = set(model.state_dict())
    assert not any(k.startswith("diff_encoder.W_o") or k.startswith("diff_encoder.W_h") for k in keys)
    opt = build_optimizer(model)
    sched = build_lr_scheduler(opt, warmup_epochs=1, total_epochs=3, train_data_size=len(train_df), batch_size=60, init_lr=1e-4, max_lr=1e-3,
                               final_lr=1e-4)
    path = os.path.join(str(tmp_path), "0.pt")
    train(model, sched, train_df, val_df, path, opt, 3, fz, batch_size=60, seed=0, gpu=GPU, task_type="mle", writer=None, target_name="lgk",
          smiles_list=["rsmi_mapped", "psmi_mapped"], add_features_name="temp")
    assert os.path.exists(path)
    state = load_checkpoint(path)["state_dict"]
    assert set(state) == keys
    assert all(bool(torch.isfinite(v).all()) for v in state.values())
    m2 = variant_model(c, (0.1, 0.2, 0.1))
    m2.load_state_dict(state)
    m2 = m2.cuda(GPU).eval()
    model.load_state_dict(state)
    model.eval()
    r_b, p_b = BatchMolGraph([ds.mols[t] for t in ds.rsmi[:20]]), BatchMolGraph([ds.mols[t] for t in ds.psmi[:20]])
    with torch.no_grad():
        a = model(r_b, p_b, gpu=GPU, add_features=ds.temp[:20].reshape(-1, 1))
        b = m2(r_b, p_b, gpu=GPU, add_features=ds.temp[:20].reshape(-1, 1))
    assert torch.equal(a, b)
