"""Models that build_model does not make but ReactionModel does: diff depth 0 (no message passing in the difference encoder, mpn.py:220-221),
separate hidden sizes for the encoder / diff encoder / FFN, and biases switched off in one sub-module only.  No GPU here: the oracle reads
every parameter of each configuration, the C ABI sizes and refuses configurations without a device, and, where the reference is
installed, the oracle equals the reference's own modules.  tests/test_gpu_model_variants.py runs the same configurations on the GPU."""
import contextlib
import ctypes
import io
import os
import sys

import numpy as np
import pytest
import torch

from oracle import ref_loader
from oracle import reactranker_oracle as O
from reactranker_b200 import _lib, synthetic
from helpers import add_features

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# he / hd / hf: encoder, diff encoder and FFN hidden sizes; bias_e / bias_d / bias_f: mpnn_bias, mpnn_diff_bias, ffn_bias.
VARIANT_DEFAULTS = dict(he=40, hd=40, hf=40, depth=3, ddepth=3, ffn_depth=3, bias_e=True, bias_d=True, bias_f=True, add=1, task_num=1,
                        sizes=(7, 5, 9, 4), atoms=(12, 28))
VARIANTS = {
    "ddepth0": dict(ddepth=0),
    "ddepth0_depth1_ffn1": dict(ddepth=0, depth=1, ffn_depth=1),
    "ddepth0_ffn4": dict(ddepth=0, ffn_depth=4),
    "w40_64_24": dict(hd=64, hf=24),
    # >= 320 reactions: the FFN weight gradients run on the tensor cores too, so forward, dgrad and wgrad all meet non-square weights
    "w300_600_300_n320": dict(he=300, hd=600, hf=300, atoms=(3, 6), sizes=(40,) * 8),
    "w600_300_128_n320": dict(he=600, hd=300, hf=128, atoms=(3, 6), sizes=(40,) * 8),
    # encoder wider than the row pipeline takes (first-generation gathers), diff encoder on the row pipeline
    "w1040_300_300": dict(he=1040, hd=300, hf=300, depth=2, ddepth=2, sizes=(3, 2, 4)),
    # the readout vector hd + 3 add features crosses the padded width of hd (302 + 3 -> vp 320)
    "hd302_add3": dict(he=64, hd=302, hf=48, add=3, atoms=(3, 6)),
    "nobias_enc": dict(bias_e=False, hd=48),
    "nobias_diff": dict(bias_d=False, hd=48),
    "nobias_ffn": dict(bias_f=False, hf=24),
}


def variant(name, **over):
    """VARIANTS[name] with the defaults filled in (and ``over`` on top)."""
    c = dict(VARIANT_DEFAULTS, **VARIANTS[name])
    c.update(over)
    return c


def variant_model(c, p=(0.0, 0.0, 0.0)):
    """ReactionModel for a filled-in variant with dropouts p = (mpnn, mpnn_diff, ffn); the head is the raw output."""
    from reactranker_b200.models.base_model import ReactionModel
    return ReactionModel(mpnn_hidden_size=c["he"], mpnn_bias=c["bias_e"], mpnn_depth=c["depth"], mpnn_dropout=p[0],
                         mpnn_diff_hidden_size=c["hd"], mpnn_diff_bias=c["bias_d"], mpnn_diff_depth=c["ddepth"], mpnn_diff_dropout=p[1],
                         ffn_hidden_size=c["hf"], ffn_bias=c["bias_f"], ffn_dropout=p[2], ffn_depth=c["ffn_depth"], task_num=c["task_num"],
                         task_type="with_softplus", addtion_react_featrues=c["add"])


def variant_dataset(c, seed=61):
    ds = synthetic.make_dataset(seed, list(c["sizes"]), atoms_lo=c["atoms"][0], atoms_hi=c["atoms"][1])
    return ds, add_features(ds, c["add"])


def oracle_forward(sd, c, r_batch, p_batch, feats, training=False, trace=None):
    """The oracle's model_forward for a variant; its widths follow the shapes in ``sd``.  ``training`` makes it call its dropout at every
    site with p = 0: a caller that replaces the oracle's ``_drop`` gives each site its own module's mask and p
    (tests/test_gpu_model_variants.py::oracle_drops)."""
    return O.model_forward(sd, r_batch, p_batch, feats, mpnn_depth=c["depth"], mpnn_diff_depth=c["ddepth"], ffn_depth=c["ffn_depth"],
                           head="with_softplus", training=training, trace=trace)


@pytest.mark.parametrize("name", list(VARIANTS))
def test_oracle_reads_every_parameter_of_each_variant(name):
    """The fp64 oracle run on the model's state_dict gives every trainable parameter a gradient and reads no key the model lacks (at diff
    depth 0 there is no diff_encoder.W_o / W_h); the parameter shapes are the reference's for separate widths."""
    c = variant(name)
    ds, feats = variant_dataset(c)
    torch.manual_seed(3)
    model = variant_model(c)
    sd = {k: v.double() for k, v in model.state_dict().items()}
    he, hd, hf = c["he"], c["hd"], c["hf"]
    assert tuple(sd["diff_encoder.W_i.weight"].shape) == (hd, he)
    assert tuple(sd["diff_encoder.cached_zero_vector"].shape) == (hd,)
    assert tuple(sd["ffn.ffn.1.weight"].shape) == ((c["task_num"] if c["ffn_depth"] == 1 else hf), hd + c["add"])
    assert ("diff_encoder.W_o.weight" in sd) == (c["ddepth"] > 0) and ("diff_encoder.W_h.weight" in sd) == (c["ddepth"] > 1)
    if c["ddepth"] > 0:
        assert tuple(sd["diff_encoder.W_o.weight"].shape) == (hd, he + hd)
    if c["ddepth"] > 1:
        assert tuple(sd["diff_encoder.W_h.weight"].shape) == (hd, hd + O.FBOND_TOTAL)
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items() if "cached_zero" not in k}
    full = dict(sd, **params)
    read = set()

    class Tracking(dict):
        def __getitem__(self, k):
            read.add(k)
            return dict.__getitem__(self, k)

        def get(self, k, default=None):
            if k in self:
                read.add(k)
            return dict.get(self, k, default)
    out = oracle_forward(Tracking(full), c, O.OracleBatch([ds.mols[t] for t in ds.rsmi]), O.OracleBatch([ds.mols[t] for t in ds.psmi]), feats)
    n = sum(c["sizes"])
    assert tuple(out.shape) == ((n,) if c["task_num"] == 1 else (n, c["task_num"]))
    (out * torch.randn(out.shape, generator=torch.Generator().manual_seed(1), dtype=torch.float64)).sum().backward()
    trainable = {k for k, q in model.named_parameters() if q.requires_grad}
    assert trainable == set(params)
    assert read - set(sd) == set() and trainable <= read, (sorted(trainable - read), sorted(read - set(sd)))
    for k in sorted(trainable):
        assert params[k].grad is not None, k
        assert bool(torch.isfinite(params[k].grad).all()), k


# ------------------------------------------------------------------------------------------------
# C ABI without a device: sizing and argument checks run on the host before anything is enqueued
# ------------------------------------------------------------------------------------------------
def _graphs(n_atoms=40, n_bonds=70, n_mols=6):
    from reactranker_b200.features.featurization import RRGraph
    r, p = RRGraph(), RRGraph()
    for q in (r, p):
        q.n_atoms, q.n_bonds, q.n_mols, q.wmax, q.n_segments = n_atoms, n_bonds, n_mols, 4, 1
    return r, p


def _cfg_ex(hidden=300, diff_hidden=300, ffn_hidden=300, dropout=0.1, diff_dropout=0.1, ffn_dropout=0.1, diff_depth=3, training=1):
    base = _lib.RRModelCfg(hidden, 3, diff_depth, 3, 1, 1, _lib.HEAD_RAW, training, dropout, 7)
    return _lib.RRModelCfgEx(base, diff_hidden, ffn_hidden, diff_dropout, ffn_dropout)


def _ws_ex(cfg, r, p):
    return _lib.lib().rr_model_workspace_bytes_ex(ctypes.byref(cfg), ctypes.byref(r), ctypes.byref(p))


def test_tied_extension_sizes_the_abi3_workspace():
    """rr_model_workspace_bytes_ex with diff/ffn widths and dropouts equal to the encoder's gives rr_model_workspace_bytes, in both
    deterministic settings; the ex struct's base is an rr_model_cfg the ABI-3 entry point reads as is."""
    L = _lib.lib()
    r, p = _graphs()
    try:
        for det in (0, 1):
            _lib.check(L.rr_set_deterministic(det))
            for h, dd in ((300, 3), (40, 1), (1040, 2), (302, 0)):
                cfg = _cfg_ex(h, h, h, diff_depth=dd)
                want = L.rr_model_workspace_bytes(ctypes.byref(cfg.base), ctypes.byref(r), ctypes.byref(p))
                assert want > 0
                assert _ws_ex(cfg, r, p) == want
                assert L.rr_model_workspace_bytes(ctypes.byref(cfg), ctypes.byref(r), ctypes.byref(p)) == want
    finally:
        _lib.check(L.rr_set_deterministic(0))


def test_diff_depth_zero_workspace_is_smaller():
    """At diff depth 0 the diff encoder keeps no inp2 / nf / am2 / messages: its workspace is smaller than depth 1's, and the names of
    those buffers are refused (-1 with a message) while hid2 is still there."""
    L = _lib.lib()
    r, p = _graphs()
    for widths in ((300, 300, 300), (64, 128, 32)):
        d0, d1 = _cfg_ex(*widths, diff_depth=0), _cfg_ex(*widths, diff_depth=1)
        assert 0 < _ws_ex(d0, r, p) < _ws_ex(d1, r, p)
        for name in (b"inp2", b"nf", b"am2"):
            assert L.rr_model_buffer_offset_ex(ctypes.byref(d0), ctypes.byref(r), ctypes.byref(p), name) == -1
            assert name.decode() in L.rr_last_error().decode()
            assert L.rr_model_buffer_offset_ex(ctypes.byref(d1), ctypes.byref(r), ctypes.byref(p), name) > 0
        assert L.rr_model_buffer_offset_ex(ctypes.byref(d0), ctypes.byref(r), ctypes.byref(p), b"hid2") > 0


def test_untied_workspace_follows_each_width():
    """Growing one sub-module's width grows the workspace; the same widths in another order give another size."""
    r, p = _graphs()
    base = _ws_ex(_cfg_ex(64, 64, 64), r, p)
    for w in ((128, 64, 64), (64, 128, 64), (64, 64, 128)):
        assert _ws_ex(_cfg_ex(*w), r, p) > base, w
    assert _ws_ex(_cfg_ex(64, 128, 32), r, p) != _ws_ex(_cfg_ex(32, 128, 64), r, p)


BAD = [("diff_hidden", dict(diff_hidden=0), "diff_hidden"), ("diff_hidden", dict(diff_hidden=4097), "diff_hidden"),
       ("ffn_hidden", dict(ffn_hidden=-1), "ffn_hidden"), ("ffn_hidden", dict(ffn_hidden=5000), "ffn_hidden"),
       ("diff_dropout", dict(diff_dropout=1.0), "diff_dropout"), ("diff_dropout", dict(diff_dropout=-0.1), "diff_dropout"),
       ("ffn_dropout", dict(ffn_dropout=1.5), "ffn_dropout"), ("ffn_dropout", dict(ffn_dropout=float("nan")), "ffn_dropout")]


@pytest.mark.parametrize("field,kw,msg", BAD, ids=[f"{f}={list(k.values())[0]}" for f, k, _ in BAD])
def test_out_of_range_extension_is_refused_before_any_launch(field, kw, msg):
    """rr_model_forward_ex / rr_model_backward_ex refuse an out-of-range width or dropout with RR_ERR_INVALID and a message naming the
    field, before anything is enqueued (the pointers here are not device memory, and the launch counter does not move)."""
    L = _lib.lib()
    r, p = _graphs()
    fake = 1 << 20                                  # 16-byte aligned, never dereferenced: the checks run first
    for q in (r, p):
        q.f_atoms = q.f_bonds = fake
    w = _lib.RRParams()
    for slot in ("enc_Wi", "enc_Wh", "enc_Wo", "enc_bo", "dif_Wi", "dif_Wh", "dif_Wo", "dif_bo"):
        setattr(w, slot, fake)
    for l in range(3):
        w.ffn_W[l] = fake
    cfg = _cfg_ex(**kw)
    L.rr_launch_count_reset()
    big = 1 << 40
    st = L.rr_model_forward_ex(ctypes.byref(cfg), ctypes.byref(w), ctypes.byref(r), ctypes.byref(p), fake, fake, fake, big, None)
    assert st == -1 and msg in L.rr_last_error().decode(), (st, L.rr_last_error())
    st = L.rr_model_backward_ex(ctypes.byref(cfg), ctypes.byref(w), ctypes.byref(r), ctypes.byref(p), fake, ctypes.byref(w), fake, big, None)
    assert st == -1 and msg in L.rr_last_error().decode(), (st, L.rr_last_error())
    assert L.rr_launch_count() == 0
    if "hidden" in field:
        assert _ws_ex(cfg, r, p) == -1 and msg in L.rr_last_error().decode()


def test_dedup_refused_while_any_module_trains_with_dropout():
    """r_atom_map (de-duplicated reactants) is refused in training whenever any sub-module has dropout, and allowed in eval mode."""
    L = _lib.lib()
    r, p = _graphs()
    amap = (ctypes.c_int32 * 40)()
    for d in ((0.0, 0.0, 0.2), (0.0, 0.2, 0.0), (0.2, 0.0, 0.0)):
        for training, ok in ((1, False), (0, True)):
            cfg = _cfg_ex(64, 48, 32, *d, training=training)
            cfg.r_atom_map = ctypes.addressof(amap)
            assert (_ws_ex(cfg, r, p) > 0) == ok, (d, training)
    cfg = _cfg_ex(64, 48, 32, 0.0, 0.0, 0.0)
    cfg.r_atom_map = ctypes.addressof(amap)
    assert _ws_ex(cfg, r, p) > 0


def test_reaction_model_builds_every_variant_and_keeps_build_model_tied():
    """ReactionModel accepts separate widths, dropouts and biases and diff depth 0; build_model still ties them."""
    from reactranker_b200.models.base_model import build_model, reactant_dedup_exact
    c = variant("w40_64_24")
    m = variant_model(c, p=(0.0, 0.0, 0.3))
    assert (m._he, m._hd, m._hf, m._pe, m._pd, m._pf) == (40, 64, 24, 0.0, 0.0, 0.3)
    assert reactant_dedup_exact(m.eval()) and not reactant_dedup_exact(m.train())
    m0 = variant_model(variant("ddepth0"))
    assert not hasattr(m0.diff_encoder, "W_o") and [k for k, _ in m0._named_slots()][-8:-6] == ["dif_Wi", "dif_bi"]
    b = build_model(hidden_size=32, mpnn_diff_depth=0, dropout=0.1)
    assert (b._he, b._hd, b._hf, b._pe, b._pd, b._pf) == (32, 32, 32, 0.1, 0.1, 0.1) and not hasattr(b.diff_encoder, "W_o")
    cfg = b._cfg(training=True)
    assert (cfg.hidden, cfg.diff_hidden, cfg.ffn_hidden, cfg.diff_depth) == (32, 32, 32, 0)
    assert cfg.seed != 0 and abs(cfg.dropout - 0.1) < 1e-7 and abs(cfg.ffn_dropout - 0.1) < 1e-7


# ------------------------------------------------------------------------------------------------
# the oracle against the reference's own modules, where the reference is installed
# ------------------------------------------------------------------------------------------------
@pytest.mark.skipif(not ref_loader.available(), reason="needs the original ReactRanker source (set RR_REFERENCE_ROOT)")
@pytest.mark.parametrize("name", ["ddepth0", "w40_64_24"])
def test_oracle_equals_live_reference(name):
    """The reference's own ReactionModel built with the variant's widths, depths and biases (mpn.py:220-221 at diff depth 0), in fp64:
    the oracle on its state_dict gives its scores and, under a fixed random weighting of the outputs, its gradients."""
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_golden as MG
    c = variant(name)
    bm = ref_loader.ref("models.base_model")
    torch.manual_seed(3)
    model = bm.ReactionModel(mpnn_hidden_size=c["he"], mpnn_bias=c["bias_e"], mpnn_depth=c["depth"], mpnn_dropout=0.0,
                             mpnn_diff_hidden_size=c["hd"], mpnn_diff_bias=c["bias_d"], mpnn_diff_depth=c["ddepth"], mpnn_diff_dropout=0.0,
                             ffn_hidden_size=c["hf"], ffn_bias=c["bias_f"], ffn_dropout=0.0, ffn_depth=c["ffn_depth"], task_num=c["task_num"],
                             task_type="with_softplus", addtion_react_featrues=c["add"]).to(torch.float64).train()
    ds, fz = MG.dataset_case(404, [4, 1, 7, 3], {2: 6})
    r_g, p_g = fz.parsing_reactions(np.stack([ds.rsmi, ds.psmi], axis=1))
    for g in (r_g, p_g):
        g.f_atoms, g.f_bonds = g.f_atoms.to(torch.float64), g.f_bonds.to(torch.float64)
    feats = add_features(ds, c["add"])
    orig = torch.FloatTensor            # mpn.py:183 casts add_features with FloatTensor (fp32); lift the result to fp64
    torch.FloatTensor = lambda x: torch.tensor(np.asarray(x, np.float32), dtype=torch.float64)  # type: ignore
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            want = model(r_g, p_g, gpu=None, add_features=feats)
    finally:
        torch.FloatTensor = orig  # type: ignore
    up = torch.randn(want.shape, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    (want * up).sum().backward()
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items() if "cached_zero" not in k}
    full = dict(sd, **params)
    got = oracle_forward(full, c, O.OracleBatch([ds.mols[t] for t in ds.rsmi]), O.OracleBatch([ds.mols[t] for t in ds.psmi]), feats)
    assert tuple(got.shape) == tuple(want.shape)
    assert float((got - want).abs().max()) <= 1e-10 * max(1.0, float(want.abs().max()))
    (got * up).sum().backward()
    ref_grads = {k: q.grad for k, q in model.named_parameters() if q.grad is not None}
    assert set(ref_grads) == set(params)
    gscale = max(float(g.abs().max()) for g in ref_grads.values())
    for k, g in ref_grads.items():
        assert float((params[k].grad - g).abs().max()) <= 1e-9 * gscale, k
