"""CPU tests of the host-side mirror: bit-exact batching vs the reference goldens, the device
packing, the C-ABI surface (symbols only -- no compute without a GPU) and the schedule."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from reactranker_b200 import _lib, synthetic
from reactranker_b200.features.featurization import BatchMolGraph, DeviceGraph, MolGraph
from helpers import star_dict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_batching_bit_exact_vs_reference_golden(golden):
    g = golden("batching")
    for name in ("plain", "star"):
        ds = synthetic.make_dataset(int(g[name + ".seed"]), [int(x) for x in g[name + ".sizes"]],
                                    star_leaves_in_group=star_dict(g[name + ".star"]))
        for side, col in (("r", ds.rsmi), ("p", ds.psmi)):
            b = BatchMolGraph([ds.mols[t] for t in col])
            pre = f"{name}.{side}."
            fa, fb, a2b, b2a, b2revb, a_scope, b_scope = b.get_components()
            for got, key in ((fa, "f_atoms"), (fb, "f_bonds"), (a2b, "a2b"), (b2a, "b2a"), (b2revb, "b2revb"), (b.get_a2a(), "a2a")):
                want = g[pre + key]
                assert got.numpy().dtype == want.dtype and np.array_equal(got.numpy(), want), key
            assert np.array_equal(np.asarray(a_scope), g[pre + "a_scope"])
            assert np.array_equal(np.asarray(b_scope), g[pre + "b_scope"])
            assert b.max_num_bonds == int(g[pre + "max_num_bonds"])
            assert b.n_atoms == want_rows(g, pre, "f_atoms") and b.n_bonds == want_rows(g, pre, "f_bonds")


def want_rows(g, pre, key):
    return g[pre + key].shape[0]


def test_molgraph_list_roundtrip():
    """A molecule given as python lists (the reference's MolGraph attributes) batches identically."""
    ds = synthetic.make_dataset(3, [2, 2])
    class Lists:  # what a reference MolGraph looks like
        pass
    mols = []
    for t in ds.psmi:
        m = ds.mols[t]
        o = Lists()
        o.smiles, o.n_atoms, o.n_bonds = m.smiles, m.n_atoms, m.n_bonds
        o.f_atoms, o.f_bonds, o.a2b, o.b2a, o.b2revb = m.f_atoms, m.f_bonds, m.a2b, m.b2a, m.b2revb
        mols.append(o)
    a = BatchMolGraph(mols)
    b = BatchMolGraph([ds.mols[t] for t in ds.psmi])
    for x, y in zip(a.get_components()[:5], b.get_components()[:5]):
        assert torch.equal(x, y)


def test_empty_and_degenerate_batches():
    rng = np.random.default_rng(0)
    single = synthetic.make_molecule(rng, 1, "lonely")        # one atom, no bonds
    b = BatchMolGraph([single])
    assert b.n_atoms == 2 and b.n_bonds == 1 and b.max_num_bonds == 1
    assert b.a2b.shape == (2, 1) and int(b.a2b.abs().sum()) == 0
    e = BatchMolGraph([])
    assert e.n_atoms == 1 and e.n_bonds == 1 and e.a_scope == []


def test_device_graph_layout_single_and_multi_segment():
    ds = synthetic.make_dataset(5, [3, 2], star_leaves_in_group={1: 6})
    b1 = BatchMolGraph([ds.mols[t] for t in ds.psmi[:3]])
    b2 = BatchMolGraph([ds.mols[t] for t in ds.rsmi[3:]])       # the star reactant, repeated per candidate
    one = DeviceGraph.from_batches([b1], "cpu")
    meta = one.section("a_meta", torch.int32, (b1.n_atoms, 4)).numpy()
    assert meta[0, 0] == 0x100 and meta[0, 1] == b1.max_num_bonds
    assert np.array_equal(meta[1:, 0], b1._deg[1:]) and np.array_equal(meta[:, 1], b1.max_num_bonds - b1._deg)
    a2b = one.section("a2b", torch.int32, (b1.n_atoms, one.c.wmax)).numpy()
    assert np.array_equal(a2b, b1.a2b.numpy()[:, :one.c.wmax])
    fb = one.section("f_bonds", torch.float32, (b1.n_bonds, 88)).numpy()
    assert np.array_equal(fb[:, :83], b1.f_bonds.numpy()) and not fb[:, 83:].any()
    both = DeviceGraph.from_batches([b1, b2], "cpu")
    assert both.c.n_segments == 2 and both.n_atoms == b1.n_atoms + b2.n_atoms
    meta = both.section("a_meta", torch.int32, (both.n_atoms, 4)).numpy()
    assert meta[b1.n_atoms, 0] == 0x100 and meta[b1.n_atoms, 2] == b1.n_bonds and meta[b1.n_atoms, 3] == b1.n_atoms
    assert meta[b1.n_atoms, 1] == b2.max_num_bonds == 6           # each segment keeps ITS max_num_bonds
    a2a = both.section("a2a", torch.int32, (both.n_atoms, both.c.wmax)).numpy()
    d2 = b2._deg
    want = b2.get_a2a().numpy() + b1.n_atoms
    for a in range(b2.n_atoms):
        assert np.array_equal(a2a[b1.n_atoms + a, :d2[a]], want[a, :d2[a]])
    with pytest.raises(ValueError):
        DeviceGraph.from_batches([b2], "cpu", [3])


def test_c_abi_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "rr_sm100.h")).read()
    declared = set(re.findall(r"\b(rr_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    _lib.build()
    L = ctypes.CDLL(_lib.SO_PATH)
    for name in declared:
        assert hasattr(L, name), name
    assert L.rr_version() == 3
    assert L.rr_padded(300) == 304 and L.rr_padded(600) == 608 and L.rr_padded(40) == 48
    L.rr_loss_max_group.restype = ctypes.c_int
    assert L.rr_loss_max_group() >= 500           # config 5 sweeps groups of 50..500 candidates


def test_no_cpu_fallback():
    from reactranker_b200.models.base_model import build_model
    ds = synthetic.make_dataset(1, [2])
    m = build_model(hidden_size=16, task_num=1, add_features_dim=0, dropout=0.0)
    b = BatchMolGraph([ds.mols[t] for t in ds.psmi])
    with pytest.raises(_lib.RRError):
        m(b, b, gpu=None)
    if not torch.cuda.is_available():
        with pytest.raises(_lib.RRError):
            m(b, b, gpu=0)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "reactranker_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "/root/reference" not in src, f


def test_noam_matches_reference_golden(golden):
    from reactranker_b200.train.utils import build_lr_scheduler, build_optimizer
    g = golden("steps")
    lin = torch.nn.Linear(2, 2)
    opt = build_optimizer(lin)
    sched = build_lr_scheduler(opt, warmup_epochs=2, total_epochs=4, train_data_size=30, batch_size=10,
                               init_lr=1e-4, max_lr=1e-3, final_lr=1e-4)
    lrs = [opt.param_groups[0]["lr"]]
    for _ in range(3):
        sched.step()
        lrs.append(opt.param_groups[0]["lr"])
    assert np.allclose(lrs, g["lrs"], rtol=1e-12)
    assert opt.defaults["weight_decay"] == 0 and opt.param_groups[0]["weight_decay"] == 0


def test_state_dict_keys_and_init_match_reference_golden(golden):
    """Same 20 keys/shapes as the reference and, under the same torch seed, the same default init."""
    from reactranker_b200.models.base_model import build_model
    g = golden("model")
    name = "mle.h40"
    hidden, seed, depth, ddepth = (int(x) for x in g[name + ".meta"])
    torch.manual_seed(seed)
    m = build_model(hidden_size=hidden, mpnn_depth=depth, mpnn_diff_depth=ddepth, ffn_depth=3, use_bias=True, dropout=0.0,
                    task_num=1, ffn_last_layer="with_softplus", add_features_dim=1)
    sd = m.state_dict()
    want = {k[len(name) + 4:]: g[k] for k in g.files if k.startswith(name + ".sd.")}
    assert set(sd) == set(want) and len(sd) == 20
    for k, v in want.items():
        assert np.array_equal(sd[k].numpy(), v), k


def test_planner_bit_exact_vs_reference_golden(golden):
    """DataProcessor.generate_batch_reactions / generate_batch_per_query reproduce the row order and
    scope the reference produced (incl. the truncating `sample(n=idx)` branch) for several seeds."""
    from reactranker_b200.data.load_reactions import DataProcessor
    g = golden("planner")
    ds = synthetic.make_dataset(int(g["seed"]), [int(x) for x in g["sizes"]], atoms_lo=3, atoms_hi=4)
    df = ds.to_dataframe()
    row_of = {p: i for i, p in enumerate(ds.psmi)}
    dp = DataProcessor(df)
    for bs in (50, 24, 64):
        for seed in (0, 1, 5):
            rows, scopes, steps = [], [], []
            for smiles, targets, scope, feats in dp.generate_batch_reactions(
                    smiles_list=["rsmi_mapped", "psmi_mapped"], target_name="lgk", batch_size=bs, seed=seed, add_features_name="temp"):
                ids = [row_of[s[1]] for s in smiles]
                assert targets.shape == (len(ids), 1) and feats.shape == (len(ids), 1)
                assert np.array_equal(targets[:, 0], ds.lgk[ids]) and np.array_equal(feats[:, 0], ds.temp[ids])
                rows += ids
                scopes += list(scope)
                steps.append((len(ids), len(scope)))
            key = f"reactions.bs{bs}.seed{seed}."
            assert np.array_equal(rows, g[key + "rows"]) and np.array_equal(scopes, g[key + "scope"])
            assert np.array_equal(np.asarray(steps), g[key + "steps"])
    for seed in (0, 3):
        rows, lens = [], []
        for smiles, targets, feats in dp.generate_batch_per_query(smiles_list=["rsmi_mapped", "psmi_mapped"], target_name="lgk",
                                                                  seed=seed, add_features_name="temp"):
            ids = [row_of[s[1]] for s in smiles]
            assert np.array_equal(feats[:, 0], ds.lgk[ids])        # the target-column leak is preserved
            rows += ids
            lens.append(len(ids))
        assert np.array_equal(rows, g[f"per_query.seed{seed}.rows"]) and np.array_equal(lens, g[f"per_query.seed{seed}.lens"])


def test_parsing_features_builds_reference_batches():
    from reactranker_b200.data.load_reactions import Parsing_features
    ds = synthetic.make_dataset(8, [3, 2])
    fz = Parsing_features(ds.mols)
    r, p = fz.parsing_reactions(np.stack([ds.rsmi, ds.psmi], 1))
    assert r.n_mols == p.n_mols == 5 and r.n_atoms == p.n_atoms
    assert fz.parsing_reactions(None) == [None, None] and fz.parsing_smiles(None) is None


def test_lookahead_prepares_one_batch_ahead():
    """data/prefetch.py: ``current`` is ready at construction, ``advance`` prepares exactly one more item, exhaustion gives None."""
    from reactranker_b200.data.prefetch import Lookahead
    seen = []

    def prep(x):
        seen.append(x)
        return x * 10
    feed = Lookahead(iter(range(3)), prep)
    assert feed.current == 0 and seen == [0]
    feed.advance()
    assert feed.current == 10 and seen == [0, 1]
    feed.advance()
    feed.advance()
    assert feed.current is None and seen == [0, 1, 2]
    with pytest.raises(ValueError):
        Lookahead(iter([1]), lambda x: (_ for _ in ()).throw(ValueError("bad batch")))


def test_molecule_store_registration_is_thread_safe():
    """Molecules may be registered from a data-loading thread while the training thread reads the store tables."""
    import threading
    from reactranker_b200 import synthetic
    from reactranker_b200.data.load_reactions import Parsing_features
    ds = synthetic.make_dataset(5, [40, 40, 40])
    fz = Parsing_features()
    for tok, m in ds.mols.items():
        fz.add(tok, m)
    toks = list(ds.psmi)
    out = {}

    def run(k):
        out[k] = fz.parsing_smiles(toks[k::4])
    threads = [threading.Thread(target=run, args=(k,)) for k in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    st = fz.store
    n = len(st)
    assert n == len(set(toks)) and len({id(p) for p in st.packs}) == n
    assert np.array_equal(st.aoff[:n], np.concatenate(([0], np.cumsum(st.nA[:n])[:-1])))
    for k in range(4):
        want = BatchMolGraph([ds.mols[t] for t in toks[k::4]])
        assert out[k].n_atoms == want.n_atoms and torch.equal(out[k].a2b, want.a2b) and torch.equal(out[k].f_bonds, want.f_bonds)


# ---- evaluation metrics vs the reference's own functions (tests/golden/metrics.npz: tests/golden/make_golden.py golden_metrics) ----------
class _StubScorer(torch.nn.Module):
    """Same deterministic scorer the golden was generated with (scores from the product token + the extra feature)."""

    def __init__(self, two):
        super().__init__()
        self.two = two

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
        return torch.stack((base, 0.5 + base.abs()), dim=1) if self.two else base


@pytest.mark.parametrize("two", [False, True])
def test_eval_metrics_match_reference_golden(two):
    """The oracle's per-group metric restatement (what the GPU kernel rr_rank_metrics is checked against) reproduces the reference's
    ranking_metrics / evaluate_top_scores return values, and calculate_ndcg (host report arithmetic) its tables."""
    from oracle import reactranker_oracle as O
    from reactranker_b200.data.load_reactions import DataProcessor, Parsing_features
    from reactranker_b200.train import eval as E
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "metrics.npz"))
    ds = synthetic.make_dataset(int(g["seed"]), [int(x) for x in g["sizes"]], atoms_lo=3, atoms_hi=4)
    fz = Parsing_features(ds.mols)
    dp = DataProcessor(ds.to_dataframe())
    cols = ["rsmi_mapped", "psmi_mapped"]
    m = _StubScorer(two).eval()
    tag = "two." if two else "one."

    def score(X, feats):
        p = m(None, fz.parsing_smiles([s[1] for s in X]), add_features=feats)
        return (p[:, 0] if p.dim() > 1 else p).numpy()
    rows = []
    for X, t, scope, feats in dp.generate_batch_querys(smiles_list=cols, target_name="lgk", batch_size=3, shuffle_query=False, shuffle_batch=False,
                                                       add_features_name="temp"):
        p, t, o = score(X, feats), np.asarray(t, np.float64).reshape(-1), 0
        for n in scope:
            rows.append(O.group_metrics(p[o:o + n], t[o:o + n], 0.25))
            o += n
    rows = np.asarray(rows)
    assert np.allclose([rows[:, 0].mean(), rows[:, 1].mean(), rows[:, 3].mean()], g[tag + "top_scores"], rtol=0, atol=1e-12)
    rows = np.asarray([O.group_metrics(score(X, feats), np.asarray(t, np.float64).reshape(-1), 0.25)
                       for X, t, feats in dp.generate_batch_per_query(smiles_list=cols, target_name="lgk", shuffle_query=False, shuffle_batch=False,
                                                                      add_features_name="temp")])
    got = [rows[:, 0].mean(), rows[:, 1].mean(), rows[:, 2].mean()] + list(rows[:, 4:8].mean(axis=0))
    assert np.allclose(got, g[tag + "ranking"], rtol=1e-12, atol=1e-12)
    for means, stds, name in ((None, None, "raw"), (0.7, 1.9, "scaled")):
        nd, kl, order, smi = E.calculate_ndcg(m, gpu=None, data_processor=dp, smiles2graph_dic=fz, batch_size=3, NDCG_cut=0.25, smiles_list=cols,
                                              target_name="lgk", means=means, stds=stds, add_features_name="temp")
        assert np.allclose([nd, kl], g[tag + name + ".ndcg_kl"], rtol=1e-6)
        assert np.allclose(np.asarray(order), g[tag + name + ".order"], rtol=1e-6, atol=1e-6)
        assert [x[0] for x in smi] == g[tag + name + ".smi_iter"].tolist() and [x[2] for x in smi] == g[tag + name + ".smi_p"].tolist()
    nd, kl, rows, smi = E.calculate_ndcg(m, gpu=None, data_processor=dp, smiles2graph_dic=fz, batch_size=3, NDCG_cut=0.25, smiles_list=cols,
                                         target_name="lgk", is_order=False, add_features_name="temp")
    assert nd is None and kl is None
    assert np.allclose(np.asarray(rows), g[tag + "unordered.rows"], rtol=1e-6, atol=1e-6) and [x[1] for x in smi] == g[tag + "unordered.smi_p"].tolist()


def test_dedup_plan_maps_every_product_atom_to_its_reactant_row():
    """DeviceGraph.dedup_plan: unique reactants per segment in order of first appearance, padding rows map to padding rows, and every
    product atom row maps to the row its own (repeated) reactant would have had."""
    from reactranker_b200.data.load_reactions import Parsing_features
    ds = synthetic.make_dataset(12, [4, 1, 3])
    fz = Parsing_features(ds.mols)
    groups = [(0, 4), (4, 5), (5, 8)]
    r_b = [fz.parsing_smiles(list(ds.rsmi[a:b])) for a, b in groups]
    p_b = [fz.parsing_smiles(list(ds.psmi[a:b])) for a, b in groups]
    uniq, w, amap = DeviceGraph.dedup_plan(r_b, p_b)
    assert [u.n_mols for u in uniq] == [1, 1, 1] and w == [b.max_num_bonds for b in r_b]
    assert amap.shape[0] == sum(b.n_atoms for b in p_b)
    # brute force: features of the mapped reactant row == features of the row in the un-deduplicated reactant batch
    full = np.concatenate([b.f_atoms.numpy() for b in r_b])
    dedup = np.concatenate([u.f_atoms.numpy() for u in uniq])
    assert np.array_equal(dedup[amap], full)
    a0_p = np.cumsum([0] + [b.n_atoms for b in p_b])[:-1]
    a0_u = np.cumsum([0] + [u.n_atoms for u in uniq])[:-1]
    assert np.array_equal(amap[a0_p], a0_u)                       # segment padding atoms
    # nothing repeats -> no plan; a whole batch with two different reactants keeps both, first appearance first
    assert DeviceGraph.dedup_plan([fz.parsing_smiles([ds.rsmi[0]])], [fz.parsing_smiles([ds.psmi[0]])]) is None
    rb, pb = fz.parsing_smiles(list(ds.rsmi)), fz.parsing_smiles(list(ds.psmi))
    uniq, w, amap = DeviceGraph.dedup_plan([rb], [pb])
    assert uniq[0].n_mols == 3 and uniq[0].smiles_batch == [ds.rsmi[0], ds.rsmi[4], ds.rsmi[5]]
    assert np.array_equal(uniq[0].f_atoms.numpy()[amap], rb.f_atoms.numpy())


def test_buffer_pool_best_fit_and_event_guard():
    """features/featurization.py _BufferPool: best-fit reuse by identity, head-room on fresh allocations, pinned buffers held back until
    their copy event has completed."""
    from reactranker_b200.features.featurization import _BufferPool
    pool = _BufferPool()
    made = []

    def make(n):
        made.append(n)
        return torch.empty(n, dtype=torch.uint8)
    a = pool.take(1000, "k", make)
    assert a.numel() >= 1000 and made == [a.numel()] and a.numel() <= 1000 * 1.31 + 256
    b = pool.take(5000, "k", make)
    pool.give(a, "k")
    pool.give(b, "k")
    assert pool.take(900, "k", make) is a and pool.take(900, "k", make) is b and len(made) == 2      # best fit first, then whatever fits

    class Ev:
        def __init__(self, done):
            self.done = done

        def query(self):
            return self.done
    ev = Ev(False)
    pool.give(a, "pinned", ev)
    c = pool.take(10, "pinned", make)
    assert c is not a                      # copy still in flight: a fresh buffer instead
    ev.done = True
    assert pool.take(10, "pinned", make) is a
    # device blobs: take() relies on stream order (no host-side wait); take_device() hands the "freed" event to the caller, whose
    # side stream waits for it
    ev2 = Ev(False)
    pool.give(b, "cuda:0", ev2)
    got, freed = pool.take_device(100, "cuda:0", make)
    assert got is b and freed is ev2
    fresh, none = pool.take_device(100, "cuda:0", make)
    assert fresh is not b and none is None


def test_train_state_round_trip_resumes_adam_and_noam(tmp_path):
    """save_train_state / load_train_state (SURVEY.md §8f row 3) on a plain torch module: 3 + 3 steps through a saved state are bit-identical
    to 6 uninterrupted steps, the reference's loader still finds 'state_dict' / 'data_scaler', and weights-only files are refused."""
    import torch
    from reactranker_b200 import _lib
    from reactranker_b200.train.utils import NoamLR
    from reactranker_b200.utils import load_checkpoint, load_train_state, save_checkpoint, save_train_state

    def fresh():
        torch.manual_seed(3)
        m = torch.nn.Linear(5, 3)
        o = torch.optim.Adam([{"params": list(m.parameters()), "lr": 1e-4, "weight_decay": 0}])
        return m, o, NoamLR(o, warmup_epochs=1, total_epochs=3, steps_per_epoch=2, init_lr=1e-4, max_lr=1e-2, final_lr=1e-3)

    def steps(m, o, s, lo, hi):
        for k in range(lo, hi):
            x = torch.randn(7, 5, generator=torch.Generator().manual_seed(k))
            o.zero_grad()
            (m(x) ** 2).mean().backward()
            o.step()
            s.step()

    m1, o1, s1 = fresh()
    steps(m1, o1, s1, 0, 6)
    m2, o2, s2 = fresh()
    steps(m2, o2, s2, 0, 3)
    path = str(tmp_path / "state.pt")
    save_train_state(path, m2, o2, s2, epoch=0, means=1.5, stds=0.5, best=[0.1, 0.2, 0.3])
    m3, o3, s3 = fresh()
    nxt, best, scaler = load_train_state(path, m3, o3, s3)
    assert nxt == 1 and best == [0.1, 0.2, 0.3] and scaler == {"means": 1.5, "stds": 0.5}
    assert s3.current_step == s2.current_step and o3.param_groups[0]["lr"] == o2.param_groups[0]["lr"]
    steps(m3, o3, s3, 3, 6)
    for a, b in zip(m1.parameters(), m3.parameters()):
        assert torch.equal(a, b)
    assert set(load_checkpoint(path)) >= {"state_dict", "data_scaler"}
    weights_only = str(tmp_path / "w.pt")
    save_checkpoint(weights_only, m1, 1.0, 2.0)
    with pytest.raises(_lib.RRError):
        load_train_state(weights_only, m3, o3, s3)


def test_vectorised_control_block_equals_the_per_batch_layout():
    """DeviceGraph.control_block (ids + segment lengths, vectorised) against the per-BatchMolGraph bookkeeping it replaced: every segment
    is a reference-shaped batch (one padding row, running a_start / b_start, its own max_num_bonds), offsets accumulate over segments."""
    from reactranker_b200.data.load_reactions import Parsing_features
    ds = synthetic.make_dataset(21, [5, 1, 7, 3], star_leaves_in_group={2: 8})
    fz = Parsing_features(ds.mols)
    groups = [(0, 5), (5, 6), (6, 13), (13, 16)]
    for override in (None, [None, 9, None, 12]):
        batches = [fz.parsing_smiles(list(ds.rsmi[a:b])) for a, b in groups]     # the star molecule is a reactant
        nM, S = sum(b.n_mols for b in batches), len(batches)
        want = np.empty(6 * nM + 3 * S, np.int32)
        ids, a_st, b_st, mW, mpb, mpa = (want[i * nM:(i + 1) * nM] for i in range(6))
        seg = want[6 * nM:].reshape(3, S)
        a0 = b0 = m0 = 0
        for s_i, b in enumerate(batches):
            W = b.max_num_bonds if not (override and override[s_i]) else override[s_i]
            n = b.n_mols
            ids[m0:m0 + n] = b._ids
            a_st[m0:m0 + n] = b._a_start + a0
            b_st[m0:m0 + n] = b._b_start + b0
            mW[m0:m0 + n], mpb[m0:m0 + n], mpa[m0:m0 + n] = W, b0, a0
            seg[0, s_i], seg[1, s_i], seg[2, s_i] = a0, b0, W
            a0 += b.n_atoms
            b0 += b.n_bonds
            m0 += n
        W = None if override is None else [b.max_num_bonds if o is None else o for b, o in zip(batches, override)]
        got, (nA, nB, nM2, wmax, S2), (A_s, B_s, W_s) = DeviceGraph.control_block(fz.store, np.concatenate([b._ids for b in batches]),
                                                                                  [b.n_mols for b in batches], W)
        assert np.array_equal(got, want)
        assert (nA, nB, nM2, S2) == (a0, b0, nM, S) and wmax == max(1, max(b._max_deg for b in batches))
        assert A_s.tolist() == [b.n_atoms for b in batches] and B_s.tolist() == [b.n_bonds for b in batches]
    assert [b.max_num_bonds for b in batches] == [4, 4, 8, 4]    # the star molecule widens its own segment only
    with pytest.raises(ValueError):
        DeviceGraph.control_block(fz.store, np.concatenate([b._ids for b in batches]), [b.n_mols for b in batches], [1, 1, 1, 1])
    # an empty segment is a lone padding row
    got, (nA, nB, nM2, wmax, S2), (A_s, B_s, W_s) = DeviceGraph.control_block(fz.store, batches[0]._ids, [0, batches[0].n_mols])
    assert A_s.tolist() == [1, batches[0].n_atoms] and W_s.tolist() == [1, batches[0].max_num_bonds] and got[6 * nM2:].reshape(3, 2)[0].tolist() == [0, 1]


def test_dedup_ids_equals_dedup_plan():
    """The vectorised reactant de-duplication on store ids gives the same unique reactants, segment lengths and atom map as the
    per-BatchMolGraph dedup_plan, on groups with one reactant each, on a whole batch as one segment and on a group with two reactants."""
    from reactranker_b200.data.load_reactions import Parsing_features
    ds = synthetic.make_dataset(12, [4, 1, 3, 6])
    fz = Parsing_features(ds.mols)
    layouts = [[(0, 4), (4, 5), (5, 8), (8, 14)], [(0, 14)], [(0, 6), (6, 14)]]       # the last two mix reactants inside a segment
    for groups in layouts:
        r_b = [fz.parsing_smiles(list(ds.rsmi[a:b])) for a, b in groups]
        p_b = [fz.parsing_smiles(list(ds.psmi[a:b])) for a, b in groups]
        uniq, w, amap = DeviceGraph.dedup_plan(r_b, p_b)
        r_ids, p_ids = fz.parsing_ids(list(ds.rsmi)), fz.parsing_ids(list(ds.psmi))
        u_ids, u_lens, amap2 = DeviceGraph.dedup_ids(fz.store, r_ids, p_ids, [b - a for a, b in groups])
        assert np.array_equal(u_ids, np.concatenate([u._ids for u in uniq])) and u_lens.tolist() == [u.n_mols for u in uniq]
        assert np.array_equal(amap2, amap)
        # the widths the unique segments get by default are the widths the full reactant segments had
        _, _, (_, _, W_s) = DeviceGraph.control_block(fz.store, u_ids, u_lens)
        assert W_s.tolist() == w
    # nothing repeats -> None
    assert DeviceGraph.dedup_ids(fz.store, fz.parsing_ids([ds.rsmi[0]]), fz.parsing_ids([ds.psmi[0]]), [1]) is None


def test_control_block_and_dedup_ids_on_random_layouts():
    """Property check over random segmentations (incl. empty and single-molecule segments, repeated and interleaved reactants): the
    vectorised host code agrees with a direct per-segment construction of the same quantities."""
    from reactranker_b200.data.load_reactions import Parsing_features
    ds = synthetic.make_dataset(77, [3, 5, 2, 6, 4])
    fz = Parsing_features(ds.mols)
    all_r, all_p = fz.parsing_ids(list(ds.rsmi)), fz.parsing_ids(list(ds.psmi))
    rng = np.random.default_rng(5)
    store = fz.store
    for trial in range(40):
        n = int(rng.integers(1, 20))
        pick = rng.integers(0, len(all_r), size=n)
        r_ids, p_ids = all_r[pick], all_p[pick]
        cuts = np.sort(rng.integers(0, n + 1, size=int(rng.integers(0, 5))))
        lens = np.diff(np.concatenate(([0], cuts, [n])))
        ctl, (nA, nB, nM, wmax, S), (A_s, B_s, W_s) = DeviceGraph.control_block(store, p_ids, lens)
        m = ctl[:6 * nM].reshape(6, nM)
        a0 = b0 = o = 0
        for s_i, ln in enumerate(lens.tolist()):
            ids = p_ids[o:o + ln]
            na, nb = store.nA[ids].astype(np.int64), store.nB[ids].astype(np.int64)
            W = max(1, int(store.maxdeg[ids].max())) if ln else 1
            assert (A_s[s_i], B_s[s_i], W_s[s_i]) == (1 + na.sum(), 1 + nb.sum(), W)
            assert m[1, o:o + ln].tolist() == (a0 + 1 + np.cumsum(na) - na).tolist()
            assert m[2, o:o + ln].tolist() == (b0 + 1 + np.cumsum(nb) - nb).tolist()
            assert set(m[3, o:o + ln].tolist()) <= {W} and set(m[4, o:o + ln].tolist()) <= {b0} and set(m[5, o:o + ln].tolist()) <= {a0}
            a0, b0, o = a0 + 1 + int(na.sum()), b0 + 1 + int(nb.sum()), o + ln
        assert (nA, nB) == (a0, b0)
        plan = DeviceGraph.dedup_ids(store, r_ids, p_ids, lens)
        uniq_per_seg, o = [], 0
        for ln in lens.tolist():
            seen = []
            for x in r_ids[o:o + ln].tolist():
                if x not in seen:
                    seen.append(x)
            uniq_per_seg.append(seen)
            o += ln
        if sum(len(u) for u in uniq_per_seg) == n:
            assert plan is None
            continue
        u_ids, u_lens, amap = plan
        assert u_ids.tolist() == [x for u in uniq_per_seg for x in u] and u_lens.tolist() == [len(u) for u in uniq_per_seg]
        # atom map by brute force: row of atom k of product molecule j -> row of atom k of its reactant inside the de-duplicated graph
        want, a0_p, a0_u, o = [], 0, 0, 0
        for ln, useg in zip(lens.tolist(), uniq_per_seg):
            u_na = store.nA[np.asarray(useg, dtype=np.int64)].astype(np.int64) if useg else np.zeros(0, np.int64)
            u_start = a0_u + 1 + np.cumsum(u_na) - u_na
            want.append(a0_u)
            for x in r_ids[o:o + ln].tolist():
                st = int(u_start[useg.index(x)])
                want.extend(range(st, st + int(store.nA[x])))
            a0_p += 1 + int(store.nA[p_ids[o:o + ln]].sum())
            a0_u += 1 + int(u_na.sum())
            o += ln
        assert amap.tolist() == want


def test_rr_batch_build_equals_the_numpy_restatement_and_reports_errors():
    """The C++ host batcher behind DeviceGraph.control_block (rr_batch_build, csrc/rr_host.cu; host pointers only, runs without a GPU)
    against the vectorised numpy restatement, bit for bit, on random segment layouts incl. empty segments, an empty batch and
    max_num_bonds overrides; bad arguments come back as messages, not crashes."""
    from reactranker_b200 import synthetic
    from reactranker_b200.data.load_reactions import Parsing_features
    from reactranker_b200.features.featurization import DeviceGraph
    rng = np.random.default_rng(5)
    ds = synthetic.make_dataset(71, [6, 9, 4, 11, 3], star_leaves_in_group={2: 9})
    fz = Parsing_features(ds.mols)
    all_ids = np.concatenate([fz.parsing_ids(list(ds.rsmi)), fz.parsing_ids(list(ds.psmi))])
    for trial in range(40):
        n = int(rng.integers(0, 60))
        ids = rng.choice(all_ids, size=n)
        S = int(rng.integers(1, 7))
        cuts = np.sort(rng.integers(0, n + 1, size=S - 1))
        lens = np.diff(np.concatenate(([0], cuts, [n])))
        W = None
        if trial % 3 == 0:
            _, _, (_, _, W_min) = DeviceGraph.control_block_numpy(fz.store, ids, lens)
            W = W_min + rng.integers(0, 3, size=S)
        a = DeviceGraph.control_block(fz.store, ids, lens, W)
        b = DeviceGraph.control_block_numpy(fz.store, ids, lens, W)
        assert np.array_equal(a[0], b[0]) and a[1] == b[1], trial
        assert all(np.array_equal(x, y) for x, y in zip(a[2], b[2])), trial
    staging = np.zeros(6 * 4 + 3 + 5, np.int32)                      # written in place (the pinned staging buffer of the product path)
    ctl, dims, _ = DeviceGraph.control_block(fz.store, all_ids[:4], [4], out=staging)
    assert ctl.base is staging or ctl is staging or np.shares_memory(ctl, staging)
    with pytest.raises(ValueError, match="override"):
        DeviceGraph.control_block(fz.store, all_ids, [len(all_ids)], [1])
    with pytest.raises(ValueError, match="segment lengths"):
        DeviceGraph.control_block(fz.store, all_ids[:5], [2, 2])
    with pytest.raises(ValueError, match="outside the store"):
        DeviceGraph.control_block(fz.store, np.asarray([10 ** 6], np.int32), [1])


def test_frame_ids_equal_per_token_lookups_and_follow_the_frame():
    """Parsing_features.frame_ids: the store id of every row's molecule, computed once per (frame, column); a batch's molecules are then
    frame_ids[rows].  Must equal the per-SMILES dictionary path, survive new frames and not be confused by a dead frame's recycled id()."""
    from reactranker_b200 import synthetic
    from reactranker_b200.data.load_reactions import DataProcessor, Parsing_features
    ds = synthetic.make_dataset(81, [5, 3, 6, 4])
    fz = Parsing_features(ds.mols)
    df = ds.to_dataframe()
    for col in ("rsmi_mapped", "psmi_mapped"):
        ids = fz.frame_ids(df, col)
        assert ids.dtype == np.int32 and np.array_equal(ids, fz.parsing_ids(list(df[col].values)))
        assert fz.frame_ids(df, col) is ids                                  # cached
    proc = DataProcessor(df)
    for rows, scope in proc.plan_batch_reactions(batch_size=9, seed=3):
        smiles, _, _ = proc._gather(df, rows, ["rsmi_mapped", "psmi_mapped"], "lgk", None)
        assert np.array_equal(fz.frame_ids(df, "psmi_mapped")[rows], fz.parsing_ids(smiles[:, 1].tolist()))
    sub = df.iloc[5:].reset_index(drop=True)
    assert np.array_equal(fz.frame_ids(sub, "psmi_mapped"), fz.parsing_ids(list(sub["psmi_mapped"].values)))
