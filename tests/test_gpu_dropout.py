"""Dropout, checked exactly: the Philox4x32-7 masks of rr_common.cuh regenerated on the host bit for bit, and the training step with
dropout against the fp64 oracle run under exactly those masks.

Every dropout mask of a step is a function of (seed, stream id, element index): element ``c & 3`` of the draw at counter
``(row * ld + c) >> 2`` is kept iff it is >= floor(fp32(p) * 2^32).  So the masks need not be checked statistically: the numpy port below
(``keep_mask``) gives every one of them, the kernels must reproduce them entry for entry, and the oracle (oracle/reactranker_oracle.py, its
``_drop`` replaced by multiplication with the host mask / (1 - p)) then makes the step with dropout as checkable as the step without.

Stream ids follow rr_model.cu ``model_forward``: one id per dense layer (with or without dropout), in launch order, the readout taking its
own (``stream_ids``); the encoder's layers draw over the joint rows [reactant rows | product rows]."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import reactranker_oracle as O
from reactranker_b200 import _lib, synthetic
from reactranker_b200.features.featurization import BatchMolGraph, DeviceGraph
from reactranker_b200.models.base_model import build_model
from reactranker_b200.train import loss as RL
from helpers import KINK, TOL, add_features, forced_relu_masks, grads_close, rel_err

GPU = 0
DEV = "cuda:0"
SEED = 0x2F3A_96C1_D45B_7E08          # above 2^32: both key words matter
SID = (5 << 32) | 0x9D                # above 2^32: both stream-id counter words matter

# ------------------------------------------------------------------------------------------------
# host port of rr_common.cuh philox4x32 / dropout4
# ------------------------------------------------------------------------------------------------
_U32 = np.uint64(0xFFFFFFFF)
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)


def philox4x32_7(seed: int, stream_id: int, idx) -> np.ndarray:
    """Philox4x32-7 of counters (idx lo, idx hi, stream lo, stream hi) under key (seed lo, seed hi) -> uint32 [len(idx), 4].
    32 x 32 -> 64-bit products are exact in uint64, so mulhi / mullo are the two halves of one product."""
    idx = np.asarray(idx, dtype=np.uint64)
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    c0, c1 = idx & _U32, idx >> np.uint64(32)
    c2 = np.full(idx.shape, stream_id & 0xFFFFFFFF, dtype=np.uint64)
    c3 = np.full(idx.shape, (stream_id >> 32) & 0xFFFFFFFF, dtype=np.uint64)
    for _ in range(7):
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0), p1 & _U32, (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1), p0 & _U32
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def keep_threshold(p: float) -> np.uint32:
    """uint32(fminf(p, 1) * 4294967295.f): the float constant rounds to 2^32, so the product is exact and the cast truncates."""
    return np.uint32(np.floor(float(np.float32(p)) * 2.0 ** 32))


def keep_mask(seed: int, stream_id: int, rows: int, cols: int, ld: int, p: float) -> np.ndarray:
    """bool [rows, cols]: which entries of a [rows, ld]-strided output the dropout of (seed, stream_id, p) keeps."""
    assert ld % 4 == 0 and cols <= ld
    r = philox4x32_7(seed, stream_id, np.arange(rows * ld // 4, dtype=np.uint64))
    return (r.reshape(rows, ld) >= keep_threshold(p))[:, :cols]


def _philox_scalar(seed, stream_id, idx):
    """The same function in Python integers, one counter at a time (cross-check of the vectorised port)."""
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32 & 0xFFFFFFFF
    c = [idx & 0xFFFFFFFF, idx >> 32 & 0xFFFFFFFF, stream_id & 0xFFFFFFFF, stream_id >> 32 & 0xFFFFFFFF]
    for _ in range(7):
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [(p1 >> 32) ^ c[1] ^ k0, p1 & 0xFFFFFFFF, (p0 >> 32) ^ c[3] ^ k1, p0 & 0xFFFFFFFF]
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return c


def test_host_philox_keep_rate_and_high_words():
    """No GPU: the numpy port agrees with a scalar restatement, keeps 1 - p of the entries within binomial bounds, and uses all four
    key / counter words (the model's seeds come from randint(0, 2**62), the stream ids of a test go above 2^32)."""
    idx = [0, 1, 2 ** 32 - 1, 2 ** 32, 2 ** 40 + 12345, 2 ** 63 + 7]
    got = philox4x32_7(SEED, SID, idx)
    for i, x in enumerate(idx):
        assert [int(v) for v in got[i]] == _philox_scalar(SEED, SID, x)
    assert keep_threshold(0.1) == np.uint32(429496736)          # fp32(0.1) = 0.100000001490116..., times 2^32, truncated
    rows, cols = 512, 304
    n = rows * cols
    for p in (0.1, 0.2, 0.5):
        keep = keep_mask(SEED, SID, rows, cols, cols, p)
        drop = 1.0 - float(keep.mean())
        assert abs(drop - p) < 5 * np.sqrt(p * (1 - p) / n), (p, drop)
        per_col = 1.0 - keep.mean(0)                          # every column position of the 4-wide draw is used, none is stuck
        assert abs(per_col.reshape(-1, 4).mean(0) - p).max() < 5 * np.sqrt(p * (1 - p) / (n / 4))
    p = 0.5
    base = keep_mask(SEED, SID, rows, cols, cols, p)
    for s, sid in ((SEED + 1, SID), (SEED + (1 << 32), SID), (SEED ^ (1 << 61), SID), (SEED, SID + 1), (SEED, SID + (1 << 32)),
                   (SEED, SID ^ (1 << 60))):
        other = keep_mask(s, sid, rows, cols, cols, p)
        assert abs(float((other != base).mean()) - 2 * p * (1 - p)) < 0.02, (hex(s), hex(sid))
    # rows past 2^32 / 4 draws: the high counter word
    far = philox4x32_7(SEED, SID, np.arange(4096, dtype=np.uint64) + np.uint64(1 << 32))
    near = philox4x32_7(SEED, SID, np.arange(4096, dtype=np.uint64))
    assert float((far != near).mean()) > 0.99


# ------------------------------------------------------------------------------------------------
# kernel level: dense layer epilogue (SIMT and tcgen05) and the readout
# ------------------------------------------------------------------------------------------------
def S():
    return torch.cuda.current_stream().cuda_stream


def _set_path(path):
    L = _lib.lib()
    _lib.check(L.rr_set_gemm_mode(0 if path == "simt" else 1))
    return L


def _assert_zero_pattern(got, want, z, what):
    """(got == 0) == (want == 0) wherever |z| exceeds 1e-5 of its row's largest magnitude (a pre-activation that close to zero may take
    either ReLU decision on an fp32 path)."""
    far = z.abs() > 1e-5 * z.abs().amax(dim=1, keepdim=True)
    bad = ((got == 0) != (want == 0)) & far
    assert not bool(bad.any()), (what, int(bad.sum()), [tuple(x) for x in bad.nonzero()[:5].tolist()])


@pytest.mark.gpu
@pytest.mark.parametrize("M,n,k1,k2,ldy", [(5, 16, 304, 0, 16), (130, 48, 64, 48, 48), (130, 48, 64, 48, 64), (777, 304, 304, 88, 304),
                                           (777, 304, 304, 88, 320), (4100, 608, 608, 608, 608)])
@pytest.mark.parametrize("path", ["simt", "tc16"])
def test_linear_dropout_mask_is_bit_exact(path, M, n, k1, k2, ldy):
    """rr_linear_fwd with flags 3 (ReLU + dropout) and 2 (dropout only) on the SIMT kernel and on the tcgen05 kernel (16 epilogue warps):
    relu(z) * keep / (1 - p) with the host's keep mask, p in {0.1, 0.2, 0.5}, seed and stream id above 2^32.  With ldy > n the
    counter runs over the output stride: the columns [n, ldy) are never written."""
    L = _set_path(path)
    g = torch.Generator().manual_seed(M + n + ldy)
    X1, W1 = torch.randn(M, k1, generator=g), torch.randn(n, k1, generator=g) / k1 ** 0.5
    X2 = torch.randn(M, k2, generator=g) if k2 else None
    W2 = torch.randn(n, k2, generator=g) / k2 ** 0.5 if k2 else None
    bias, resid = torch.randn(n, generator=g), torch.randn(M, n, generator=g)
    z = X1.double() @ W1.double().T + bias.double() + resid.double()
    if k2:
        z = z + X2.double() @ W2.double().T
    d = {k: (v.to(DEV) if v is not None else None) for k, v in dict(X1=X1, W1=W1, X2=X2, W2=W2, bias=bias, resid=resid).items()}
    tol = 3e-6 if path == "simt" else (1e-5 if k1 + k2 > 1000 else 5e-6)
    for i, p in enumerate((0.1, 0.2, 0.5)):
        seed, sid = SEED + 977 * i, SID + 31 * i
        keep = torch.from_numpy(keep_mask(seed, sid, M, n, ldy, p))
        for flags in (3, 2):
            Y = torch.full((M, ldy), float("nan"), device=DEV)
            _lib.check(L.rr_linear_fwd(M, n, d["X1"].data_ptr(), k1, d["W1"].data_ptr(), k1, _lib.ptr(d["X2"]), k2, _lib.ptr(d["W2"]), k2,
                                       d["bias"].data_ptr(), d["resid"].data_ptr(), n, Y.data_ptr(), ldy, flags, p, seed, sid, S()))
            Y = Y.double().cpu()
            assert bool(torch.isnan(Y[:, n:]).all())
            got = Y[:, :n]
            want = (torch.relu(z) if flags & 1 else z) * keep / (1 - p)
            assert not bool(((got != 0) & ~keep).any()), (p, flags, "an entry the host mask drops survived")
            _assert_zero_pattern(got, want, z, (p, flags))
            assert rel_err(got, want) < tol, (p, flags, rel_err(got, want))


def _graph(seed, sizes, star=None, segments=1):
    ds = synthetic.make_dataset(seed, list(sizes), star_leaves_in_group=star)
    mols = [ds.mols[t] for t in ds.psmi]
    cuts = np.linspace(0, len(mols), segments + 1).astype(int)
    batches = [BatchMolGraph(mols[a:b]) for a, b in zip(cuts[:-1], cuts[1:])]
    scopes = []
    o = 0
    for b in batches:                       # (first atom row, atom count) of every molecule in the joint atom rows
        scopes += [(o + s, m) for s, m in b.a_scope]
        o += b.n_atoms
    return ds, DeviceGraph.from_batches(batches, DEV), sum(b.n_atoms for b in batches), scopes


@pytest.mark.gpu
@pytest.mark.parametrize("h,sizes,star,segments", [(40, (3, 4), None, 1), (300, (6, 1, 5), {1: 7}, 3)])
def test_readout_dropout_is_bit_exact_forward_and_backward(h, sizes, star, segments):
    """rr_readout_fwd with dropout: vec = [scope mean of hid | add feature | 0] * keep / (1 - p), the counter (mol * vp + c) >> 2 and the
    mask covering the add-feature column, columns [h + 1, vp) zero.  rr_readout_bwd with dropout against autograd of
    drop_vec(mean(drop_hid(relu(z)))) built with the host masks: the gradient reaches z through both masks, scaled by 1 / (1 - p) twice."""
    L = _lib.lib()
    ds, dg, A, scopes = _graph(3, sizes, star, segments)
    hp, vp, f = L.rr_padded(h), L.rr_padded(h + 1), 1
    N = len(scopes)
    feats = torch.tensor(ds.temp.reshape(-1, 1), dtype=torch.float32)
    g = torch.Generator().manual_seed(h)
    z0 = torch.randn(A, hp, generator=g)
    z0[:, h:] = 0
    for i, p in enumerate((0.1, 0.2, 0.5)):
        seed, sid_h, sid_v = SEED + 5 * i, SID + 2 * i, SID + 2 * i + 1
        keep_h = torch.from_numpy(keep_mask(seed, sid_h, A, hp, hp, p))
        keep_v = torch.from_numpy(keep_mask(seed, sid_v, N, vp, vp, p))
        z = z0.double().requires_grad_(True)
        hid = torch.relu(z) * keep_h / (1 - p)
        mean = torch.stack([hid[s:s + m].sum(0) / m for s, m in scopes])[:, :h]
        full = torch.cat([mean, feats.double(), torch.zeros(N, vp - h - f, dtype=torch.double)], 1)
        want = full * keep_v / (1 - p)
        hd, fd = hid.detach().float().to(DEV), feats.to(DEV)
        vec = torch.full((N, vp), float("nan"), device=DEV)
        _lib.check(L.rr_readout_fwd(ctypes.byref(dg.c), hd.data_ptr(), hp, h, fd.data_ptr(), f, vec.data_ptr(), vp, p, seed, sid_v, S()))
        got = vec.double().cpu()
        assert not bool(got[:, h + f:].any())
        assert torch.equal(got != 0, want.detach() != 0), (p, int(((got != 0) != (want.detach() != 0)).sum()))
        assert rel_err(got, want.detach()) < 3e-6
        up = torch.randn(N, vp, generator=g)
        want.backward(up.double())
        dz, upd = torch.full((A, hp), float("nan"), device=DEV), up.to(DEV)
        _lib.check(L.rr_readout_bwd(ctypes.byref(dg.c), upd.data_ptr(), vp, vec.data_ptr(), hd.data_ptr(), dz.data_ptr(), hp, p, S()))
        got = dz.double().cpu()
        assert rel_err(got, z.grad) < 3e-6, (p, rel_err(got, z.grad))
        assert torch.equal(got != 0, z.grad != 0)


# ------------------------------------------------------------------------------------------------
# model level: the training step with dropout against the fp64 oracle under the same masks
# ------------------------------------------------------------------------------------------------
def stream_ids(depth, ddepth, ffn_depth=3):
    """model_forward's stream id of every dropout site: ``sid`` starts at 1 and each ``lin`` call takes the next (dropout or not), the
    readout takes its own.  Depth 3 / 3: encoder W_h 2, 3, encoder W_o 4, diff W_h 6, 7, diff W_o 8, readout 9, FFN hidden layers 10, 11."""
    sid = iter(range(1, 1 << 10))
    next(sid)                                                    # encoder W_i (ReLU only, applied by its consumers)
    ids = {f"enc.m{t}": next(sid) for t in range(1, depth)}
    ids["enc.hid"] = next(sid)
    next(sid)                                                    # diff encoder W_i
    ids.update({f"m2_{t}": next(sid) for t in range(1, ddepth)})
    ids["hid2"] = next(sid)
    ids["vec"] = next(sid)
    ids.update({f"x{l}": next(sid) for l in range(ffn_depth - 1)})
    return ids


class Layout:
    """Row ranges of a (possibly multi-segment) reactant / product batch pair: one entry per group of the oracle, which runs one forward
    per group (the reference's per-group forward)."""

    def __init__(self, r_batches, p_batches):
        self.groups = []
        ra = rb = pa = pb = m = 0
        for r, p in zip(r_batches, p_batches):
            self.groups.append(dict(rb=slice(rb, rb + r.n_bonds), ra=slice(ra, ra + r.n_atoms), pb=slice(pb, pb + p.n_bonds),
                                    pa=slice(pa, pa + p.n_atoms), m=slice(m, m + p.n_mols)))
            ra, rb, pa, pb, m = ra + r.n_atoms, rb + r.n_bonds, pa + p.n_atoms, pb + p.n_bonds, m + p.n_mols
        self.A_r, self.B_r, self.A_p, self.B_p, self.N = ra, rb, pa, pb, m


def site_keeps(seed, p, hidden, depth, ddepth, lay, hp, vp, ids, add=1, ffn_depth=3):
    """{saved buffer name: host keep mask [rows, cols]} of every dropout site of one forward."""
    def km(sid, rows, cols, ld):
        return torch.from_numpy(keep_mask(seed, sid, rows, cols, ld, p))
    keeps = {}
    for t in range(1, depth):
        j = km(ids[f"enc.m{t}"], lay.B_r + lay.B_p, hidden, hp)          # joint rows [reactant bonds | product bonds]
        keeps[f"enc0.m{t}"], keeps[f"enc1.m{t}"] = j[:lay.B_r], j[lay.B_r:]
    j = km(ids["enc.hid"], lay.A_r + lay.A_p, hidden, hp)
    keeps["enc0.hid"], keeps["enc1.hid"] = j[:lay.A_r], j[lay.A_r:]
    for t in range(1, ddepth):
        keeps[f"m2_{t}"] = km(ids[f"m2_{t}"], lay.A_p, hidden, hp)
    keeps["hid2"] = km(ids["hid2"], lay.A_p, hidden, hp)
    keeps["vec"] = km(ids["vec"], lay.N, hidden + add, vp)
    for l in range(ffn_depth - 1):
        keeps[f"x{l}"] = km(ids[f"x{l}"], lay.N, hidden, hp)
    return keeps


def saved_buffers(model, out, lay, hidden, depth, ddepth, add=1, ffn_depth=3):
    """Every forward activation a ReLU or a dropout acted on, read from the autograd node's workspace (call BEFORE backward)."""
    hp, vp = _lib.lib().rr_padded(hidden), _lib.lib().rr_padded(hidden + add)

    def act(name, rows, ld=hp, cols=hidden):
        return model.saved_activation(out, name, rows, ld)[:, :cols].detach().cpu()
    buf = {}
    for k, (na, nb) in enumerate(((lay.A_r, lay.B_r), (lay.A_p, lay.B_p))):
        buf[f"enc{k}.inp"] = act(f"enc{k}.inp", nb)
        for t in range(1, depth):
            buf[f"enc{k}.m{t}"] = act(f"enc{k}.m{t}", nb)
        buf[f"enc{k}.hid"] = act(f"enc{k}.hid", na)
    buf["inp2"] = act("inp2", lay.A_p)
    for t in range(1, ddepth):
        buf[f"m2_{t}"] = act(f"m2_{t}", lay.A_p)
    buf["hid2"] = act("hid2", lay.A_p)
    buf["vec"] = act("vec", lay.N, vp, hidden + add)
    for l in range(ffn_depth - 1):
        buf[f"x{l}"] = act(f"x{l}", lay.N)
    return buf


def site_order(depth, ddepth, ffn_depth=3):
    """(buffer name, row-range key of Layout) in the order of the oracle's torch.relu and _drop calls for one group: mpn_forward(r),
    mpn_forward(p), mpndiff_forward, ffn_forward.  ``enc*.inp`` / ``inp2`` only feed a ReLU, ``vec`` only a dropout, the others both."""
    order = []
    for k, (a, b) in enumerate((("ra", "rb"), ("pa", "pb"))):
        order += [(f"enc{k}.inp", b)] + [(f"enc{k}.m{t}", b) for t in range(1, depth)] + [(f"enc{k}.hid", a)]
    order += [("inp2", "pa")] + [(f"m2_{t}", "pa") for t in range(1, ddepth)] + [("hid2", "pa"), ("vec", "m")]
    order += [(f"x{l}", "m") for l in range(ffn_depth - 1)]
    return order


def relu_masks_and_keeps(buf, keeps, lay, depth, ddepth, ffn_depth=3):
    """The dropout-aware counterpart of helpers.gpu_relu_masks: per group of ``lay``, the GPU's ReLU decisions in the oracle's torch.relu
    order and the keep mask of each (None for the un-dropped inputs ``enc.inp`` / ``inp2``, whose mask is [pre-activation > 0]).  A dropped
    entry is 0 whatever its ReLU decided, so only the kept entries carry the GPU's decision (forced_relu_masks(masks, keeps=...))."""
    masks, kps = [], []
    for grp in lay.groups:
        for name, rows in site_order(depth, ddepth, ffn_depth):
            if name == "vec":                                    # the readout has no ReLU
                continue
            x = buf[name][grp[rows]]
            pre = name.endswith("inp") or name == "inp2"
            masks.append(x > 0 if pre else x != 0)
            kps.append(None if pre else keeps[name][grp[rows]])
    return masks, kps


def check_sites(buf, keeps, seed, p, lay, hidden, hp, vp, ids, add=1):
    """Nothing the host mask drops survives in the GPU's activations.  On a miss, name the stream ids in 1..64 whose mask the site's zero
    pattern does fit, so that a change of the launch schedule is told apart from a wrong counter."""
    for name, keep in keeps.items():
        got = buf[name]
        bad = (got != 0) & ~keep
        if not bool(bad.any()):
            continue
        cols, ld = (hidden + add, vp) if name == "vec" else (hidden, hp)
        base = name.split(".")[-1]
        joint = name.startswith("enc")
        sid_key = f"enc.{base}" if joint else name
        rows = (lay.B_r + lay.B_p if base.startswith("m") else lay.A_r + lay.A_p) if joint else got.shape[0]
        r0 = 0 if name.startswith("enc0") else (rows - got.shape[0])
        fits = [s for s in range(1, 65)
                if not bool(((got != 0) & ~torch.from_numpy(keep_mask(seed, s, rows, cols, ld, p))[r0:r0 + got.shape[0]]).any())]
        pytest.fail(f"{name}: {int(bad.sum())} entries survive that stream id {ids[sid_key]} drops; "
                    f"stream ids in 1..64 whose mask fits: {fits}")


def run_oracle(monkeypatch, sd, groups, drop_keeps, p, depth, ddepth, head, loss_fn, relu=None, ffn_depth=3, kink=KINK):
    """fp64 oracle forward (one per group) + loss + backward, ``_drop`` multiplying by the host keep masks / (1 - p) in call order; with
    ``relu`` = (masks, keeps) the kept entries' ReLU decisions are the GPU's (helpers.forced_relu_masks asserts each differing one sits
    within ``kink`` of a kink).  Returns (scores, loss, {name: gradient}, [every _drop output in call order], flips, the largest relative
    pre-activation of a differing decision)."""
    sd64 = {k: v.double().cpu() for k, v in sd.items()}
    params = {k: v.clone().requires_grad_(True) for k, v in sd64.items() if "cached_zero" not in k}
    full = dict(sd64)
    full.update(params)
    it, outs = iter(drop_keeps), []

    def drop(x, p_, training):
        keep = next(it)
        assert tuple(keep.shape) == tuple(x.shape), (len(outs), tuple(keep.shape), tuple(x.shape))
        y = x * keep.to(x.dtype) / (1 - p)
        outs.append(y.detach())
        return y
    monkeypatch.setattr(O, "_drop", drop)

    def fwd():
        return torch.cat([O.model_forward(full, r, q, f, mpnn_depth=depth, mpnn_diff_depth=ddepth, ffn_depth=ffn_depth, head=head, dropout=p,
                                          training=True) for r, q, f in groups])
    flips, worst = 0, 0.0
    if relu is None:
        scores = fwd()
    else:
        with forced_relu_masks(relu[0], kink=kink, keeps=relu[1]) as fm:
            scores = fwd()
        flips, worst = fm.flips, fm.worst
    monkeypatch.undo()
    assert next(it, None) is None
    loss = loss_fn(scores)
    loss.backward(torch.ones_like(loss))
    return scores.detach().numpy(), loss.detach().numpy(), {k: v.grad.numpy() for k, v in params.items()}, outs, flips, worst


BENCH_TOL = {0: dict(max_rel=4e-3, l2=2e-3), 1: dict(max_rel=2.5e-2, l2=6e-3)}     # as test_gpu_model.py::BENCH_TOL


def step_vs_oracle(monkeypatch, gemm_mode, *, task, hidden, depth, p, mols, feats, gpu_loss, oracle_loss, last="with_softplus", bench=False,
                   ddepth=None, ffn_depth=3, use_bias=True, add=1, score_tol=None, kink=KINK):
    """One training step with dropout p on the GPU and the fp64 oracle under the same dropout masks (see the module docstring).
    ``mols``: [(reactant molecules, product molecules)] per group; several groups run as the segments of one launch.  ``ddepth``
    defaults to ``depth``; ``feats`` must have ``add`` columns.  ``score_tol`` (default TOL[gemm_mode]['score']) bounds the scores and the
    saved activations, ``kink`` the pre-activation of a ReLU decision the GPU takes differently.  Returns the measured figures."""
    tn, tt = {"mle": (1, None), "evidential_ranking": (2, "evidential_ranking")}[task]
    ddepth = depth if ddepth is None else ddepth
    L = _lib.lib()
    hp, vp = L.rr_padded(hidden), L.rr_padded(hidden + add)
    torch.manual_seed(3)
    model = build_model(hidden_size=hidden, mpnn_depth=depth, mpnn_diff_depth=ddepth, ffn_depth=ffn_depth, use_bias=use_bias, dropout=p,
                        task_num=tn, ffn_last_layer=last, task_type=tt, add_features_dim=add).cuda(GPU).train()
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    r_batches, p_batches = [BatchMolGraph(r) for r, _ in mols], [BatchMolGraph(q) for _, q in mols]
    lay = Layout(r_batches, p_batches)
    if len(mols) == 1:
        rg, pg = r_batches[0], p_batches[0]
    else:
        dev = torch.device("cuda", GPU)
        rg, pg = DeviceGraph.from_batches(r_batches, dev), DeviceGraph.from_batches(p_batches, dev)
    torch.manual_seed(17)
    out = model(rg, pg, gpu=GPU, add_features=feats)
    seed = int(out.grad_fn.cfg.seed)
    assert seed != 0
    ids = stream_ids(depth, ddepth, ffn_depth)
    keeps = site_keeps(seed, p, hidden, depth, ddepth, lay, hp, vp, ids, add, ffn_depth)
    buf = saved_buffers(model, out, lay, hidden, depth, ddepth, add, ffn_depth)
    check_sites(buf, keeps, seed, p, lay, hidden, hp, vp, ids, add)
    relu = relu_masks_and_keeps(buf, keeps, lay, depth, ddepth, ffn_depth)
    loss = gpu_loss(out)
    loss.backward()
    got = {k: q.grad.double().cpu().numpy() for k, q in model.named_parameters() if q.requires_grad}

    head = O.resolve_task_type(tn, last, tt)
    groups, drops, names = [], [], []
    for grp, (r, q) in zip(lay.groups, mols):
        groups.append((O.OracleBatch(r), O.OracleBatch(q), None if feats is None else feats[grp["m"]]))
        for name, rows in site_order(depth, ddepth, ffn_depth):
            if name in keeps:
                drops.append(keeps[name][grp[rows]])
                names.append((name, rows, grp))
    ws, wl, wg, outs, flips, kink_seen = run_oracle(monkeypatch, sd, groups, drops, p, depth, ddepth, head, oracle_loss, relu, ffn_depth, kink)

    tol = dict(TOL[gemm_mode])
    if score_tol is not None:
        tol["score"] = score_tol
    measured = dict(flips=flips, worst_kink=kink_seen, act_rel={})
    # every saved activation a dropout acted on, padding rows included: same zero pattern (nothing the host drops survives: check_sites;
    # every kept ReLU decision on a kink: forced_relu_masks) and the same values
    per_site = {}
    for (name, rows, grp), y in zip(names, outs):
        per_site.setdefault(name, []).append((grp[rows], y))
    for name, parts in per_site.items():
        want = torch.cat([y for _, y in parts])
        gotb = torch.cat([buf[name][s] for s, _ in parts]).double()
        assert torch.equal(gotb != 0, want != 0), (name, int(((gotb != 0) != (want != 0)).sum()))
        measured["act_rel"][name] = rel_err(gotb, want)
        assert rel_err(gotb, want) < tol["score"], (name, rel_err(gotb, want))
    e_s, e_l = rel_err(out.detach().cpu().numpy(), ws), rel_err(loss.detach().cpu().numpy(), wl)
    measured.update(score_rel=e_s, loss_rel=e_l)
    assert e_s < tol["score"] and e_l < tol["loss"], (e_s, e_l)
    gscale = max(float(np.abs(v).max()) for v in wg.values())
    live = {k: wg[k] for k in got if float(np.abs(wg[k]).max()) >= 1e-6 * gscale}
    n_pre = sum(int(m.numel()) for m in relu[0])
    assert flips <= max(8, 2e-4 * n_pre), (flips, n_pre)
    bad = grads_close(got, live, 2e-4)
    assert not bad, (flips, bad)
    if bench:
        # the unconditional bounds of test_gpu_model.py::test_gradients_at_bench_scale_vs_fp64_oracle, against the oracle's own ReLU
        # decisions under the same dropout masks
        ws0, wl0, wg0, _, _, _ = run_oracle(monkeypatch, sd, groups, drops, p, depth, ddepth, head, oracle_loss, ffn_depth=ffn_depth)
        e_s, e_l = rel_err(out.detach().cpu().numpy(), ws0), rel_err(loss.detach().cpu().numpy(), wl0)
        assert e_s < 1e-4 and e_l < 1e-4, (e_s, e_l)
        worst = max(float(np.abs(got[k] - wg0[k]).max() / np.abs(wg0[k]).max()) for k in live)
        worst_l2 = max(float(np.linalg.norm(got[k] - wg0[k]) / np.linalg.norm(wg0[k])) for k in live)
        assert worst <= BENCH_TOL[gemm_mode]["max_rel"] and worst_l2 <= BENCH_TOL[gemm_mode]["l2"], (worst, worst_l2)
    return measured


def _listwise_case(task, seed, sizes, add=1):
    from reactranker_b200.train.train_listwise import batch_loss
    ds = synthetic.make_dataset(seed, sizes)
    targets = ds.lgk.astype(np.float32)
    return dict(mols=[([ds.mols[t] for t in ds.rsmi], [ds.mols[t] for t in ds.psmi])], feats=add_features(ds, add),
                gpu_loss=lambda out: batch_loss(task, out, sizes, torch.tensor(targets), GPU),
                oracle_loss=lambda s: O.loss_for_task(task, s, sizes, torch.tensor(targets).double()))


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.1, 0.5])
def test_listmle_step_with_dropout_vs_fp64_oracle(monkeypatch, gemm_mode, p):
    """ListMLE, hidden 300, depth 3 (the c5 model) at p = 0.1 and at p = 0.5, where any masking or scaling error is macroscopic."""
    step_vs_oracle(monkeypatch, gemm_mode, task="mle", hidden=300, depth=3, p=p, **_listwise_case("mle", 77, [7, 5, 9, 4]))


@pytest.mark.gpu
def test_evidential_ranking_step_with_dropout_vs_fp64_oracle(monkeypatch):
    """UC-Listwise (evidential_ranking), hidden 600, depth 5 (the c4 model) at p = 0.1 on the product path: stream ids 2-15."""
    step_vs_oracle(monkeypatch, 1, task="evidential_ranking", hidden=600, depth=5, p=0.1,
                   **_listwise_case("evidential_ranking", 78, [6, 8, 5]))


@pytest.mark.gpu
def test_ranknet_window_step_with_dropout_vs_fp64_oracle(monkeypatch, gemm_mode):
    """A RankNet accumulation window (main_ranknet.py: p = 0.2) of four groups as four segments of one launch, one with a star molecule:
    every segment's padding rows, and on the tensor-core path their exact-arithmetic fix-up (k_pad_rows_linear) with its own Philox draw.
    The oracle runs one forward per group on that group's rows of the window's masks."""
    sizes = [6, 4, 5, 3]
    ds = synthetic.make_dataset(91, sizes, star_leaves_in_group={1: 7})
    cuts = np.cumsum([0] + sizes)
    mols = [([ds.mols[t] for t in ds.rsmi[a:b]], [ds.mols[t] for t in ds.psmi[a:b]]) for a, b in zip(cuts[:-1], cuts[1:])]
    targets = ds.lgk.astype(np.float32)
    pairs = sum(RL.count_ordered_pairs(targets[a:b]) for a, b in zip(cuts[:-1], cuts[1:]))

    def oracle_loss(s):
        total = 0
        for a, b in zip(cuts[:-1], cuts[1:]):
            c, _ = O.ranknet_group_cost(s[a:b], targets[a:b])
            if c is not None:
                total = total + c
        return total / pairs
    step_vs_oracle(monkeypatch, gemm_mode, task="mle", hidden=300, depth=3, p=0.2, mols=mols, feats=ds.temp.reshape(-1, 1), last="no_softplus",
                   gpu_loss=lambda y: RL.ranknet_window_loss(y, sizes, targets, pairs, sigma=1.0, gpu=GPU), oracle_loss=oracle_loss)


@pytest.mark.gpu
def test_c5_batch_step_with_dropout_vs_fp64_oracle(monkeypatch):
    """A c5-shaped batch (24 groups x 50 candidates, ListMLE h300 d3, p = 0.1) on the product path, under the bench-scale bounds of the
    dropout-free test as well as the exact statement given the GPU's ReLU decisions."""
    step_vs_oracle(monkeypatch, 1, task="mle", hidden=300, depth=3, p=0.1, bench=True, **_listwise_case("mle", 4242, [50] * 24))


# Models whose number of dense layers differs from the c5 model's, and with it the stream id of every later dropout site; one without the
# W_i / W_h / FFN biases (the padding-row fix-up then adds no bias); one whose readout dropout runs over three add features that cross the
# padded hidden width (hidden 46 + 3 -> vp 64).
DROPOUT_CONFIGS = {"ffn1": dict(ffn_depth=1), "ffn4": dict(ffn_depth=4), "depth1_diff2": dict(depth=1, ddepth=2), "nobias": dict(use_bias=False),
                   "add3": dict(hidden=46, add=3)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(DROPOUT_CONFIGS))
def test_listmle_step_with_dropout_at_other_configurations_vs_fp64_oracle(monkeypatch, gemm_mode, name):
    """p = 0.2 at FFN depth 1 and 4, encoder depth 1 with diff depth 2, no biases and three add features: the stream-id schedule, the
    readout mask over every add-feature column and the training step against the oracle wherever the layer count changes."""
    c = dict(dict(hidden=40, depth=3), **DROPOUT_CONFIGS[name])
    step_vs_oracle(monkeypatch, gemm_mode, task="mle", p=0.2, **c, **_listwise_case("mle", 79, [7, 5, 9, 4], add=c.get("add", 1)))


@pytest.fixture
def precision_switches():
    """The process-wide operand-split switches of rr_model_forward / rr_model_backward, put back as found after the test."""
    L = _lib.lib()
    prev = L.rr_get_forward_bf16(), L.rr_get_backward_bf16()
    yield L
    L.rr_set_forward_bf16(prev[0])
    L.rr_set_backward_bf16(prev[1])


# The forward GEMMs on the 3 x bf16 split (rr_set_forward_bf16(1)): the k_tc_gemm2 epilogue with bias, residual, ReLU and Philox dropout.
# Its forward error is larger than the 3 x TF32 split's, so the scores / saved activations and the distance from zero at which a ReLU
# decision may differ from the fp64 oracle's get bounds of their own.  Measured on this case and on three more batches of the same model
# (seeds 78, 80, 81) on one B200 (1000 W power limit): scores within 1.25e-5 of the oracle (3 x TF32: 1.1e-5), saved activations within
# 7.7e-6 of their maximum (3 x TF32: 6.7e-6), differing ReLU decisions at most 1.95e-6 (relative to the row) from zero, gradients given the
# GPU's masks within 2.4e-5.  The bounds are 4x the measured score and activation error, as helpers.KINK is for the 3 x TF32 split:
FWD_BF16_SCORE_TOL = 5e-5
FWD_BF16_KINK = 3e-5


@pytest.mark.gpu
@pytest.mark.parametrize("fwd_bf16,bwd_bf16", [(1, 1), (0, 0)], ids=["forward_bf16", "backward_tf32"])
def test_listmle_step_with_dropout_under_the_precision_switches(monkeypatch, precision_switches, fwd_bf16, bwd_bf16):
    """ListMLE h300 d3 at p = 0.1 on the tensor-core path with the forward GEMMs on the 3 x bf16 split, and with the backward GEMMs on the
    3 x TF32 split: the dropout zero pattern of every site bit for bit, and every gradient, given the GPU's ReLU decisions, to 2e-4."""
    L = precision_switches
    L.rr_set_forward_bf16(fwd_bf16)
    L.rr_set_backward_bf16(bwd_bf16)
    kw = dict(score_tol=FWD_BF16_SCORE_TOL, kink=FWD_BF16_KINK) if fwd_bf16 else {}
    step_vs_oracle(monkeypatch, 1, task="mle", hidden=300, depth=3, p=0.1, **kw, **_listwise_case("mle", 77, [7, 5, 9, 4]))


@pytest.mark.gpu
def test_training_forward_is_reproducible_under_the_torch_seed():
    """The dropout seed is drawn from torch's generator: the same torch.manual_seed gives bit-identical scores, another one other scores."""
    ds = synthetic.make_dataset(5, [8, 6, 7])
    torch.manual_seed(0)
    model = build_model(hidden_size=300, mpnn_depth=3, mpnn_diff_depth=3, ffn_depth=3, use_bias=True, dropout=0.1, task_num=1,
                        ffn_last_layer="with_softplus", add_features_dim=1).cuda(GPU).train()
    r_g, p_g = BatchMolGraph([ds.mols[t] for t in ds.rsmi]), BatchMolGraph([ds.mols[t] for t in ds.psmi])
    runs = []
    for s in (7, 7, 8):
        torch.manual_seed(s)
        with torch.no_grad():
            runs.append(model(r_g, p_g, gpu=GPU, add_features=ds.temp.reshape(-1, 1)).cpu())
    assert torch.equal(runs[0], runs[1])
    assert not torch.equal(runs[0], runs[2])
