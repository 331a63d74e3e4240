"""GPU parity of every kernel behind the C ABI against the CPU oracle
(oracle/reactranker_oracle.py) on the same seeded inputs.  fp32 tolerances are stated per test."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import reactranker_oracle as O
from reactranker_b200 import _lib, synthetic
from reactranker_b200.features.featurization import BatchMolGraph, DeviceGraph

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def S():
    return torch.cuda.current_stream().cuda_stream


def graphs(seed=7, sizes=(4, 3, 5), star=None, side="p"):
    ds = synthetic.make_dataset(seed, list(sizes), star_leaves_in_group=star)
    col = ds.psmi if side == "p" else ds.rsmi
    b = BatchMolGraph([ds.mols[t] for t in col])
    return ds, b, DeviceGraph.from_batches([b], DEV)


def rand(rows, hp, h, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(rows, hp, generator=g)
    x[:, h:] = 0
    return x


def close(got, want, tol=2e-6):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    scale = max(float(want.abs().max()), 1e-30)
    err = float((got - want).abs().max()) / scale
    assert err < tol, err


@pytest.mark.parametrize("h,star", [(300, None), (40, {1: 9}), (24, {0: 11})])
def test_bond_message_fwd_bwd(h, star):
    L = _lib.lib()
    ds, b, dg = graphs(star=star, side="r" if star else "p")
    hp = L.rr_padded(h)
    for relu in (0, 1):
        m = rand(b.n_bonds, hp, h, 1).requires_grad_(True)
        src = torch.relu(m) if relu else m
        a_msg = O.gather_sum(src.double(), b.a2b)                       # mpn.py:89-90
        want = a_msg[b.b2a] - src.double()[b.b2revb]                    # mpn.py:91-92
        pre = torch.empty(b.n_bonds, hp, device=DEV)
        md = m.detach().to(DEV)
        _lib.check(L.rr_bond_message_fwd(ctypes.byref(dg.c), md.data_ptr(), pre.data_ptr(), hp, relu, S()))
        close(pre, want.detach())
    up = rand(b.n_bonds, hp, h, 2)
    m = rand(b.n_bonds, hp, h, 3).double().requires_grad_(True)
    (O.gather_sum(m, b.a2b)[b.b2a] - m[b.b2revb]).backward(up.double())
    dm = torch.full((b.n_bonds, hp), float("nan"), device=DEV)
    upd = up.to(DEV)
    _lib.check(L.rr_bond_message_bwd(ctypes.byref(dg.c), upd.data_ptr(), dm.data_ptr(), hp, S()))
    close(dm, m.grad, 5e-6)


@pytest.mark.parametrize("which", [0, 1])
@pytest.mark.parametrize("h,star", [(300, None), (40, {2: 10})])
def test_neighbor_sum_fwd_bwd(which, h, star):
    L = _lib.lib()
    ds, b, dg = graphs(star=star, side="r" if star else "p")
    hp = L.rr_padded(h)
    rows = b.n_atoms if which else b.n_bonds
    table = b.get_a2a() if which else b.a2b
    src = rand(rows, hp, h, 4).double().requires_grad_(True)
    want = O.gather_sum(src, table)
    out = torch.empty(b.n_atoms, hp, device=DEV)
    sd = src.detach().float().to(DEV)
    _lib.check(L.rr_neighbor_sum_fwd(ctypes.byref(dg.c), which, sd.data_ptr(), out.data_ptr(), hp, 0, S()))
    close(out, want.detach())
    up = rand(b.n_atoms, hp, h, 5)
    want.backward(up.double())
    dsrc = torch.full((rows, hp), float("nan"), device=DEV)
    upd = up.to(DEV)
    _lib.check(L.rr_neighbor_sum_bwd(ctypes.byref(dg.c), which, upd.data_ptr(), dsrc.data_ptr(), hp, S()))
    close(dsrc, src.grad, 5e-6)


def test_neighbor_sum_of_bond_features():
    """nf = sum_k f_bonds[a2b[a,k]] (mpn.py:202-206) over the 88-wide padded feature rows."""
    L = _lib.lib()
    ds, b, dg = graphs()
    out = torch.empty(b.n_atoms, 88, device=DEV)
    _lib.check(L.rr_neighbor_sum_fwd(ctypes.byref(dg.c), 0, dg.c.f_bonds, out.data_ptr(), 88, 0, S()))
    close(out[:, :83], O.gather_sum(b.f_bonds.double(), b.a2b))
    assert not out[:, 83:].any()


def test_multi_segment_launch_equals_separate_batches():
    """Two reference batches with different max_num_bonds (4 and 9) in ONE launch reproduce the two
    separately-batched results, padding rows included (SURVEY.md §7 'pad-row recurrence')."""
    L = _lib.lib()
    ds = synthetic.make_dataset(9, [3, 3], star_leaves_in_group={1: 9})
    b1 = BatchMolGraph([ds.mols[t] for t in ds.rsmi[:3]])
    b2 = BatchMolGraph([ds.mols[t] for t in ds.rsmi[3:]])
    assert b1.max_num_bonds != b2.max_num_bonds
    dg = DeviceGraph.from_batches([b1, b2], DEV)
    h, hp = 40, 48
    m1, m2 = rand(b1.n_bonds, hp, h, 1), rand(b2.n_bonds, hp, h, 2)
    want = torch.cat([O.gather_sum(m.double(), b.a2b)[b.b2a] - m.double()[b.b2revb] for m, b in ((m1, b1), (m2, b2))])
    md = torch.cat([m1, m2]).to(DEV)
    pre = torch.empty_like(md)
    _lib.check(L.rr_bond_message_fwd(ctypes.byref(dg.c), md.data_ptr(), pre.data_ptr(), hp, 0, S()))
    close(pre, want)
    ups = [rand(b1.n_bonds, hp, h, 3), rand(b2.n_bonds, hp, h, 4)]
    grads = []
    for m, b, up in ((m1, b1, ups[0]), (m2, b2, ups[1])):
        x = m.double().requires_grad_(True)
        (O.gather_sum(x, b.a2b)[b.b2a] - x[b.b2revb]).backward(up.double())
        grads.append(x.grad)
    upd = torch.cat(ups).to(DEV)
    dm = torch.empty_like(upd)
    _lib.check(L.rr_bond_message_bwd(ctypes.byref(dg.c), upd.data_ptr(), dm.data_ptr(), hp, S()))
    close(dm, torch.cat(grads), 5e-6)
    # atom-level (a2a) gather across segments
    x1, x2 = rand(b1.n_atoms, hp, h, 5), rand(b2.n_atoms, hp, h, 6)
    want = torch.cat([O.gather_sum(x.double(), b.get_a2a()) for x, b in ((x1, b1), (x2, b2))])
    xd = torch.cat([x1, x2]).to(DEV)
    out = torch.empty_like(xd)
    _lib.check(L.rr_neighbor_sum_fwd(ctypes.byref(dg.c), 1, xd.data_ptr(), out.data_ptr(), hp, 0, S()))
    close(out, want)


def test_max_num_bonds_override_matches_bigger_batch():
    """A shard packed with the GLOBAL batch's max_num_bonds equals its rows inside the global batch
    (data-parallel sharding, SURVEY.md §8e)."""
    L = _lib.lib()
    ds = synthetic.make_dataset(10, [2, 2], star_leaves_in_group={1: 8})
    mols = [ds.mols[t] for t in ds.rsmi]
    whole, shard = BatchMolGraph(mols), BatchMolGraph(mols[:2])
    assert whole.max_num_bonds == 8 and shard.max_num_bonds < 8
    dg = DeviceGraph.from_batches([shard], DEV, [whole.max_num_bonds])
    h, hp = 24, 32
    m = rand(whole.n_bonds, hp, h, 1)
    want = (O.gather_sum(m.double(), whole.a2b)[whole.b2a] - m.double()[whole.b2revb])[:shard.n_bonds]
    md = m[:shard.n_bonds].contiguous().to(DEV)
    pre = torch.empty_like(md)
    _lib.check(L.rr_bond_message_fwd(ctypes.byref(dg.c), md.data_ptr(), pre.data_ptr(), hp, 0, S()))
    close(pre, want)


@pytest.mark.parametrize("M,n,k1,k2", [(1000, 304, 88, 0), (777, 304, 304, 88), (130, 48, 64, 48), (5, 16, 304, 0), (4100, 608, 608, 608)])
def test_linear_fwd_dgrad_wgrad(M, n, k1, k2):
    L = _lib.lib()
    g = torch.Generator().manual_seed(M)
    X1, W1 = torch.randn(M, k1, generator=g), torch.randn(n, k1, generator=g) / k1 ** 0.5
    X2 = torch.randn(M, k2, generator=g) if k2 else None
    W2 = torch.randn(n, k2, generator=g) / k2 ** 0.5 if k2 else None
    bias, resid = torch.randn(n, generator=g), torch.randn(M, n, generator=g)
    z = X1.double() @ W1.double().T + bias.double() + resid.double()
    if k2:
        z = z + X2.double() @ W2.double().T
    d = {k: (v.to(DEV) if v is not None else None) for k, v in dict(X1=X1, W1=W1, X2=X2, W2=W2, bias=bias, resid=resid).items()}
    Y = torch.empty(M, n, device=DEV)
    for flags, want in ((0, z), (1, torch.relu(z))):
        _lib.check(L.rr_linear_fwd(M, n, d["X1"].data_ptr(), k1, d["W1"].data_ptr(), k1, _lib.ptr(d["X2"]), k2, _lib.ptr(d["W2"]), k2,
                                   d["bias"].data_ptr(), d["resid"].data_ptr(), n, Y.data_ptr(), n, flags, 0.0, 0, 0, S()))
        close(Y, want, 3e-6)
    dZ = torch.randn(M, n, generator=g)
    dZd = dZ.to(DEV)
    dX = torch.empty(M, k1, device=DEV)
    _lib.check(L.rr_linear_dgrad(M, n, k1, dZd.data_ptr(), n, d["W1"].data_ptr(), k1, dX.data_ptr(), k1, 0, S()))
    close(dX, dZ.double() @ W1.double(), 3e-6)
    _lib.check(L.rr_linear_dgrad(M, n, k1, dZd.data_ptr(), n, d["W1"].data_ptr(), k1, dX.data_ptr(), k1, 1, S()))
    close(dX, 2 * (dZ.double() @ W1.double()), 3e-6)
    dW = torch.zeros(n, k1, device=DEV)
    db = torch.zeros(n, device=DEV)
    _lib.check(L.rr_linear_wgrad(M, n, k1, dZd.data_ptr(), n, d["X1"].data_ptr(), k1, dW.data_ptr(), k1, db.data_ptr(), S()))
    close(dW, dZ.double().T @ X1.double(), 1e-5)
    close(db, dZ.double().sum(0), 1e-5)


def test_dropout_epilogue_statistics_and_backward_mask():
    L = _lib.lib()
    M, n, k, p = 4096, 304, 64, 0.25
    X = torch.randn(M, k, device=DEV)
    W = torch.randn(n, k, device=DEV)
    Y0, Y1, Y2 = (torch.empty(M, n, device=DEV) for _ in range(3))
    for Y, flags, seed in ((Y0, 1, 0), (Y1, 3, 11), (Y2, 3, 12)):
        _lib.check(L.rr_linear_fwd(M, n, X.data_ptr(), k, W.data_ptr(), k, None, 0, None, 0, None, None, 0, Y.data_ptr(), n, flags, p, seed, 5, S()))
    pos = Y0 > 0
    dropped = (Y1 == 0) & pos
    frac = float(dropped.sum()) / float(pos.sum())
    assert abs(frac - p) < 0.01, frac
    kept = (Y1 != 0)
    close(Y1[kept], Y0[kept] / (1 - p), 1e-6)
    assert float(((Y1 == 0) != (Y2 == 0)).float().mean()) > 0.1      # another seed, another mask
    # relu_bwd regenerates nothing: mask = [y != 0], scale = 1/(1-p)
    dy = torch.randn(M, n, device=DEV)
    dz = torch.empty_like(dy)
    acc = torch.ones_like(dy)
    _lib.check(L.rr_relu_bwd(M, n, dy.data_ptr(), Y1.data_ptr(), 1 / (1 - p), 0, dz.data_ptr(), acc.data_ptr(), 2, S()))
    close(dz, dy * kept / (1 - p), 1e-6)
    close(acc, 1 + dy * kept / (1 - p), 1e-6)


def test_readout_fwd_bwd():
    L = _lib.lib()
    ds, b, dg = graphs(sizes=(3, 4))
    h, hp, vp, f = 40, 48, 48, 1
    hid = torch.relu(rand(b.n_atoms, hp, h, 1)).double().requires_grad_(True)
    feats = torch.tensor(ds.temp.reshape(-1, 1), dtype=torch.float32)
    vec = torch.stack([hid[s:s + n].sum(0) / n for s, n in b.a_scope])[:, :h]        # mpn.py:224-235
    want = torch.cat([vec, feats.double()], 1)                                          # mpn.py:237-238
    out = torch.full((b.n_mols, vp), float("nan"), device=DEV)
    hd, fd = hid.detach().float().to(DEV), feats.to(DEV)
    _lib.check(L.rr_readout_fwd(ctypes.byref(dg.c), hd.data_ptr(), hp, h, fd.data_ptr(), f, out.data_ptr(), vp, 0.0, 0, 0, S()))
    close(out[:, :h + f], want.detach())
    assert not out[:, h + f:].any()
    up = torch.randn(b.n_mols, vp)
    want.backward(up[:, :h + f].double())
    dz = torch.full((b.n_atoms, hp), float("nan"), device=DEV)
    upd = up.to(DEV)
    _lib.check(L.rr_readout_bwd(ctypes.byref(dg.c), upd.data_ptr(), vp, out.data_ptr(), hd.data_ptr(), dz.data_ptr(), hp, 0.0, S()))
    mask = (hid.detach() != 0)
    close(dz[:, :h], (hid.grad * mask)[:, :h], 3e-6)
    assert not dz[0].any()                                                              # the padding atom gets no gradient


LOSSES = [("mle", _lib.LOSS_LISTMLE, 1), ("listnet", _lib.LOSS_LISTNET, 1), ("evidential_ranking", _lib.LOSS_EVIDENTIAL, 2),
          ("gauss_regression", _lib.LOSS_GAUSS, 2), ("regression", _lib.LOSS_MSE, 1)]


@pytest.mark.parametrize("task,kind,cols", LOSSES)
@pytest.mark.parametrize("scope", [[5, 3, 6], [1, 2, 1], [32] * 8, [50, 100, 200, 500], [2048]])
def test_losses_match_oracle(task, kind, cols, scope):
    L = _lib.lib()
    N, G = sum(scope), len(scope)
    g = torch.Generator().manual_seed(N + kind)
    s = torch.randn(N, cols, generator=g)
    if cols == 2:
        s[:, 1] = torch.nn.functional.softplus(s[:, 1]) + 1e-3
    else:
        s = s[:, 0]
    t = torch.randn(N, generator=g)
    sx = s.double().requires_grad_(True)
    want = O.loss_for_task(task, sx, scope, t.double())
    want.backward(torch.ones_like(want))
    norm = {"mle": G, "evidential_ranking": G}.get(task, N)
    seg = torch.tensor(np.concatenate([[0], np.cumsum(scope)]), dtype=torch.int32, device=DEV)
    sd, td = s.to(DEV), t.to(DEV)
    loss, ds_ = torch.empty(1, device=DEV), torch.full_like(sd, float("nan"))
    _lib.check(L.rr_loss_fwdbwd(kind, N, G, sd.data_ptr(), td.data_ptr(), seg.data_ptr(), float(norm), 1.0, loss.data_ptr(), ds_.data_ptr(), S()))
    close(loss, want.detach().reshape(1), 2e-6)
    close(ds_, sx.grad, 2e-5)


@pytest.mark.parametrize("task,kind", [("mle", _lib.LOSS_LISTMLE), ("evidential_ranking", _lib.LOSS_EVIDENTIAL), ("ranknet", _lib.LOSS_RANKNET)])
@pytest.mark.parametrize("scope", [[3000, 5], [8192], [2049, 64, 1]])
def test_large_groups_through_the_sized_entry(task, kind, scope):
    """rr_loss_fwdbwd_ex sizes the per-group shared arrays from max_group (up to rr_loss_max_group() = 8192): groups beyond the plain
    entry's 2048 match the fp64 oracle; the plain entry answers NaN for them (never an overrun); max_group > 8192 is refused."""
    L = _lib.lib()
    assert L.rr_loss_max_group() == 8192
    N, G = sum(scope), len(scope)
    g = torch.Generator().manual_seed(N + kind)
    cols = 2 if task == "evidential_ranking" else 1
    s = torch.randn(N, cols, generator=g)
    if cols == 2:
        s[:, 1] = torch.nn.functional.softplus(s[:, 1]) + 1e-3
    else:
        s = s[:, 0]
    t = torch.randn(N, generator=g)
    sx = s.double().requires_grad_(True)
    if task == "ranknet":
        total, pairs, o = 0, 0.0, 0
        for n in scope:
            c, npairs = O.ranknet_group_cost(sx[o:o + n], t[o:o + n].numpy())
            if c is not None:
                total, pairs = total + c, pairs + npairs
            o += n
        want, norm = total / pairs, pairs
    else:
        want, norm = O.loss_for_task(task, sx, scope, t.double()), G
    want.backward(torch.ones_like(want))
    seg = torch.tensor(np.concatenate([[0], np.cumsum(scope)]), dtype=torch.int32, device=DEV)
    sd, td = s.to(DEV), t.to(DEV)
    loss, ds_ = torch.empty(1, device=DEV), torch.full_like(sd, float("nan"))
    _lib.check(L.rr_loss_fwdbwd_ex(kind, N, G, sd.data_ptr(), td.data_ptr(), seg.data_ptr(), max(scope), float(norm), 1.0,
                                   loss.data_ptr(), ds_.data_ptr(), S()))
    close(loss, want.detach().reshape(1), 5e-6)
    close(ds_, sx.grad, 5e-5)
    _lib.check(L.rr_loss_fwdbwd(kind, N, G, sd.data_ptr(), td.data_ptr(), seg.data_ptr(), float(norm), 1.0, loss.data_ptr(), ds_.data_ptr(), S()))
    torch.cuda.synchronize()
    if task == "evidential_ranking":                            # streams its groups through registers: no capacity to exceed
        close(loss, want.detach().reshape(1), 5e-6)
    else:
        assert bool(torch.isnan(loss).all()) and bool(torch.isnan(ds_[:scope[0]]).all())
    assert L.rr_loss_fwdbwd_ex(kind, N, G, sd.data_ptr(), td.data_ptr(), seg.data_ptr(), 8193, float(norm), 1.0,
                               loss.data_ptr(), ds_.data_ptr(), S()) != 0


def test_loss_modules_take_groups_beyond_2048():
    """The Python loss layer passes the batch's largest group down (rr_loss_fwdbwd_ex): MLEloss on a 3000-candidate group matches the fp64
    oracle in value and gradient; a group beyond rr_loss_max_group() is refused with RRError before any launch."""
    from reactranker_b200.train.loss import MLEloss
    scope = [3000, 40, 7]
    N = sum(scope)
    g = torch.Generator().manual_seed(5)
    s, t = torch.randn(N, generator=g), torch.randn(N, generator=g)
    sx = s.double().requires_grad_(True)
    want = O.listmle_loss(sx, scope, t.double())
    want.backward()
    sd = s.to(DEV).requires_grad_(True)
    loss = MLEloss()(sd, scope, t, 0)
    loss.backward()
    close(loss.detach().reshape(1), want.detach().reshape(1), 5e-6)
    close(sd.grad, sx.grad, 5e-5)
    big = [9000]
    with pytest.raises(_lib.RRError):
        MLEloss()(torch.zeros(9000, device=DEV), big, torch.zeros(9000), 0)


@pytest.mark.parametrize("scope", [[5, 4, 6], [64] * 4, [3, 500]])
def test_ranknet_window_matches_oracle(scope):
    L = _lib.lib()
    N, G = sum(scope), len(scope)
    g = torch.Generator().manual_seed(N)
    s, t = torch.randn(N, generator=g), torch.randn(N, generator=g)
    t[:3] = 0.5                                                  # a group whose targets tie: no pairs, skipped (train_pairwise.py:103-104)
    sx = s.double().requires_grad_(True)
    total, pairs, o = 0, 0.0, 0
    for n in scope:
        c, npairs = O.ranknet_group_cost(sx[o:o + n], t[o:o + n].numpy())
        if c is not None:
            total = total + c
            pairs += npairs
        o += n
    want = total / pairs
    want.backward()
    seg = torch.tensor(np.concatenate([[0], np.cumsum(scope)]), dtype=torch.int32, device=DEV)
    sd, td = s.to(DEV), t.to(DEV)
    loss, ds_ = torch.empty(1, device=DEV), torch.empty_like(sd)
    _lib.check(L.rr_loss_fwdbwd(_lib.LOSS_RANKNET, N, G, sd.data_ptr(), td.data_ptr(), seg.data_ptr(), pairs, 1.0, loss.data_ptr(), ds_.data_ptr(), S()))
    close(loss, want.detach().reshape(1), 2e-6)
    close(ds_, sx.grad, 2e-5)


def test_listmle_sortedness_and_shift_invariance_at_full_size():
    """Size-independent properties at config-5 scale (82 groups x 50, 8 x 500): the loss is invariant to a
    per-group shift of the scores, its gradient sums to zero per group, and a perfectly ordered group with
    widely separated scores has ~zero loss."""
    L = _lib.lib()
    for scope in ([50] * 82, [500] * 8):
        N, G = sum(scope), len(scope)
        s, t = torch.randn(N, device=DEV), torch.randn(N, device=DEV)
        seg = torch.tensor(np.concatenate([[0], np.cumsum(scope)]), dtype=torch.int32, device=DEV)
        shift = torch.repeat_interleave(torch.randn(G, device=DEV) * 3, torch.tensor(scope, device=DEV))
        out = []
        for sc in (s, s + shift, t * 50):
            loss, d = torch.empty(1, device=DEV), torch.empty(N, device=DEV)
            _lib.check(L.rr_loss_fwdbwd(_lib.LOSS_LISTMLE, N, G, sc.contiguous().data_ptr(), t.data_ptr(), seg.data_ptr(), float(G), 1.0,
                                        loss.data_ptr(), d.data_ptr(), S()))
            out.append((float(loss), d))
        assert abs(out[0][0] - out[1][0]) < 1e-4 * abs(out[0][0])
        persum = torch.stack([x.sum() for x in out[0][1].split(scope)])
        assert float(persum.abs().max()) < 1e-6
        assert out[2][0] < 0.05


def test_argument_errors_are_reported_not_crashed():
    L = _lib.lib()
    x = torch.zeros(8, 6, device=DEV)
    st = L.rr_linear_fwd(8, 6, x.data_ptr(), 6, x.data_ptr(), 6, None, 0, None, 0, None, None, 0, x.data_ptr(), 6, 0, 0.0, 0, 0, S())
    assert st == -1 and b"multiples of 4" in L.rr_last_error()
    with pytest.raises(_lib.RRError):
        _lib.check(L.rr_loss_fwdbwd(99, 4, 1, x.data_ptr(), x.data_ptr(), x.data_ptr(), 1.0, 1.0, x.data_ptr(), x.data_ptr(), S()))


@pytest.mark.parametrize("M,n,k1,k2", [(128, 48, 64, 0), (1000, 304, 88, 0), (777, 304, 304, 88), (130, 48, 64, 48), (5, 16, 304, 0),
                                       (4100, 608, 608, 608), (40000, 304, 304, 0), (300, 304, 16, 0)])
def test_tcgen05_linear_matches_fp64(tc_mode, M, n, k1, k2):
    """tcgen05 3xTF32 forward GEMM (bias + residual + ReLU epilogue, two-source K) against an fp64 matmul:
    fp32-class accuracy, 5e-6 of the largest output."""
    L = _lib.lib()
    g = torch.Generator().manual_seed(M + n)
    X1, W1 = torch.randn(M, k1, generator=g), torch.randn(n, k1, generator=g) / k1 ** 0.5
    X2 = torch.randn(M, k2, generator=g) if k2 else None
    W2 = torch.randn(n, k2, generator=g) / k2 ** 0.5 if k2 else None
    bias, resid = torch.randn(n, generator=g), torch.randn(M, n, generator=g)
    z = X1.double() @ W1.double().T + bias.double() + resid.double()
    if k2:
        z = z + X2.double() @ W2.double().T
    d = {k: (v.to(DEV) if v is not None else None) for k, v in dict(X1=X1, W1=W1, X2=X2, W2=W2, bias=bias, resid=resid).items()}
    Y = torch.full((M, n), float("nan"), device=DEV)
    for flags, want in ((0, z), (1, torch.relu(z))):
        _lib.check(L.rr_linear_fwd(M, n, d["X1"].data_ptr(), k1, d["W1"].data_ptr(), k1, _lib.ptr(d["X2"]), k2, _lib.ptr(d["W2"]), k2,
                                   d["bias"].data_ptr(), d["resid"].data_ptr(), n, Y.data_ptr(), n, flags, 0.0, 0, 0, S()))
        torch.cuda.synchronize()
        close(Y, want, 1e-5 if k1 + k2 > 1000 else 5e-6)
    # no bias / residual, plain product
    _lib.check(L.rr_linear_fwd(M, n, d["X1"].data_ptr(), k1, d["W1"].data_ptr(), k1, None, 0, None, 0, None, None, 0, Y.data_ptr(), n, 0, 0.0, 0, 0, S()))
    close(Y, X1.double() @ W1.double().T, 1e-5 if k1 > 500 else 5e-6)


def test_tcgen05_and_simt_draw_the_same_dropout_mask(tc_mode):
    L = _lib.lib()
    M, n, k, p = 1024, 304, 64, 0.3
    X, W = torch.randn(M, k, device=DEV), torch.randn(n, k, device=DEV)
    Yt, Ys = torch.empty(M, n, device=DEV), torch.empty(M, n, device=DEV)
    _lib.check(L.rr_linear_fwd(M, n, X.data_ptr(), k, W.data_ptr(), k, None, 0, None, 0, None, None, 0, Yt.data_ptr(), n, 3, p, 7, 9, S()))
    _lib.check(L.rr_set_gemm_mode(0))
    _lib.check(L.rr_linear_fwd(M, n, X.data_ptr(), k, W.data_ptr(), k, None, 0, None, 0, None, None, 0, Ys.data_ptr(), n, 3, p, 7, 9, S()))
    assert float(((Yt == 0) != (Ys == 0)).float().mean()) < 1e-4        # only entries whose pre-activation is ~0 may differ
    close(Yt, Ys.double(), 5e-6)


@pytest.mark.parametrize("M,n,k", [(1000, 304, 304), (4100, 304, 88), (777, 304, 64), (40000, 304, 304), (1000, 608, 608), (300, 16, 304),
                                   (513, 48, 48)])
@pytest.mark.parametrize("bf16", [1, 0])
def test_tcgen05_wgrad_matches_fp64(tc_mode, M, n, k, bf16):
    """tcgen05 wgrad (dZ through TMEM, X MN-major, split over the row range, vector reductions into dW) and its fused bias gradient,
    in both operand splits: 3 x bf16 (default for the backward pass, 16 significand bits per operand: 3e-5) and 3 x tf32 (1e-5)."""
    L = _lib.lib()
    L.rr_set_backward_bf16(bf16)
    tol = 3e-5 if bf16 else 1e-5
    g = torch.Generator().manual_seed(M + k)
    dZ, X = torch.randn(M, n, generator=g), torch.randn(M, k, generator=g)
    dZ[0] *= 50.0
    dZd, Xd = dZ.to(DEV), X.to(DEV)
    dW = torch.zeros(n, k, device=DEV)
    db = torch.zeros(n, device=DEV)
    _lib.check(L.rr_linear_wgrad(M, n, k, dZd.data_ptr(), n, Xd.data_ptr(), k, dW.data_ptr(), k, db.data_ptr(), S()))
    L.rr_set_backward_bf16(1)
    close(dW, dZ.double().T @ X.double(), tol)
    close(db, dZ.double().sum(0), 1e-5)
    L.rr_set_backward_bf16(bf16)
    _lib.check(L.rr_linear_wgrad(M, n, k, dZd.data_ptr(), n, Xd.data_ptr(), k, dW.data_ptr(), k, None, S()))   # accumulates
    L.rr_set_backward_bf16(1)
    close(dW, 2 * (dZ.double().T @ X.double()), tol)


@pytest.mark.parametrize("M,n,k", [(1000, 304, 304), (4100, 304, 304), (777, 304, 64), (40000, 304, 304), (1000, 608, 608), (300, 304, 16),
                                   (513, 48, 48), (129, 16, 320)])
@pytest.mark.parametrize("bf16", [1, 0])
def test_tcgen05_dgrad_matches_fp64(tc_mode, M, n, k, bf16):
    """The tensor-core dgrad of rr_model_backward (k_tc_gemm2<16, BF> with the transposed, pre-split weight images; 14 launches of every
    training step) through its own C-ABI entry point, dX (+)= dZ W, in both operand splits: 3 x bf16 (the default of the backward pass:
    16 significand bits per operand) and 3 x tf32, overwrite and accumulate."""
    L = _lib.lib()
    tol = 3e-5 if bf16 else 1e-5
    g = torch.Generator().manual_seed(M + n + k)
    dZ, W = torch.randn(M, n, generator=g), torch.randn(n, k, generator=g) / n ** 0.5
    dZ[0] *= 50.0                                   # one row two orders of magnitude larger (a padding row's gradient)
    dZd, Wd = dZ.to(DEV), W.to(DEV)
    nbytes = int(L.rr_linear_dgrad_tc_scratch_bytes(n, k))
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    dX = torch.full((M, k), float("nan"), device=DEV)
    want = dZ.double() @ W.double()
    row_scale = want.abs().amax(dim=1, keepdim=True).clamp_min(1e-30)
    try:
        L.rr_set_backward_bf16(bf16)
        _lib.check(L.rr_linear_dgrad_tc(M, n, k, dZd.data_ptr(), n, Wd.data_ptr(), k, dX.data_ptr(), k, 0, scratch.data_ptr(), nbytes, S()))
        torch.cuda.synchronize()
        assert float(((dX.double().cpu() - want).abs() / row_scale).max()) < tol          # per row: the large row must not hide the others
        _lib.check(L.rr_linear_dgrad_tc(M, n, k, dZd.data_ptr(), n, Wd.data_ptr(), k, dX.data_ptr(), k, 1, scratch.data_ptr(), nbytes, S()))
        assert float(((dX.double().cpu() - 2 * want).abs() / (2 * row_scale)).max()) < tol
        st = L.rr_linear_dgrad_tc(M, n, 12, dZd.data_ptr(), n, Wd.data_ptr(), k, dX.data_ptr(), k, 0, scratch.data_ptr(), nbytes, S())
        assert st == -4 and b"tensor-core" in L.rr_last_error()                             # RR_ERR_UNSUPPORTED, reported not crashed
    finally:
        L.rr_set_backward_bf16(1)


def test_device_assembly_equals_host_packing():
    """rr_graph_assemble (molecule store in HBM, ids + offsets from the host) writes exactly the arrays the host packer
    ships, for a single batch, for a multi-segment launch and with a max_num_bonds override."""
    from reactranker_b200.data.load_reactions import Parsing_features
    ds = synthetic.make_dataset(17, [5, 3, 6], star_leaves_in_group={1: 8})
    fz = Parsing_features(ds.mols)
    cases = []
    whole_r, whole_p = fz.parsing_reactions(np.stack([ds.rsmi, ds.psmi], 1))
    cases.append(([whole_r], None))
    cases.append(([whole_p], [whole_p.max_num_bonds + 2]))
    groups = [fz.parsing_smiles(list(ds.rsmi[a:b])) for a, b in ((0, 5), (5, 8), (8, 14))]
    cases.append((groups, None))
    for batches, w in cases:
        assert all(b._ids is not None for b in batches)
        dev_g = DeviceGraph.from_batches(batches, DEV, w)                       # assembled on the GPU
        host_g = DeviceGraph.from_batches([BatchMolGraph([ds.mols[s] for s in b.smiles_batch]) for b in batches], DEV, w)   # packed on the host
        assert dev_g.h2d_bytes < host_g.h2d_bytes / 50
        nA, nB, nM, wmax, S_ = dev_g.n_atoms, dev_g.n_bonds, dev_g.n_mols, dev_g.c.wmax, dev_g.c.n_segments
        assert (nA, nB, nM, wmax, S_) == (host_g.n_atoms, host_g.n_bonds, host_g.n_mols, host_g.c.wmax, host_g.c.n_segments)
        for name, dt, shape in (("f_atoms", torch.float32, (nA, 64)), ("f_bonds", torch.float32, (nB, 88)), ("a_meta", torch.int32, (nA, 4)),
                                ("a2b", torch.int32, (nA, wmax)), ("a2b_rev", torch.int32, (nA, wmax)), ("a2a", torch.int32, (nA, wmax)),
                                ("mol_start", torch.int32, (nM,)), ("mol_size", torch.int32, (nM,)), ("pad_bonds", torch.int32, (S_,)),
                                ("pad_atoms", torch.int32, (S_,))):
            assert torch.equal(dev_g.section(name, dt, shape), host_g.section(name, dt, shape)), name


# ---- gather backward fused with the ReLU / dropout backward that follows it (rr_mp_pipe.cu) ---------------------------------------
def _act_reference(d, y, scale, preact, acc0, acc_mode):
    mask = (y > 0) if preact else (y != 0)
    dz = d * mask * scale
    acc = dz if acc_mode == 1 else (acc0 + dz if acc_mode == 2 else None)
    return dz, acc


@pytest.mark.parametrize("acc_mode,skip_out,preact", [(1, 0, 0), (2, 0, 0), (2, 1, 1), (0, 0, 0)])
@pytest.mark.parametrize("h,star,segments", [(300, None, 1), (40, {1: 9}, 1), (40, {1: 9}, 2)])
def test_bond_message_bwd_act(h, star, segments, acc_mode, skip_out, preact):
    L = _lib.lib()
    ds = synthetic.make_dataset(11, [3, 3], star_leaves_in_group=star)
    mols = [ds.mols[t] for t in ds.rsmi]
    batches = [BatchMolGraph(mols)] if segments == 1 else [BatchMolGraph(mols[:3]), BatchMolGraph(mols[3:])]
    dg = DeviceGraph.from_batches(batches, DEV)
    hp = L.rr_padded(h)
    B = sum(b.n_bonds for b in batches)
    up, y, acc0 = rand(B, hp, h, 2), torch.relu(rand(B, hp, h, 6)), rand(B, hp, h, 7)
    grads, o = [], 0
    for b in batches:
        x = torch.zeros(b.n_bonds, hp, dtype=torch.double, requires_grad=True)
        (O.gather_sum(x, b.a2b)[b.b2a] - x[b.b2revb]).backward(up[o:o + b.n_bonds].double())
        grads.append(x.grad)
        o += b.n_bonds
    ysrc = (rand(B, hp, h, 6) if preact else y)
    want_dz, want_acc = _act_reference(torch.cat(grads), ysrc.double(), 0.8, preact, acc0.double(), acc_mode)
    dm = torch.full((B, hp), float("nan"), device=DEV)
    acc = acc0.to(DEV).clone()
    upd, yd = up.to(DEV), ysrc.to(DEV)
    _lib.check(L.rr_bond_message_bwd_act(ctypes.byref(dg.c), upd.data_ptr(), dm.data_ptr(), hp, yd.data_ptr(), 0.8, preact,
                                         acc.data_ptr() if acc_mode else None, acc_mode, skip_out, S()))
    if not skip_out:
        close(dm, want_dz, 5e-6)
    if acc_mode:
        close(acc, want_acc, 5e-6)


@pytest.mark.parametrize("which", [0, 1])
@pytest.mark.parametrize("acc_mode,skip_out,preact", [(1, 0, 0), (2, 0, 0), (1, 1, 1), (2, 1, 1)])
@pytest.mark.parametrize("h,star", [(300, None), (40, {2: 10})])
def test_neighbor_sum_bwd_act(which, h, star, acc_mode, skip_out, preact):
    L = _lib.lib()
    ds, b, dg = graphs(star=star, side="r" if star else "p")
    hp = L.rr_padded(h)
    rows = b.n_atoms if which else b.n_bonds
    table = b.get_a2a() if which else b.a2b
    src = torch.zeros(rows, hp, dtype=torch.double, requires_grad=True)
    up = rand(b.n_atoms, hp, h, 5)
    O.gather_sum(src, table).backward(up.double())
    ysrc = rand(rows, hp, h, 8) if preact else torch.relu(rand(rows, hp, h, 8))
    acc0 = rand(rows, hp, h, 9)
    want_dz, want_acc = _act_reference(src.grad, ysrc.double(), 1.25, preact, acc0.double(), acc_mode)
    dsrc = torch.full((rows, hp), float("nan"), device=DEV)
    acc = acc0.to(DEV).clone()
    upd, yd = up.to(DEV), ysrc.to(DEV)
    _lib.check(L.rr_neighbor_sum_bwd_act(ctypes.byref(dg.c), which, upd.data_ptr(), dsrc.data_ptr(), hp, yd.data_ptr(), 1.25, preact,
                                         acc.data_ptr(), acc_mode, skip_out, S()))
    if not skip_out:
        close(dsrc, want_dz, 5e-6)
    close(acc, want_acc, 5e-6)


def test_first_generation_gather_kernels_agree(monkeypatch):
    """RR_MP_V1=1 selects the register-gather kernels of rr_mp.cu; both generations give the same rows (bit-exact for the pure
    gathers, which add in the same order)."""
    L = _lib.lib()
    ds, b, dg = graphs(seed=21, sizes=(6, 5, 7))
    h, hp = 300, 304
    m = rand(b.n_bonds, hp, h, 1).to(DEV)
    outs = {}
    for v1 in ("0", "1"):
        monkeypatch.setenv("RR_MP_V1", v1)
        _lib.lib().rr_reload_switches()
        pre = torch.empty_like(m)
        am = torch.empty(b.n_atoms, hp, device=DEV)
        _lib.check(L.rr_bond_message_fwd(ctypes.byref(dg.c), m.data_ptr(), pre.data_ptr(), hp, 1, S()))
        _lib.check(L.rr_neighbor_sum_fwd(ctypes.byref(dg.c), 0, m.data_ptr(), am.data_ptr(), hp, 0, S()))
        outs[v1] = (pre.cpu(), am.cpu())
    assert torch.equal(outs["0"][0], outs["1"][0]) and torch.equal(outs["0"][1], outs["1"][1])


@pytest.mark.parametrize("seed,h,sizes,star,segments", [
    (101, 8, (1, 1, 1), None, 1), (102, 16, (3, 2), {0: 12}, 2), (103, 600, (5, 4, 3), None, 1), (104, 1000, (2, 2), {1: 6}, 1),
    (105, 300, (9, 1, 7, 2), {2: 5}, 4), (106, 44, (30, 20), None, 2)])
def test_row_pipeline_matches_first_generation_on_odd_shapes(monkeypatch, seed, h, sizes, star, segments):
    """Every gather op of the TMA-bulk row pipeline against the register-gather kernels (RR_MP_V1=1) over widths from 8 to 1000 floats,
    in-degrees above the four staged neighbours, single-molecule groups and multi-segment launches; fused variants against
    gather + rr_relu_bwd."""
    L = _lib.lib()
    ds = synthetic.make_dataset(seed, list(sizes), star_leaves_in_group=star)
    mols = [ds.mols[t] for t in ds.psmi]
    if segments == 1:
        batches = [BatchMolGraph(mols)]
    else:
        cuts = np.linspace(0, len(mols), segments + 1).astype(int)
        batches = [BatchMolGraph(mols[a:b]) for a, b in zip(cuts[:-1], cuts[1:]) if b > a]
    dg = DeviceGraph.from_batches(batches, DEV)
    hp = L.rr_padded(h)
    A, B = dg.n_atoms, dg.n_bonds
    g = ctypes.byref(dg.c)
    mB, upB, yB, accB0 = (rand(B, hp, h, seed + i).to(DEV) for i in range(4))
    mA, upA, yA, accA0 = (rand(A, hp, h, seed + 10 + i).to(DEV) for i in range(4))
    res = {}
    for v1 in ("1", "0"):
        monkeypatch.setenv("RR_MP_V1", v1)
        _lib.lib().rr_reload_switches()
        out = {}
        t = torch.empty(B, hp, device=DEV)
        _lib.check(L.rr_bond_message_fwd(g, mB.data_ptr(), t.data_ptr(), hp, 1, S()))
        out["bond_fwd"] = t
        t = torch.empty(B, hp, device=DEV)
        _lib.check(L.rr_bond_message_bwd(g, upB.data_ptr(), t.data_ptr(), hp, S()))
        out["bond_bwd"] = t
        for which, src in ((0, mB), (1, mA)):
            t = torch.empty(A, hp, device=DEV)
            _lib.check(L.rr_neighbor_sum_fwd(g, which, src.data_ptr(), t.data_ptr(), hp, 0, S()))
            out[f"nbr_fwd{which}"] = t
            rows = A if which else B
            t = torch.empty(rows, hp, device=DEV)
            _lib.check(L.rr_neighbor_sum_bwd(g, which, upA.data_ptr(), t.data_ptr(), hp, S()))
            out[f"nbr_bwd{which}"] = t
            y, acc0 = (yA, accA0) if which else (yB, accB0)
            for mode, skip in ((1, 0), (2, 0), (2, 1)):
                dz, acc = torch.zeros(rows, hp, device=DEV), acc0.clone()
                _lib.check(L.rr_neighbor_sum_bwd_act(g, which, upA.data_ptr(), dz.data_ptr(), hp, y.data_ptr(), 0.9, 0, acc.data_ptr(), mode, skip, S()))
                out[f"nbr_act{which}.{mode}{skip}"] = acc if skip else torch.cat([dz, acc])
        for mode, skip, pre in ((1, 0, 0), (2, 0, 0), (2, 1, 1)):
            dz, acc = torch.zeros(B, hp, device=DEV), accB0.clone()
            _lib.check(L.rr_bond_message_bwd_act(g, upB.data_ptr(), dz.data_ptr(), hp, yB.data_ptr(), 1.1, pre, acc.data_ptr(), mode, skip, S()))
            out[f"bond_act.{mode}{skip}"] = acc if skip else torch.cat([dz, acc])
        res[v1] = {k: v.cpu() for k, v in out.items()}
    for k in res["0"]:
        a, b = res["0"][k], res["1"][k]
        if "act" in k or "bwd" in k:          # padding rows are reduced with atomics (order), fused accumulators may use a reduction
            close(a, b, 2e-6)
        else:
            assert torch.equal(a, b), k


@pytest.mark.parametrize("which", ["mledis", "listnet_gauss", "expmse"])
@pytest.mark.parametrize("scope", [[5, 3, 6], [1, 2, 1], [32] * 8, [50, 100, 200]])
def test_distribution_valued_losses_match_the_reference_form(which, scope):
    """RR_LOSS_LISTMLE_DIS / RR_LOSS_LISTNET_DIS against the oracle's literal n x n restatement of MLEDisLoss / Listnet_For_Gauss
    (loss.py:102-141, 233-272), and RR_LOSS_EXPMSE, on ragged groups, in fp64 on the host."""
    L = _lib.lib()
    N, G = sum(scope), len(scope)
    g = torch.Generator().manual_seed(N + len(which))
    m = torch.randn(N, generator=g) * 0.7
    v = torch.nn.functional.softplus(torch.randn(N, generator=g)) * 0.5 + 1e-3
    t = torch.randn(N, generator=g)
    seg = torch.tensor(np.concatenate([[0], np.cumsum(scope)]), dtype=torch.int32, device=DEV)
    if which == "expmse":
        sx = m.double().requires_grad_(True)
        want = torch.mean((torch.exp(t.double()) - torch.exp(sx)) ** 2)
        want.backward()
        sd, kind, norm, wgrad = m.to(DEV), _lib.LOSS_EXPMSE, float(N), sx.grad
    else:
        mx, vx = m.double().requires_grad_(True), v.double().requires_grad_(True)
        fn = O.mledis_loss if which == "mledis" else O.listnet_gauss_loss
        want = fn(mx, vx, scope, t.double())
        want.backward(torch.ones_like(want))
        sd = torch.stack((m, v), 1).contiguous().to(DEV)
        kind = _lib.LOSS_LISTMLE_DIS if which == "mledis" else _lib.LOSS_LISTNET_DIS
        norm, wgrad = float(G), torch.stack((mx.grad, vx.grad), 1)
    td = t.to(DEV)
    loss, ds_ = torch.empty(1, device=DEV), torch.full_like(sd, float("nan"))
    _lib.check(L.rr_loss_fwdbwd(kind, N, G, sd.data_ptr(), td.data_ptr(), seg.data_ptr(), norm, 1.0, loss.data_ptr(), ds_.data_ptr(), S()))
    close(loss, want.detach().reshape(1), 3e-6)
    close(ds_, wgrad, 2e-5)


@pytest.mark.parametrize("coef", [0.0, 0.0216, 0.5])
@pytest.mark.parametrize("scope", [[5, 3, 6], [1, 2, 1], [32] * 8, [50, 100, 200]])
def test_listnet_uq_matches_the_reference_form(coef, scope):
    """RR_LOSS_LISTNET_UQ (annealing coefficient through `sigma`) against the oracle's restatement of Listnet_with_uq (loss.py:355-399),
    scores on both sides of 1 so that the |.| penalty changes sign inside a group."""
    L = _lib.lib()
    N, G = sum(scope), len(scope)
    g = torch.Generator().manual_seed(N)
    s = torch.nn.functional.softplus(torch.randn(N, generator=g) * 1.5) + 1e-2
    t = torch.randn(N, generator=g)
    seg = torch.tensor(np.concatenate([[0], np.cumsum(scope)]), dtype=torch.int32, device=DEV)
    sx = s.double().requires_grad_(True)
    want = O.listnet_uq_loss(sx, scope, t.double(), coef, 1, 2)          # (epoch / (epochs - 1)) ** 3 = 1
    want.backward(torch.ones_like(want))
    sd, td = s.to(DEV), t.to(DEV)
    loss, ds_ = torch.empty(1, device=DEV), torch.full_like(sd, float("nan"))
    _lib.check(L.rr_loss_fwdbwd(_lib.LOSS_LISTNET_UQ, N, G, sd.data_ptr(), td.data_ptr(), seg.data_ptr(), float(G), coef, loss.data_ptr(),
                                ds_.data_ptr(), S()))
    close(loss, want.detach().reshape(1), 3e-6)
    close(ds_, sx.grad, 2e-5)


@pytest.mark.parametrize("coef", [0.0, 0.0216])
@pytest.mark.parametrize("scope", [[5, 3, 6], [1, 2, 1], [32] * 8, [50, 100, 200]])
def test_dirichlet_uq_matches_the_reference_form(coef, scope):
    """RR_LOSS_DIRICHLET_UQ against the oracle's restatement of Dirichlet_uq (loss.py:440-474), concentrations on both sides of 1."""
    L = _lib.lib()
    N, G = sum(scope), len(scope)
    g = torch.Generator().manual_seed(N + 1)
    a = torch.nn.functional.softplus(torch.randn(N, generator=g) * 1.5) + 1e-2
    t = torch.randn(N, generator=g)
    seg = torch.tensor(np.concatenate([[0], np.cumsum(scope)]), dtype=torch.int32, device=DEV)
    ax = a.double().requires_grad_(True)
    want = O.dirichlet_uq_loss(ax, scope, t.double(), coef, 1, 2)
    want.backward(torch.ones_like(want))
    ad, td = a.to(DEV), t.to(DEV)
    loss, ds_ = torch.empty(1, device=DEV), torch.full_like(ad, float("nan"))
    _lib.check(L.rr_loss_fwdbwd(_lib.LOSS_DIRICHLET_UQ, N, G, ad.data_ptr(), td.data_ptr(), seg.data_ptr(), float(G), coef, loss.data_ptr(),
                                ds_.data_ptr(), S()))
    close(loss, want.detach().reshape(1), 3e-6)
    close(ds_, ax.grad, 2e-5)


@pytest.mark.parametrize("N", [1, 14, 128, 513, 1500])
@pytest.mark.parametrize("lam", [0.1, 0.2])
def test_nig_all_pairs_matches_the_reference_broadcast(N, lam):
    """RR_LOSS_NIG against evidential_loss_new evaluated with the shapes of its call sites ([N,1] parameters, [N] targets -> [N,N]),
    across row-block and column-tile boundaries (128 / 512)."""
    L = _lib.lib()
    g = torch.Generator().manual_seed(N)
    sp = torch.nn.functional.softplus
    mu = torch.randn(N, 1, generator=g)
    v = sp(torch.randn(N, 1, generator=g)) + 1e-6
    al = sp(torch.randn(N, 1, generator=g) * 2) + 1 + 1e-6
    be = sp(torch.randn(N, 1, generator=g)) + 1e-6
    t = torch.randn(N, generator=g)
    xs = [x.double().requires_grad_(True) for x in (mu, v, al, be)]
    want = O.nig_loss(*xs, t.double(), lam=lam)
    want.backward()
    sd = torch.cat((mu, v, al, be), 1).contiguous().to(DEV)
    td = t.to(DEV)
    loss, ds_ = torch.empty(1, device=DEV), torch.full_like(sd, float("nan"))
    _lib.check(L.rr_loss_fwdbwd(_lib.LOSS_NIG, N, 0, sd.data_ptr(), td.data_ptr(), None, float(N) * float(N), lam, loss.data_ptr(),
                                ds_.data_ptr(), S()))
    close(loss, want.detach().reshape(1), 5e-6)
    close(ds_, torch.cat([x.grad for x in xs], 1), 2e-5)


@pytest.mark.parametrize("N", [1, 14, 5000])
def test_lognorm_matches_the_reference_form(N):
    L = _lib.lib()
    g = torch.Generator().manual_seed(N)
    sp = torch.nn.functional.softplus
    m, v, t = sp(torch.randn(N, generator=g)) + 1e-6, sp(torch.randn(N, generator=g)) + 1e-6, torch.randn(N, generator=g)
    mx, vx = m.double().requires_grad_(True), v.double().requires_grad_(True)
    want = O.lognorm_loss(mx, vx, t.double())
    want.backward()
    sd, td = torch.stack((m, v), 1).contiguous().to(DEV), t.to(DEV)
    loss, ds_ = torch.empty(1, device=DEV), torch.full_like(sd, float("nan"))
    _lib.check(L.rr_loss_fwdbwd(_lib.LOSS_LOGNORM, N, 0, sd.data_ptr(), td.data_ptr(), None, float(N), 1.0, loss.data_ptr(), ds_.data_ptr(), S()))
    close(loss, want.detach().reshape(1), 3e-6)
    close(ds_, torch.stack((mx.grad, vx.grad), 1), 2e-5)


@pytest.mark.parametrize("task_type,last,task", [("listnetdis_lognorm", "with_softplus", 2), ("listnetdis_lognorm", "with_softplus", 6),
                                                 ("listnet", "with_uncertainty", 1), ("evidential", "with_softplus", 4),
                                                 ("evidential", "with_softplus", 8)])
def test_new_heads_against_the_oracle(task_type, last, task):
    """The FFN heads of base_model.py:61-70, 83-90, 101-104 through the whole model, also on wider-than-minimal task_num
    (the stack(..., dim=2).view interleave), forward and backward with a random upstream gradient."""
    from helpers import grads_close
    from reactranker_b200.models.base_model import build_model
    ds = synthetic.make_dataset(5, [4, 3])
    torch.manual_seed(task)
    model = build_model(hidden_size=24, mpnn_depth=2, mpnn_diff_depth=2, ffn_depth=2, use_bias=True, dropout=0.0, task_num=task,
                        ffn_last_layer=last, task_type=task_type, add_features_dim=1).cuda(0)
    sd64 = {k: v.double().cpu() for k, v in model.state_dict().items()}
    params = {k: v.clone().requires_grad_(True) for k, v in sd64.items() if "cached_zero" not in k}
    full = dict(sd64)
    full.update(params)
    r_g, p_g = O.OracleBatch([ds.mols[t] for t in ds.rsmi]), O.OracleBatch([ds.mols[t] for t in ds.psmi])
    want = O.model_forward(full, r_g, p_g, ds.temp.reshape(-1, 1), mpnn_depth=2, mpnn_diff_depth=2, ffn_depth=2,
                           head=O.resolve_task_type(task, last, task_type))
    got = model(BatchMolGraph([ds.mols[t] for t in ds.rsmi]), BatchMolGraph([ds.mols[t] for t in ds.psmi]), gpu=0,
                add_features=ds.temp.reshape(-1, 1))
    assert tuple(got.shape) == tuple(want.shape)
    close(got, want.detach(), 2e-5)
    w = torch.randn(got.shape, generator=torch.Generator().manual_seed(1))
    (want * w.double()).sum().backward()
    (got * w.to(got.device)).sum().backward()
    got_g = {k: p.grad.cpu().numpy() for k, p in model.named_parameters() if p.requires_grad}
    assert not grads_close(got_g, {k: params[k].grad.numpy() for k in got_g}, 2e-4)


@pytest.mark.parametrize("ratio", [0.25, 0.5])
@pytest.mark.parametrize("scope,ld", [([1, 2, 3, 6, 10, 14], 1), ([7, 1, 64, 300], 2), ([5000, 9], 1), ([33] * 200, 4)])
def test_rank_metrics_kernel_matches_the_host_restatement(scope, ld, ratio):
    """rr_rank_metrics against oracle.group_metrics (pinned to the reference's ranking_metrics / evaluate_top_scores goldens on the host):
    group sizes where n * ratio is exactly half way (2, 6, 10, 14: Python rounds half to even), tied scores AND tied targets (stable
    order), a group beyond the loss kernels' 2048 limit, strided score columns.  Hits are exact, NDCGs to 1e-12."""
    from reactranker_b200.train.eval import group_metrics
    N = sum(scope)
    g = torch.Generator().manual_seed(N + ld)
    s = torch.randn(N, ld, generator=g)
    s[:, 0] = torch.round(s[:, 0] * 4) / 4                      # plenty of exact ties
    t = np.round(torch.randn(N, generator=g).double().numpy() * 3) / 3
    got = group_metrics(s.to(DEV) if ld > 1 else s[:, 0].to(DEV), scope, t, ratio).cpu().numpy()
    want, o = [], 0
    for n in scope:
        want.append(O.group_metrics(s[o:o + n, 0].numpy(), t[o:o + n], ratio))
        o += n
    want = np.asarray(want)
    assert np.array_equal(got[:, [0, 2, 3]], want[:, [0, 2, 3]])
    assert np.allclose(got[:, 1], want[:, 1], rtol=0, atol=1e-15)
    assert np.allclose(got[:, 4:], want[:, 4:], rtol=1e-12, atol=0)


def test_rank_metrics_refuses_an_understated_max_group():
    """Shared memory is sized from max_group: a larger group must come back as NaN, not as an overrun."""
    L = _lib.lib()
    s = torch.randn(40, device=DEV)
    t = torch.randn(40, dtype=torch.float64, device=DEV)
    seg = torch.tensor([0, 8, 40], dtype=torch.int32, device=DEV)
    out = torch.zeros(2, 8, dtype=torch.float64, device=DEV)
    _lib.check(L.rr_rank_metrics(40, 2, s.data_ptr(), 1, t.data_ptr(), seg.data_ptr(), 8, 0.25, out.data_ptr(), S()))
    o = out.cpu()
    assert bool(torch.isfinite(o[0]).all()) and bool(torch.isnan(o[1]).all())


@pytest.mark.parametrize("dedup", [False, True])
def test_id_vector_assembly_equals_per_group_batches(dedup):
    """DeviceGraph.from_id_groups (store ids + segment lengths, no BatchMolGraph per group) builds byte-identical device graphs to
    from_batches / from_batches_dedup: every section of the blob, the sizes and the reactant atom map."""
    from reactranker_b200.data.load_reactions import Parsing_features
    ds = synthetic.make_dataset(31, [6, 1, 9, 4], star_leaves_in_group={2: 7})
    fz = Parsing_features(ds.mols)
    groups = [(0, 6), (6, 7), (7, 16), (16, 20)]
    r_b = [fz.parsing_smiles(list(ds.rsmi[a:b])) for a, b in groups]
    p_b = [fz.parsing_smiles(list(ds.psmi[a:b])) for a, b in groups]
    if dedup:
        rg1, pg1 = DeviceGraph.from_batches_dedup(r_b, p_b, DEV)
    else:
        rg1, pg1 = DeviceGraph.from_batches(r_b, DEV), DeviceGraph.from_batches(p_b, DEV)
    rg2, pg2 = DeviceGraph.from_id_groups(fz.store, fz.parsing_ids(list(ds.rsmi)), fz.parsing_ids(list(ds.psmi)), [b - a for a, b in groups], DEV, dedup)
    torch.cuda.synchronize()
    for g1, g2 in ((rg1, rg2), (pg1, pg2)):
        assert (g1.n_atoms, g1.n_bonds, g1.n_mols, g1.c.wmax, g1.c.n_segments) == (g2.n_atoms, g2.n_bonds, g2.n_mols, g2.c.wmax, g2.c.n_segments)
        sizes = dict(DeviceGraph._sections(g1.n_atoms, g1.n_bonds, g1.n_mols, g1.c.wmax, g1.c.n_segments))
        for name in sizes:          # same bytes in every section (a pair's blob lays its sections out differently: adjacent feature arrays)
            o1, o2 = g1._offs[name], g2._offs[name]
            assert torch.equal(g1.blob[o1:o1 + sizes[name]], g2.blob[o2:o2 + sizes[name]]), name
    if dedup:
        assert rg2.n_mols == 4 and torch.equal(rg1.atom_map, rg2.atom_map)
