"""Fine-tuning with frozen tensors on the GPU: rr_model_backward computes only the gradients autograd asks for (a NULL pointer for a
frozen tensor) and launches nothing below the lowest trainable layer.  The trainable gradients are the full backward's bit for bit in
deterministic mode, match the fp64 oracle, the launch counts follow the configuration, and main.py / predict.py fine-tune and rank."""
import ctypes

import numpy as np
import pytest
import torch

from reactranker_b200 import _lib, parallel, synthetic
from reactranker_b200.features.featurization import DeviceGraph
from helpers import check_grads, rel_err, TOL
from test_gpu_dropout import Layout
from test_gpu_model_variants import _case, oracle_run, relu_masks_and_keeps, saved_buffers
from test_gpu_train import _loss_curve, run
from test_model_variants_cpu import variant

pytestmark = pytest.mark.gpu
GPU = 0

# frozen state_dict names of each pattern (FFN Linear layers sit at ffn.ffn.1 / .4 / .7); "ddepth0_*" run the diff-depth-0 model
PATTERNS = {
    "encoder": lambda n: n.startswith("encoder."),
    "encoder_diff": lambda n: n.startswith(("encoder.", "diff_encoder.")),
    "encoder_diff_ffn1": lambda n: n.startswith(("encoder.", "diff_encoder.", "ffn.ffn.1.")),
    "last_ffn_only": lambda n: not n.startswith("ffn.ffn.7."),
    "middle_ffn": lambda n: n.startswith("ffn.ffn.4."),
    "encoder_Wi": lambda n: n.startswith("encoder.W_i."),
    "bias_only": lambda n: n in ("encoder.W_h.weight", "diff_encoder.W_o.weight", "ffn.ffn.4.weight"),
    "ddepth0_encoder": lambda n: n.startswith("encoder."),
    "ddepth0_bias_only": lambda n: n.startswith("encoder.") or n == "diff_encoder.W_i.weight",
}


@pytest.fixture(autouse=True)
def _modes_back_afterwards():
    yield
    torch.use_deterministic_algorithms(False)
    _lib.check(_lib.lib().rr_set_deterministic(0))


def _config(pattern):
    return variant("ddepth0") if pattern.startswith("ddepth0") else variant("w40_64_24", hd=40, hf=40)


def _freeze(model, pattern):
    """requires_grad per PATTERNS[pattern]; returns (frozen names, bias-only names: biases that train under a frozen weight)."""
    frozen, names = PATTERNS[pattern], dict(model.named_parameters())
    for n, p in names.items():
        if "cached_zero" not in n:
            p.requires_grad_(not frozen(n))
    frozen_names = [n for n, p in names.items() if not p.requires_grad and "cached_zero" not in n]
    bias_only = [n for n in names if n.endswith(".bias") and names[n].requires_grad and n[:-4] + "weight" in frozen_names]
    return frozen_names, bias_only


def _grads(model, rb, pb, feats, w, seed=11):
    for p in model.parameters():
        p.grad = None
    torch.manual_seed(seed)
    out = model(rb[0], pb[0], gpu=GPU, add_features=feats)
    (out * w.to(out.device)).sum().backward()
    torch.cuda.synchronize()
    return {n: (None if p.grad is None else p.grad.clone()) for n, p in model.named_parameters() if "cached_zero" not in n}


@pytest.mark.parametrize("bf16", [1, 0], ids=["bwd_bf16", "bwd_tf32"])
@pytest.mark.parametrize("mode", [0, 1, 2, 3])
@pytest.mark.parametrize("pattern", list(PATTERNS))
def test_trainable_gradients_equal_the_full_backward_bit_for_bit(pattern, mode, bf16):
    """Deterministic mode, dropout 0.1 in every module: every trainable gradient of the frozen backward is the full backward's tensor
    bit for bit; frozen tensors get no gradient.  A bias that trains under a frozen weight comes from its own column-sum kernel (other
    bits than the weight gradient's fused sum): two frozen runs agree bit for bit, and the oracle test below checks its value."""
    L = _lib.lib()
    L.rr_set_gemm_mode(mode)
    L.rr_set_backward_bf16(bf16)
    torch.use_deterministic_algorithms(True)
    c = _config(pattern)
    model, sd, ds, feats, rb, pb, groups, w = _case(c, (0.1, 0.1, 0.1))
    model.train()
    full = _grads(model, rb, pb, feats, w)
    frozen, bias_only = _freeze(model, pattern)
    got = _grads(model, rb, pb, feats, w)
    assert frozen and all(got[n] is None for n in frozen)
    for n, g in got.items():
        if n not in frozen and n not in bias_only:
            assert torch.equal(g, full[n]), n
    if bias_only:
        again = _grads(model, rb, pb, feats, w)
        assert all(torch.equal(again[n], got[n]) for n in bias_only)


@pytest.mark.parametrize("pattern", list(PATTERNS))
def test_trainable_gradients_match_the_fp64_oracle(pattern, gemm_mode):
    """Dropout 0, the flags of the pattern on the model; the oracle's gradients of the same tensors (autograd's values do not depend on
    which other tensors require one), at the model tests' tolerances.  The bias-only kernel repeats bit for bit in the default mode too,
    where its input does: in the FFN (the encoders' gathers sum padding rows with atomics in this mode)."""
    c = _config(pattern)
    model, sd, ds, feats, rb, pb, groups, w = _case(c, (0.0, 0.0, 0.0))
    model.train()
    frozen, bias_only = _freeze(model, pattern)
    lay = Layout(rb, pb)
    out = model(rb[0], pb[0], gpu=GPU, add_features=feats)
    masks = relu_masks_and_keeps(saved_buffers(model, out, c, lay), {}, c, lay) if gemm_mode == 1 else None
    (out * w.to(out.device)).sum().backward()
    ws, wg, _ = oracle_run(sd, c, groups, w)
    assert rel_err(out.detach().cpu().numpy(), ws) < TOL[gemm_mode]["score"]
    got = {k: q.grad.cpu().numpy() for k, q in model.named_parameters() if q.requires_grad}
    assert set(got) == set(wg) - set(frozen)
    assert all(q.grad is None for k, q in model.named_parameters() if k in frozen)

    def redo():
        _, g, flips = oracle_run(sd, c, groups, w, relu=masks)
        return {k: g[k] for k in got}, flips
    check_grads(gemm_mode, got, {k: wg[k] for k in got}, redo if masks else None)
    if bias_only:
        again = _grads(model, rb, pb, feats, w, seed=0)
        assert all(np.array_equal(again[k].cpu().numpy(), got[k]) for k in bias_only if k.startswith("ffn."))


# ------------------------------------------------------------------------------------------------
# launch counts of the backward pass
# ------------------------------------------------------------------------------------------------
CLASSES = ("gemm_dgrad", "gemm_wgrad", "bond_bwd", "nbr_bwd", "readout", "elementwise")


def launch_plan(c, trainable):
    """Per-class launches of rr_model_backward (default mode, no de-duplication) for the set of trainable state_dict names, following
    the rule of include/rr_sm100.h: a weight gradient per requested weight (two for a split weight), the two bias-only kernels for a
    bias that trains under a frozen weight, and the dgrad chain only while some layer below trains."""
    n = dict.fromkeys(CLASSES, 0)
    F, T, Td = c["ffn_depth"], c["depth"] - 1, c["ddepth"] - 1
    layers = ["encoder.W_i", "encoder.W_h", "encoder.W_o", "diff_encoder.W_i", "diff_encoder.W_h", "diff_encoder.W_o"]
    layers += [f"ffn.ffn.{1 + 3 * l}" for l in range(F)]
    w = [m + ".weight" in trainable for m in layers]
    b = [m + ".bias" in trainable for m in layers]
    below = [any(w[:i]) or any(b[:i]) for i in range(len(layers) + 1)]

    def grads(i, splits=1):
        n["gemm_wgrad"] += splits if w[i] else (2 if b[i] else 0)
    for l in range(F - 1, -1, -1):
        grads(6 + l)
        if not below[6 + l]:
            return n
        n["gemm_dgrad"] += 1
        n["elementwise"] += 1 if l > 0 else 0
    n["readout"] += 1
    if c["ddepth"] > 0:
        grads(5, 2)
        if not below[5]:
            return n
        n["gemm_dgrad"] += 2 if below[3] else 1
        n["nbr_bwd"] += 1
        for t in range(Td, 0, -1):
            grads(4, 2)
            if t == 1 and not below[4]:
                return n
            n["gemm_dgrad"] += 1
            n["nbr_bwd"] += 1
    grads(3)
    if not below[3]:
        return n
    n["gemm_dgrad"] += 1
    n["elementwise"] += 2
    grads(2, 2)
    if not below[2]:
        return n
    n["gemm_dgrad"] += 1
    n["nbr_bwd"] += 1
    for t in range(T, 0, -1):
        grads(1)
        if t == 1 and not below[1]:
            return n
        n["gemm_dgrad"] += 1
        n["bond_bwd"] += 1
    grads(0)
    return n


def _backward_launches(model, rb, pb, feats, w):
    for p in model.parameters():
        p.grad = None
    out = model(rb[0], pb[0], gpu=GPU, add_features=feats)
    torch.cuda.synchronize()
    _lib.profile_begin()
    (out * w.to(out.device)).sum().backward()
    torch.cuda.synchronize()
    prof = _lib.profile_end()
    return {k: prof[k][1] for k in CLASSES}


@pytest.mark.parametrize("pattern", ["none"] + list(PATTERNS))
def test_launch_counts_follow_the_frozen_set(pattern, gemm_mode):
    c = _config(pattern)
    model, sd, ds, feats, rb, pb, groups, w = _case(c, (0.1, 0.1, 0.1))
    model.train()
    if pattern != "none":
        _freeze(model, pattern)
    trainable = {n for n, p in model.named_parameters() if p.requires_grad}
    got = _backward_launches(model, rb, pb, feats, w)
    assert got == launch_plan(c, trainable), (got, launch_plan(c, trainable))
    if pattern.endswith("encoder"):
        assert got["bond_bwd"] == 0 and got["nbr_bwd"] == c["ddepth"]


def test_nothing_requested_launches_nothing_and_the_all_null_struct_is_ok():
    c = _config("encoder")
    model, sd, ds, feats, rb, pb, groups, w = _case(c, (0.0, 0.0, 0.0))
    for p in model.parameters():
        p.requires_grad_(False)
    out = model(rb[0], pb[0], gpu=GPU, add_features=feats)
    assert out.grad_fn is None                                    # nothing requires a gradient: autograd records no node
    # the C ABI directly: an all-NULL gradient struct returns RR_OK without a launch
    next(model.ffn.linears()[-1].parameters()).requires_grad_(True)
    out = model(rb[0], pb[0], gpu=GPU, add_features=feats)
    node = out.grad_fn
    L = _lib.lib()
    params = [p for _, p in model._named_slots()]
    pw = model._param_struct(params)
    nothing = _lib.RRParams()
    dscores = torch.ones_like(out)
    L.rr_launch_count_reset()
    _lib.check(L.rr_model_backward_ex(ctypes.byref(node.cfg), ctypes.byref(pw), ctypes.byref(node.rg.c), ctypes.byref(node.pg.c),
                                      dscores.data_ptr(), ctypes.byref(nothing), node.ws.data_ptr(), node.ws.numel(), _lib.stream_ptr()))
    assert L.rr_launch_count() == 0


def test_deterministic_backward_with_shared_reactants_and_a_frozen_encoder():
    """r_atom_map (each reactant encoded once) in deterministic mode: with the encoder frozen the backward runs -- the atomic sum over
    shared rows lives in the encoder's backward only -- and repeats bit for bit; asking for an encoder gradient is still refused."""
    from reactranker_b200.data.load_reactions import Parsing_features
    c = _config("encoder")
    ds = synthetic.make_dataset(61, [6, 5, 7])
    feats = torch.as_tensor(ds.temp.reshape(-1, 1), dtype=torch.float32, device="cuda")
    torch.manual_seed(3)
    from test_model_variants_cpu import variant_model
    model = variant_model(c).cuda(GPU).train()
    fz = Parsing_features(ds.mols)
    r_b, p_b = fz.parsing_smiles(list(ds.rsmi)), fz.parsing_smiles(list(ds.psmi))
    rg, pg = DeviceGraph.from_batches_dedup([r_b], [p_b], torch.device("cuda", GPU))
    assert rg.atom_map is not None
    L = _lib.lib()
    _lib.check(L.rr_set_deterministic(1))
    cfg = model._cfg(training=True)
    cfg.r_atom_map = rg.atom_map.data_ptr()
    params = [p for _, p in model._named_slots()]
    pw = model._param_struct(params)
    need = L.rr_model_workspace_bytes_ex(ctypes.byref(cfg), ctypes.byref(rg.c), ctypes.byref(pg.c))
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    scores = torch.empty(pg.n_mols, device="cuda")
    dscores = torch.linspace(-1, 1, pg.n_mols, device="cuda")

    def backward(names):
        grads = [torch.full_like(p, 7.0) if n in names else None for n, p in model._named_slots()]
        _lib.check(L.rr_model_forward_ex(ctypes.byref(cfg), ctypes.byref(pw), ctypes.byref(rg.c), ctypes.byref(pg.c), feats.data_ptr(),
                                         scores.data_ptr(), ws.data_ptr(), need, _lib.stream_ptr()))
        st = L.rr_model_backward_ex(ctypes.byref(cfg), ctypes.byref(pw), ctypes.byref(rg.c), ctypes.byref(pg.c), dscores.data_ptr(),
                                    ctypes.byref(model._param_struct(grads)), ws.data_ptr(), need, _lib.stream_ptr())
        torch.cuda.synchronize()
        return st, [g for g in grads if g is not None]
    slots = [n for n, _ in model._named_slots()]
    trainable = [n for n in slots if not str(n).startswith("enc_")]
    st, g1 = backward(trainable)
    assert st == 0 and all(not bool((g == 7.0).all()) for g in g1)
    st, g2 = backward(trainable)
    assert all(torch.equal(a, b) for a, b in zip(g1, g2))
    st, _ = backward(slots)
    assert st == -4                                                    # RR_ERR_UNSUPPORTED


def test_main_fine_tunes_a_pretrained_checkpoint_and_predict_ranks_with_it(tmp_path):
    """main.py --pretrained ckpt --freeze encoder,diff_encoder for two epochs: the frozen tensors of the written checkpoint are the
    pretrained ones bit for bit, the trainable ones moved; predict.py ranks with the result."""
    import main
    import pandas as pd
    from reactranker_b200.utils import load_checkpoint, save_checkpoint
    torch.manual_seed(5)
    pre = main.make_model("listnet", 64, 3, 0.1)
    ckpt = str(tmp_path / "pre.pt")
    save_checkpoint(ckpt, pre)
    args = ["--synthetic", "40,10", "--task_type", "listnet", "--hidden_size", "64", "--batch_size", "100", "--gpu", "0"]
    run(["main.py"] + args + ["--total_epochs", "3", "--stop_after", "2", "--save_metric", "average_score", "--path", str(tmp_path / "ft"), "--pretrained", ckpt,
                              "--freeze", "encoder,diff_encoder"])
    out_ckpt = str(tmp_path / "ft" / "0.pt")
    got, want = load_checkpoint(out_ckpt)["state_dict"], pre.state_dict()
    for k in want:
        if k.startswith(("encoder.", "diff_encoder.")):
            assert torch.equal(got[k], want[k]), k
        else:
            assert not torch.equal(got[k], want[k]), k
    log = open(str(tmp_path / "ft" / "output.log")).read()
    assert "Frozen tensors" in log and "encoder.W_i.weight" in log
    out = str(tmp_path / "ranked.csv")
    run(["predict.py", "--checkpoint", out_ckpt, "--synthetic", "40,10", "--out", out, "--hidden_size", "64", "--task_type", "listnet"])
    assert len(pd.read_csv(out)) == 400


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_torchrun_fine_tune_reproduces_the_one_gpu_loss_curve(tmp_path):
    """--freeze encoder under torchrun (2 ranks, in-place all-reduce of the trainable tensors only) trains as the one-GPU run does."""
    import main
    from reactranker_b200.utils import save_checkpoint
    torch.manual_seed(5)
    ckpt = str(tmp_path / "pre.pt")
    save_checkpoint(ckpt, main.make_model("mle", 64, 3, 0.0))
    args = ["main.py", "--synthetic", "40,10", "--task_type", "mle", "--batch_size", "100", "--total_epochs", "4", "--hidden_size", "64",
            "--max_lr", "3e-3", "--dropout", "0.0", "--pretrained", ckpt, "--freeze", "encoder"]
    one = run(args + ["--gpu", "0", "--path", str(tmp_path / "one")])
    two = run(["-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29641"]
              + args + ["--path", str(tmp_path / "two")])
    want, got = _loss_curve(one), _loss_curve(two)
    assert len(want) == 4 and np.allclose(got, want, rtol=1e-4), (got, want)


def test_train_step_all_reduce_carries_the_trainable_tensors_only():
    """TrainStep's GradSync over a frozen model: the in-place buffer of the backward pass has GradSync's layout (its element count is
    the aligned trainable count) and is aliased by every trainable p.grad, so a data-parallel step takes the in-place path."""
    c = _config("encoder")
    model, sd, ds, feats, rb, pb, groups, w = _case(c, (0.0, 0.0, 0.0))
    _freeze(model, "encoder")
    sync = parallel.GradSync(model.parameters(), None, model)
    _grads(model, rb, pb, feats, w)
    assert sync.numel == parallel.flat_layout(model.hot_parameters())[1] == model._grad_flat.numel()
    assert list(model._grad_offsets) == sync.offsets
    assert sync._aliased() is model._grad_flat
