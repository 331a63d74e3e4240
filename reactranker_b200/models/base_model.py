"""``build_model`` / ``ReactionModel`` with the reference's signature, defaults, module tree
and ``state_dict`` keys (models/base_model.py:10-171, 235-297), executing on sm_100a kernels.

``model(r_inputs, p_inputs, gpu, add_features)`` takes two ``BatchMolGraph`` objects exactly
like the reference (base_model.py:150-154).  ``gpu=None`` raises: there is no CPU path.
"""
from __future__ import annotations

import ctypes
from typing import List, Optional

import numpy as np
import torch
import torch.nn as nn

from .. import _lib
from ..parallel import flat_layout
from ..features.featurization import ATOM_FDIM, BOND_FDIM, BatchMolGraph, DeviceGraph
from .mpn import MPN, MPNDiff

_HEADS = {
    "evidential_ranking": _lib.HEAD_EVIDENTIAL_RANKING,
    "gauss_regression_with_softplus": _lib.HEAD_GAUSS_SOFTPLUS,
    "gaussian_with_softplus": _lib.HEAD_GAUSS_SOFTPLUS,
    "listnet_with_softplus": _lib.HEAD_SOFTPLUS,
    "listnetdis_lognorm_with_softplus": _lib.HEAD_LOGNORM,     # base_model.py:83-90 (without its debugging print of the whole output)
    "listnet_with_uncertainty": _lib.HEAD_SOFTPLUS_P1,         # base_model.py:101-102
    "evidential": _lib.HEAD_SOFTPLUS_P1,                       # base_model.py:103-104
    "evidential_with_softplus": _lib.HEAD_NIG,                 # base_model.py:61-70
}
_UNBUILT_HEADS = ()


class FFN(nn.Module):
    """Same Sequential layout as the reference (base_model.py:32-57) so the Linear layers sit
    at indices 1, 4, 7 of ``ffn.ffn``; evaluated by the fused model kernel sequence."""

    def __init__(self, reacvec_fdim: int, ffn_hidden_size: int, ffn_dropout: float = 0.2, ffn_num_layers: int = 3,
                 task_num: int = 2, ffn_bias: bool = True, task_type: str = 'gaussian'):
        super().__init__()
        self.hidden_size, self.ffn_hidden_size = reacvec_fdim, ffn_hidden_size
        self.dropout, self.ffn_num_layers, self.task_type, self.bias = ffn_dropout, ffn_num_layers, task_type, ffn_bias
        self.activation = nn.ReLU()
        self.output = None
        drop = nn.Dropout(self.dropout)
        if ffn_num_layers == 1:
            layers = [drop, nn.Linear(reacvec_fdim, task_num, bias=ffn_bias)]
        else:
            layers = [drop, nn.Linear(reacvec_fdim, ffn_hidden_size, bias=ffn_bias)]
            for _ in range(ffn_num_layers - 2):
                layers += [self.activation, drop, nn.Linear(ffn_hidden_size, ffn_hidden_size, bias=ffn_bias)]
            layers += [self.activation, drop, nn.Linear(ffn_hidden_size, task_num, bias=ffn_bias)]
        self.ffn = nn.Sequential(*layers)

    def linears(self) -> List[nn.Linear]:
        return [m for m in self.ffn if isinstance(m, nn.Linear)]

    def forward(self, *args, **kwargs):
        raise NotImplementedError("FFN runs fused inside ReactionModel.forward (reactranker_b200/csrc/rr_model.cu)")


def reactant_dedup_exact(model) -> bool:
    """Whether ``model`` may encode each distinct reactant once (rr_model_cfg.r_atom_map) instead of once per candidate.  The scores are the
    same in eval mode and at dropout 0 (with dropout the reference draws a mask per copy).  Under torch.use_deterministic_algorithms it is
    used only where no backward pass can follow (eval mode with grad disabled): the gradient of a shared row is a sum over its copies
    that rr_model_backward forms with atomics, so the deterministic backward refuses it."""
    if not getattr(model, "dedup_reactants", False):
        return False
    if model.training and model.any_dropout():
        return False
    return not _lib.deterministic_requested() or (not model.training and not torch.is_grad_enabled())


class _WorkspacePool:
    """Saved-for-backward workspaces (3-7 GB per step) recycled between steps.  Batch composition changes every step, so
    the exact size does too: asking the caching allocator for a fresh block per step ends in cudaMalloc / cudaFree
    round trips (tens of ms).  A forward takes the smallest free buffer that fits (allocating with head-room when none
    does); the backward gives it back.  A graph that is never back-propagated simply drops its buffer.
    Head-room 30 %: a data-parallel shard is a run of whole groups, so with a few large groups per rank (8 x 500 candidates) its size
    moves by a group (+-12.5 %) from step to step, and every growth is a cudaFree + cudaMalloc of GBs with the device drained."""

    def __init__(self, headroom: float = 1.3):
        self.free: List[torch.Tensor] = []
        self.headroom = headroom

    def take(self, nbytes: int, dev: torch.device) -> torch.Tensor:
        fits = [t for t in self.free if t.device == dev and t.numel() >= nbytes]
        if fits:
            best = min(fits, key=lambda t: t.numel())
            self.free = [t for t in self.free if t is not best]
            return best
        self.free = [t for t in self.free if t.device != dev]      # too small for the batches now arriving: let them go
        return torch.empty(int(nbytes * self.headroom) + 256, dtype=torch.uint8, device=dev)

    def give(self, t: torch.Tensor) -> None:
        if len(self.free) < 4:
            self.free.append(t)


class _ReactionFn(torch.autograd.Function):
    """One autograd node for the whole model: rr_model_forward / rr_model_backward."""

    @staticmethod
    def forward(ctx, model, rg: DeviceGraph, pg: DeviceGraph, addf, *params):
        L = _lib.lib()
        # torch.use_deterministic_algorithms(True) selects the library's deterministic mode for this step: set before the workspace is
        # sized (it then includes the backward's scratch) and recorded, so that the backward runs in the same mode
        det = _lib.deterministic_requested()
        _lib.set_deterministic(det)
        cfg = model._cfg(training=model.training)
        amap = getattr(rg, "atom_map", None)
        if amap is not None:
            if model.training and model.any_dropout():
                raise _lib.RRError("de-duplicated reactants are exact only without dropout (eval mode or dropout = 0)")
            cfg.r_atom_map = amap.data_ptr()
        w = model._param_struct(params)
        ws_bytes = L.rr_model_workspace_bytes_ex(ctypes.byref(cfg), ctypes.byref(rg.c), ctypes.byref(pg.c))
        if ws_bytes < 0:
            _lib.check(-1)
        dev = params[0].device
        ws = model._ws_pool.take(int(ws_bytes), dev)
        n = pg.n_mols
        scores = torch.empty((n,) if cfg.task_num == 1 else (n, cfg.task_num), dtype=torch.float32, device=dev)
        _lib.check(L.rr_model_forward_ex(ctypes.byref(cfg), ctypes.byref(w), ctypes.byref(rg.c), ctypes.byref(pg.c),
                                      _lib.ptr(addf), scores.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr()))
        if not any(ctx.needs_input_grad):        # inference: nothing will come back for the activations
            model._ws_pool.give(ws)
            ws = None
        ctx.model, ctx.rg, ctx.pg, ctx.cfg, ctx.ws, ctx.addf, ctx.det = model, rg, pg, cfg, ws, addf, det
        ctx.save_for_backward(*params)
        return scores

    @staticmethod
    def backward(ctx, dscores):
        L = _lib.lib()
        params = ctx.saved_tensors
        model = ctx.model
        w = model._param_struct(params)
        # All gradients are written into ONE flat buffer (state_dict layout, parameter order of _named_slots, each tensor 16-byte aligned)
        # and handed to autograd as views of it: p.grad then aliases the buffer, and the data-parallel gradient exchange is a single
        # all-reduce of `model._grad_flat` in place -- no flatten / unflatten copies (parallel.GradSync).  Only the tensors autograd asks
        # for are in it: a frozen one gets a NULL pointer, which rr_model_backward neither computes nor writes.
        needs = ctx.needs_input_grad[4:]
        hot = [p for p, n in zip(params, needs) if n]
        offs, total = flat_layout(hot)
        flat = torch.empty(total, dtype=torch.float32, device=params[0].device)
        if total != sum(p.numel() for p in hot):
            flat.zero_()                                     # alignment gaps take part in the all-reduce
        views = iter([flat[o:o + p.numel()].view(p.shape) for o, p in zip(offs, hot)])
        grads = [next(views) if n else None for n in needs]
        gw = model._param_struct(grads)
        dscores = dscores.contiguous().float()
        _lib.set_deterministic(ctx.det)
        _lib.check(L.rr_model_backward_ex(ctypes.byref(ctx.cfg), ctypes.byref(w), ctypes.byref(ctx.rg.c), ctypes.byref(ctx.pg.c),
                                       dscores.data_ptr(), ctypes.byref(gw), ctx.ws.data_ptr(), ctx.ws.numel(), _lib.stream_ptr()))
        model._ws_pool.give(ctx.ws)
        ctx.ws = None
        model._grad_flat, model._grad_offsets = flat, offs
        return (None, None, None, None) + tuple(grads)


class ReactionModel(nn.Module):
    """r/p encode -> atom-wise difference -> diff encoder -> FFN (base_model.py:111-171)."""

    def __init__(self, mpnn_hidden_size: int = 300, mpnn_bias: bool = True, mpnn_depth: int = 3, mpnn_dropout=0.2,
                 mpnn_diff_hidden_size: int = 300, mpnn_diff_bias: bool = True, mpnn_diff_depth: int = 3, mpnn_diff_dropout=0.2,
                 ffn_hidden_size: int = 300, ffn_bias: bool = True, ffn_dropout=0.2, ffn_depth: int = 3, task_num: int = 2,
                 task_type: str = 'no_softplus', addtion_react_featrues: int = 0):
        super().__init__()
        if task_type in _UNBUILT_HEADS:
            raise NotImplementedError(f"FFN head '{task_type}' is outside the five north-star task keys")
        self.encoder = MPN(bond_fdim=ATOM_FDIM + BOND_FDIM, atom_fdim=ATOM_FDIM, MPN_hidden_size=mpnn_hidden_size, MPN_bias=mpnn_bias,
                           MPN_depth=mpnn_depth, MPN_dropout=mpnn_dropout, return_atom_hiddens=True)
        self.diff_encoder = MPNDiff(atom_fdim=mpnn_hidden_size, bond_fdim=ATOM_FDIM + BOND_FDIM, MPNDiff_hidden_size=mpnn_diff_hidden_size,
                                    MPNDiff_bias=mpnn_diff_bias, MPNDiff_depth=mpnn_diff_depth, MPNDiff_dropout=mpnn_diff_dropout)
        self.ffn = FFN(reacvec_fdim=mpnn_diff_hidden_size + addtion_react_featrues, ffn_hidden_size=ffn_hidden_size,
                       ffn_dropout=ffn_dropout, ffn_num_layers=ffn_depth, task_num=task_num, ffn_bias=ffn_bias, task_type=task_type)
        self._he, self._hd, self._hf = mpnn_hidden_size, mpnn_diff_hidden_size, ffn_hidden_size
        self._pe, self._pd, self._pf = float(mpnn_dropout), float(mpnn_diff_dropout), float(ffn_dropout)
        self._depth, self._diff_depth, self._ffn_depth = mpnn_depth, mpnn_diff_depth, ffn_depth
        self._task_num, self._add = task_num, addtion_react_featrues
        self._head = _HEADS.get(task_type, _lib.HEAD_RAW)     # every other name returns the raw output (base_model.py:105-106)
        self.last_h2d_bytes = 0
        self.dedup_reactants = True      # encode repeated reactants once whenever that is exact (eval mode, dropout 0)
        self._ws_pool = _WorkspacePool()
        self._grad_flat, self._grad_offsets = None, None     # the newest backward's flat gradient buffer (see _ReactionFn.backward)

    # ---- plumbing to the C ABI -----------------------------------------------------------
    def _named_slots(self):
        e, d = self.encoder, self.diff_encoder
        slots = [("enc_Wi", e.W_i.weight), ("enc_bi", e.W_i.bias),
                 ("enc_Wh", getattr(e, "W_h", None) and e.W_h.weight), ("enc_bh", getattr(e, "W_h", None) and e.W_h.bias),
                 ("enc_Wo", e.W_o.weight), ("enc_bo", e.W_o.bias),
                 ("dif_Wi", d.W_i.weight), ("dif_bi", d.W_i.bias),
                 ("dif_Wh", getattr(d, "W_h", None) and d.W_h.weight), ("dif_bh", getattr(d, "W_h", None) and d.W_h.bias),
                 ("dif_Wo", getattr(d, "W_o", None) and d.W_o.weight), ("dif_bo", getattr(d, "W_o", None) and d.W_o.bias)]
        for i, lin in enumerate(self.ffn.linears()):
            slots += [(("ffn_W", i), lin.weight), (("ffn_b", i), lin.bias)]
        return [(k, v) for k, v in slots if v is not None]

    def _param_struct(self, tensors) -> _lib.RRParams:
        """The C struct of one tensor per slot of _named_slots; None leaves the slot NULL."""
        s = _lib.RRParams()
        for (slot, _), t in zip(self._named_slots(), tensors):
            if t is None:
                continue
            if isinstance(slot, tuple):
                getattr(s, slot[0])[slot[1]] = t.data_ptr()
            else:
                setattr(s, slot, t.data_ptr())
        return s

    def any_dropout(self) -> bool:
        return max(self._pe, self._pd, self._pf) > 0

    def _cfg(self, training: bool) -> _lib.RRModelCfgEx:
        seed = 0
        if training and self.any_dropout():
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())        # follows torch.manual_seed
        base = _lib.RRModelCfg(self._he, self._depth, self._diff_depth, self._ffn_depth, self._task_num, self._add,
                               self._head, int(training), self._pe, seed)
        return _lib.RRModelCfgEx(base, self._hd, self._hf, self._pd, self._pf)

    def hot_parameters(self):
        """The trainable parameters in the order of the flat gradient buffer."""
        return [p for _, p in self._named_slots() if p.requires_grad]

    def saved_activation(self, out: torch.Tensor, name: str, rows: int, cols: int) -> torch.Tensor:
        """A forward activation kept in the workspace of the autograd node behind ``out`` (per-layer parity tests):
        see rr_model_buffer_offset for the names."""
        node = out.grad_fn
        off = _lib.lib().rr_model_buffer_offset_ex(ctypes.byref(node.cfg), ctypes.byref(node.rg.c), ctypes.byref(node.pg.c), name.encode())
        if off < 0:
            _lib.check(-1)
        return node.ws[off:off + rows * cols * 4].view(torch.float32).reshape(rows, cols)

    # ---- reference call signature (base_model.py:150-154) ----------------------------------
    def forward(self, r_inputs, p_inputs, gpu, add_features: Optional[List[np.ndarray]] = None):
        dev_idx = _lib.require_device(gpu)
        dev = torch.device("cuda", dev_idx)
        params = [p for _, p in self._named_slots()]
        if params[0].device != dev:
            raise _lib.RRError(f"model parameters live on {params[0].device}, expected {dev}: call model.cuda({dev_idx}) first")
        if (reactant_dedup_exact(self) and isinstance(r_inputs, BatchMolGraph)
                and isinstance(p_inputs, BatchMolGraph) and r_inputs._ids is not None and p_inputs._ids is not None):
            # every candidate of a group repeats the reactant graph (load_reactions.py:574-576): without dropout the copies are identical,
            # so each distinct reactant is encoded once (rr_model_cfg.r_atom_map); with dropout the reference draws a mask per copy
            rg, pg = DeviceGraph.from_batches_dedup([r_inputs], [p_inputs], dev)
        elif isinstance(r_inputs, BatchMolGraph) and isinstance(p_inputs, BatchMolGraph):
            # one blob with adjacent feature arrays: the shared-weight encoder runs once over both batches without copying a feature row
            rg, pg = DeviceGraph.pair_from_batches([r_inputs], [p_inputs], dev)
        else:
            rg = r_inputs if isinstance(r_inputs, DeviceGraph) else r_inputs.to_device(dev)
            pg = p_inputs if isinstance(p_inputs, DeviceGraph) else p_inputs.to_device(dev)
        addf = None
        h2d = rg.h2d_bytes + pg.h2d_bytes
        if self._add > 0:
            if add_features is None:
                raise _lib.RRError(f"model was built with add_features_dim={self._add} but add_features is None")
            if isinstance(add_features, torch.Tensor) and add_features.is_cuda:
                addf = add_features.float().contiguous()
            else:
                host = torch.as_tensor(np.asarray(add_features, dtype=np.float32)).reshape(pg.n_mols, self._add)   # FloatTensor cast, mpn.py:183
                addf = host.pin_memory().to(dev, non_blocking=True)
                h2d += host.numel() * 4
        self.last_h2d_bytes = h2d
        if getattr(rg, "atom_map", None) is not None and torch.is_grad_enabled() and _lib.deterministic_requested():
            raise _lib.RRError("deterministic mode (torch.use_deterministic_algorithms) has no backward pass for de-duplicated reactants: "
                               "build the graphs with one reactant row per candidate (DeviceGraph.from_batches / pair_from_batches), "
                               "or run the forward under torch.no_grad()")
        with torch.cuda.device(dev):
            return _ReactionFn.apply(self, rg, pg, addf, *params)


def build_model(hidden_size: int = 300, mpnn_depth: int = 3, mpnn_diff_depth: int = 3, ffn_depth: int = 3, use_bias: bool = True,
                dropout=0.2, task_num: int = 2, ffn_last_layer: str = 'no_softplus', task_type=None, bimolecule=False,
                add_features_dim=0):
    """Same resolution of the FFN head name as the reference (base_model.py:252-264).  As in the
    reference, ``bimolecule=True`` builds the same model without ``add_features_dim`` (281-295)."""
    if task_type is None:
        if task_num == 2:
            task_type = 'gaussian_' + ffn_last_layer
        elif task_num == 4:
            task_type = 'evidential_' + ffn_last_layer
        else:
            task_type = ffn_last_layer
    elif task_type != 'evidential_ranking':
        task_type = task_type + '_' + ffn_last_layer
    return ReactionModel(mpnn_hidden_size=hidden_size, mpnn_bias=use_bias, mpnn_depth=mpnn_depth, mpnn_dropout=dropout,
                         mpnn_diff_hidden_size=hidden_size, mpnn_diff_bias=use_bias, mpnn_diff_depth=mpnn_diff_depth,
                         mpnn_diff_dropout=dropout, ffn_hidden_size=hidden_size, ffn_bias=use_bias, ffn_dropout=dropout,
                         ffn_depth=ffn_depth, task_num=task_num, task_type=task_type,
                         addtion_react_featrues=0 if bimolecule else add_features_dim)


_FREEZE_MODULES = ("encoder", "diff_encoder")


def parse_freeze(spec: str) -> dict:
    """``freeze()``'s keyword arguments from the command-line form ``encoder[,diff_encoder][,ffn:N]`` (any order); ValueError on anything
    else, so that argparse reports it."""
    kw = dict(encoder=False, diff_encoder=False, ffn_layers=0)
    for tok in (t.strip() for t in spec.split(",")):
        if tok in _FREEZE_MODULES:
            kw[tok] = True
        elif tok.startswith("ffn:") and tok[4:].isdigit() and int(tok[4:]) > 0:
            kw["ffn_layers"] = int(tok[4:])
        else:
            raise ValueError(f"unknown module {tok!r} in --freeze {spec!r}: expected encoder, diff_encoder or ffn:N (N >= 1)")
    return kw


def freeze(model: ReactionModel, encoder: bool = False, diff_encoder: bool = False, ffn_layers: int = 0) -> List[str]:
    """Fine-tuning: ``requires_grad = False`` on the encoder, the diff encoder and / or the first ``ffn_layers`` Linear layers of
    ``ffn.ffn`` (chemprop's frozen MPN / frozen FFN layers).  Their gradients are then neither computed nor written by the backward pass,
    and everything below the lowest trainable layer is skipped (rr_model_backward).  Setting ``requires_grad_(False)`` on single tensors
    by hand works the same way.  Every frozen tensor must have been loaded by ``load_pretrained`` (freezing random weights is always a
    mistake): raises ``ValueError`` otherwise.  Returns the frozen ``state_dict`` names."""
    linears = model.ffn.linears()
    if not 0 <= ffn_layers <= len(linears):
        raise ValueError(f"ffn_layers = {ffn_layers}: the FFN has {len(linears)} Linear layers")
    mods = [m for m, on in (("encoder", encoder), ("diff_encoder", diff_encoder)) if on]
    names = dict(model.named_parameters())
    frozen = [n for n in names if n.split(".")[0] in mods and "cached_zero" not in n]
    ffn_ids = {id(p) for lin in linears[:ffn_layers] for p in lin.parameters()}
    frozen += [n for n, p in names.items() if id(p) in ffn_ids]
    loaded = getattr(model, "pretrained_names", set())
    missing = [n for n in frozen if n not in loaded]
    if missing:
        raise ValueError(f"freeze: {len(missing)} tensors to freeze were not loaded from a pretrained checkpoint (load_pretrained): "
                         f"{missing}")
    for n in frozen:
        names[n].requires_grad_(False)
    return frozen
