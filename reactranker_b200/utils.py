"""``save_checkpoint`` and ``index_select_ND`` with the reference's signatures (utils.py:152-193)."""
import ctypes

import torch

from . import _lib


def save_checkpoint(path, model, means=None, stds=None):
    """Same dict layout as the reference (utils.py:152-173): ``{'state_dict', 'data_scaler': {'means','stds'}}``.
    ``means``/``stds`` are stored as python floats so that ``torch.load(weights_only=True)`` (the default since
    torch 2.6) can read the file; numerically identical to the reference's numpy scalars."""
    scaler = {'means': float(means), 'stds': float(stds)} if means is not None and stds is not None else None
    torch.save({'state_dict': model.state_dict(), 'data_scaler': scaler}, path)


def save_train_state(path, model, optimizer, scheduler, epoch, means=None, stds=None, best=None):
    """A checkpoint one can RESUME from (SURVEY.md §8f row 3; the reference saves weights only and restarts from scratch).
    A superset of ``save_checkpoint``'s dict, so the reference's loaders (test_listwise.py:27-38) read it unchanged; the extra keys carry
    Adam's moments and step, the NoamLR position, the last finished epoch, the best validation scores so far and torch's host RNG state
    (dropout seeds are drawn from it).  Batches are planned from ``seed=epoch`` (train_listwise.py:179-182), so a resumed run sees the
    same batches as an uninterrupted one.  Written to a temporary name and renamed: a crash mid-write cannot destroy the last state."""
    import os
    scaler = {'means': float(means), 'stds': float(stds)} if means is not None and stds is not None else None
    # plain Python numbers only (no numpy scalars), so that the file loads with torch.load's safe default weights_only=True
    if isinstance(best, (list, tuple)):
        best = [float(b) for b in best]
    elif best is not None:
        best = float(best)
    state = {'state_dict': model.state_dict(), 'data_scaler': scaler, 'optimizer': optimizer.state_dict(),
             'scheduler': {k: _plain(v) for k, v in scheduler.state_dict().items() if not k.startswith('_')} if scheduler is not None else None,
             'epoch': int(epoch), 'best': best, 'rng_state': torch.get_rng_state()}
    tmp = str(path) + '.tmp'
    torch.save(state, tmp)
    os.replace(tmp, path)


def load_train_state(path, model, optimizer, scheduler=None):
    """Inverse of ``save_train_state``: restores model / optimizer / scheduler in place and returns ``(next_epoch, best, data_scaler)``."""
    state = load_checkpoint(path)
    if 'optimizer' not in state:
        raise _lib.RRError(f"{path} is a weights-only checkpoint (save_checkpoint); resuming needs one written by save_train_state")
    model.load_state_dict(state['state_dict'])
    optimizer.load_state_dict(state['optimizer'])
    if scheduler is not None and state.get('scheduler') is not None:
        for k, v in state['scheduler'].items():
            setattr(scheduler, k, v)
        optimizer.param_groups[0]['lr'] = scheduler.lr
    torch.set_rng_state(state['rng_state'])
    return state['epoch'] + 1, state.get('best'), state['data_scaler']


def _plain(v):
    """numpy scalars / arrays -> Python numbers / lists (what torch.load(weights_only=True) accepts)."""
    import numpy as np
    if isinstance(v, np.generic):
        return v.item()
    if isinstance(v, np.ndarray):
        return v.tolist()
    if isinstance(v, (list, tuple)):
        return [_plain(x) for x in v]
    return v


def load_checkpoint(path, allow_unsafe_pickle=None):
    """Reads checkpoints written by this package or by the reference.

    Always ``torch.load(weights_only=True)``: tensors, Python containers and numbers, plus an allow-list of exactly what the reference's
    own files add -- numpy scalars for ``data_scaler['means' / 'stds']`` (utils.py:165-173 stores ``np.float64``).  Anything else in the
    pickle stream is refused; a corrupt or hostile file can therefore not execute code.  Full unpickling is an explicit opt-in
    (``allow_unsafe_pickle=True`` or ``RR_UNSAFE_CHECKPOINTS=1``) for files from a source you trust."""
    import os
    import pickle
    import numpy as np
    if allow_unsafe_pickle is None:
        allow_unsafe_pickle = os.environ.get("RR_UNSAFE_CHECKPOINTS", "0") == "1"
    loc = lambda storage, _loc: storage  # noqa: E731
    safe = [np.dtype, np.float64, np.float32, np.int64, np.int32, np.bool_, np.ndarray]
    try:
        from numpy._core.multiarray import scalar as _np_scalar, _reconstruct as _np_reconstruct
    except Exception:  # numpy < 2
        from numpy.core.multiarray import scalar as _np_scalar, _reconstruct as _np_reconstruct
    safe += [_np_scalar, _np_reconstruct]
    for name in ("Float64DType", "Float32DType", "Int64DType", "Int32DType", "BoolDType"):
        t = getattr(getattr(np, "dtypes", None), name, None)
        if t is not None:
            safe.append(t)
    try:
        with torch.serialization.safe_globals(safe):
            return torch.load(path, map_location=loc, weights_only=True)
    except pickle.UnpicklingError:
        if not allow_unsafe_pickle:
            raise
        return torch.load(path, map_location=loc, weights_only=False)


def load_pretrained(model, path):
    """Start fine-tuning from a pretrained checkpoint: copies every ``state_dict`` tensor of ``path`` whose name and shape match the
    model's (read through ``load_checkpoint``, same ``weights_only`` policy) and records the copied names in ``model.pretrained_names``,
    which ``freeze`` checks.  A different ``task_num`` or ``add_features_dim`` changes the shape of the last or the first FFN layer only,
    so e.g. a model pretrained with 'mle' fine-tunes as 'evidential_ranking' with those layers left as initialised.  Returns the
    ``(name, reason)`` pairs that were not copied."""
    state = load_checkpoint(path)
    src = state["state_dict"] if isinstance(state, dict) and "state_dict" in state else state
    own = model.state_dict()
    skipped, loaded = [], set()
    with torch.no_grad():
        for name, t in own.items():
            if name not in src:
                skipped.append((name, "not in the checkpoint"))
            elif tuple(src[name].shape) != tuple(t.shape):
                skipped.append((name, f"shape {tuple(src[name].shape)} in the checkpoint, {tuple(t.shape)} in the model"))
            else:
                t.copy_(src[name])
                loaded.add(name)
    skipped += [(name, "not in the model") for name in src if name not in own]
    model.pretrained_names = getattr(model, "pretrained_names", set()) | loaded
    return skipped


def index_select_ND(source: torch.Tensor, index: torch.Tensor) -> torch.Tensor:
    """``source[index]`` with the reference's shape contract (utils.py:176-193): [R, h], [A, W] -> [A, W, h].
    The hot path never materialises this tensor (the gather kernels sum on the fly); kept for API parity."""
    if not source.is_cuda:
        raise _lib.RRError("index_select_ND: reactranker_b200 tensors live on the GPU (no CPU fallback)")
    return source.index_select(0, index.reshape(-1).to(source.device)).view(index.shape + source.shape[1:])
