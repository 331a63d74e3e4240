"""ctypes binding of ``librr_sm100.so`` (include/rr_sm100.h) and its in-tree build.

There is no CPU fallback: ``lib()`` raises when the shared library is missing or a call
fails, and every compute entry point needs a CUDA device of compute capability 10.x.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import threading
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
CSRC = os.path.join(_HERE, "csrc")
SO_PATH = os.path.join(_HERE, "librr_sm100.so")
SOURCES = ["rr_api.cu", "rr_host.cu", "rr_mp.cu", "rr_mp_pipe.cu", "rr_gemm_simt.cu", "rr_gemm_tc.cu", "rr_linear.cu", "rr_assemble.cu", "rr_loss.cu", "rr_model.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC"]

RR_MAX_FFN = 4
RR_OUT_LD = 16
FA_LD, FB_LD = 64, 88
HEAD_RAW, HEAD_EVIDENTIAL_RANKING, HEAD_GAUSS_SOFTPLUS, HEAD_SOFTPLUS, HEAD_LOGNORM, HEAD_SOFTPLUS_P1, HEAD_NIG = range(7)
LOSS_LISTMLE, LOSS_LISTNET, LOSS_EVIDENTIAL, LOSS_RANKNET, LOSS_GAUSS, LOSS_MSE, LOSS_EXPMSE, LOSS_LISTMLE_DIS, LOSS_LISTNET_DIS, LOSS_LISTNET_UQ, LOSS_RANKNET_ACC, LOSS_LOGNORM, LOSS_DIRICHLET_UQ, LOSS_NIG = range(14)
LOSS_LAMBDARANK, LOSS_LAMBDARANK_TOP = 14, 15

c_f32p = ctypes.c_void_p   # device pointers travel as plain integers


class RRModelCfg(ctypes.Structure):
    _fields_ = [("hidden", ctypes.c_int32), ("depth", ctypes.c_int32), ("diff_depth", ctypes.c_int32),
                ("ffn_depth", ctypes.c_int32), ("task_num", ctypes.c_int32), ("add_features", ctypes.c_int32),
                ("head", ctypes.c_int32), ("training", ctypes.c_int32), ("dropout", ctypes.c_float),
                ("seed", ctypes.c_uint64), ("r_atom_map", ctypes.c_void_p)]


class RRModelCfgEx(ctypes.Structure):
    """rr_model_cfg_ex: ``base`` is anonymous, so ``cfg.seed`` etc. read through, and ``byref(cfg)`` is also a valid ``rr_model_cfg*``."""
    _anonymous_ = ("base",)
    _fields_ = [("base", RRModelCfg), ("diff_hidden", ctypes.c_int32), ("ffn_hidden", ctypes.c_int32),
                ("diff_dropout", ctypes.c_float), ("ffn_dropout", ctypes.c_float)]


class RRMolStore(ctypes.Structure):
    _fields_ = [(k, ctypes.c_void_p) for k in ("f_atoms", "f_bonds", "n_atoms", "n_bonds", "atom_off", "bond_off", "deg", "a2b_start", "a2b_flat", "b2a")]


class RRParams(ctypes.Structure):
    _fields_ = [("enc_Wi", c_f32p), ("enc_bi", c_f32p), ("enc_Wh", c_f32p), ("enc_bh", c_f32p), ("enc_Wo", c_f32p), ("enc_bo", c_f32p),
                ("dif_Wi", c_f32p), ("dif_bi", c_f32p), ("dif_Wh", c_f32p), ("dif_bh", c_f32p), ("dif_Wo", c_f32p), ("dif_bo", c_f32p),
                ("ffn_W", c_f32p * RR_MAX_FFN), ("ffn_b", c_f32p * RR_MAX_FFN)]


EXPORTS = [
    "rr_version", "rr_last_error", "rr_device_check", "rr_padded",
    "rr_graph_assemble", "rr_batch_build", "rr_bond_message_fwd", "rr_bond_message_bwd", "rr_neighbor_sum_fwd", "rr_neighbor_sum_bwd",
    "rr_bond_message_bwd_act", "rr_neighbor_sum_bwd_act", "rr_readout_fwd", "rr_readout_bwd", "rr_linear_fwd", "rr_linear_dgrad", "rr_linear_dgrad_tc", "rr_linear_dgrad_tc_scratch_bytes", "rr_linear_wgrad", "rr_relu_bwd", "rr_sub",
    "rr_loss_fwdbwd", "rr_loss_fwdbwd_ex", "rr_loss_max_group", "rr_rank_metrics", "rr_rank_predict",
    "rr_model_workspace_bytes", "rr_model_buffer_offset", "rr_model_forward", "rr_model_backward", "rr_model_workspace_bytes_ex",
    "rr_model_buffer_offset_ex", "rr_model_forward_ex", "rr_model_backward_ex", "rr_launch_count", "rr_launch_count_reset",
    "rr_profile_begin", "rr_profile_end", "rr_profile_classes", "rr_set_gemm_mode", "rr_get_gemm_mode", "rr_set_backward_bf16", "rr_get_backward_bf16",
    "rr_set_forward_bf16", "rr_get_forward_bf16", "rr_reload_switches", "rr_set_deterministic", "rr_get_deterministic",
]
KERNEL_CLASSES = ["gemm_fwd", "gemm_dgrad", "gemm_wgrad", "bond_fwd", "bond_bwd", "nbr_fwd", "nbr_bwd", "readout", "elementwise", "loss", "misc"]


def source_hash() -> str:
    """sha256 over every CUDA source, header and the compiler flags: what the built library must correspond to."""
    import hashlib
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h"))]
    files.append(os.path.join(_ROOT, "include", "rr_sm100.h"))
    for f in files:
        h.update(os.path.basename(f).encode() + b"\0")
        with open(f, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS + SOURCES).encode())
    return h.hexdigest()


HASH_PATH = SO_PATH + ".hash"


def build(verbose: bool = False, force: bool = False) -> str:
    """Compile the CUDA sources for sm_100a into ``reactranker_b200/librr_sm100.so`` (nvcc cross-compiles without a GPU).
    Skipped only when the library on disk was built from exactly these sources and flags: the hash of the sources is stored next to the
    ``.so`` and compared, so a prebuilt library that travelled with the tree can never silently disagree with the sources beside it."""
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    want = source_hash()
    if not force and os.path.exists(SO_PATH) and os.path.exists(HASH_PATH):
        with open(HASH_PATH) as fh:
            if fh.read().strip() == want:
                return SO_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-I", os.path.join(_ROOT, "include"), "-shared", "-o", SO_PATH] + srcs
    if verbose:
        print(" ".join(cmd))
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    with open(HASH_PATH, "w") as fh:
        fh.write(want + "\n")
    return SO_PATH


_lock = threading.Lock()
_lib: Optional[ctypes.CDLL] = None


class RRError(RuntimeError):
    pass


def lib() -> ctypes.CDLL:
    """The loaded library.  Raises (loudly) if it has not been built: the product path never
    falls back to a CPU implementation."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(SO_PATH):
                    raise RRError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                  "(reactranker_b200 has no CPU fallback)")
                L = ctypes.CDLL(SO_PATH)
                L.rr_last_error.restype = ctypes.c_char_p
                L.rr_model_workspace_bytes.restype = ctypes.c_int64
                L.rr_launch_count.restype = ctypes.c_int64
                L.rr_launch_count_reset.restype = None
                L.rr_reload_switches.restype = None
                i32, i64, u64, f32, vp = ctypes.c_int, ctypes.c_int64, ctypes.c_uint64, ctypes.c_float, ctypes.c_void_p
                L.rr_device_check.argtypes = [i32]
                L.rr_padded.argtypes = [i32]
                L.rr_graph_assemble.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp]
                L.rr_batch_build.argtypes = [i32, vp, i32, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp]
                L.rr_bond_message_fwd.argtypes = [vp, vp, vp, i32, i32, vp]
                L.rr_bond_message_bwd.argtypes = [vp, vp, vp, i32, vp]
                L.rr_neighbor_sum_fwd.argtypes = [vp, i32, vp, vp, i32, i32, vp]
                L.rr_neighbor_sum_bwd.argtypes = [vp, i32, vp, vp, i32, vp]
                L.rr_bond_message_bwd_act.argtypes = [vp, vp, vp, i32, vp, f32, i32, vp, i32, i32, vp]
                L.rr_neighbor_sum_bwd_act.argtypes = [vp, i32, vp, vp, i32, vp, f32, i32, vp, i32, i32, vp]
                L.rr_readout_fwd.argtypes = [vp, vp, i32, i32, vp, i32, vp, i32, f32, u64, u64, vp]
                L.rr_readout_bwd.argtypes = [vp, vp, i32, vp, vp, vp, i32, f32, vp]
                L.rr_linear_fwd.argtypes = [i32, i32, vp, i32, vp, i32, vp, i32, vp, i32, vp, vp, i32, vp, i32, i32, f32, u64, u64, vp]
                L.rr_linear_dgrad.argtypes = [i32, i32, i32, vp, i32, vp, i32, vp, i32, i32, vp]
                L.rr_linear_dgrad_tc.argtypes = [i32, i32, i32, vp, i32, vp, i32, vp, i32, i32, vp, i64, vp]
                L.rr_linear_dgrad_tc_scratch_bytes.argtypes = [i32, i32]
                L.rr_linear_dgrad_tc_scratch_bytes.restype = ctypes.c_int64
                L.rr_linear_wgrad.argtypes = [i32, i32, i32, vp, i32, vp, i32, vp, i32, vp, vp]
                L.rr_relu_bwd.argtypes = [i64, i32, vp, vp, f32, i32, vp, vp, i32, vp]
                L.rr_sub.argtypes = [i64, vp, vp, vp, vp]
                L.rr_loss_fwdbwd.argtypes = [i32, i32, i32, vp, vp, vp, f32, f32, vp, vp, vp]
                L.rr_loss_fwdbwd_ex.argtypes = [i32, i32, i32, vp, vp, vp, i32, f32, f32, vp, vp, vp]
                L.rr_rank_metrics.argtypes = [i32, i32, vp, i32, vp, vp, i32, ctypes.c_double, vp, vp]
                L.rr_rank_predict.argtypes = [i32, i32, i32, vp, i64, i32, vp, i32, vp, vp]
                L.rr_model_workspace_bytes.argtypes = [vp, vp, vp]
                L.rr_model_buffer_offset.argtypes = [vp, vp, vp, ctypes.c_char_p]
                L.rr_model_buffer_offset.restype = ctypes.c_int64
                L.rr_model_forward.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, vp]
                L.rr_model_backward.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, vp]
                L.rr_model_workspace_bytes_ex.argtypes = [vp, vp, vp]
                L.rr_model_workspace_bytes_ex.restype = ctypes.c_int64
                L.rr_model_buffer_offset_ex.argtypes = [vp, vp, vp, ctypes.c_char_p]
                L.rr_model_buffer_offset_ex.restype = ctypes.c_int64
                L.rr_model_forward_ex.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, vp]
                L.rr_model_backward_ex.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, vp]
                L.rr_profile_end.argtypes = [vp, vp, i32]
                L.rr_set_gemm_mode.argtypes = [i32]
                # dense layers: tcgen05 tensor cores (3xTF32 split) unless RR_GEMM_MODE=0 asks for the exact-fp32 SIMT kernels
                L.rr_set_gemm_mode(int(os.environ.get("RR_GEMM_MODE", "1")))
                L.rr_set_backward_bf16.argtypes = [i32]
                L.rr_set_backward_bf16(int(os.environ.get("RR_BWD_BF16", "1")))
                L.rr_set_forward_bf16.argtypes = [i32]
                L.rr_set_forward_bf16(int(os.environ.get("RR_FWD_BF16", "0")))
                L.rr_set_deterministic.argtypes = [i32]
                L.rr_get_deterministic.argtypes = []
                _lib = L
    return _lib


def check(status: int) -> None:
    if status != 0:
        raise RRError(f"librr_sm100 error {status}: {lib().rr_last_error().decode(errors='replace')}")


_checked_devices = set()


def require_device(device) -> int:
    """Resolve ``gpu`` (int / torch.device / str) to a CUDA ordinal that passes rr_device_check."""
    import torch
    if device is None:
        raise RRError("gpu=None: reactranker_b200 runs on a B200 only (no CPU fallback); pass gpu=<cuda ordinal>")
    if not torch.cuda.is_available():
        raise RRError("CUDA is not available: reactranker_b200 has no CPU fallback")
    idx = device if isinstance(device, int) else torch.device(device).index
    if idx is None:
        idx = torch.cuda.current_device()
    if idx not in _checked_devices:
        check(lib().rr_device_check(int(idx)))
        _checked_devices.add(idx)
    return int(idx)


def deterministic_requested() -> bool:
    """torch.use_deterministic_algorithms(True) (also with warn_only=True) asks for bit-identical results."""
    import torch
    return bool(torch.are_deterministic_algorithms_enabled())


def set_deterministic(on: bool) -> None:
    """The library's process-wide deterministic switch (rr_set_deterministic)."""
    check(lib().rr_set_deterministic(1 if on else 0))


def ptr(t) -> Optional[int]:
    return None if t is None else t.data_ptr()


def stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


def profile_begin() -> None:
    check(lib().rr_profile_begin())


def profile_end() -> dict:
    """{class: (milliseconds, launches)} of every kernel launched since profile_begin()."""
    n = lib().rr_profile_classes()
    ms = (ctypes.c_double * n)()
    cnt = (ctypes.c_int64 * n)()
    check(lib().rr_profile_end(ms, cnt, n))
    return {KERNEL_CLASSES[i]: (float(ms[i]), int(cnt[i])) for i in range(n)}
