"""GPU micro-benchmark of the dense-layer kernels through the C ABI at the model's shapes (c5 batch: 160 889 bond rows, 82 001 atom rows):
the forward GEMM with its epilogues, the tensor-core dgrad (rr_linear_dgrad_tc), and the weight gradient in both backward operand splits
(rr_set_backward_bf16 1 / 0).

rr_linear_fwd is handed fp32 weights and splits them inside the kernel, while the model's own launches take weight images split once per
step; the per-launch times of the model's GEMMs are in bench.py's roofline."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from reactranker_b200 import _lib

L = _lib.lib()
dev = torch.device("cuda:0")
torch.manual_seed(0)
st = _lib.stream_ptr


def timeit(fn, iters=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e3  # us


def fwd_case(M, n, k1, k2=0, epi=True, p=0.1):
    X1 = torch.relu(torch.randn(M, k1, device=dev))
    W1 = torch.randn(n, k1, device=dev) * 0.05
    X2 = torch.randn(M, k2, device=dev) if k2 else None
    W2 = torch.randn(n, k2, device=dev) * 0.05 if k2 else None
    bias = torch.randn(n, device=dev) if epi else None
    R = torch.randn(M, n, device=dev) if epi else None
    Y = torch.empty(M, n, device=dev)
    flags = (1 | (2 if p > 0 else 0)) if epi else 0

    def run():
        _lib.check(L.rr_linear_fwd(M, n, X1.data_ptr(), k1, W1.data_ptr(), k1, _lib.ptr(X2), k2, _lib.ptr(W2), k2, _lib.ptr(bias), _lib.ptr(R), n,
                                   Y.data_ptr(), n, flags, p, 1234, 7, st()))
    return run, 2.0 * M * n * (k1 + k2), (M * (k1 + k2) + M * n * (2 if epi else 1)) * 4.0, (X1, W1, X2, W2, bias, R, Y)


def dgrad_case(M, n, k, accumulate):
    dZ = torch.randn(M, n, device=dev)
    W = torch.randn(n, k, device=dev) * 0.05
    dX = torch.zeros(M, k, device=dev)
    scratch = torch.empty(int(L.rr_linear_dgrad_tc_scratch_bytes(n, k)), dtype=torch.uint8, device=dev)

    def run():
        _lib.check(L.rr_linear_dgrad_tc(M, n, k, dZ.data_ptr(), n, W.data_ptr(), k, dX.data_ptr(), k, accumulate, scratch.data_ptr(), scratch.numel(), st()))
    return run, 2.0 * M * n * k, (M * n + M * k * (2 if accumulate else 1)) * 4.0, (dZ, W, dX, scratch)


def wgrad_case(M, n, k):
    dZ = torch.randn(M, n, device=dev)
    X = torch.randn(M, k, device=dev)
    dW = torch.zeros(n, k, device=dev)
    db = torch.zeros(n, device=dev)

    def run():
        _lib.check(L.rr_linear_wgrad(M, n, k, dZ.data_ptr(), n, X.data_ptr(), k, dW.data_ptr(), k, db.data_ptr(), st()))
    return run, 2.0 * M * n * k, (M * (n + k)) * 4.0, (dZ, X, dW, db)


def report(name, case):
    run, flops, bytes_, _ = case
    us = timeit(run)
    print(f"{name:58s} {us:8.1f} us  {flops / us * 1e-6:7.1f} TFLOP/s  {bytes_ / us * 1e-3:7.0f} GB/s (algorithmic)", flush=True)


B, A = 160889, 82001
report("W_h fwd  [B,304]x[304,304] bias+resid+relu+dropout", fwd_case(B, 304, 304))
report("W_h fwd  same, no dropout", fwd_case(B, 304, 304, p=0.0))
report("W_i fwd  [B,88]x[88,304] plain", fwd_case(B, 304, 88, epi=False))
report("W_o fwd  [A,64|304]x[.,304] two-source + relu", fwd_case(A, 304, 64, 304))
report("plain [B,304]x[304,304]", fwd_case(B, 304, 304, epi=False))
report("h600 resid [A,608]x[608,608]", fwd_case(A, 608, 608))
report("dgrad 3xbf16 accumulate [2B,304]x[304,304]", dgrad_case(2 * B, 304, 304, 1))
report("dgrad 3xbf16 plain [2B,304]x[304,304]", dgrad_case(2 * B, 304, 304, 0))
wcases = [("[B,304]^T[B,304]", (B, 304, 304)), ("[B,304]^T[B,88]", (B, 304, 88)), ("[A,304]^T[A,304]", (A, 304, 304)),
          ("h600 [A,608]^T[A,608]", (A, 608, 608))]
for bf16 in (1, 0):
    _lib.check(L.rr_set_backward_bf16(bf16))
    for name, shape in wcases:
        report(f"wgrad {'3xbf16' if bf16 else '3xtf32'} {name}", wgrad_case(*shape))
