"""GPU micro-benchmark of the message-passing gather kernels at the c5 batch shape: first generation (register gathers, RR_MP_V1=1)
against the TMA-bulk row pipeline, plain and fused with the ReLU backward."""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from reactranker_b200 import _lib, synthetic
from reactranker_b200.features.featurization import BatchMolGraph

L = _lib.lib()
dev = torch.device("cuda:0")
ds = synthetic.make_dataset(1000, [50] * 82)
b = BatchMolGraph([ds.mols[t] for t in ds.psmi])
dg = b.to_device(dev)
A, B, hp = b.n_atoms, b.n_bonds, 304
S = _lib.stream_ptr
g = ctypes.byref(dg.c)
mB, oB, yB, accB = (torch.randn(B, hp, device=dev) for _ in range(4))
mA, oA, yA, accA = (torch.randn(A, hp, device=dev) for _ in range(4))
nf = torch.empty(A, 88, device=dev)
row = hp * 4
idx = (A * dg.c.wmax + 2 * B) * 4


def timeit(fn, iters=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return a.elapsed_time(e) / iters * 1e3


cases = [
    ("bond_fwd", lambda: L.rr_bond_message_fwd(g, mB.data_ptr(), oB.data_ptr(), hp, 1, S()), 2 * B * row + idx),
    ("bond_bwd", lambda: L.rr_bond_message_bwd(g, mB.data_ptr(), oB.data_ptr(), hp, S()), 2 * B * row + idx),
    ("bond_bwd+relu_bwd(acc+=)", lambda: L.rr_bond_message_bwd_act(g, mB.data_ptr(), oB.data_ptr(), hp, yB.data_ptr(), 1.1, 0, accB.data_ptr(), 2, 0, S()),
     5 * B * row + idx),
    ("bond_bwd+relu_bwd(acc only)", lambda: L.rr_bond_message_bwd_act(g, mB.data_ptr(), oB.data_ptr(), hp, yB.data_ptr(), 1.0, 1, accB.data_ptr(), 2, 1, S()),
     4 * B * row + idx),
    ("nbr_fwd a2b", lambda: L.rr_neighbor_sum_fwd(g, 0, mB.data_ptr(), oA.data_ptr(), hp, 0, S()), (A + B) * row + idx),
    ("nbr_fwd a2a", lambda: L.rr_neighbor_sum_fwd(g, 1, mA.data_ptr(), oA.data_ptr(), hp, 0, S()), 2 * A * row + idx),
    ("nbr_fwd f_bonds", lambda: L.rr_neighbor_sum_fwd(g, 0, dg.c.f_bonds, nf.data_ptr(), 88, 0, S()), (A + B) * 88 * 4 + idx),
    ("nbr_bwd bond", lambda: L.rr_neighbor_sum_bwd(g, 0, mA.data_ptr(), oB.data_ptr(), hp, S()), (A + B) * row + idx),
    ("nbr_bwd bond+relu_bwd(acc=)", lambda: L.rr_neighbor_sum_bwd_act(g, 0, mA.data_ptr(), oB.data_ptr(), hp, yB.data_ptr(), 1.1, 0, accB.data_ptr(), 1, 0, S()),
     (A + 3 * B) * row + idx),
    ("nbr_bwd atom", lambda: L.rr_neighbor_sum_bwd(g, 1, mA.data_ptr(), oA.data_ptr(), hp, S()), 2 * A * row + idx),
    ("nbr_bwd atom+relu_bwd(acc+=)", lambda: L.rr_neighbor_sum_bwd_act(g, 1, mA.data_ptr(), oA.data_ptr(), hp, yA.data_ptr(), 1.1, 0, accA.data_ptr(), 2, 0, S()),
     5 * A * row + idx),
    ("relu_bwd [B] alone (dz, acc+=)", lambda: L.rr_relu_bwd(B, hp, mB.data_ptr(), yB.data_ptr(), 1.1, 0, oB.data_ptr(), accB.data_ptr(), 2, S()), 5 * B * row),
]
for v1 in ("1", "0"):
    os.environ["RR_MP_V1"] = v1
    L.rr_reload_switches()
    for name, fn, by in cases:
        us = timeit(lambda: _lib.check(fn()))
        print(f"{'gen1' if v1 == '1' else 'pipe'} {name:32s} {us:8.1f} us  {by / us * 1e-3:7.0f} GB/s", flush=True)
