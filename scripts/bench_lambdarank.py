"""Cost of the LambdaRank loss kernel and of a LambdaRank training step on one GPU.

    python scripts/bench_lambdarank.py [--launches 200] [--replays 20] [--steps 30] [--rounds 6] [--out result.json]

Reports, with the card's name and power limit (nvidia-smi) read in the same run:
  * device time per rr_loss_fwdbwd_ex launch (the loss zeroing memset and the kernel) of ListMLE, RankNet, LambdaRank and LambdaRank@25%
    at 82 x 50, 64 x 64, 8 x 500 and 1 x 8192 candidates: up to `--launches` launches are captured in one CUDA graph, replayed up to
    `--replays` times between CUDA events (fewer for a shape slower than 100 us), so the host's launch rate does not enter the number.
    The inputs (at most 8192 x 2 floats) stay in L2, as they do in a training step, where the loss reads the scores the forward has
    just written;
  * the median training step of c5 (h300 d3, 82 x 50, dropout 0.1) with the `mle` and the `lambdarank` task keys, two models over the
    same resident batches, alternated block by block in one process, and the loss class's device time per step (rr_profile_begin).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [(82, 50), (64, 64), (8, 500), (1, 8192)]


def card():
    res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return res.stdout.strip().splitlines()[0] if res.returncode == 0 and res.stdout.strip() else "unknown"


def kernel_us(kind, groups, n, launches, replays):
    """Microseconds per launch; `launches` and `replays` shrink for a slow shape so that one timed window stays near 0.2 s."""
    from reactranker_b200 import _lib
    L = _lib.lib()
    dev = torch.device("cuda", 0)
    N = groups * n
    g = torch.Generator().manual_seed(kind)
    s, t = torch.randn(N, generator=g).to(dev), torch.randn(N, generator=g).to(dev)
    seg = torch.arange(0, N + 1, n, dtype=torch.int32, device=dev)
    loss, ds = torch.empty(1, device=dev), torch.empty(N, device=dev)

    def one():
        _lib.check(L.rr_loss_fwdbwd_ex(kind, N, groups, s.data_ptr(), t.data_ptr(), seg.data_ptr(), n, float(groups), 1.0, loss.data_ptr(),
                                       ds.data_ptr(), torch.cuda.current_stream().cuda_stream))
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        one()                                                   # sets the kernel's shared-memory attribute outside the capture
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(3):
        one()
    b.record()
    b.synchronize()
    est_s = a.elapsed_time(b) / 3e3
    launches = max(3, min(launches, int(0.02 / est_s)))
    replays = max(3, min(replays, int(0.2 / (launches * est_s))))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(launches):
            one()
    graph.replay()
    torch.cuda.synchronize()
    a.record()
    for _ in range(replays):
        graph.replay()
    b.record()
    b.synchronize()
    assert bool(torch.isfinite(loss).all())
    return a.elapsed_time(b) * 1e3 / (launches * replays)


def timed_block(job, steps, start):
    torch.cuda.synchronize()
    t = time.perf_counter()
    for i in range(steps):
        job.step_resident(start + i)
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3 / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200, help="loss launches per CUDA graph")
    ap.add_argument("--replays", type=int, default=20, help="graph replays per timed kernel")
    ap.add_argument("--steps", type=int, default=30, help="training steps per timed block")
    ap.add_argument("--rounds", type=int, default=6, help="alternations of the two task keys")
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    a = ap.parse_args()
    import bench
    from reactranker_b200 import _lib
    kinds = {"listmle": _lib.LOSS_LISTMLE, "ranknet": _lib.LOSS_RANKNET, "lambdarank": _lib.LOSS_LAMBDARANK,
             "lambdarank_top": _lib.LOSS_LAMBDARANK_TOP}
    kern = {}
    for gr, n in SHAPES:
        kern[f"{gr}x{n}"] = {name: round(kernel_us(k, gr, n, a.launches, a.replays), 2) for name, k in kinds.items()}
        print(f"{gr}x{n}", kern[f"{gr}x{n}"], flush=True)

    bench.WORKLOADS["c5-lambdarank"] = dict(bench.WORKLOADS["c5"], task="lambdarank",
                                            desc=bench.WORKLOADS["c5"]["desc"].replace("ListMLE", "LambdaRank"))
    jobs = {"mle": bench.Job("c5", 0), "lambdarank": bench.Job("c5-lambdarank", 0)}
    for job in jobs.values():                                  # warm-up
        timed_block(job, 3, 0)
    ms = {k: [] for k in jobs}
    for r in range(a.rounds):
        for k, job in jobs.items():
            ms[k].append(timed_block(job, a.steps, r * a.steps))
    loss_ms = {}
    for k, job in jobs.items():
        torch.cuda.synchronize()
        _lib.profile_begin()
        for i in range(a.steps):
            job.step_resident(i)
        torch.cuda.synchronize()
        loss_ms[k] = round(_lib.profile_end()["loss"][0] / a.steps, 4)
    out = {"card": card(), "kernel_us_per_launch": kern, "launches_per_graph": a.launches, "replays": a.replays,
           "step_workload": bench.WORKLOADS["c5"]["desc"], "steps_per_block": a.steps, "rounds": a.rounds,
           "step_ms_median": {k: round(statistics.median(v), 3) for k, v in ms.items()},
           "step_ms_blocks": {k: [round(x, 3) for x in v] for k, v in ms.items()},
           "loss_class_ms_per_step": loss_ms}
    print(json.dumps(out))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
