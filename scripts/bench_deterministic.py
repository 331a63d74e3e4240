"""Cost of deterministic mode on the default workload (c5: ListMLE h300 d3, 82 groups x 50 candidates, dropout 0.1) on one GPU.

    python scripts/bench_deterministic.py [--steps 30] [--rounds 4] [--out result.json]

Alternates default and deterministic mode (torch.use_deterministic_algorithms) in one process over the same resident batches and reports:
  * the median step time of each mode (CUDA-synchronised wall clock per block of steps),
  * per-kernel-class device time of one profiled block per mode (rr_profile_begin / rr_profile_end),
  * how many entries of the flat gradient differ between two default-mode runs of the same step from the same weights and seed (the
    float-atomic races this mode removes), and the same count for two deterministic runs (0),
  * the card's name and power limit (nvidia-smi), read in the same run.
"""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return res.stdout.strip().splitlines()[0] if res.returncode == 0 and res.stdout.strip() else "unknown"


def timed_block(job, steps, start):
    torch.cuda.synchronize()
    t = time.perf_counter()
    for i in range(steps):
        job.step_resident(start + i)
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3 / steps


def grad_of_one_step(job, state, seed):
    """The flat gradient of resident batch 0 from the saved weights / optimiser state and torch seed."""
    job.model.load_state_dict(state["model"])
    job.opt.load_state_dict(state["opt"])
    torch.manual_seed(seed)
    job.step_resident(0)
    torch.cuda.synchronize()
    return job.model._grad_flat.clone()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30, help="steps per timed block")
    ap.add_argument("--rounds", type=int, default=4, help="alternations default / deterministic")
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    a = ap.parse_args()
    import bench
    from reactranker_b200 import _lib
    job = bench.Job("c5", 0)
    for det in (False, True, False, True):                   # warm-up: every shape and both kernel variants
        torch.use_deterministic_algorithms(det)
        timed_block(job, 3, 0)
    ms = {"default": [], "deterministic": []}
    for r in range(a.rounds):
        for det in (False, True):
            torch.use_deterministic_algorithms(det)
            ms["deterministic" if det else "default"].append(timed_block(job, a.steps, r * a.steps))
    profile = {}
    for det in (False, True):
        torch.use_deterministic_algorithms(det)
        torch.cuda.synchronize()
        _lib.profile_begin()
        for i in range(a.steps):
            job.step_resident(i)
        torch.cuda.synchronize()
        profile["deterministic" if det else "default"] = {k: round(v[0] / a.steps, 4) for k, v in _lib.profile_end().items()}
    state = {"model": copy.deepcopy(job.model.state_dict()), "opt": copy.deepcopy(job.opt.state_dict())}
    races = {}
    for det in (False, True):
        torch.use_deterministic_algorithms(det)
        g1, g2 = grad_of_one_step(job, state, 7), grad_of_one_step(job, state, 7)
        races["deterministic" if det else "default"] = int((g1 != g2).sum())
    torch.use_deterministic_algorithms(False)
    med = {k: statistics.median(v) for k, v in ms.items()}
    out = {"workload": bench.WORKLOADS["c5"]["desc"], "card": card(), "steps_per_block": a.steps, "rounds": a.rounds,
           "step_ms_median": {k: round(v, 3) for k, v in med.items()}, "step_ms_blocks": {k: [round(x, 3) for x in v] for k, v in ms.items()},
           "deterministic_cost_ms": round(med["deterministic"] - med["default"], 3),
           "kernel_ms_per_step_by_class": profile, "gradient_entries": int(g1.numel()), "gradient_entries_differing_between_two_runs": races}
    print(json.dumps(out))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
