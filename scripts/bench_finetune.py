"""Cost of a fine-tuning step with frozen sub-modules on the default workload (c5: ListMLE h300 d3, 82 groups x 50 candidates, dropout
0.1) on one GPU.

    python scripts/bench_finetune.py [--steps 30] [--rounds 4] [--out result.json]

Alternates four freeze levels in one process over the same resident batches -- nothing frozen, the encoder, the encoder and the diff
encoder, and everything but the last FFN layer -- and reports for each:
  * the median step time (CUDA-synchronised wall clock per block of steps),
  * per-kernel-class device time and launch counts of one profiled block (rr_profile_begin / rr_profile_end),
  * the trainable element count (what a data-parallel step all-reduces),
and the card's name and power limit (nvidia-smi), read in the same run.  The weights keep training between blocks; a frozen tensor's
value does not change the work of a step.
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

LEVELS = {
    "none": lambda n: False,
    "encoder": lambda n: n.startswith("encoder."),
    "encoder+diff_encoder": lambda n: n.startswith(("encoder.", "diff_encoder.")),
    "all_but_last_ffn": lambda n: not n.startswith("ffn.ffn.7."),
}


def card():
    res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return res.stdout.strip().splitlines()[0] if res.returncode == 0 and res.stdout.strip() else "unknown"


def set_level(model, level):
    for n, p in model.named_parameters():
        if "cached_zero" not in n:
            p.requires_grad_(not LEVELS[level](n))


def timed_block(job, steps, start):
    torch.cuda.synchronize()
    t = time.perf_counter()
    for i in range(steps):
        job.step_resident(start + i)
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3 / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30, help="steps per timed block")
    ap.add_argument("--rounds", type=int, default=4, help="alternations of the four levels")
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    a = ap.parse_args()
    import bench
    from reactranker_b200 import _lib
    job = bench.Job("c5", 0)
    for level in LEVELS:                                       # warm-up: every level's launch sequence
        set_level(job.model, level)
        timed_block(job, 3, 0)
    ms = {k: [] for k in LEVELS}
    for r in range(a.rounds):
        for level in LEVELS:
            set_level(job.model, level)
            ms[level].append(timed_block(job, a.steps, r * a.steps))
    profile, launches, trainable = {}, {}, {}
    for level in LEVELS:
        set_level(job.model, level)
        trainable[level] = sum(p.numel() for p in job.model.hot_parameters())
        torch.cuda.synchronize()
        _lib.profile_begin()
        for i in range(a.steps):
            job.step_resident(i)
        torch.cuda.synchronize()
        prof = _lib.profile_end()
        profile[level] = {k: round(v[0] / a.steps, 4) for k, v in prof.items()}
        launches[level] = {k: v[1] // a.steps for k, v in prof.items()}
    set_level(job.model, "none")
    med = {k: statistics.median(v) for k, v in ms.items()}
    out = {"workload": bench.WORKLOADS["c5"]["desc"], "card": card(), "steps_per_block": a.steps, "rounds": a.rounds,
           "step_ms_median": {k: round(v, 3) for k, v in med.items()}, "step_ms_blocks": {k: [round(x, 3) for x in v] for k, v in ms.items()},
           "kernel_ms_per_step_by_class": profile, "launches_per_step_by_class": launches, "trainable_elements": trainable}
    print(json.dumps(out))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
