#!/usr/bin/env python3
"""FM training-step cost of batch normalisation of the interaction vector (FM.py:111-112, batch_norm=1) at the fm_c1 shape
of scripts/bench_models.py: frappe-10 (F = 10), K = 64, B = 2^20, dense-L2 Adagrad, four device-resident batches.

    python scripts/bench_fm_bn.py [--runs 3] [--steps 20] [--profile-steps 5] [--json out.json]

Two models of the same shape and seed, batch_norm = 0 and 1, are timed in alternation in one process (run r times `steps`
whole steps of each in turn, so clock and neighbour drift hit both alike).  Reported: ms per step of every run, the
median and the ratio.  A separate torch.profiler run (its own steps, after the timed ones) gives the per-kernel device
times of one step of each model.  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

from bench_afm_dropout import gpu_info  # noqa: E402
from bench_models import frappe_rows, timed  # noqa: E402


def kernel_times(model, batches, steps):
    """Mean device time per step of every kernel over `steps` profiled steps (us)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(steps):
            model.fit_device(*batches[i % len(batches)])
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t > 0:
            out[ev.key] = round(t / steps, 2)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--profile-steps", type=int, default=5)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    from hhfm_b200.models import FM
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(1)
    B = 1 << 20
    batches = []
    for _ in range(4):
        X, M, n_user, n_item = frappe_rows(rng, B)
        batches.append((torch.from_numpy(X).to(dev), torch.from_numpy(rng.choice([1.0, 0.0], B).astype(np.float32)).to(dev)))
    models = {bn: FM(10, M, n_user, n_item, 64, 0.1, 0.1, 1, "AdagradOptimizer", bn, 0) for bn in (0, 1)}
    for m in models.values():                               # warm both (module load, hot-row plan, workspace)
        timed(lambda i: m.fit_device(*batches[i % 4]), 3, 2)
    times = {0: [], 1: []}
    for _ in range(args.runs):
        for bn, m in models.items():
            times[bn].append(timed(lambda i: m.fit_device(*batches[i % 4]), args.steps, 1))
    med = {bn: float(np.median(t)) for bn, t in times.items()}
    res = {"gpu": gpu_info(), "shape": "frappe-10 (F=10, M=%d), K=64, B=2^20, dense-L2 Adagrad" % M,
           "runs": args.runs, "steps_per_run": args.steps,
           "batch_norm0": {"ms_per_step_runs": times[0], "median": med[0]},
           "batch_norm1": {"ms_per_step_runs": times[1], "median": med[1]},
           "ratio": med[1] / med[0],
           "kernels_us_per_step": {("batch_norm%d" % bn): kernel_times(m, batches, args.profile_steps) for bn, m in models.items()}}
    line = json.dumps(res)
    print(line, flush=True)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
