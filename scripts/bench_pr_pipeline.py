#!/usr/bin/env python
"""HHFM training pass at the `bench.py` headline shape: per-launch timings of the grouped entry point and of the whole step.

    python scripts/bench_pr_pipeline.py [--reps 60] [--rounds 5]

B = 2^20 positives, K = 64, NG = 10, the eight frappe context columns pooled into two groups, hot-row plan from the first
batch, four device-resident batches cycled (320 MB of records > 126 MB of L2).  Each round times `--reps` launches of
`hhfm_pairrank_fwd_bwd` (pre-sum, `pairrank_sum_train_kernel<16,8,10,2>`, expansion, memset of the group gradients) and
`--reps` whole steps (the entry point plus the fold / Adagrad / loss kernel), each launch between two CUDA events; the two
arms alternate round by round.  A separate `torch.profiler` capture gives the per-kernel times of the step.  One JSON line
on stdout: median and p10-p90 per arm, the card's name and power limit read in the same call.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import bench  # noqa: E402
from bench_pool_groups import B, N_BATCHES, gpu_info, make_records, stats, time_launches  # noqa: E402


def setup():
    """Model, hot-row plan and batches of the headline step; returns (entry(i), step(i)) launchers."""
    import torch
    from hhfm_b200 import _lib
    from hhfm_b200.engine import NO_HOT, cur_stream, ptr
    from hhfm_b200.models import OUR
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(1234)
    n_ctx, K, NG = len(bench.CTX_CARD), bench.K_FACTOR, bench.NG
    batches = []
    for _ in range(N_BATCHES):
        rec, stride, M = make_records(rng, bench.CTX_CARD, dev)
        batches.append(rec)
    m = OUR(n_ctx, 0, M, bench.N_USER, bench.N_ITEM, K, bench.LR, bench.LAMDA, "AdagradOptimizer", True, False)
    hot = m._hot_plan(batches[0], False)
    hargs = hot.args() if hot is not None else NO_HOT
    assert m._pool_groups is not None, "the headline shape must run the grouped kernel"

    def entry(i):
        _lib.call("hhfm_pairrank_fwd_bwd", ptr(batches[i % N_BATCHES]), B, stride, n_ctx, 0, NG, 0, 0, 0,
                  ptr(m.weights["feature_embeddings"]), M, K, None, None, ptr(m._gV), ptr(m._loss_partials), None, 0, None,
                  None, *hargs, 0, cur_stream())

    def step(i):
        m._opt.begin_step()
        entry(i)
        m._finish_step(hot, False)

    return entry, step


def profile_launches(fn, n=20):
    """Average device time (us) per launch of every kernel / memset in n calls of fn, from a torch.profiler capture."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    for i in range(3):
        fn(i)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(n):
            fn(i)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type is not None and "cuda" in str(e.device_type).lower() and e.count:
            t = getattr(e, "device_time", None) or getattr(e, "cuda_time", 0.0)
            out[e.key[:90]] = {"count": e.count, "avg_us": float(t)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=60)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if args.reps < 50 or args.rounds < 3:
        ap.error("--reps must be at least 50, --rounds at least 3")
    entry, step = setup()
    ts = {"entry": [], "step": []}
    for _ in range(args.rounds):
        for name, fn in (("entry", entry), ("step", step)):
            ts[name] += time_launches(fn, args.reps)
    out = {"gpu": gpu_info(), "B": B, "K": bench.K_FACTOR, "NG": bench.NG, "reps": args.reps, "rounds": args.rounds,
           "entry": stats(ts["entry"]), "step": stats(ts["step"]), "launches_step": profile_launches(step)}
    out["samples_per_s_step"] = B / (out["step"]["median_ms"] * 1e-3)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
