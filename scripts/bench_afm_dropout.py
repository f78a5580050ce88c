#!/usr/bin/env python3
"""AFM training-step cost of dropout (AFM.py:126,134) and of attention=0 (AFM.py:132) at the afm_c3 shape of
scripts/bench_models.py: frappe-10 (P = 45 pairs), K = A = 64, B = 2^17, two device-resident batches.

    python scripts/bench_afm_dropout.py [--rounds 7] [--steps 20] [--json out.json]

Four models of the same shape and seed, one per configuration, are timed in alternation in one process (round r times
`steps` whole steps of each configuration in turn, so clock and neighbour drift hit every arm alike):
keep [1,1] (the fused tcgen05 kernel as before), [1,0.5], [0.5,0.5] (its DROP instantiation), and attention=0 with
keep [1,0.5].  Reported per configuration: the median ms per step over the rounds, the spread (min, max), and the ratio
to keep [1,1]; the card name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

from bench_models import frappe_rows, timed  # noqa: E402

CONFIGS = [("keep[1,1]", 1, [1, 1]), ("keep[1,0.5]", 1, [1, 0.5]), ("keep[0.5,0.5]", 1, [0.5, 0.5]),
           ("attention0 keep[1,0.5]", 0, [1, 0.5])]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out.splitlines()[0] if out else None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    from hhfm_b200.models import AFM
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(3)
    B, K = 1 << 17, 64
    batches = []
    for _ in range(2):
        X, M, n_user, n_item = frappe_rows(rng, B)
        batches.append((torch.from_numpy(X).to(dev), torch.from_numpy(rng.choice([1.0, -1.0], B).astype(np.float32)).to(dev)))
    models = [AFM(n_user, n_item, M, att, [K, K], "relu", 0.1, 100.0, keep, "AdagradOptimizer", 0.999, 10) for _, att, keep in CONFIGS]
    times = [[] for _ in CONFIGS]
    for m in models:                                        # warm every configuration (module load, first launches)
        timed(lambda i: m.fit_device(*batches[i % 2]), 2, 2)
    for r in range(args.rounds):
        for c, m in enumerate(models):
            times[c].append(timed(lambda i: m.fit_device(*batches[i % 2]), args.steps, 1))
    base = float(np.median(times[0]))
    res = {"gpu": gpu_info(), "shape": "frappe-10 (P=45), K=A=64, B=2^17, 2 device-resident batches",
           "rounds": args.rounds, "steps_per_round": args.steps, "configs": {}}
    for (name, att, keep), t in zip(CONFIGS, times):
        med = float(np.median(t))
        res["configs"][name] = {"attention": att, "keep": keep, "ms_per_step": med, "min": float(min(t)), "max": float(max(t)),
                                "ratio_to_keep11": med / base}
    line = json.dumps(res)
    print(line, flush=True)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
