#!/usr/bin/env python3
"""DeepFM training step and full-catalog top-N per reference option (use_fm, use_deep, loss_type) at the DeepFM shape of
scripts/bench_models.py: frappe-10, 640-150-200-150, K = 64, B = 2^17, two device-resident batches.

    python scripts/bench_dfm_modes.py [--rounds 5] [--steps 10] [--contexts 2048] [--json out.json]

One model per mode, same shape and seed, timed in alternation in one process (round r times `steps` whole steps of each
mode in turn, so clock and neighbour drift hit every arm alike).  Then `topk(A, 20)` over frappe-10's 4082 items for
`contexts` rows, per mode, alternating the same way (host clock around a call that ends in a device synchronise).
Reported per mode: median ms over the rounds, (min, max), ratio to the default mode; the card name and power limit are
read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

from bench_models import frappe_rows, timed  # noqa: E402

MODES = [("default (use_fm, use_deep, mse)", dict()),
         ("logloss", dict(loss_type="logloss")),
         ("use_deep=False (FM part only)", dict(use_deep=False)),
         ("use_fm=False (DNN part only)", dict(use_fm=False)),
         ("use_deep=False, logloss", dict(use_deep=False, loss_type="logloss")),
         ("use_fm=False, logloss", dict(use_fm=False, loss_type="logloss"))]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out.splitlines()[0] if out else None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--contexts", type=int, default=2048)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    from hhfm_b200.models import DeepFM
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(6)
    B, K, layers = 1 << 17, 64, [150, 200, 150]
    batches = []
    for _ in range(2):
        X, M, n_user, n_item = frappe_rows(rng, B)
        batches.append((torch.from_numpy(X).to(dev), torch.from_numpy(rng.choice([1.0, -1.0], B).astype(np.float32)).to(dev)))
    models = [DeepFM(n_user, n_item, M, 10, K, layers, "relu", 0.01, 0, 0.01, **kw) for _, kw in MODES]
    for m in models:                                        # warm every mode (module load, first launches)
        timed(lambda i: m.fit_device(*batches[i % 2]), 2, 2)
    step = [[] for _ in MODES]
    for r in range(args.rounds):
        for c, m in enumerate(models):
            step[c].append(timed(lambda i: m.fit_device(*batches[i % 2]), args.steps, 1))
    A = batches[0][0][:args.contexts].cpu().numpy()
    for m in models:
        m.topk(A[:64], 20)
    topn = [[] for _ in MODES]
    for r in range(args.rounds):
        for c, m in enumerate(models):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m.topk(A, 20)
            topn[c].append((time.perf_counter() - t0) * 1e3)
    res = {"gpu": gpu_info(), "shape": "frappe-10, 640-150-200-150, K=64, B=2^17, 2 device-resident batches, l2_reg=0.01",
           "topk": "%d contexts x %d items, top-20" % (len(A), n_item), "rounds": args.rounds, "steps_per_round": args.steps,
           "modes": {}}
    s0, t0 = float(np.median(step[0])), float(np.median(topn[0]))
    for (name, kw), s, t in zip(MODES, step, topn):
        res["modes"][name] = {"options": kw, "step_ms": float(np.median(s)), "step_min": float(min(s)), "step_max": float(max(s)),
                              "step_ratio": float(np.median(s)) / s0, "topk_ms": float(np.median(t)), "topk_min": float(min(t)),
                              "topk_max": float(max(t)), "topk_ratio": float(np.median(t)) / t0}
    line = json.dumps(res)
    print(line, flush=True)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
