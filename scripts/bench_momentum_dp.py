#!/usr/bin/env python3
"""MomentumOptimizer under data parallelism next to Adagrad, at two shapes, B = 2^20 rows PER RANK, four device-resident
batches per rank:

  fm_c1   FM frappe-10 (F = 10), K = 64, lamda 0.1 (scripts/bench_models.py c1): V dense with L2, feature_bias IndexedSlices
  hhfm    HHFM (OUR) frappe-10 records [user, item, 8 context] + 10 negatives, K = 64, lamda 0: V IndexedSlices

    python scripts/bench_momentum_dp.py [--runs 3] [--steps 20] [--json out.json]                      # N = 1
    torchrun --nproc_per_node N scripts/bench_momentum_dp.py [--runs 3] [--steps 20] [--json out.json]  # N = 2, 4, 8

N = 1 (no torchrun): a world-size-1 NCCL group in this process; per shape and optimizer the single-GPU model and the
model under the group (NCCL exchange; with Momentum that includes the MAX all-reduce of the stamps and the compaction) are
timed in alternation.  N > 1: per shape and optimizer the fused exchange (`fused=True`) and the NCCL exchange
(`fused=False`), ms per step from rank 0's device events around `steps` whole steps.  The card's name and power limit
are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import socket
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

from bench_afm_dropout import gpu_info  # noqa: E402
from bench_models import frappe_rows, timed  # noqa: E402

OPTS = {"adagrad": "AdagradOptimizer", "momentum": "MomentumOptimizer"}


def _data(dev, seed, B):
    import torch
    rng = np.random.default_rng(seed)
    fm, hh = [], []
    for _ in range(4):
        X, M, n_user, n_item = frappe_rows(rng, B)
        fm.append((torch.from_numpy(X).to(dev), torch.from_numpy(rng.choice([1.0, 0.0], B).astype(np.float32)).to(dev)))
        neg = n_user + rng.integers(0, n_item, (B, 10))
        hh.append((X[:, :2], X[:, 2:], neg))
    return fm, hh, (M, n_user, n_item)


def _model(kind, opt, shape, dp, hh=None):
    from hhfm_b200.models import FM, OUR
    M, n_user, n_item = shape
    if kind == "fm_c1":
        m = FM(10, M, n_user, n_item, 64, 0.1, 0.1, 1, OPTS[opt], 0, 0)
    else:
        m = OUR(8, 0, M, n_user, n_item, 64, 0.05, 0.0, OPTS[opt], True, False)
    if dp is not None:
        m.enable_data_parallel(fused=dp, sparse=False)
    if kind == "hhfm":
        recs = []
        for X, F1, neg in hh:
            idx, _ = m._upload_ids([X, F1, neg])
            recs.append((idx.clone(), 8, 0, 10))
        return m, recs
    return m, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world == 1 and "MASTER_ADDR" not in os.environ:
        s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
        os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
        os.environ["RANK"], os.environ["WORLD_SIZE"] = "0", "1"
    dist.init_process_group("nccl", device_id=dev)
    try:
        B = 1 << 20
        fm, hh, shape = _data(dev, 1 + rank, B)
        res = {"gpu": gpu_info(), "world": world, "rows_per_rank": B, "runs": args.runs, "steps_per_run": args.steps,
               "shapes": {"fm_c1": "FM frappe-10 (F=10, M=%d), K=64, lamda 0.1" % shape[0],
                          "hhfm": "HHFM frappe-10 (8 context columns, 10 negatives), K=64, lamda 0"}}
        exchanges = {"single": None, "nccl_w1": False} if world == 1 else {"fused": True, "nccl": False}
        for kind in ("fm_c1", "hhfm"):
            models = {}
            for opt in OPTS:
                for ex, dp in exchanges.items():
                    m, recs = _model(kind, opt, shape, dp, hh)
                    batches = recs if recs is not None else fm
                    models["%s/%s" % (opt, ex)] = (m, batches)
            for m, b in models.values():                    # warm all (module load, hot-row plan, communicator)
                timed(lambda i: m.fit_device(*b[i % 4]), 3, 2)
            times = {k: [] for k in models}
            for _ in range(args.runs):
                for k, (m, b) in models.items():
                    times[k].append(timed(lambda i: m.fit_device(*b[i % 4]), args.steps, 1))
            res[kind] = {k: {"ms_per_step_runs": t, "median": float(np.median(t))} for k, t in times.items()}
            del models
            torch.cuda.empty_cache()
        if rank == 0:
            line = json.dumps(res)
            print(line, flush=True)
            if args.json:
                os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
                with open(args.json, "w") as f:
                    f.write(line + "\n")
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
