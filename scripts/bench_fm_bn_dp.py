#!/usr/bin/env python3
"""FM batch_norm=1 under data parallelism with synchronised batch norm (FM.enable_data_parallel(sync_batch_norm=True)) at
the fm_c1 shape of scripts/bench_models.py: frappe-10 (F = 10), K = 64, B = 2^20 rows PER RANK, dense-L2 Adagrad, four
device-resident batches per rank.

    python scripts/bench_fm_bn_dp.py [--runs 3] [--steps 20] [--json out.json]                      # N = 1
    torchrun --nproc_per_node N scripts/bench_fm_bn_dp.py [--runs 3] [--steps 20] [--json out.json]  # N = 2, 4, 8

N = 1 (no torchrun): a world-size-1 NCCL group in this process; four models of the same shape and seed timed in
alternation (run r times `steps` whole steps of each in turn): batch_norm = 1 on one GPU (the single fused entry),
batch_norm = 1 under the world-size-1 group (the three phases and two all-gathers, and the NCCL gradient tail of a
data-parallel step), and the same two with batch_norm = 0.  The cost of the split and the two collectives is the batch_norm
= 1 difference less the batch_norm = 0 difference (the tail of the step).
N > 1: every rank trains its own 2^20 rows; ms per step and samples per second of the global batch (N * 2^20), from
rank 0's device events around `steps` whole steps (each step ends in the collectives, so every rank is in it).
The card's name and power limit are read in the same run.
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


def _batches(dev, seed, B):
    import torch
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(4):
        X, M, n_user, n_item = frappe_rows(rng, B)
        out.append((torch.from_numpy(X).to(dev), torch.from_numpy(rng.choice([1.0, 0.0], B).astype(np.float32)).to(dev)))
    return out, (M, n_user, n_item)


def _model(shape, bn, dp):
    from hhfm_b200.models import FM
    M, n_user, n_item = shape
    m = FM(10, M, n_user, n_item, 64, 0.1, 0.1, 1, "AdagradOptimizer", bn, 0)
    if dp:
        m.enable_data_parallel(sync_batch_norm=True)
    return m


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
        batches, shape = _batches(dev, 1 + rank, B)
        res = {"gpu": gpu_info(), "world": world, "shape": "frappe-10 (F=10, M=%d), K=64, B=2^20 per rank, dense-L2 Adagrad"
               % shape[0], "runs": args.runs, "steps_per_run": args.steps}
        if world == 1:
            names = {"bn1_single": (1, False), "bn1_sync_w1": (1, True), "bn0_single": (0, False), "bn0_dp_w1": (0, True)}
            models = {k: _model(shape, bn, dp) for k, (bn, dp) in names.items()}
            for m in models.values():                       # warm all (module load, hot-row plan, workspace, communicator)
                timed(lambda i: m.fit_device(*batches[i % 4]), 3, 2)
            times = {k: [] for k in models}
            for _ in range(args.runs):
                for k, m in models.items():
                    times[k].append(timed(lambda i: m.fit_device(*batches[i % 4]), args.steps, 1))
            med = {k: float(np.median(t)) for k, t in times.items()}
            res.update({k: {"ms_per_step_runs": times[k], "median": med[k]} for k in models})
            res["split_and_collectives_ms"] = (med["bn1_sync_w1"] - med["bn1_single"]) - (med["bn0_dp_w1"] - med["bn0_single"])
        else:
            m = _model(shape, 1, True)
            timed(lambda i: m.fit_device(*batches[i % 4]), 3, 2)
            runs = [timed(lambda i: m.fit_device(*batches[i % 4]), args.steps, 1) for _ in range(args.runs)]
            med = float(np.median(runs))
            res.update({"ms_per_step_runs": runs, "median": med, "samples_per_s": world * B / (med * 1e-3)})
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
