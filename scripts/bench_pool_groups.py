#!/usr/bin/env python
"""Pooled context groups of the HHFM sum-pooling training kernel (DESIGN §4, `hhfm_pool_groups_attach`): timings on the GPU.

    python scripts/bench_pool_groups.py premise [--reps 60]        # existing kernel at n_ctx = 8 / 3 / 0 (no groups)
    python scripts/bench_pool_groups.py ab [--pairs 6] [--steps 60] # HHFM_POOL_GROUPS=0 / 1 alternated in one process

`premise` times `hhfm_pairrank_fwd_bwd` at the benchmark shape (B = 2^20 positives, K = 64, NG = 10, hot-row plan from the
batch) for the frappe context columns (n_ctx = 8, cardinalities 7, 2, 3, 2, 9, 80, 233, 7), for three columns of
cardinalities (5292, 18640, 7) -- the grouped kernel's memory pattern (two pooled group rows) plus one small column -- and
for no context at all (the bound).  `ab` runs the benchmark's step (OUR.fit_device's two launches on device-resident
batches) with the grouped path switched off and on, alternating on the same batches.  Every time comes from CUDA events;
one JSON line on stdout.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (shapes and the seeded batch generator of the headline benchmark)

B = 1 << 20
N_BATCHES = 4            # 4 x 80 MB of records > 126 MB of L2, as in bench.py


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out.splitlines()[0] if out else None
    except Exception:
        return None


def make_records(rng, cards, dev):
    """Device-resident packed records [B, stride] (user, item+, one column per entry of `cards`, NG negatives)."""
    import torch
    from hhfm_b200.engine import Staging, pack_records
    M = bench.N_USER + bench.N_ITEM + sum(cards)
    X = np.stack([bench.zipf_ids(rng, bench.N_USER, B), bench.N_USER + bench.zipf_ids(rng, bench.N_ITEM, B)], 1)
    base = bench.N_USER + bench.N_ITEM
    cols = []
    for c in cards:
        cols.append(base + rng.integers(0, c, B))
        base += c
    Y = bench.N_USER + rng.integers(0, bench.N_ITEM, (B, bench.NG))
    parts = [X] + ([np.stack(cols, 1)] if cols else []) + [Y]
    stg = Staging(torch.int32, dev)
    host, stride = pack_records(parts, M, stg)
    rec = stg.upload(host.numel()).view(B, stride).clone()
    return rec, stride, M


def time_launches(fn, reps):
    """Per-launch CUDA-event times (ms) of `reps` launches of fn(i) after 5 warm-up launches."""
    import torch
    for i in range(5):
        fn(i)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for i, (a, b) in enumerate(ev):
        a.record()
        fn(i)
        b.record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev]


def stats(ts):
    ts = np.asarray(ts)
    return {"median_ms": float(np.median(ts)), "p10_ms": float(np.percentile(ts, 10)), "p90_ms": float(np.percentile(ts, 90)),
            "n": int(ts.size)}


def run_premise(args):
    import torch
    from hhfm_b200 import _lib
    from hhfm_b200.engine import NO_HOT, HotRows, cur_stream, ptr
    dev = torch.device("cuda", 0)
    K = bench.K_FACTOR
    out = {"mode": "premise", "gpu": gpu_info(), "B": B, "K": K, "NG": bench.NG, "reps": args.reps}
    for name, cards in (("n_ctx8_frappe", bench.CTX_CARD), ("n_ctx3_proxy", (5292, 18640, 7)), ("n_ctx0_bound", ())):
        rng = np.random.default_rng(1234)
        batches = []
        for _ in range(N_BATCHES):
            rec, stride, M = make_records(rng, cards, dev)
            batches.append(rec)
        g = torch.Generator(device="cpu").manual_seed(7)
        V = torch.empty(M, K).normal_(0, 0.01, generator=g).to(dev)
        gV = torch.zeros_like(V)
        lp = torch.zeros(_lib.partials_len(), dtype=torch.float32, device=dev)
        hot = HotRows.from_batch(batches[0], M, K, dev)
        hargs = hot.args() if hot is not None else NO_HOT
        n_ctx = len(cards)

        def launch(i):
            rec = batches[i % N_BATCHES]
            _lib.call("hhfm_pairrank_fwd_bwd", ptr(rec), B, stride, n_ctx, 0, bench.NG, 0, 0, 0, ptr(V), M, K, None, None,
                      ptr(gV), ptr(lp), None, 0, None, None, *hargs, 0, cur_stream())

        out[name] = dict(stats(time_launches(launch, args.reps)), cards=list(cards), stride=stride,
                         n_hot=hot.n_hot if hot is not None else 0)
        del batches, V, gV, hot
        torch.cuda.empty_cache()
    base = out["n_ctx8_frappe"]["median_ms"]
    out["proxy_speedup"] = base / out["n_ctx3_proxy"]["median_ms"]
    out["bound_speedup"] = base / out["n_ctx0_bound"]["median_ms"]
    print(json.dumps(out))


def grouped_bytes_per_sample(n_slots, K=bench.K_FACTOR, NG=bench.NG):
    """bench.py's accounting (rows gathered + 80 B of ids + rows reduced) for the grouped formulation: 2 + n_slots + NG
    gathers, 2 + n_slots + 1 reductions (user, item+, one per slot, the max negative)."""
    return 4 * K * (2 + n_slots + NG) + 80 + 4 * K * (3 + n_slots)


def run_ab(args):
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
    arms = {}
    for arm in ("0", "1"):
        os.environ["HHFM_POOL_GROUPS"] = arm                 # the planner reads it when the plan is built
        m = OUR(n_ctx, 0, M, bench.N_USER, bench.N_ITEM, K, bench.LR, bench.LAMDA, "AdagradOptimizer", True, False)
        hot = m._hot_plan(batches[0], False)
        arms[arm] = (m, hot, hot.args() if hot is not None else NO_HOT)
    os.environ.pop("HHFM_POOL_GROUPS")

    def step(arm, i, ev=None):
        m, hot, hargs = arms[arm]
        rec = batches[i % N_BATCHES]
        m._opt.begin_step()
        if ev is not None:
            ev[0].record()
        _lib.call("hhfm_pairrank_fwd_bwd", ptr(rec), B, stride, n_ctx, 0, NG, 0, 0, 0, ptr(m.weights["feature_embeddings"]), M,
                  K, None, None, ptr(m._gV), ptr(m._loss_partials), None, 0, None, None, *hargs, 0, cur_stream())
        if ev is not None:
            ev[1].record()
        m._finish_step(hot, False)
        if ev is not None:
            ev[2].record()

    def run_arm(arm, steps):
        os.environ["HHFM_POOL_GROUPS"] = arm
        for i in range(5):
            step(arm, i)
        torch.cuda.synchronize()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for i in range(steps):
            step(arm, i, ev[i])
        t1.record()
        torch.cuda.synchronize()
        return (t0.elapsed_time(t1) / steps, float(np.median([e[0].elapsed_time(e[1]) for e in ev])))

    res = {"0": {"step_ms": [], "kernel_ms": []}, "1": {"step_ms": [], "kernel_ms": []}}
    for _ in range(args.pairs):
        for arm in ("0", "1"):
            s, k = run_arm(arm, args.steps)
            res[arm]["step_ms"].append(s)
            res[arm]["kernel_ms"].append(k)
    # the launches of the grouped entry point, from a short torch.profiler capture of its own (not in the timed pairs)
    os.environ["HHFM_POOL_GROUPS"] = "1"
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(10):
            step("1", i)
        torch.cuda.synchronize()
    launches = {}
    for e in prof.key_averages():
        if e.device_type is not None and "cuda" in str(e.device_type).lower() and e.count:
            t = getattr(e, "device_time", None) or getattr(e, "cuda_time", 0.0)
            launches[e.key[:90]] = {"count": e.count, "avg_us": float(t)}
    os.environ.pop("HHFM_POOL_GROUPS")
    out = {"mode": "ab", "gpu": gpu_info(), "B": B, "K": K, "NG": NG, "pairs": args.pairs, "steps_per_arm": args.steps,
           "hot_rows": {a: (arms[a][1].n_hot if arms[a][1] is not None else 0) for a in arms},
           "pool_groups": arms["1"][0]._pool_groups.groups if arms["1"][0]._pool_groups is not None else None,
           "bytes_per_sample": {"ungrouped": bench.ALGO_BYTES_PER_SAMPLE, "grouped": grouped_bytes_per_sample(2)},
           "launches_grouped": launches}
    for arm, name in (("0", "ungrouped"), ("1", "grouped")):
        s, k = np.asarray(res[arm]["step_ms"]), np.asarray(res[arm]["kernel_ms"])
        out[name] = {"step_ms_median": float(np.median(s)), "step_ms_min": float(s.min()), "step_ms_max": float(s.max()),
                     "kernel_ms_median": float(np.median(k)), "kernel_ms_min": float(k.min()), "kernel_ms_max": float(k.max()),
                     "step_ms_per_pair": s.tolist()}
    out["step_speedup"] = out["ungrouped"]["step_ms_median"] / out["grouped"]["step_ms_median"]
    out["samples_per_s_grouped"] = B / (out["grouped"]["step_ms_median"] * 1e-3)
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("mode", choices=["premise", "ab"])
    ap.add_argument("--reps", type=int, default=60)
    ap.add_argument("--pairs", type=int, default=6)
    ap.add_argument("--steps", type=int, default=60)
    args = ap.parse_args()
    if args.reps < 50 or args.steps < 50 or args.pairs < 5:
        ap.error("--reps and --steps must be at least 50, --pairs at least 5")
    if args.mode == "premise":
        run_premise(args)
    else:
        run_ab(args)


if __name__ == "__main__":
    main()
