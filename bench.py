#!/usr/bin/env python
"""bench.py -- headline benchmark of the HHFM hot path on B200 (contract: see the task statement / DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (one process per GPU under torchrun)
    python bench.py --impl reference [--gpus N] [--steps K] ...     # the reference's CPU path (oracle restatement)
    python bench.py ... --dump-outputs DIR     # also write the last timed step's loss and weights as DIR/<name>.npy

The same arguments give the same seeded batches and initial weights on every run.  The timed step adds its gradients
with float atomics, whose rounding changes from run to run, and the max over the negatives grows that into different
training trajectories within a few steps.  With --dump-outputs the last timed step therefore starts again from the
seeded weights and Adagrad accumulators, so what it writes differs between two runs of one build by rounding only.

Workload (BASELINE.json configs[1]): OurModel7 (HHFM) training on frappe-10-shaped synthetic data -- 10 fields
(user 957, item 4082, 8 context columns, 343 values), features_M = 5382, K = 64, NG = 10 negatives, Adagrad lr 0.1,
lamda 0.01 (the reference defaults, OurModel7.py:29-41).  One step = one pass of the hot path over one batch:
fused gather + pooling + BPR max-negative loss + backward scatter, dense-L2 Adagrad update, loss reduction.
`value` = positives/s with the batch records resident in HBM; `e2e` = the same through `OUR.partial_fit` with
host numpy int64 batches (pack + H2D + kernels + loss D2H inside the timed region).
One JSON line on stdout (rank 0).  Beside the contract keys the line carries: `roofline` (the scatter kernel against the
L2 read bandwidth measured in this run -- at frappe shape the table is L2-resident), `roofline_hbm` (the same model at
the scaled c5 shape, where HBM binds), `topn` / `topn_c5` (the evaluator half of the metric), `models` (the other
BASELINE.json configs), `parity_bands` (the drop-in trainer on the reference's shipped frappe file against the bands of
the reference's result.txt, with HR@10), `e2e_epoch` (one reference-style epoch, sampler included), `dp_check` (N > 1:
replicas bit-identical, update cross-checked against an NCCL all-reduce of the same gradients).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_USER, N_ITEM = 957, 4082
CTX_CARD = (7, 2, 3, 2, 9, 80, 233, 7)      # daytime, isweekend, homework, cost, weather, country, city, cnt
K_FACTOR = 64
NG = 10
LAMDA, LR = 0.01, 0.1
FEATURES_M = N_USER + N_ITEM + sum(CTX_CARD)
# SURVEY.md 8(d): per positive, gather (F+NG)=20 rows + 80 B of ids = 5200 B, scatter 11 rows = 2816 B
ALGO_BYTES_PER_SAMPLE = 4 * 20 * K_FACTOR + 80 + 4 * 11 * K_FACTOR


def zipf_ids(rng, n, size, a=1.1):
    p = 1.0 / np.arange(1, n + 1) ** a
    p /= p.sum()
    return rng.choice(n, size=size, p=p)


def make_batch(rng, B):
    """Frappe-10-shaped HHFM batch in the reference's feed layout: X[B,2], F1[B,8], Y[B,10] (int64)."""
    X = np.stack([zipf_ids(rng, N_USER, B), N_USER + zipf_ids(rng, N_ITEM, B)], axis=1).astype(np.int64)
    base = N_USER + N_ITEM
    cols = []
    for c in CTX_CARD:
        cols.append(base + rng.integers(0, c, B))
        base += c
    F1 = np.stack(cols, axis=1).astype(np.int64)
    Y = (N_USER + rng.integers(0, N_ITEM, (B, NG))).astype(np.int64)
    return {"X": X, "F1": F1, "Y": Y}


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe).  NVML is polled from a
    thread every ~2 ms (the nvidia-smi CLI needs longer to start than a short timed region lasts); the CLI loop of the
    recipe is the fallback when pynvml is missing."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, gpu_index, uuid=None):
        self.gpu = gpu_index
        self.uuid = uuid
        self.lines = []
        self.proc = None
        self.nvml = None
        self.sm, self.reason_bits, self.power = [], 0, []
        self.max_sm = None
        self._stop = threading.Event()

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        h = None
        if self.uuid:
            for u in (self.uuid, "GPU-" + self.uuid):
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(u.encode() if isinstance(u, str) else u)
                    break
                except Exception:
                    h = None
        if h is None:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
        return pynvml, h

    def start(self):
        try:
            self.nvml, self.h = self._nvml_handle()
            self.max_sm = float(self.nvml.nvmlDeviceGetMaxClockInfo(self.h, self.nvml.NVML_CLOCK_SM))
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def sample(self):
        """One synchronous NVML sample (called by the timing loop itself while the GPU is busy)."""
        if self.nvml is None:
            return
        try:
            self.sm.append(float(self.nvml.nvmlDeviceGetClockInfo(self.h, self.nvml.NVML_CLOCK_SM)))
            try:
                self.reason_bits |= int(self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                self.reason_bits |= int(self.nvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            if len(self.sm) % 4 == 1:                    # NVML queries take milliseconds: keep the sample cheap
                self.power.append(self.nvml.nvmlDeviceGetPowerUsage(self.h) / 1e3)
        except Exception:
            pass

    def _poll(self):
        while not self._stop.is_set():
            self.sample()
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self._stop.set()
            self.th.join(timeout=2)
            reasons = sorted(k for k, b in self.BITS.items() if self.reason_bits & b)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_sm,
                    "samples": len(self.sm), "power_w_max": max(self.power) if self.power else None,
                    "reasons": reasons, "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------------
# CPU baseline: the oracle's torch-CPU mirror of the TF graph (restatement, not TF)
# ----------------------------------------------------------------------------------------------------
def cpu_baseline(budget_s=12.0, batch=1 << 20, max_steps=8):
    import torch
    from oracle import torch_cpu as T
    torch.set_num_threads(os.cpu_count() or 1)
    rng = np.random.default_rng(99)
    g = torch.Generator().manual_seed(2016)
    V = torch.empty(FEATURES_M, K_FACTOR).normal_(0, 0.01, generator=g)
    acc = torch.full_like(V, 0.1)
    b = make_batch(rng, batch)
    Pos, Fea, Neg = torch.from_numpy(b["X"]), torch.from_numpy(b["F1"]), torch.from_numpy(b["Y"])
    T.hhfm_train_step(V, acc, Pos, Neg, Fea, None, (0, 0, 0), LAMDA, LR)      # warm-up
    t0 = time.perf_counter()
    steps = 0
    while steps < max_steps and (time.perf_counter() - t0) < budget_s:
        T.hhfm_train_step(V, acc, Pos, Neg, Fea, None, (0, 0, 0), LAMDA, LR)
        steps += 1
    dt = time.perf_counter() - t0
    return {"value": steps * batch / dt, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": "%d steps of %d positives (frappe-10 HHFM, NG=10, K=64), torch-CPU op-for-op mirror of "
                      "OurModel7.py:105-189; restatement, not TF" % (steps, batch), "ms_per_step": 1e3 * dt / max(steps, 1)}


def run_reference(args):
    """The reference's CPU path for the same workload, metric and batch as our arm (same_config): the torch-CPU op-for-op
    mirror of OurModel7.py:105-189 on all host cores (TensorFlow 1.x cannot be installed here: restatement, not TF)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import torch_cpu as T
    torch.set_num_threads(os.cpu_count() or 1)
    batch = args.batch
    rng = np.random.default_rng(99)
    g = torch.Generator().manual_seed(2016)
    V = torch.empty(FEATURES_M, K_FACTOR).normal_(0, 0.01, generator=g)
    acc = torch.full_like(V, 0.1)
    b = make_batch(rng, batch)
    Pos, Fea, Neg = torch.from_numpy(b["X"]), torch.from_numpy(b["F1"]), torch.from_numpy(b["Y"])
    for _ in range(max(min(args.warmup, 2), 1)):          # a CPU step takes seconds: two warm-up steps settle the thread pool
        T.hhfm_train_step(V, acc, Pos, Neg, Fea, None, (0, 0, 0), LAMDA, LR)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        T.hhfm_train_step(V, acc, Pos, Neg, Fea, None, (0, 0, 0), LAMDA, LR)
    dt = time.perf_counter() - t0
    val = args.steps * batch / dt
    cb = {"value": val, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
          "sample": "%d steps of %d positives per step; torch-CPU mirror of OurModel7.py:105-189 (restatement, not TF: "
                    "TensorFlow 1.x cannot be installed here)" % (args.steps, batch)}
    line = {"impl": "reference", "metric": "hhfm_train_samples_per_s", "value": val, "unit": "samples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(batch, args.gpus), "cpu_baseline": cb,
            "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------
# second half of BASELINE.json's metric: full-catalog top-N scored pairs/s (item-sharded, NCCL merge)
# ----------------------------------------------------------------------------------------------------
def _tensor_peaks():
    burst, sustained = 1626.2, 1371.7
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        burst, sustained = float(d.get("bf16_tflops", burst)), float(d.get("bf16_tflops_sustained", sustained))
    return burst, sustained


def _time_prepare_items(t, V, n_user, lo, hi, K):
    """The fp32 -> bf16 item-operand preparation (once per weight version; reported beside the timed region, not in it)."""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    t._item_operand(0, V[n_user + lo:n_user + hi], None, hi - lo, K, ("bench", lo, hi), None)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def run_topn(world, rank, dev, quick):
    """C contexts x (N items per GPU) x K=128, tp=100, WEAK-scaled (10^6 items per GPU): every rank scores all contexts
    against ITS item shard with the tcgen05 filter + exact rescoring, then the [C,tp] candidates are all-gathered and merged
    (score desc, id asc).  Returns pairs/s over the whole job and stage timings."""
    import torch
    import torch.distributed as dist
    from hhfm_b200 import dist as hd
    from hhfm_b200.engine import TopN
    C, N, K, tp, n_user = (2048, 200000, 128, 100, 1024) if quick else (16384, 1000000, 128, 100, 1024)
    g = torch.Generator(device="cpu").manual_seed(4321 + rank)
    M = n_user + N
    V = torch.empty(M, K).normal_(0, 0.01, generator=g).to(dev)
    gq = torch.Generator(device="cpu").manual_seed(4321)
    V[:n_user] = torch.empty(n_user, K).normal_(0, 0.01, generator=gq).to(dev)       # same users on every rank
    A = torch.stack([torch.randint(0, n_user, (C,), generator=gq), torch.randint(n_user, M, (C,), generator=gq)], 1).to(torch.int32)
    t = TopN(dev, max_workspace_bytes=6 << 30)
    A_dev, stride = t.upload_rows(A.numpy(), M)

    def once():
        ids, sc = t.topk(0, A_dev, stride, 0, 0, (0, 0, 0), V, None, n_user, N, tp, return_scores=True, method="tc", version=1)
        ids = ids + rank * N                       # global item ids of this rank's shard
        if world > 1:
            ids, sc = hd.merge_topk(sc, ids, tp)
        return ids

    for _ in range(2):
        once()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    reps = 3 if quick else 5
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        once()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    if world > 1:
        tt = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    prep_ms = _time_prepare_items(t, V, n_user, 0, N, K)
    pairs = float(C) * N * world
    burst, sustained = _tensor_peaks()
    ach_tf = 2.0 * K * pairs / world / (ms * 1e-3) / 1e12      # per GPU, algorithmic 2*K flop per pair, whole pipeline
    return {"metric": "topn_scored_pairs_per_s", "value": pairs / (ms * 1e-3), "unit": "pairs/s", "ms_per_query_batch": ms,
            "config": {"workload": "full-catalog top-N (BPR/HHFM query kind), tcgen05 bf16 filter + exact fp32 rescoring",
                       "contexts": C, "items_per_gpu": N, "K": K, "tp": tp, "item_sharding": "N per GPU (weak), all-gather merge"},
            "overflow_rows": t.last_overflow_rows, "item_operand_prep_ms": prep_ms,
            "roofline": {"bound": "tensor", "achieved": ach_tf, "peak": burst, "unit": "TFLOP/s", "frac": ach_tf / burst,
                         "frac_of_sustained": ach_tf / sustained,
                         "note": "algorithmic 2*K flop per pair over the WHOLE pipeline (query prep, sampled max pass, cut, "
                                 "emission GEMM, candidate compaction, exact rescoring, final select, proof of the cut); the "
                                 "timed region is milliseconds, so the peak is the BURST cuBLAS bf16 figure "
                                 "(MEASURED_PEAKS.json).  The fp32 -> bf16 item-operand preparation is cached per weight "
                                 "version (an evaluation scores thousands of context rows against one set of weights) and is "
                                 "reported as item_operand_prep_ms, outside the timed region"}}


_C5_LISTS = {}


def run_topn_c5(world, rank, dev):
    """BASELINE.json configs[4] as written (SURVEY.md 8d): ONE catalog of 10^6 items, K = 128, C = 65 536 context rows,
    tp = 100; at N GPUs every rank scores all contexts against its 10^6/N items (STRONG scaling).  Contexts run in chunks;
    the exchange + merge of chunk i (all-to-all by context rows on a side stream, hhfm_b200.dist.merge_topk_sharded) overlaps
    the GEMM of chunk i+1; each rank ends with the merged lists of its C/N context rows (the HR/NDCG walk shards by rows)."""
    import torch
    import torch.distributed as dist
    from hhfm_b200 import dist as hd
    from hhfm_b200.engine import TopN
    C, N, K, tp, n_user, n_chunks = 65536, 1000000, 128, 100, 4096, 4
    g = torch.Generator(device="cpu").manual_seed(777)
    lo, hi = hd.shard_range(N, rank, world)
    M = n_user + N
    # every rank draws the same catalog and keeps users + its item range (the bench holds one shard per GPU, like the model would)
    Vfull = torch.empty(M, K).normal_(0, 0.01, generator=g)
    V = torch.cat([Vfull[:n_user], Vfull[n_user + lo:n_user + hi]]).to(dev)
    del Vfull
    n_loc = hi - lo
    A = torch.stack([torch.randint(0, n_user, (C,), generator=g), torch.full((C,), n_user, dtype=torch.int64)], 1).to(torch.int32)
    t = TopN(dev, max_workspace_bytes=6 << 30)
    A_dev, stride = t.upload_rows(A.numpy(), n_user + n_loc)
    side = torch.cuda.Stream(device=dev)
    per = C // n_chunks

    def once():
        outs = []
        main = torch.cuda.current_stream()
        for c in range(n_chunks):
            ids, sc = t.topk(0, A_dev[c * per:(c + 1) * per], stride, 0, 0, (0, 0, 0), V, None, n_user, n_loc, tp,
                             return_scores=True, method="tc", version=1)
            ids = ids + lo
            if world > 1:
                ready = torch.cuda.Event()
                ready.record(main)
                with torch.cuda.stream(side):
                    side.wait_event(ready)
                    ids.record_stream(side); sc.record_stream(side)
                    outs.append(hd.merge_topk_sharded(sc, ids, tp)[0])
            else:
                outs.append(ids)
        if world > 1:
            main.wait_stream(side)
        return outs

    for _ in range(2):
        once()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    reps = 3
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        last = once()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    if world > 1:
        tt = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
        # kept for the cross-check against the context-sharded evaluator: chunk c leaves rank r with rows
        # [c*per + r*per/world, c*per + (r+1)*per/world) of the merged lists
        _C5_LISTS["item_sharded"] = [x.clone() for x in last]
    prep_ms = _time_prepare_items(t, V, n_user, 0, n_loc, K)
    pairs = float(C) * N
    burst, sustained = _tensor_peaks()
    ach_tf = 2.0 * K * pairs / world / (ms * 1e-3) / 1e12
    return {"metric": "topn_scored_pairs_per_s", "value": pairs / (ms * 1e-3), "unit": "pairs/s", "ms_per_query_batch": ms,
            "scaling": "strong",
            "config": {"workload": "BASELINE configs[4]: 10^6-item catalog TOTAL, K=128, top-100, item-sharded, context-sharded all-to-all merge "
                                   "overlapped with the next chunk's GEMM", "contexts": C, "items_total": N, "items_per_gpu": n_loc,
                       "K": K, "tp": tp, "context_chunks": n_chunks},
            "overflow_rows": t.last_overflow_rows, "item_operand_prep_ms": prep_ms,
            "roofline": {"bound": "tensor", "achieved": ach_tf, "peak": burst, "unit": "TFLOP/s", "frac": ach_tf / burst,
                         "frac_of_sustained": ach_tf / sustained,
                         "note": "per GPU, algorithmic 2*K flop per pair over the whole pipeline incl. exchange + merge; burst bf16 peak"}}


def run_topn_c5_ctx(world, rank, dev):
    """The same evaluation (10^6-item catalog, K = 128, 65 536 context rows, tp = 100) with the CONTEXT rows sharded: every
    rank holds the whole table (it does under data-parallel training: 0.5 GB + 0.26 GB of bf16 operand) and scores its
    65 536/N rows against all 10^6 items; the [C/N, tp] lists are all-gathered inside the timed region.  No candidate exchange,
    no merge, and the per-row stages shard with the rows (`models.enable_context_sharding`)."""
    import torch
    import torch.distributed as dist
    from hhfm_b200 import dist as hd
    from hhfm_b200.engine import TopN
    C, N, K, tp, n_user = 65536, 1000000, 128, 100, 4096
    g = torch.Generator(device="cpu").manual_seed(777)
    V = torch.empty(n_user + N, K).normal_(0, 0.01, generator=g).to(dev)
    A = torch.stack([torch.randint(0, n_user, (C,), generator=g), torch.full((C,), n_user, dtype=torch.int64)], 1).to(torch.int32)
    lo, hi = hd.shard_range(C, rank, world)
    t = TopN(dev, max_workspace_bytes=6 << 30)
    A_dev, stride = t.upload_rows(A[lo:hi].numpy(), n_user + N)
    chunk = 16384

    def once():
        outs = []
        for c0 in range(0, hi - lo, chunk):
            outs.append(t.topk(0, A_dev[c0:c0 + chunk], stride, 0, 0, (0, 0, 0), V, None, n_user, N, tp, method="tc", version=1))
        ids = torch.cat(outs) if len(outs) > 1 else outs[0]
        return hd.gather_rows(ids, None, sizes) if world > 1 else ids

    sizes = [hd.shard_range(C, r, world)[1] - hd.shard_range(C, r, world)[0] for r in range(world)]
    for _ in range(2):
        once()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    reps = 3
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = once()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    if world > 1:
        tt = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    pairs = float(C) * N
    burst, sustained = _tensor_peaks()
    ach_tf = 2.0 * K * pairs / world / (ms * 1e-3) / 1e12
    # N > 1 evidence: the two decompositions of the same evaluation (same catalog, same context rows) must give the same lists
    same = None
    if world > 1 and "item_sharded" in _C5_LISTS:
        chunks = _C5_LISTS.pop("item_sharded")
        per = C // len(chunks)
        ok = True
        for c, lst in enumerate(chunks):
            r0 = c * per + rank * (per // world)
            ok = ok and bool(torch.equal(lst.to(torch.int32), out[r0:r0 + per // world].to(torch.int32)))
        tt = torch.tensor([1.0 if ok else 0.0], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MIN)
        same = bool(tt.item() == 1.0)
    return {"metric": "topn_scored_pairs_per_s", "value": pairs / (ms * 1e-3), "unit": "pairs/s", "ms_per_query_batch": ms,
            "scaling": "strong", "lists_gathered": [int(out.shape[0]), int(out.shape[1])],
            "lists_identical_to_item_sharded": same,
            "config": {"workload": "BASELINE configs[4]: 10^6-item catalog, K=128, top-100, CONTEXT rows sharded (table replicated), "
                                   "lists all-gathered inside the timed region", "contexts": C, "contexts_per_gpu": hi - lo,
                       "items_total": N, "K": K, "tp": tp},
            "overflow_rows": t.last_overflow_rows,
            "roofline": {"bound": "tensor", "achieved": ach_tf, "peak": burst, "unit": "TFLOP/s", "frac": ach_tf / burst,
                         "frac_of_sustained": ach_tf / sustained,
                         "note": "per GPU, algorithmic 2*K flop per pair over the whole pipeline incl. the all-gather of the lists; burst bf16 peak"}}


def workload_config(batch, n_gpus):
    return {"workload": "OurModel7 (HHFM) train step, frappe-10 shape: 10 fields, features_M=%d, K=%d, NG=%d, "
                        "Adagrad lr=0.1, lamda=0.01 (dense L2 update)" % (FEATURES_M, K_FACTOR, NG),
            "batch_per_gpu": batch, "global_batch": batch * n_gpus, "parallelism": "dp%d" % n_gpus,
            "l2_policy": "device-resident batches cycled; 4 x 84 MB of records > 126 MB L2"}


# ----------------------------------------------------------------------------------------------------
def l2_read_peak(dev):
    """L2 -> SM read bandwidth measured in this run (hhfm_l2_read_sweep: L1-bypassing 16-byte loads over a 48 MB buffer that
    stays L2-resident): the denominator of the L2-bound gather kernels' roofline.  GB/s."""
    import torch
    from hhfm_b200 import _lib
    from hhfm_b200.engine import cur_stream, ptr
    n = (48 << 20) // 4
    buf = torch.ones(n, dtype=torch.float32, device=dev)
    sink = torch.zeros(1, dtype=torch.float32, device=dev)
    iters = 20
    _lib.call("hhfm_l2_read_sweep", ptr(buf), n, 4, ptr(sink), cur_stream())
    torch.cuda.synchronize()
    best = 0.0
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.call("hhfm_l2_read_sweep", ptr(buf), n, iters, ptr(sink), cur_stream())
        e1.record()
        torch.cuda.synchronize()
        best = max(best, 4.0 * n * iters / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    return best


def measured_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/traffic.json names the capture)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None, None
    d = json.load(open(p)).get(kernel)
    if not d:
        return None, None
    return d.get("dram_bytes_per_launch"), d.get("capture")


def dump_outputs(out_dir, arrays):
    """Write every array as `out_dir/<name>.npy` (float64 stays float64, everything else becomes float32), so that two
    builds run with the same arguments -- and therefore the same seeded inputs -- can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64 if a.dtype == np.float64 else np.float32))


def dp_check(model, rec, n_ctx, world, dev):
    """N > 1 correctness evidence carried by the bench line itself (the driver's test box has one GPU): one more step whose
    update is recomputed from an NCCL all-reduce of the ranks' gradients, and a bit-comparison of the replicas."""
    import torch
    import torch.distributed as dist
    from hhfm_b200 import _lib
    from hhfm_b200.engine import NO_HOT, cur_stream, ptr
    V = model.weights["feature_embeddings"]
    acc = model._opt.slots("feature_embeddings", V)[0]
    V0, acc0 = V.clone(), acc.clone()
    # this rank's gradient of `rec` at the current weights, into a scratch arena (no hot replicas: plain scatter)
    g = torch.zeros_like(V)
    lp = torch.zeros(_lib.partials_len(), dtype=torch.float32, device=dev)
    B, stride = rec.shape
    _lib.call("hhfm_pairrank_fwd_bwd", ptr(rec), B, stride, n_ctx, 0, NG, 0, 0, 0, ptr(V), FEATURES_M, K_FACTOR, None, None,
              ptr(g), ptr(lp), None, 0, None, None, *NO_HOT, 0, cur_stream())
    loss_local = lp.double().sum()
    dist.all_reduce(g)
    dist.all_reduce(loss_local)
    reg = 0.5 * LAMDA * float((V0.double() ** 2).sum())
    ge = g + LAMDA * V0
    acc1 = acc0 + ge * ge
    V1 = V0 - LR * ge / torch.sqrt(acc1)
    model.fit_device(rec, n_ctx, 0, NG)                      # the product's step (fused exchange) on the same records
    loss = model._read_loss()
    upd = (V1 - V0).abs()
    scale = float(torch.sqrt((upd * upd).mean()))
    err = float(((V - V1).abs() / torch.clamp(upd, min=scale)).max())
    gathered = [torch.empty_like(V) for _ in range(world)]
    dist.all_gather(gathered, V)
    same = all(bool(torch.equal(gathered[0], t)) for t in gathered)
    ga = [torch.empty_like(acc) for _ in range(world)]
    dist.all_gather(ga, acc)
    same = same and all(bool(torch.equal(ga[0], t)) for t in ga)
    loss_ref = float(loss_local) + reg
    return {"replicas_bit_identical": same, "update_max_rel_err_vs_nccl_allreduce": err,
            "loss": loss, "loss_from_nccl_allreduce": loss_ref, "loss_rel_err": abs(loss - loss_ref) / abs(loss_ref),
            "exchange": "fused symmetric-memory kernel (%s)" % ("multimem" if (model._dpx is not None and model._dpx.multicast) else "peer loads/stores")
                        if model._dpx is not None else "NCCL all-reduce of the arena",
            "ok": bool(same and err <= 2e-4 and abs(loss - loss_ref) <= 2e-5 * abs(loss_ref))}


def parity_bands(seeds=2, epochs=30):
    """BASELINE.json's third term ("HR@10 parity").  The reference cannot run here and seeds nothing, so the evidence it holds
    is its shipped data + the HR / NDCG / AUC lines of its result.txt: the drop-in `M7_main` path is trained on the shipped
    frappe.libfm with the reference defaults and its metrics are placed against those bands (scripts/reference_bands.py)."""
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import reference_bands as rb
    runs = [rb.run_one("M7", "frappe", 100 + s, epochs, K_FACTOR) for s in range(seeds)]
    out = rb.summarize("M7", "frappe", runs)
    return {"model": "OurModel7 (HHFM) via the drop-in M7_main path", "dataset": "frappe.libfm as shipped by the reference",
            "epochs": epochs, "seeds": seeds, "hr_at_5": out["mean"]["hr"], "ndcg_at_5": out["mean"]["ndcg"],
            "hr_at_10": out["mean"]["hr_at_10"], "ndcg_at_10": out["mean"]["ndcg_at_10"], "test_auc": out["mean"]["auc"],
            "reference_band": out["band"], "in_band": out["in_band"], "ok": out["ok"],
            "band_source": "result.txt:433-435,453-455,472,540-542,582-584,601-603,611-613,617-619,656-658 (HR@5 / NDCG@5 / AUC; "
                           "the reference logs no HR@10)", "train_s_per_run": float(np.mean([r["train_s"] for r in runs]))}


def e2e_epoch():
    """One reference-style epoch of the drop-in HHFM trainer on the shipped frappe file, sampler and batch assembly
    included (OurModel7.py:369-387; result.txt:431-435 logs 3.7-4.1 s per epoch for the reference), with the host sampler
    (the reference's numpy stream) and with the device sampler, next to the CPU port's epoch on the same batches."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import reference_bands as rb
    from hhfm_b200 import trainer
    from hhfm_b200.Newcode import OurModel7 as M7
    out = {"dataset": "frappe.libfm (shipped)", "reference_result_txt_epoch_s": "3.7-4.1 (result.txt:431-435, hardware unknown)"}
    os.environ.setdefault("HHFM_RESULT_FILE", os.devnull)
    sess = None
    saved_default = trainer.BaseTrain.device_sampler
    for name, dev_sampler in (("host_sampler", False), ("device_sampler", True)):
        trainer.BaseTrain.device_sampler = dev_sampler
        np.random.seed(1)
        args = M7.parse_args("frappe", K_FACTOR, 5, ["--path", rb.DATA, "--epoch", "2", "--Result", "2"])
        sess = M7.Train(args)
        sess.run_epoch()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            sess.run_epoch()
        torch.cuda.synchronize()
        out[name + "_epoch_s"] = (time.perf_counter() - t0) / 3
    trainer.BaseTrain.device_sampler = saved_default
    out["train_rows"] = int(len(sess.data.Train_data))
    out["samples_per_s_device_sampler"] = out["train_rows"] / out["device_sampler_epoch_s"]
    # CPU port: the same epoch (vectorised reference sampler + 18 steps of 5000) with the torch-CPU mirror
    from oracle import torch_cpu as T
    torch.set_num_threads(os.cpu_count() or 1)
    V = sess.model.weights["feature_embeddings"].cpu().clone()
    acc = torch.full_like(V, 0.1)
    t0 = time.perf_counter()
    pos = np.array(sess.data.Train_data.values[:, 1:])
    np.random.shuffle(pos)
    neg = sess.sample_negative(pos, 10)
    for c0 in range(0, len(pos), 5000):
        d = sess.split(pos[c0:c0 + 5000])
        T.hhfm_train_step(V, acc, torch.from_numpy(d["X"]), torch.from_numpy(np.array(neg[c0:c0 + 5000], dtype=np.int64)),
                          torch.from_numpy(d["F1"]), None, (0, 0, 0), LAMDA, LR)
    out["cpu_port_epoch_s"] = time.perf_counter() - t0
    out["cpu_port_note"] = "oracle/torch_cpu.py on %d threads with the vectorised sampler; restatement, not TF" % torch.get_num_threads()
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    from hhfm_b200 import _lib
    from hhfm_b200.engine import NO_HOT, Staging, cur_stream, pack_records, ptr
    from hhfm_b200.models import OUR

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    B = args.batch
    n_batches = 4
    rng = np.random.default_rng(1234 + rank)
    model = OUR(len(CTX_CARD), 0, FEATURES_M, N_USER, N_ITEM, K_FACTOR, LR, LAMDA, "AdagradOptimizer", True, False)
    if args.no_hot:
        model.hot_rows = None
    if world > 1:
        model.enable_data_parallel()
    host_batches = [make_batch(rng, B) for _ in range(n_batches)]
    # --dump-outputs: the seeded weights the last timed step restarts from (see the module docstring)
    V_seed = model.weights["feature_embeddings"].clone() if args.dump_outputs else None

    # device-resident records (the `value` arm): same packing as partial_fit, done once
    dev_batches = []
    stride = None
    for hb in host_batches:
        stg = Staging(torch.int32, dev)
        host, stride = pack_records([hb["X"], hb["F1"], hb["Y"]], FEATURES_M, stg)
        dev_batches.append(stg.upload(host.numel()).view(B, stride).clone())
    torch.cuda.synchronize()
    V = model.weights["feature_embeddings"]
    n_ctx = len(CTX_CARD)
    hot = model._hot_plan(dev_batches[0], False)
    hot_args = hot.args() if hot is not None else NO_HOT

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * (args.steps + 1))]

    def device_step(i, timed_idx=None):
        """OUR.fit_device (models.py) with CUDA events around its scatter kernel."""
        rec = dev_batches[i % n_batches]
        model._opt.begin_step()
        if timed_idx is not None:
            ev[2 * timed_idx].record()
        _lib.call("hhfm_pairrank_fwd_bwd", ptr(rec), B, stride, n_ctx, 0, NG, 0, 0, 0, ptr(V), FEATURES_M, K_FACTOR,
                  None, None, ptr(model._gV), ptr(model._loss_partials), None, 0, None, None, *hot_args, 0, cur_stream())
        if timed_idx is not None:
            ev[2 * timed_idx + 1].record()
        model._finish_step(hot, False)       # one kernel: replica fold + (N > 1: multimem all-reduce) + Adagrad + loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        device_step(i)
    barrier()
    try:
        uuid = str(torch.cuda.get_device_properties(local).uuid)
    except Exception:
        uuid = None
    sampler = ClockSampler(local, uuid)
    if rank == 0:
        sampler.start()                  # NVML init + thread start BEFORE the barrier: it must not delay rank 0's first step
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    calls0 = dict(_lib.CALLS)
    t_start.record()
    for i in range(args.steps):
        if V_seed is not None and i == args.steps - 1:
            model.weights["feature_embeddings"].copy_(V_seed)
            model._opt.slots("feature_embeddings", model.weights["feature_embeddings"])[0].fill_(model._opt.acc0)
        device_step(args.warmup + i, timed_idx=i)
    t_end.record()
    calls1 = dict(_lib.CALLS)
    if rank == 0:
        sampler.sample()                 # the queue is still draining here: at least one sample under load
    barrier()
    total_ms = t_start.elapsed_time(t_end)
    kern_ms = sum(ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(args.steps)) / args.steps
    loss_value = model._read_loss()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # what a caller of the timed step holds after its last step: that step's loss and the updated weights
        # (the replicas are bit-identical under data parallelism, so rank 0 speaks for all)
        outs = {"loss": np.array([loss_value], dtype=np.float32)}
        outs.update(model.get_weights())
        dump_outputs(args.dump_outputs, outs)
    # every timed entry point launches exactly one kernel (pairrank_sum_train_kernel, dp_step_kernel; without the fused
    # tail: hot_fold, opt_dense, loss_finalize)
    launches = sum(calls1.get(k, 0) - calls0.get(k, 0) for k in calls1)
    launch_names = sorted(k for k in calls1 if calls1.get(k, 0) != calls0.get(k, 0))

    # e2e arm: the user-facing call with host numpy batches (int64 ids as the reference feeds them)
    e2e_steps = 0 if args.quick else max(3, min(args.steps, 10))
    for i in range(0 if args.quick else 2):
        model.partial_fit(host_batches[i % n_batches])
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        model.partial_fit(host_batches[i % n_batches])
    barrier()
    e2e_s = max(time.perf_counter() - t0, 1e-9)
    # the same with one step in flight (`partial_fit_async`): every step still packs and copies its own host batch and its
    # loss still comes back to the host, but the loss of step i is waited for after step i+1 has been enqueued, so the host
    # packs batch i+1 while the GPU runs batch i
    e2e_pipe_s = None
    if e2e_steps:
        barrier()
        t0 = time.perf_counter()
        prev, acc_loss = None, 0.0
        for i in range(e2e_steps):
            h = model.partial_fit_async(host_batches[i % n_batches])
            if prev is not None:
                acc_loss += prev.result()
            prev = h
        acc_loss += prev.result()
        barrier()
        e2e_pipe_s = max(time.perf_counter() - t0, 1e-9)

    if world > 1:
        t = torch.tensor([total_ms, kern_ms, e2e_s, e2e_pipe_s or 0.0], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, kern_ms, e2e_s, e2e_pipe_s = [float(x) for x in t.tolist()]
    check = dp_check(model, dev_batches[0], n_ctx, world, dev) if world > 1 else None
    wire_bytes = int(_lib.load().hhfm_pack_upload_staging_bytes(B, stride, FEATURES_M))
    exchange = None
    if world > 1:
        exchange = ("fused dp_step_kernel over symmetric memory, " + ("multimem.ld_reduce/st" if model._dpx.multicast else
                    "peer loads/stores")) if model._dpx is not None else "NCCL all-reduce of the arena"

    # free the training buffers before the evaluator half of the metric
    del dev_batches, host_batches
    torch.cuda.empty_cache()
    topn = None if args.no_topn else run_topn(world, rank, dev, args.quick)
    topn_c5 = None if (args.no_topn or args.quick) else run_topn_c5(world, rank, dev)
    topn_c5_ctx = None if (args.no_topn or args.quick or world == 1) else run_topn_c5_ctx(world, rank, dev)
    models = None
    l2_peak = bands = epoch = None
    if world == 1 and not args.quick and not args.no_models:
        # the other BASELINE.json configs (device-resident batches, whole step): the scaled c5 lines are the HBM-bound ones
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import bench_models as bm
        margs = argparse.Namespace(steps=10)
        models = {}
        for name in ("hhfm_c5", "fm_c1", "fm_c5", "fm_c5_l2", "bpr_c4", "afm_c3", "dfm"):
            try:
                models[name] = bm.RUNNERS[name](margs, dev)
            except Exception as e:                      # a secondary line must not take the headline line down
                models[name] = {"error": repr(e)[:200]}
            torch.cuda.empty_cache()
    if rank == 0 and not args.quick:
        try:
            l2_peak = l2_read_peak(dev)
        except Exception as e:
            l2_peak = None
    if world == 1 and not args.quick and not args.no_bands:
        try:
            bands = parity_bands()
        except Exception as e:
            bands = {"error": repr(e)[:300]}
        try:
            epoch = e2e_epoch()
        except Exception as e:
            epoch = {"error": repr(e)[:300]}

    if rank == 0:
        hbm_peak, peak_src = measured_peaks()
        ms_per_step = total_ms / args.steps
        value = world * B * args.steps / (total_ms * 1e-3)
        achieved = B * ALGO_BYTES_PER_SAMPLE / (kern_ms * 1e-3) / 1e9
        traffic, capture = measured_traffic("pairrank_sum_train_kernel")
        cb = cpu_baseline() if (world == 1 and not args.quick) else None
        roof = {"bound": "l2", "kernel": "pairrank_sum_train_kernel<16,8,10>", "achieved": achieved, "peak": l2_peak,
                "unit": "GB/s", "frac": (achieved / l2_peak) if l2_peak else None, "traffic": traffic, "traffic_capture": capture,
                "peak_source": "hhfm_l2_read_sweep measured in this run (L1-bypassing 16-byte loads over an L2-resident 48 MB buffer)",
                "algorithmic_bytes_per_sample": ALGO_BYTES_PER_SAMPLE, "kernel_ms": kern_ms,
                "hbm": {"peak": hbm_peak, "peak_source": peak_src,
                        "frac_of_hbm_by_measured_traffic": (traffic / (kern_ms * 1e-3) / 1e9 / hbm_peak) if traffic else None},
                "note": "frappe shape: the 1.4 MB table and the hot-row replicas are L2 / L1 resident, only the 80 B record per "
                        "positive streams from HBM, so HBM does not bound this kernel; the 8016 algorithmic B/sample are served by "
                        "L1 (repeated context rows) and L2 (gathers, REDs) -- a fraction above 1 of the L2 sweep peak means L1 hits. "
                        "The HBM-bound evidence is `roofline_hbm` (the same model at the scaled c5 shape)."}
        line = {
            "metric": "hhfm_train_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(B, world),
            "e2e": {"value": world * B * e2e_steps / (e2e_pipe_s or e2e_s), "unit": "samples/s", "h2d_bytes_per_step": wire_bytes,
                    "d2h_bytes_per_step": 4, "steps": e2e_steps,
                    "api": "OUR.partial_fit_async(host int64 numpy batch), one step in flight: the loss of step i is read back "
                           "after step i+1 is enqueued (the drop-in trainers' epoch loop, hhfm_b200/trainer.py _PipelinedFit)",
                    "value_blocking_partial_fit": world * B * e2e_steps / e2e_s,
                    "note": "the host reads %d B of int64 ids per step and sends %d B of 16-bit wire records; every step copies "
                            "its own batch H2D and its loss D2H in both variants" % (B * 20 * 8, wire_bytes)},
            "gpu_launches": launches, "gpu_launch_entry_points": launch_names,
            "hot_rows": {"n_hot": hot.n_hot, "n_rep": hot.n_rep} if hot is not None else None,
            "roofline": roof, "clocks": clocks, "final_loss": loss_value,
        }
        if exchange is not None:
            line["dp_exchange"] = exchange
        if check is not None:
            line["dp_check"] = check
        if models is not None and isinstance(models.get("hhfm_c5"), dict) and "roofline" in models["hhfm_c5"]:
            line["roofline_hbm"] = dict(models["hhfm_c5"]["roofline"], config=models["hhfm_c5"]["config"])
        if topn is not None:
            line["topn"] = topn
        if topn_c5 is not None:
            line["topn_c5"] = topn_c5
        if topn_c5_ctx is not None:
            line["topn_c5_context_sharded"] = topn_c5_ctx
        if models is not None:
            line["models"] = models
        if bands is not None:
            line["parity_bands"] = bands
            if "hr_at_10" in bands:
                line["hr_at_10"] = bands["hr_at_10"]
        if epoch is not None:
            line["e2e_epoch"] = epoch
        if cb is not None:
            line["cpu_baseline"] = cb
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1 << 20, help="positives per GPU per step")
    ap.add_argument("--no-hot", dest="no_hot", action="store_true", help="disable the two-level hot-row scatter")
    ap.add_argument("--no-topn", dest="no_topn", action="store_true", help="skip the top-N half of the metric")
    ap.add_argument("--no-models", dest="no_models", action="store_true", help="skip the per-model secondary lines")
    ap.add_argument("--no-bands", dest="no_bands", action="store_true", help="skip the reference-band / epoch legs")
    ap.add_argument("--quick", action="store_true", help="profiling aid: skip the e2e and cpu_baseline legs")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's loss and the updated weights as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the timed GPU step computed; it needs --impl ours")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_ours(args)


if __name__ == "__main__":
    main()
