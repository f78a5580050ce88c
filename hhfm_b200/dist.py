"""torch.distributed plumbing for the two places the path exchanges data (SURVEY.md 8e):

  training   batch rows sharded across ranks; ONE all-reduce of the flat gradient arena per step
             ([gV | gbias | gb0 | loss partials], 1.4 MB at frappe shape), then every rank applies the identical update.
  evaluation item catalog sharded in contiguous id ranges; every rank scores all contexts against its items, keeps its
             local top-tp with GLOBAL ids, all-gather of [C, tp] (score, id), and a merge under the comparator
             (score desc, id asc) -- the lists are bit-identical to a single-GPU run.

`SymmExchange` is the training exchange on one NVLink box: every rank's exchange buffer lives in symmetric memory (mapped
into every peer, multicast-bound on NVSwitch) and ONE kernel per step folds, all-reduces (multimem.ld_reduce / multimem.st)
and applies the optimizer (csrc/p2p.cu).  `allreduce_arena` (NCCL / gloo) remains the fallback and what the CPU tests
exercise.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.distributed as dist


def world(group=None):
    if not dist.is_available() or not dist.is_initialized():
        return 0, 1
    return dist.get_rank(group), dist.get_world_size(group)


def shard_range(n, rank, world_size):
    """Contiguous, balanced [lo, hi) of n units for `rank` (sizes differ by at most one)."""
    base, rem = divmod(n, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def allreduce_arena(arena, group=None):
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(arena, op=dist.ReduceOp.SUM, group=group)
    return arena


def union_touched(stamp_arr, group=None):
    """Rows touched on any rank (TF1 SparseApplyMomentum over the global batch): every rank stamps the rows its shard touched
    with the step's stamp, which is the same on every rank and larger than any earlier one, so an element-wise MAX over the
    ranks carries the stamp exactly on the union.  One all-reduce of the int32 stamp array (4 B per row), in place; the
    arrays are identical on every rank afterwards."""
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(stamp_arr, op=dist.ReduceOp.MAX, group=group)
    return stamp_arr


def gather_candidates(local_scores, local_ids, group=None):
    """All-gather of the per-shard candidate lists: [C, tl] per rank -> [C, ws*tl] (rank order).  torch.distributed
    plumbing only (NCCL on the GPUs, gloo in the CPU tests)."""
    rank, ws = world(group)
    if ws == 1:
        return local_scores, local_ids
    sc = [torch.empty_like(local_scores) for _ in range(ws)]
    ids = [torch.empty_like(local_ids) for _ in range(ws)]
    dist.all_gather(sc, local_scores.contiguous(), group=group)
    dist.all_gather(ids, local_ids.contiguous(), group=group)
    return torch.cat(sc, dim=1), torch.cat(ids, dim=1)


def exchange_candidates_sharded(local_scores, local_ids, group=None):
    """All-to-all of the candidate lists with the CONTEXT rows sharded for the merge: rank r receives every rank's candidates
    for context rows [r*C/ws, (r+1)*C/ws) -> [C/ws, ws*tl].  Each rank receives C*tl candidates instead of the ws*C*tl of
    the all-gather.  C must be a multiple of the world size."""
    rank, ws = world(group)
    if ws == 1:
        return local_scores, local_ids
    C_rows, tl = local_scores.shape
    if C_rows % ws != 0:
        raise ValueError("exchange_candidates_sharded: %d context rows are not a multiple of the world size %d" % (C_rows, ws))
    per = C_rows // ws
    sc_in, id_in = local_scores.contiguous(), local_ids.contiguous()
    sc_out, id_out = torch.empty_like(sc_in), torch.empty_like(id_in)
    dist.all_to_all_single(sc_out, sc_in, group=group)          # block r of the output = rank r's candidates for my rows
    dist.all_to_all_single(id_out, id_in, group=group)
    return (sc_out.view(ws, per, tl).transpose(0, 1).reshape(per, ws * tl),
            id_out.view(ws, per, tl).transpose(0, 1).reshape(per, ws * tl))


def merge_topk(local_scores, local_ids, tp, group=None):
    """All-gather the per-shard candidate lists and keep the tp best per row under (score desc, id asc) with the device
    selector.  local_scores f32 [C, tp_local], local_ids int [C, tp_local] (global ids; -1 = padding), CUDA tensors."""
    if not local_scores.is_cuda:
        raise RuntimeError("merge_topk: candidates must be CUDA tensors (the selector is a device kernel; there is no CPU path)")
    scores, idx = gather_candidates(local_scores, local_ids, group)
    return _select_merged(scores, idx, tp)


def merge_topk_sharded(local_scores, local_ids, tp, group=None):
    """Item-sharded top-N merge that leaves the result sharded by context rows: one all-to-all
    (`exchange_candidates_sharded`), then rank r re-selects tp of the ws*tp candidates of ITS rows [r*C/ws, (r+1)*C/ws) --
    the HR / NDCG walk shards by context rows anyway (SURVEY.md 8e, `allreduce_metrics`).  Same lists, bit for bit, as
    `merge_topk` restricted to the slice."""
    if not local_scores.is_cuda:
        raise RuntimeError("merge_topk_sharded: candidates must be CUDA tensors")
    scores, idx = exchange_candidates_sharded(local_scores.float(), local_ids.to(torch.int32), group)
    return _select_merged(scores, idx, tp)


def _select_merged(scores, idx, tp):
    from . import _lib
    from .engine import cur_stream, ptr
    C_rows, n = scores.shape
    out_ids = torch.empty(C_rows, tp, dtype=torch.int32, device=scores.device)
    out_sc = torch.empty(C_rows, tp, dtype=torch.float32, device=scores.device)
    scores = scores.contiguous().float(); idx = idx.contiguous().to(torch.int32)
    # padding entries carry id -1: give them the lowest possible score so they sort last
    scores = torch.where(idx < 0, torch.full_like(scores, float("-inf")), scores)
    idx = torch.where(idx < 0, torch.full_like(idx, 2 ** 31 - 1), idx)
    _lib.call("hhfm_topn_select", ptr(scores), ptr(idx), None, C_rows, n, n, tp, 0, ptr(out_sc), ptr(out_ids), cur_stream())
    out_ids = torch.where(out_ids == 2 ** 31 - 1, torch.full_like(out_ids, -1), out_ids)
    return out_ids, out_sc


def gather_rows(t, group=None, sizes=None):
    """Concatenate per-rank row blocks of possibly different length (rank order).  `sizes`: the ranks' row counts when the
    caller knows them (e.g. `shard_range` shards) -- saves the size exchange and its host synchronisation; equal blocks then
    go through one all_gather_into_tensor straight into the result."""
    rank, ws = world(group)
    if ws == 1:
        return t
    if sizes is None:
        n = torch.tensor([t.shape[0]], dtype=torch.int64, device=t.device)
        got = [torch.zeros_like(n) for _ in range(ws)]
        dist.all_gather(got, n, group=group)
        sizes = [int(s.item()) for s in got]
    else:
        sizes = [int(x) for x in sizes]
        if len(sizes) != ws or sizes[rank] != t.shape[0]:
            raise ValueError("gather_rows: sizes %r do not describe this rank's block of %d rows" % (sizes, t.shape[0]))
    if min(sizes) == max(sizes) and hasattr(dist, "all_gather_into_tensor"):
        out = torch.empty((sizes[0] * ws,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(out, t.contiguous(), group=group)
        return out
    mx = max(sizes)
    pad = torch.zeros((mx,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    pad[:t.shape[0]] = t
    outs = [torch.empty_like(pad) for _ in range(ws)]
    dist.all_gather(outs, pad, group=group)
    return torch.cat([o[:s] for o, s in zip(outs, sizes)], dim=0)


class DpSegment(C.Structure):
    """hhfm_dp_segment (include/hhfm_sm100.h, K12)."""
    _fields_ = [("w", C.c_void_p), ("s1", C.c_void_p), ("s2", C.c_void_p), ("offset", C.c_int64), ("n", C.c_int64),
                ("lamda", C.c_float), ("reserved", C.c_int32)]


class SymmExchange:
    """The exchange buffer of the fused data-parallel step (csrc/p2p.cu): `n_floats` fp32 + a flag array per rank in
    SYMMETRIC memory -- same size on every rank, mapped into every peer of the box and, where the NVSwitch offers it,
    bound to one multicast object.  Allocation, handle exchange and mapping are torch.distributed plumbing
    (`torch.distributed._symmetric_memory`); what moves through the buffers is the kernel's business.

    x            this rank's buffer (float32 tensor, n_floats)
    x_table      host int64[ws]: address of every rank's buffer in this process (rank order, own one included)
    flag_table   host int64[ws]: address of every rank's flag array (hhfm_dp_flag_ints() int32, zero-initialised)
    multicast    address of the multicast alias of `x`, or 0
    """

    MAX_RANKS = 16

    def __init__(self, n_floats, device, group=None):
        import torch.distributed._symmetric_memory as symm
        self.rank, self.ws = world(group)
        if self.ws > self.MAX_RANKS:
            raise RuntimeError("SymmExchange: at most %d ranks" % self.MAX_RANKS)
        self.n = int(n_floats)
        from . import _lib
        self.FLAG_INTS = int(_lib.load().hhfm_dp_flag_ints())   # two phases x CTAs x ranks
        flag_off = (self.n + 63) // 64 * 64                     # flags start on a 256-byte boundary behind the floats
        total = flag_off + self.FLAG_INTS
        grp = group if group is not None else dist.group.WORLD
        self._buf = symm.empty(total, dtype=torch.float32, device=device)
        self._buf.zero_()
        torch.cuda.synchronize(device)
        self._hdl = symm.rendezvous(self._buf, grp.group_name)
        base = [int(p) for p in self._hdl.buffer_ptrs]
        off = int(self._buf.data_ptr()) - base[self.rank]        # the tensor's offset inside its allocation block
        if off < 0:
            raise RuntimeError("SymmExchange: tensor lies outside its symmetric block")
        self.x = self._buf[:self.n]
        self.x_table = (C.c_int64 * self.ws)(*[b + off for b in base])
        self.flag_table = (C.c_int64 * self.ws)(*[b + off + 4 * flag_off for b in base])
        mc = 0
        try:
            if bool(getattr(self._hdl, "has_multicast_support", False)):
                mc = int(self._hdl.multicast_ptr)
        except Exception:
            mc = 0
        self.multicast = (mc + off) if mc else 0
        dist.barrier(group=group)                                # every rank has zeroed its buffer before anyone signals

    def close(self):
        self._hdl = None
        self._buf = None
        self.x = None


def allreduce_metrics(codes, group=None):
    """HR / NDCG / reciprocal-rank over context rows sharded across ranks (SURVEY.md 8e): every rank walks its rows
    (rank codes from `engine.metrics_walk`: -2 row dropped, -1 miss, n >= 0 hit at rank n), the three sums and the count
    of contributing rows are all-reduced (the count varies per rank: FM.py:336-357 drops rows), then divided.
    float64 sums: identical to np.average over the concatenated rows up to summation order."""
    import numpy as np
    c = np.asarray(codes).reshape(-1)
    hit = c >= 0
    n = c[hit].astype(np.float64)
    local = torch.tensor([float(hit.sum()), float((np.log(2.0) / np.log(n + 2.0)).sum()), float((1.0 / (n + 1.0)).sum()),
                          float((c != -2).sum())], dtype=torch.float64)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        backend = dist.get_backend(group)
        t = local.cuda() if backend == "nccl" else local
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        local = t.cpu()
    cnt = float(local[3])
    if cnt == 0:
        return [float("nan")] * 3
    return [float(local[0]) / cnt, float(local[1]) / cnt, float(local[2]) / cnt]


def allgather_rows(ids, cols, group=None):
    """Coalesced-sparse exchange (SURVEY 8e): every rank contributes `ids` [n] (int32, unique) and per-row payloads
    `cols` = list of tensors with leading dimension n; returns, for every rank r in rank order, (ids_r, [payload_r, ...]).
    The counts differ between ranks, so the lists travel padded to the longest one (one host sync to learn the counts).
    Pure torch.distributed plumbing: works on gloo (CPU tests) and NCCL alike."""
    import torch.distributed as dist
    ws = dist.get_world_size(group)
    n = int(ids.shape[0])
    cnt = torch.tensor([n], dtype=torch.int64, device=ids.device)
    counts = [torch.zeros_like(cnt) for _ in range(ws)]
    dist.all_gather(counts, cnt, group=group)
    counts = [int(c.item()) for c in counts]
    maxc = max(counts)
    if maxc == 0:
        return [(ids[:0], [c[:0] for c in cols]) for _ in range(ws)]

    def gather(t, fill):
        pad = torch.full((maxc,) + tuple(t.shape[1:]), fill, dtype=t.dtype, device=t.device)
        pad[:n] = t
        outs = [torch.empty_like(pad) for _ in range(ws)]
        dist.all_gather(outs, pad, group=group)
        return outs

    g_ids = gather(ids, -1)
    g_cols = [gather(c, 0) for c in cols]
    return [(g_ids[r][:counts[r]], [g[r][:counts[r]] for g in g_cols]) for r in range(ws)]
