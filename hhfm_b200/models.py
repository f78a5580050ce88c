"""Model classes with the reference's `Newcode` API, running on libhhfm_sm100.so.

Each class keeps the reference constructor signature, `partial_fit(data) -> loss`, `topk(A, tp) -> int32[C,tp]`,
the `weights` dict and a minimal `sess.run(handle, feed_dict)` shim for what the reference `Train` classes
reach into (FM.py:313-319, OurModel7.py:441-455, BPR.py:247-252).  The TensorFlow graph + session of the
reference (`_init_graph`) is replaced by device tensors and C-ABI kernel launches; there is no CPU path.

  FM    Newcode/FM.py:59-198          MF   Newcode/MF.py:43-149
  OUR   Newcode/OurModel7.py:50-307   BPR  Newcode/BPR.py:45-136
  AFM   Newcode/AFM.py:63-246          DeepFM  Newcode/DFM.py:50-232
  CARS2 Newcode/CARS2.py:45-187        WD   Newcode/WDMF.py:51-126 (TF canned estimator restated; parity unpinned)
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

from . import _lib
from .engine import (NO_HOT, NO_HOT_BIAS, POOL_SUM, QUERY_FM, QUERY_HHFM, QUERY_USER, HotRows, Optimizer, PoolGroups,
                     RecordUploader, SingleTouchPlan, Staging, TopN, TouchTracker, cur_stream, pack_records, ptr, require_cuda)


class PendingLoss:
    """The loss of a step enqueued by `partial_fit_async`."""

    def __init__(self, model, slot, event):
        self._model, self._slot, self._event = model, slot, event

    def result(self):
        self._event.synchronize()
        m = self._model
        if m._dpx is not None and int(m._dp_state_host[1]) != 0:
            raise _lib.HhfmError("data-parallel step: a peer did not reach the cross-GPU barrier within HHFM_DP_TIMEOUT_S; "
                                 "the replicas are no longer in step (the CUDA context is intact)")
        return float(m._loss_ring[self._slot])


class Handle:
    """Stand-in for a tf.placeholder / graph tensor: only its identity matters (feed_dict key, fetch)."""

    def __init__(self, name):
        self.name = name

    def __repr__(self):
        return "<hhfm handle %s>" % self.name


class Session:
    """`model.sess` shim: `run(fetches, feed_dict)` dispatches to the owning model."""

    def __init__(self, model):
        self._model = model

    def run(self, fetches, feed_dict=None):
        return self._model._run(fetches, feed_dict or {})

    def close(self):
        pass


class _Base:
    """Shared device state: embedding table, gradient arena, loss partial buffers, staging, optimizer."""

    _supports_sparse_dp = False     # True where fit_device ends in _apply_table(sparse_ok=True) with touched-row tracking

    def _setup(self, features_M, K, seed, with_bias, optimizer_type, learning_rate, acc0, lamda):
        self.device = require_cuda()
        if K % 4 != 0 or K > 512:
            raise _lib.HhfmError("hidden_factor=%d unsupported: the sm_100a kernels need K %% 4 == 0 and K <= 512" % K)
        self._M, self._K = int(features_M), int(K)
        gen = torch.Generator(device="cpu")
        gen.manual_seed(int(seed))
        V = torch.empty(self._M, self._K, dtype=torch.float32).normal_(0.0, 0.01, generator=gen)
        self.weights = {"feature_embeddings": V.to(self.device)}          # FM.py:152-154
        if with_bias:
            self.weights["feature_bias"] = torch.zeros(self._M, 1, dtype=torch.float32, device=self.device)  # :155-156
        P = _lib.partials_len()
        self._P = P
        # one flat gradient arena so a data-parallel step needs a single exchange
        n_v = self._M * self._K
        n_b = self._M if with_bias else 0
        self._arena_layout = (n_v, n_b, P)
        self._with_bias_grad = with_bias
        self._dpx = None            # dist.SymmExchange once enable_data_parallel() mapped the peers
        self._fused = os.environ.get("HHFM_FUSED_STEP", "1") != "0"      # fold + exchange + optimizer + loss in one kernel
        self._dp_state = torch.zeros(4, dtype=torch.int32, device=self.device)      # [step counter, sticky error, -, -]
        self._dp_state_host = torch.zeros(4, dtype=torch.int32, pin_memory=True)
        self._reg_ws = torch.zeros(512, dtype=torch.float32, device=self.device)
        self._x_local = None
        self._segs = None
        # lazy-exact dense L2 (DESIGN.md 4): "auto" = tables of 96 MB and more with lamda > 0 on one GPU; True / False force it
        self.lazy_l2 = {"0": False, "1": True}.get(os.environ.get("HHFM_LAZY_L2", ""), "auto")
        self._last_step = None
        self._lazy_reg = None
        self._bind_arena(torch.zeros(n_v + n_b + 4 + P, dtype=torch.float32, device=self.device))
        self._sq_partials = torch.zeros(P, dtype=torch.float32, device=self.device)
        self._loss_dev = torch.zeros(1, dtype=torch.float32, device=self.device)
        self._loss_host = torch.zeros(1, dtype=torch.float32, pin_memory=True)
        self._opt = Optimizer(optimizer_type, learning_rate, initial_accumulator_value=acc0)
        self._lamda = float(lamda)
        self._touch = TouchTracker(self._M, self.device)
        self._idx_stage = Staging(torch.int32, self.device)
        self._uploader = RecordUploader(self.device)
        self._f32_stage = Staging(torch.float32, self.device)
        self._topn = TopN(self.device)
        self._dp_group = None
        self._dp_sparse = False
        self._version = 0           # bumped whenever the weights change (invalidates cached top-N item operands)
        self.topn_method = "auto"   # "auto" | "exact" | "tc"
        self.deterministic = False
        self.hot_rows = "auto"      # "auto": plan from the first batch; None: off; or an explicit id list
        self._hot = None
        self._hot_planned = False
        self.sess = Session(self)

    def _bind_arena(self, arena):
        """Point the gradient views at `arena` ([gV | gbias | gb0 (4) | loss partials])."""
        n_v, n_b, P = self._arena_layout
        self._arena = arena
        self._gV = arena[:n_v].view(self._M, self._K)
        self._gb = arena[n_v:n_v + n_b] if (n_b and self._with_bias_grad) else None
        self._gb0 = arena[n_v + n_b:n_v + n_b + 1]
        self._loss_local = arena[n_v + n_b + 1:n_v + n_b + 2]        # this rank's reduced loss (peer exchange)
        self._loss_partials = arena[n_v + n_b + 4:n_v + n_b + 4 + P]

    def _drop_args(self):
        """(keep, seed) of this step's dropout mask (FM.py:114 / MF.py:87; training only -- the reference evaluates with
        dropout_keep = 1).  Counter-based masks: the seed is a pure function of (random_seed, step), so a run is reproducible
        and the oracle can restate the mask; it is statistically TF's dropout, not its random stream."""
        keep = float(getattr(self, "keep", 1.0))
        if keep >= 1.0:
            return 1.0, 0
        return keep, self._drop_seed()

    def _drop_seed(self):
        seed = (int(getattr(self, "random_seed", 2016)) * 0x9E3779B97F4A7C15 + self._opt.t) & 0xFFFFFFFFFFFFFFFF
        self._last_drop_seed = seed
        return seed

    # ---- single-touch rows (include/hhfm_sm100.h K14) ---------------------------------------------------------------
    def _single_touch(self, ids_dev, n_cols, with_bias, keep=1.0):
        """The hhfm_single_touch plan of this step, or None.  Applicable when the staged (large-table) kernels run and the
        rows optimizer is one under which untouched rows stay put: lamda == 0, Adagrad / SGD, one GPU, no dropout; the
        reference counts of the step's ids are taken first (hhfm_count_refs)."""
        # OFF by default: measured at the c5 shapes (profiles/r2_single_touch_summary.md) the reference count pass (0.5 ms: 10^7
        # scattered 4-byte atomics run at the L2 atomic rate) and the 2 GB of extra traffic in the scatter kernel outweigh the
        # 0.9 ms the rows optimizer saves.  HHFM_SINGLE_TOUCH=auto: on for large tables, =1: on for every table size (tests).
        mode = os.environ.get("HHFM_SINGLE_TOUCH", "0")
        if mode not in ("1", "auto"):
            return None
        if (self._lamda > 0 or self._opt.kind not in ("adagrad", "sgd") or self._dp_group is not None or self.deterministic
                or keep < 1.0 or (mode != "1" and self._M * self._K * 4 < (96 << 20))):
            return None
        V = self.weights["feature_embeddings"]
        if getattr(self, "_ref_count", None) is None:
            self._ref_count = torch.empty(self._M, dtype=torch.int32, device=self.device)
        B, stride = ids_dev.shape
        _lib.call("hhfm_count_refs", ptr(ids_dev), B, stride, n_cols, self._M, ptr(self._ref_count), cur_stream())
        plan = SingleTouchPlan()
        plan.ref_count = ptr(self._ref_count)
        plan.V = ptr(V)
        plan.acc = ptr(self._opt.slots("feature_embeddings", V)[0]) if self._opt.kind == "adagrad" else None
        bias = self.weights.get("feature_bias") if with_bias else None
        if bias is not None:
            plan.bias = ptr(bias)
            plan.bias_acc = ptr(self._opt.slots("feature_bias", bias)[0]) if self._opt.kind == "adagrad" else None
        plan.lr = self._opt.lr
        plan.opt_kind = Optimizer.KIND_ID[self._opt.kind]
        return plan

    # ---- lazy-exact dense L2 -----------------------------------------------------------------------------------------
    def _lazy(self):
        """True when the dense L2 update of the table runs lazily: only the rows a batch gathers are brought up to date
        (replay of their missed `g = lamda*w` steps, bit-identical to the dense kernel) and updated; everything else waits
        for `flush()`.  Adagrad (the reference default), one GPU, lamda > 0."""
        if self._lamda <= 0 or self._opt.kind != "adagrad" or self._dp_group is not None:
            return False
        if self.lazy_l2 == "auto":
            return self._M * self._K * 4 >= (96 << 20)
        return bool(self.lazy_l2)

    def _lazy_prepare(self, ids_dev):
        """Before the forward of step t: the distinct rows of the batch -> touched list, replayed up to step t-1."""
        if self._last_step is None:
            self._last_step = torch.zeros(self._M, dtype=torch.int32, device=self.device)
        t = self._touch
        t.begin_step()
        flat = ids_dev.reshape(-1)
        st = cur_stream()
        _lib.call("hhfm_mark_rows", ptr(flat), flat.numel(), ptr(t.stamp_arr), t.stamp, self._M, ptr(t.rows), ptr(t.count), st)
        V = self.weights["feature_embeddings"]
        acc, _ = self._opt.slots("feature_embeddings", V)
        _lib.call("hhfm_opt_adagrad_l2_replay", ptr(V), ptr(acc), ptr(self._last_step), ptr(t.rows), ptr(t.count), self._M, self._M,
                  self._K, self._opt.lr, self._lamda, self._opt.t - 1, st)

    def _lazy_apply(self):
        """Step t on the gathered rows (g + lamda*w), stamped with t.  The regulariser term of the reported loss is the one of
        the last flush (the untouched rows are not materialised between flushes)."""
        t = self._touch
        V = self.weights["feature_embeddings"]
        acc, _ = self._opt.slots("feature_embeddings", V)
        _lib.call("hhfm_opt_adagrad_rows_l2", ptr(V), ptr(acc), ptr(self._gV), ptr(t.rows), ptr(t.count), self._M, self._K,
                  self._opt.lr, self._lamda, 1, ptr(self._last_step), self._opt.t, cur_stream())

    def flush(self):
        """Bring every row of the table to the current optimizer step (no-op outside the lazy mode).  Called by everything
        that reads the table: topk, predict / score_device, get_weights."""
        if self._last_step is None:
            return
        V = self.weights["feature_embeddings"]
        acc, _ = self._opt.slots("feature_embeddings", V)
        _lib.call("hhfm_opt_adagrad_l2_replay", ptr(V), ptr(acc), ptr(self._last_step), None, None, 0, self._M, self._K,
                  self._opt.lr, self._lamda, self._opt.t, cur_stream())
        self._lazy_reg = (0.5 * self._lamda) * V.square().sum(dtype=torch.float32)

    def _hot_plan(self, idx_dev, with_bias):
        """Hot-row plan for the two-level scatter (engine.HotRows), built once from the first batch."""
        if not self._hot_planned:
            self._hot_planned = True
            groups = self._pool_groups_plan(idx_dev)
            if self.hot_rows is None or self.deterministic:
                self._hot = None
            elif isinstance(self.hot_rows, str):
                exclude = torch.from_numpy(groups.member_rows()) if groups is not None else None
                self._hot = HotRows.from_batch(idx_dev, self._M, self._K, self.device, with_bias, exclude)
            else:
                self._hot = HotRows(self.hot_rows, self._M, self._K, self.device, with_bias)
        return self._hot

    def _pool_groups_plan(self, idx_dev):
        """Pooled context groups of the table (engine.PoolGroups), planned with the hot rows; None where not applicable."""
        return None

    # ---- data parallel (SURVEY.md 8e): batch rows sharded across ranks, one all-reduce of the arena ----
    def enable_data_parallel(self, group=None, fused="auto", sparse="auto", p2p=None):
        """Batch rows sharded across the ranks of `group`, weights replicated (SURVEY.md 8e).  On one NVLink box the gradient
        exchange is fused with the hot-replica fold, the optimizer and the loss reduction into ONE kernel over symmetric
        memory (dist.SymmExchange, csrc/p2p.cu: multimem.ld_reduce / multimem.st through the NVSwitch, peer loads / stores
        without multicast); `fused=False`, `HHFM_DP_FUSED=0`, a model with further dense variables (AFM, DeepFM) or a box
        where symmetric memory cannot be mapped use one NCCL all-reduce of the arena per step.  `p2p` is the old name of
        `fused`.

        `sparse`: exchange the COALESCED touched rows (row id + gradient row, all-gather) instead of the dense [M, K]
        gradient, then add the ranks' lists in rank order and run the touched-row optimizer on the union.  Only for
        lamda == 0 (IndexedSlices semantics; a dense L2 term touches every row anyway).  "auto": tables above 64 MB
        (SURVEY 8e); `HHFM_DP_SPARSE=0/1` forces either."""
        import torch.distributed as dist
        from . import dist as hd
        if not dist.is_initialized():
            raise RuntimeError("enable_data_parallel: torch.distributed is not initialised")
        if p2p is not None:
            fused = p2p
        self._dp_group = group if group is not None else dist.group.WORLD
        for w in self.weights.values():
            dist.broadcast(w, src=0, group=self._dp_group)
        self._version += 1           # the broadcast changed the weights: cached top-N item operands are stale
        self._dpx = None
        self._segs = None
        ws = dist.get_world_size(self._dp_group)
        env_s = os.environ.get("HHFM_DP_SPARSE")
        if env_s in ("0", "1"):
            sparse = env_s == "1"
        elif sparse == "auto":
            sparse = self._M * self._K * 4 > (64 << 20)
        self._dp_sparse = bool(sparse) and self._lamda <= 0 and ws > 1 and self._supports_sparse_dp
        if self._dp_sparse:
            if self._opt.kind == "momentum":
                raise NotImplementedError("sparse Momentum under data parallelism is not implemented")
            return
        env = os.environ.get("HHFM_DP_FUSED", os.environ.get("HHFM_DP_P2P"))      # 0 / 1 force NCCL / the fused exchange
        if env == "0":
            fused = False
        elif env == "1":
            fused = True
        want = bool(fused) and ws > 1 and self.device.type == "cuda" and self._fused_segments() is not None \
            and self._opt.kind != "momentum"
        if not want:
            if fused is True and ws > 1:
                raise _lib.HhfmError("enable_data_parallel: the fused exchange does not cover this model / optimizer")
            return
        # every phase that can fail on one rank only is followed by ONE all-reduce that agrees on the outcome, so the
        # ranks never sit in different collectives
        def agree(ok):
            flag = torch.tensor([1 if ok else 0], device=self.device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self._dp_group)
            return int(flag.item()) == 1

        dpx, err = None, None
        try:
            import torch.distributed._symmetric_memory  # noqa: F401  (phase 1: is the facility there at all)
        except Exception as e:                           # pragma: no cover
            err = e
        if agree(err is None):
            try:
                n_v, n_b, _ = self._arena_layout
                n_x = int(_lib.load().hhfm_dp_exchange_floats(n_v + n_b + 1))
                dpx = hd.SymmExchange(n_x, self.device, self._dp_group)      # collective (phase 2)
            except Exception as e:
                err = e
            if not agree(dpx is not None):
                if dpx is not None:
                    dpx.close()
                dpx = None
        if dpx is None:
            if fused is True:
                raise _lib.HhfmError("enable_data_parallel: symmetric memory is unavailable on this box (%r)" % (err,))
            return
        self._dpx = dpx
        self._dp_state.zero_()

    def _fused_segments(self):
        """[(name, weight, gradient offset in the arena, n, lamda)] of the variables the fused tail updates, or None when
        the model has dense variables outside the arena (AFM, DeepFM, WD)."""
        return None

    def _use_fused_tail(self):
        """The one-kernel tail (csrc/p2p.cu) replaces hot_fold + [all-reduce] + dense optimizer + loss_finalize whenever the
        dense optimizer kernels would run; the touched-row (IndexedSlices) path and Momentum keep their own kernels."""
        if not self._fused or self._fused_segments() is None or self._opt.kind == "momentum":
            return False
        if self._dp_group is not None:
            return self._dpx is not None
        return self._lamda > 0 and not self._lazy()

    def _fused_tail(self, hot, with_hot_bias):
        from . import dist as hd
        import ctypes as C
        if self._segs is None:
            segs = self._fused_segments()
            arr = (hd.DpSegment * len(segs))()
            keep = []
            for i, (name, w, off, n, lam) in enumerate(segs):
                s1, s2 = self._opt.slots(name, w)
                arr[i].w, arr[i].s1, arr[i].s2 = w.data_ptr(), (s1.data_ptr() if s1 is not None else None), \
                    (s2.data_ptr() if s2 is not None else None)
                arr[i].offset, arr[i].n, arr[i].lamda = int(off), int(n), float(lam)
                keep.append((w, s1, s2))
            self._segs = (arr, len(segs), keep)
        arr, n_seg, _ = self._segs
        n_v, n_b, _ = self._arena_layout
        n_g = n_v + n_b + 1
        o = self._opt
        lr = o._lr_t() if o.kind == "adam" else o.lr
        dpx = self._dpx
        if dpx is None:
            if self._x_local is None:
                self._x_local = torch.zeros(int(_lib.load().hhfm_dp_exchange_floats(n_g)), dtype=torch.float32, device=self.device)
            x, mc, xt, ft, rank, ws = self._x_local, None, None, None, 0, 1
        else:
            x, mc, xt, ft, rank, ws = dpx.x, (C.c_void_p(dpx.multicast) if dpx.multicast else None), dpx.x_table, dpx.flag_table, \
                dpx.rank, dpx.ws
        if hot is not None:
            hargs = (ptr(hot.ghot), ptr(hot.ghot_bias) if with_hot_bias else None, hot.n_rep, hot.n_hot, self._K, self._M,
                     ptr(hot.slot), n_v)
        else:
            hargs = (None, None, 0, 0, self._K, self._M, None, n_v)
        _lib.call("hhfm_dp_step", o.KIND_ID[o.kind], C.cast(arr, C.c_void_p), n_seg, ptr(self._arena), n_g, *hargs,
                  ptr(self._loss_partials), ptr(x), mc, xt, ft, rank, ws, ptr(self._dp_state), lr, o.beta1, o.beta2, o.eps,
                  ptr(self._reg_ws), ptr(self._loss_dev), float(os.environ.get("HHFM_DP_TIMEOUT_S", "120")), cur_stream())
        self._version += 1

    def _finish_step(self, hot, with_hot_bias, bias_step=None):
        """Everything after the scatter kernels of a step: fold, exchange, optimizer, loss."""
        if self._lazy():
            if hot:
                hot.fold(self._gV, self._gb if with_hot_bias else None)
            self._lazy_apply()
            if bias_step is not None:
                bias_step()
            self._enqueue_loss(False)
            if self._lazy_reg is not None:
                self._loss_dev += self._lazy_reg
            return
        if self._use_fused_tail():
            self._fused_tail(hot, with_hot_bias)
            return
        if hot:
            hot.fold(self._gV, self._gb if with_hot_bias else None)
        self._allreduce_grads()
        with_reg = self._apply_table(sparse_ok=True)
        if bias_step is not None:
            bias_step()
        self._enqueue_loss(with_reg)

    def _allreduce_grads(self):
        """NCCL path: one all-reduce of the arena (dense) or the coalesced-sparse row exchange."""
        if self._dp_group is None:
            return
        if self._dp_sparse:
            self._exchange_sparse_rows()
            return
        import torch.distributed as dist
        dist.all_reduce(self._arena, group=self._dp_group)

    def _exchange_sparse_rows(self):
        """SURVEY 8e, tables too large for a dense all-reduce: all-gather the coalesced (row id, gradient row) lists, clear
        the local rows, add every rank's list (own one included) in rank order -- each row then holds the same fp32 sum on
        every rank, so the replicas stay bit-identical -- and extend the touched-row list to the union for the optimizer.
        The small dense tail of the arena (scalar bias gradient, loss partials) is all-reduced."""
        import torch.distributed as dist
        from . import dist as hd
        t = self._touch
        n = int(t.count.item())
        ids = t.rows[:n]
        st = cur_stream()
        rows = torch.empty(n, self._K, dtype=torch.float32, device=self.device)
        _lib.call("hhfm_gather_rows", ptr(self._gV), ptr(ids), n, self._K, self._M, ptr(rows), 1, st)
        cols = [rows]
        if self._with_bias_grad:
            gb = torch.empty(n, dtype=torch.float32, device=self.device)
            _lib.call("hhfm_gather_rows", ptr(self._gb), ptr(ids), n, 1, self._M, ptr(gb), 1, st)
            cols.append(gb)
        for ids_r, cols_r in hd.allgather_rows(ids, cols, self._dp_group):
            m = int(ids_r.shape[0])
            if m == 0:
                continue
            ids_r = ids_r.contiguous()
            _lib.call("hhfm_scatter_add_rows", ptr(ids_r), ptr(cols_r[0].contiguous()), m, self._K, ptr(self._gV), self._M, st)
            if self._with_bias_grad:
                _lib.call("hhfm_scatter_add_rows", ptr(ids_r), ptr(cols_r[1].contiguous()), m, 1, ptr(self._gb), self._M, st)
            _lib.call("hhfm_touch_rows", ptr(ids_r), m, ptr(t.stamp_arr), t.stamp, ptr(t.rows), ptr(t.count), st)
        n_v, n_b, _ = self._arena_layout
        dist.all_reduce(self._arena[n_v + n_b:], group=self._dp_group)

    def _apply_arena_dense(self, name, w, g, lamda, sq):
        """Dense optimizer step for a tensor whose gradient `g` is a slice of the arena."""
        self._opt.apply_dense(name, w, g, lamda, sq)

    def enable_item_sharding(self, group=None):
        """Full-catalog top-N with the item catalog sharded across the ranks of `group` (SURVEY.md 8e): every rank
        scores all contexts against its contiguous item range, then the candidates are all-gathered and merged."""
        import torch.distributed as dist
        if not dist.is_initialized():
            raise RuntimeError("enable_item_sharding: torch.distributed is not initialised")
        self._eval_group = group if group is not None else dist.group.WORLD

    def enable_context_sharding(self, group=None):
        """Full-catalog top-N with the CONTEXT rows sharded across the ranks of `group`: rank r scores rows
        shard_range(C, r, ws) against the WHOLE catalog and the lists are concatenated in rank order.  This is the
        evaluator's decomposition whenever the table is replicated (it is under data-parallel training): no candidate
        exchange, no merge, and the per-row work (rescoring, selection) shards with the rows -- strong scaling is the row
        split.  Item sharding (`enable_item_sharding`) is for catalogs that do not fit one GPU.  Lists are bit-identical."""
        import torch.distributed as dist
        if not dist.is_initialized():
            raise RuntimeError("enable_context_sharding: torch.distributed is not initialised")
        if getattr(self, "_eval_group", None) is not None:
            raise RuntimeError("enable_context_sharding: item sharding is already enabled on this model")
        self._eval_ctx_group = group if group is not None else dist.group.WORLD

    def _topk(self, kind, A, n_ctx, n_time, pools, bias, tp):
        from . import dist as hd
        A = np.asarray(A)
        self.flush()
        cgrp = getattr(self, "_eval_ctx_group", None)
        if cgrp is not None:
            rank, ws = hd.world(cgrp)
            lo, hi = hd.shard_range(A.shape[0], rank, ws)
            V = self.weights["feature_embeddings"]
            if hi > lo:
                A_dev, stride = self._topn.upload_rows(A[lo:hi], self._M)
                ids = self._topn.topk(kind, A_dev, stride, n_ctx, n_time, pools, V, bias, self.n_user, self.n_item, tp,
                                      method=self.topn_method, version=self._version)
            else:
                ids = torch.empty(0, tp, dtype=torch.int32, device=V.device)
            sizes = [hd.shard_range(A.shape[0], r, ws)[1] - hd.shard_range(A.shape[0], r, ws)[0] for r in range(ws)]
            return hd.gather_rows(ids, cgrp, sizes).cpu().numpy()
        A_dev, stride = self._topn.upload_rows(A, self._M)
        V = self.weights["feature_embeddings"]
        grp = getattr(self, "_eval_group", None)
        if grp is None:
            ids = self._topn.topk(kind, A_dev, stride, n_ctx, n_time, pools, V, bias, self.n_user, self.n_item, tp,
                                  method=self.topn_method, version=self._version)
            return ids.cpu().numpy()
        rank, ws = hd.world(grp)
        lo, hi = hd.shard_range(self.n_item, rank, ws)
        ids, sc = self._topn.topk(kind, A_dev, stride, n_ctx, n_time, pools, V, bias, self.n_user, self.n_item, tp,
                                  item_lo=lo, item_hi=hi, return_scores=True, method=self.topn_method,
                                  version=self._version)
        ids, _ = hd.merge_topk(sc, ids, tp, grp)
        return ids.cpu().numpy()

    def _touch_args(self, extra=False):
        """Touched-row tracking is only paid for when a *_rows optimizer will consume the list."""
        need = (self._dp_group is None or self._dp_sparse) and (self._lamda <= 0 or extra)
        if not need or self._lazy():            # lazy mode: the list was built from the ids before the forward
            return (None, 0, None, None)
        self._touch.begin_step()
        return (ptr(self._touch.stamp_arr), self._touch.stamp, ptr(self._touch.rows), ptr(self._touch.count))

    # ---- optimizer step on the embedding table (+ optional bias rows) ----
    def _apply_table(self, sparse_ok):
        """lamda > 0: aggregated dense gradient g + lamda*V over all rows (FM.py:124 regulariser).
        lamda == 0: IndexedSlices semantics; Adagrad/SGD/Adam dense kernels are exactly equivalent on untouched
        rows (g = 0), Momentum needs the touched-row list."""
        V = self.weights["feature_embeddings"]
        use_rows = sparse_ok and self._lamda <= 0 and (self._dp_group is None or self._dp_sparse)
        if use_rows:
            self._opt.apply_rows("feature_embeddings", V, self._gV, self._touch.rows, self._touch.count, self._K)
            return False
        if self._lamda <= 0 and self._opt.kind == "momentum":
            raise NotImplementedError("sparse Momentum under data parallelism is not implemented")
        sq = self._sq_partials if self._lamda > 0 else None
        self._apply_arena_dense("feature_embeddings", V, self._gV, self._lamda if self._lamda > 0 else 0.0, sq)
        return self._lamda > 0

    def _enqueue_loss(self, with_reg, half_lamda=None):
        """Deterministic reduction of the per-CTA loss partials (+ regulariser) into `_loss_dev`; no host sync.  Under data
        parallelism the partials were all-reduced with the arena, so the loss is the sum over all ranks (the reference loss
        is a sum over the batch, FM.py:124)."""
        self._version += 1
        hl = (0.5 * self._lamda) if half_lamda is None else half_lamda
        sq = ptr(self._sq_partials) if with_reg else None
        _lib.call("hhfm_loss_finalize", ptr(self._loss_partials), sq, hl if with_reg else 0.0, ptr(self._loss_dev),
                  cur_stream())

    def partial_fit_async(self, data):
        """`partial_fit` without the wait: the step (host packing, H2D copy, kernels, D2H copy of the loss into a pinned slot)
        is enqueued and a `PendingLoss` comes back; `.result()` waits for that step alone and returns the float that
        `partial_fit` would have returned.  Keeping one step in flight lets the host pack batch i+1 while the GPU runs batch i
        (the reference's loop only sums the losses of an epoch, FM.py:251-256).  At most 4 results may be outstanding."""
        self._defer_loss = True
        try:
            return self.partial_fit(data)
        finally:
            self._defer_loss = False

    def _read_loss(self):
        if getattr(self, "_defer_loss", False):
            if getattr(self, "_loss_ring", None) is None:
                self._loss_ring = torch.empty(4, dtype=torch.float32, pin_memory=True)
                self._loss_ring_n = 0
            slot = self._loss_ring_n % 4
            self._loss_ring_n += 1
            self._loss_ring[slot:slot + 1].copy_(self._loss_dev, non_blocking=True)
            if self._dpx is not None:
                self._dp_state_host.copy_(self._dp_state, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            return PendingLoss(self, slot, ev)
        self._loss_host.copy_(self._loss_dev, non_blocking=True)
        if self._dpx is not None:
            self._dp_state_host.copy_(self._dp_state, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        if self._dpx is not None and int(self._dp_state_host[1]) != 0:
            raise _lib.HhfmError("data-parallel step: a peer did not reach the cross-GPU barrier within HHFM_DP_TIMEOUT_S; "
                                 "the replicas are no longer in step (the CUDA context is intact)")
        return float(self._loss_host[0])

    def _upload_rows(self, X):
        return self._uploader.upload([np.asarray(X)], self._M, align=1)[0]

    def _upload_ids(self, parts):
        return self._uploader.upload(parts, self._M)

    def _upload_f32(self, arr):
        arr = np.ascontiguousarray(np.asarray(arr, dtype=np.float32).reshape(-1))
        host = self._f32_stage.ensure(arr.size)
        host.copy_(torch.from_numpy(arr))
        return self._f32_stage.upload(arr.size)

    def load_weights(self, weights):
        """Inject weights (numpy arrays or tensors keyed like `self.weights`) -- parity tests use this because
        the reference initialises unseeded (FM.py:153)."""
        for k, v in weights.items():
            if k not in self.weights:
                raise KeyError(k)
            t = torch.as_tensor(np.asarray(v, dtype=np.float32)).reshape(self.weights[k].shape)
            self.weights[k].copy_(t.to(self.device))
        self._version += 1
        if self._last_step is not None:
            self._last_step.fill_(self._opt.t)       # injected weights are current as of this step

    def get_weights(self):
        self.flush()
        return {k: v.detach().cpu().numpy().copy() for k, v in self.weights.items()}

    def invalidate(self):
        """Call after editing `model.weights[...]` in place: cached top-N item operands are keyed on the weight version."""
        self._version += 1


# ====================================================================================================
class FM(_Base):
    """Factorization machine, Newcode/FM.py:59-198."""

    _supports_sparse_dp = True

    interaction = 0
    _bn = False
    BN_EPS, BN_DECAY = 1e-3, 0.9          # batch_norm_layer: decay=0.9, epsilon left at the tf.contrib.layers.batch_norm default

    def __init__(self, valid_dimension, features_M, n_user, n_item, hidden_factor, learning_rate, lamda_bilinear, keep,
                 optimizer_type, batch_norm, verbose, random_seed=2016):
        self.valid_dimension = valid_dimension
        self.n_user = n_user
        self.n_item = n_item
        self.learning_rate = learning_rate
        self.hidden_factor = hidden_factor
        self.features_M = features_M
        self.lamda_bilinear = lamda_bilinear
        self.keep = keep
        self.random_seed = random_seed
        self.optimizer_type = optimizer_type
        self.batch_norm = batch_norm
        self.verbose = verbose
        self.train_rmse, self.valid_rmse, self.test_rmse = [], [], []
        self._init_graph()

    def _init_graph(self):
        if not (0.0 < float(self.keep) <= 1.0):
            raise ValueError("keep must be in (0, 1]")
        self.train_features = Handle("train_features_fm")    # FM.py:89-92
        self.train_labels = Handle("train_labels_fm")
        self.dropout_keep = Handle("dropout_keep_fm")
        self.train_phase = Handle("train_phase_fm")
        self.out = Handle("out")
        self.loss = Handle("loss")
        self.optimizer = Handle("optimizer")
        self._setup(self.features_M, self.hidden_factor, self.random_seed, True, self.optimizer_type,
                    self.learning_rate, 0.1, self.lamda_bilinear)
        self._b0 = torch.zeros(1, dtype=torch.float32, device=self.device)
        self.weights["bias"] = self._b0.view(())                                   # FM.py:157
        self._bn = bool(self.batch_norm)
        if self._bn:
            # FM.py:111-112 batch_norm_layer(scope='bn_fm'): scale gamma = 1, offset beta = 0, moving mean 0, moving variance 1
            K, dev = self._K, self.device
            self.weights["bn_fm/gamma"] = torch.ones(K, dtype=torch.float32, device=dev)
            self.weights["bn_fm/beta"] = torch.zeros(K, dtype=torch.float32, device=dev)
            self.weights["bn_fm/moving_mean"] = torch.zeros(K, dtype=torch.float32, device=dev)
            self.weights["bn_fm/moving_variance"] = torch.ones(K, dtype=torch.float32, device=dev)
            self._g_bn = torch.zeros(2, K, dtype=torch.float32, device=dev)         # d gamma, d beta
            self._bn_ws = None

    def enable_data_parallel(self, *args, **kwargs):
        if self._bn:
            raise NotImplementedError("batch_norm=1 under data parallelism: per-rank batch statistics are not the single-GPU "
                                      "step, and global statistics need two more collectives per step")
        return super().enable_data_parallel(*args, **kwargs)

    def _bn_args(self):
        w = self.weights
        return (ptr(w["bn_fm/gamma"]), ptr(w["bn_fm/beta"]), ptr(w["bn_fm/moving_mean"]), ptr(w["bn_fm/moving_variance"]))

    # -- forward only: `sess.run(model.out, ...)` of evaluate_AUC (FM.py:313-319) --
    def score_device(self, idx):
        """Scores [n] (device) for device-resident id rows idx int32 [n, F]."""
        self.flush()
        B, F = idx.shape
        out = torch.empty(B, dtype=torch.float32, device=self.device)
        if self._bn:                  # train_phase=False: the moving statistics (FM.py:111, is_training=train_phase)
            _lib.call("hhfm_fm_bn_fwd", ptr(idx), B, F, ptr(self.weights["feature_embeddings"]), ptr(self.weights["feature_bias"]),
                      ptr(self._b0), self._M, self._K, *self._bn_args(), self.BN_EPS, ptr(out), cur_stream())
            return out
        _lib.call("hhfm_fm_fwd", None, ptr(idx), None, B, F, ptr(self.weights["feature_embeddings"]),
                  ptr(self.weights.get("feature_bias")), ptr(self._b0), self._M, self._K, self.interaction, ptr(out),
                  cur_stream())
        return out

    def predict(self, X):
        return self.score_device(self._upload_rows(np.asarray(X))).cpu().numpy().reshape(-1, 1)

    def partial_fit(self, data):
        """One minibatch step (FM.py:168-171): forward, squared loss, backward, optimizer.  Returns the loss."""
        idx = self._upload_rows(data["X"])
        y = self._upload_f32(data["Y"])
        self.fit_device(idx, y)
        return self._read_loss()

    def fit_device(self, idx, y):
        """The step on device-resident inputs (idx int32 [B,F], y fp32 [B]); everything is enqueued on the current
        stream and nothing synchronises -- `partial_fit` = upload + fit_device + loss read-back."""
        B, F = idx.shape
        self._opt.begin_step()
        V = self.weights["feature_embeddings"]
        bias = self.weights.get("feature_bias")
        if self._lazy():
            self._lazy_prepare(idx)
        ts, stamp, tr, tc = self._touch_args(extra=self._opt.kind == "momentum")
        hot = self._hot_plan(idx, True)
        keep, dseed = self._drop_args()
        if self._bn:
            self._fit_bn(idx, y, ts, stamp, tr, tc, hot, keep, dseed)
            return
        plan = self._single_touch(idx, F, True, keep) if ts is not None else None
        _lib.call("hhfm_fm_fwd_bwd_sqloss_st", None, ptr(idx), None, B, F, ptr(V), ptr(bias), ptr(self._b0), self._M,
                  self._K, self.interaction, ptr(y), None, ptr(self._gV), ptr(self._gb), ptr(self._gb0),
                  ptr(self._loss_partials), ts, stamp, tr, tc, *(hot.args(True) if hot else NO_HOT_BIAS),
                  1 if self.deterministic else 0, keep, dseed, C.addressof(plan) if plan is not None else None, cur_stream())
        self._finish_step(hot, True, self._apply_bias if bias is not None else None)

    def _fit_bn(self, idx, y, ts, stamp, tr, tc, hot, keep, dseed):
        """The step with batch normalisation (csrc/fm_bn.cu): V, feature_bias and the scalar bias go through the usual tail;
        gamma and beta are dense variables without L2, stepped after it.  Single-touch rows (K14) stay off."""
        B, F = idx.shape
        nbytes = int(_lib.load().hhfm_workspace_bytes_fm_bn(B, self._K))
        if self._bn_ws is None or self._bn_ws.numel() < nbytes:
            self._bn_ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        V = self.weights["feature_embeddings"]
        _lib.call("hhfm_fm_bn_fwd_bwd_sqloss", None, ptr(idx), None, B, F, ptr(V), ptr(self.weights["feature_bias"]), ptr(self._b0),
                  self._M, self._K, 0, ptr(y), None, ptr(self._gV), ptr(self._gb), ptr(self._gb0), ptr(self._loss_partials),
                  ts, stamp, tr, tc, *(hot.args(True) if hot else NO_HOT_BIAS), 1 if self.deterministic else 0, keep, dseed,
                  *self._bn_args(), ptr(self._g_bn[0]), ptr(self._g_bn[1]), self.BN_EPS, self.BN_DECAY, ptr(self._bn_ws),
                  self._bn_ws.numel(), cur_stream())
        self._finish_step(hot, True, self._apply_bias)
        self._opt.apply_dense("bn_fm/gamma", self.weights["bn_fm/gamma"], self._g_bn[0], 0.0, None)
        self._opt.apply_dense("bn_fm/beta", self.weights["bn_fm/beta"], self._g_bn[1], 0.0, None)

    def _fused_segments(self):
        n_v, n_b, _ = self._arena_layout
        segs = [("feature_embeddings", self.weights["feature_embeddings"], 0, n_v, self._lamda if self._lamda > 0 else 0.0)]
        if self._with_bias_grad and n_b:
            # feature_bias receives IndexedSlices; for Adagrad / SGD rows with g = 0 do not move and TF1's sparse Adam
            # moves every row, so the dense update is exact for the optimizers the fused tail covers
            segs.append(("feature_bias", self.weights["feature_bias"], n_v, n_b, 0.0))
        if getattr(self, "_b0", None) is not None:
            segs.append(("bias", self._b0, n_v + n_b, 1, 0.0))
        return segs

    def _apply_bias(self):
        # feature_bias receives IndexedSlices (only touched rows move); the scalar bias is dense.
        bias = self.weights["feature_bias"]
        if self._opt.kind == "momentum":
            if self._dp_group is not None:
                raise NotImplementedError("sparse Momentum under data parallelism is not implemented")
            self._opt.apply_rows("feature_bias", bias, self._gb, self._touch.rows, self._touch.count, 1)
        else:
            self._apply_arena_dense("feature_bias", bias, self._gb, 0.0, None)
        self._apply_arena_dense("bias", self._b0, self._gb0, 0.0, None)

    def topk(self, A, tp):
        """Full-catalog top-N (FM.py:172-185): indices relative to the item id range."""
        A = np.asarray(A)
        return self._topk(QUERY_FM, A, A.shape[1] - 2, 0, (0, 0, 0), self.weights["feature_bias"], tp)

    def _run(self, fetches, feed):
        if fetches is self.out:
            return self.predict(feed[self.train_features])
        if isinstance(fetches, (tuple, list)) and len(fetches) == 2 and fetches[0] is self.loss:
            loss = self.partial_fit({"X": feed[self.train_features], "Y": feed[self.train_labels]})
            return loss, None
        raise NotImplementedError("sess.run: unsupported fetch %r" % (fetches,))


# ====================================================================================================
class MF(FM):
    """Pointwise matrix factorisation, Newcode/MF.py:43-149: out = sum_k V[u]*V[i] (the bias term is computed but
    not added, MF.py:91-92); Adagrad accumulator starts at 1e-8 (MF.py:104); topk retrieves 100 (MF.py:147)."""

    interaction = 1

    def __init__(self, features_M, n_user, n_item, hidden_factor, learning_rate, lamda_bilinear, keep, optimizer_type,
                 batch_norm, verbose, random_seed=2016):
        self.n_user = n_user
        self.n_item = n_item
        self.learning_rate = learning_rate
        self.hidden_factor = hidden_factor
        self.features_M = features_M
        self.lamda_bilinear = lamda_bilinear
        self.keep = keep
        self.random_seed = random_seed
        self.optimizer_type = optimizer_type
        self.batch_norm = batch_norm
        self.verbose = verbose
        self.train_rmse, self.valid_rmse, self.test_rmse = [], [], []
        self._init_graph()

    def _init_graph(self):
        if self.batch_norm:
            raise NotImplementedError("batch_norm=1 is not on the accelerated path")
        if not (0.0 < float(self.keep) <= 1.0):
            raise ValueError("keep must be in (0, 1]")
        self.train_features = Handle("train_features_fm")
        self.train_labels = Handle("train_labels_fm")
        self.dropout_keep = Handle("dropout_keep_fm")
        self.train_phase = Handle("train_phase_fm")
        self.out = Handle("out")
        self.loss = Handle("loss")
        self.optimizer = Handle("optimizer")
        self._setup(self.features_M, self.hidden_factor, self.random_seed, True, self.optimizer_type,
                    self.learning_rate, 1e-8, self.lamda_bilinear)
        self._b0 = None

    def score_device(self, idx):
        self.flush()
        B = idx.shape[0]
        idx2 = idx[:, :2].contiguous() if idx.shape[1] != 2 else idx
        out = torch.empty(B, dtype=torch.float32, device=self.device)
        _lib.call("hhfm_fm_fwd", None, ptr(idx2), None, B, 2, ptr(self.weights["feature_embeddings"]), None, None,
                  self._M, self._K, 1, ptr(out), cur_stream())
        return out

    def predict(self, X):
        return self.score_device(self._upload_rows(np.asarray(X)[:, :2])).cpu().numpy().reshape(-1, 1)

    def partial_fit(self, data):
        idx = self._upload_rows(np.asarray(data["X"])[:, :2])
        y = self._upload_f32(data["Y"])
        self.fit_device(idx, y)
        return self._read_loss()

    def fit_device(self, idx, y):
        B = idx.shape[0]
        self._opt.begin_step()
        V = self.weights["feature_embeddings"]
        if self._lazy():
            self._lazy_prepare(idx)
        ts, stamp, tr, tc = self._touch_args()
        hot = self._hot_plan(idx, False)
        keep, dseed = self._drop_args()
        _lib.call("hhfm_fm_fwd_bwd_sqloss_dropout", None, ptr(idx), None, B, 2, ptr(V), None, None, self._M, self._K, 1, ptr(y),
                  None, ptr(self._gV), None, None, ptr(self._loss_partials), ts, stamp, tr, tc,
                  *(hot.args(True) if hot else NO_HOT_BIAS), 1 if self.deterministic else 0, keep, dseed, cur_stream())
        self._finish_step(hot, False)

    def _fused_segments(self):
        n_v = self._arena_layout[0]
        return [("feature_embeddings", self.weights["feature_embeddings"], 0, n_v, self._lamda if self._lamda > 0 else 0.0)]

    def topk(self, A, tp=100):
        """MF.py:144-149: top-100 items per row of A by u . v (the rows may carry context columns; the table holds users and
        items only, MF.py:171)."""
        return self._topk(QUERY_USER, np.asarray(A)[:, :2], 0, 0, (0, 0, 0), None, tp)


# ====================================================================================================
class _PairRank(_Base):
    """Shared HHFM / BPR machinery: record packing, fused forward+backward kernel, scoring, top-N."""

    _supports_sparse_dp = True

    def _groups(self):
        raise NotImplementedError

    def _fit_records(self, parts, n_ctx, n_time, n_neg):
        idx, stride = self._upload_ids(parts)
        self.fit_device(idx, n_ctx, n_time, n_neg)
        return self._read_loss()

    def fit_device(self, idx, n_ctx, n_time, n_neg):
        """The step on device-resident records (int32 [B,stride], layout: include/hhfm_sm100.h K3); no host sync."""
        B, stride = idx.shape
        self._opt.begin_step()
        V = self.weights["feature_embeddings"]
        pc, pt, pf = self.pools
        if self._lazy():
            self._lazy_prepare(idx)                  # padding ids (-1) are skipped
        ts, stamp, tr, tc = self._touch_args()
        hot = self._hot_plan(idx, False)
        plan = self._single_touch(idx, 2 + n_ctx + n_time + n_neg, False) if ts is not None else None
        _lib.call("hhfm_pairrank_fwd_bwd_st", ptr(idx), B, stride, n_ctx, n_time, n_neg, pc, pt, pf, ptr(V), self._M,
                  self._K, None, None, ptr(self._gV), ptr(self._loss_partials), ts, stamp, tr, tc,
                  *(hot.args() if hot else NO_HOT), 1 if self.deterministic else 0,
                  C.addressof(plan) if plan is not None else None, cur_stream())
        self._finish_step(hot, False)

    def _fused_segments(self):
        n_v = self._arena_layout[0]
        return [("feature_embeddings", self.weights["feature_embeddings"], 0, n_v, self._lamda if self._lamda > 0 else 0.0)]

    def _positive_feedback(self, parts, n_ctx, n_time):
        idx, stride = self._upload_ids(parts)
        return self._positive_feedback_dev(idx, n_ctx, n_time).cpu().numpy().reshape(-1, 1)

    def _positive_feedback_dev(self, idx, n_ctx, n_time):
        self.flush()
        B, stride = idx.shape
        pos = torch.empty(B, dtype=torch.float32, device=self.device)
        pc, pt, pf = self.pools
        _lib.call("hhfm_pairrank_fwd", ptr(idx), B, stride, n_ctx, n_time, 0, pc, pt, pf,
                  ptr(self.weights["feature_embeddings"]), self._M, self._K, ptr(pos), None, cur_stream())
        return pos


class OUR(_PairRank):
    """HHFM ("OurModel7"), Newcode/OurModel7.py:50-307."""

    def __init__(self, feature_dimension, time_dimension, features_M, n_user, n_item, hidden_factor, learning_rate,
                 lamda_bilinear, optimizer_type, context, time, pooling=(POOL_SUM, POOL_SUM, POOL_SUM), random_seed=2016):
        self.feature_dimension = feature_dimension
        self.time_dimension = time_dimension
        self.n_user = n_user
        self.n_item = n_item
        self.learning_rate = learning_rate
        self.hidden_factor = hidden_factor
        self.features_M = features_M
        self.lamda_bilinear = lamda_bilinear
        self.optimizer_type = optimizer_type
        self.context = context
        self.time = time
        # Pooling1C / Pooling1T / Pooling1F: module-level globals in the reference (OurModel7.py:14-19)
        self.pools = tuple(int(p) for p in pooling)
        self.random_seed = random_seed
        self._init_graph()

    def _init_graph(self):
        self.Pos, self.Fea, self.Tim, self.Neg = Handle("Pos"), Handle("Fea"), Handle("Tim"), Handle("Neg")
        self.PositiveFeadback = Handle("PositiveFeadback")
        self.loss, self.optimizer = Handle("loss"), Handle("optimizer")
        self.num = 1 + (1 if self.context else 0) + (1 if self.time else 0)      # OurModel7.py:89,94
        self._n_ctx = int(self.feature_dimension) if self.context else 0
        self._n_time = int(self.time_dimension) if self.time else 0
        self._setup(self.features_M, self.hidden_factor, self.random_seed, True, self.optimizer_type,
                    self.learning_rate, 0.1, self.lamda_bilinear)
        # feature_bias exists in the reference graph (OurModel7.py:213-214) but receives no gradient
        self._with_bias_grad = False
        self._gb = None

    def _pool_groups_plan(self, idx_dev):
        """Sum pooling everywhere (the reference default): low-cardinality context / time columns are pre-pooled into
        group tables (engine.PoolGroups), so each positive gathers and reduces one row per group instead of one per
        column.  Not for the deterministic kernel or tables large enough for the staged kernel."""
        n_pool = self._n_ctx + self._n_time
        self._pool_groups = None
        if (self.deterministic or n_pool == 0 or any(p != POOL_SUM for p in self.pools) or self.device.type != "cuda"
                or self._M * self._K * 4 >= (96 << 20)):
            return None
        self._pool_groups = PoolGroups.from_batch(self.weights["feature_embeddings"], idx_dev, n_pool)
        return self._pool_groups

    def _parts(self, X, F1, F2, Y=None):
        parts = [np.asarray(X)[:, :2]]
        if self.context:
            parts.append(np.asarray(F1))
        if self.time:
            parts.append(np.asarray(F2))
        if Y is not None:
            parts.append(np.asarray(Y))
        return parts

    def partial_fit(self, data):
        """OurModel7.py:219-228: data = {'X':[B,2], 'F1':[B,fc], 'F2':[B,ft], 'Y':[B,NG]}."""
        Y = np.asarray(data["Y"])
        parts = self._parts(data["X"], data.get("F1"), data.get("F2"), Y)
        return self._fit_records(parts, self._n_ctx, self._n_time, Y.shape[1])

    def positive_feedback(self, X, F1=None, F2=None):
        return self._positive_feedback(self._parts(X, F1, F2), self._n_ctx, self._n_time)

    def score_device(self, idx):
        """PositiveFeadback (OurModel7.py:171) for device-resident rows [n, >= 2+n_ctx+n_time] = [user, item, ctx.., time..]."""
        return self._positive_feedback_dev(idx, self._n_ctx, self._n_time)

    def topk(self, A, tp):
        """OurModel7.py:229-295: A = [user, item, ctx.., time..]."""
        return self._topk(QUERY_HHFM, A, self._n_ctx, self._n_time, self.pools, None, tp)

    def _run(self, fetches, feed):
        if fetches is self.PositiveFeadback:
            return self.positive_feedback(feed[self.Pos], feed.get(self.Fea), feed.get(self.Tim))
        if isinstance(fetches, (tuple, list)) and len(fetches) == 2 and fetches[0] is self.loss:
            d = {"X": feed[self.Pos], "Y": feed[self.Neg]}
            if self.Fea in feed:
                d["F1"] = feed[self.Fea]
            if self.Tim in feed:
                d["F2"] = feed[self.Tim]
            return self.partial_fit(d), None
        raise NotImplementedError("sess.run: unsupported fetch %r" % (fetches,))


class BPR(_PairRank):
    """BPR-MF with max-negative, Newcode/BPR.py:45-136 (Adagrad accumulator starts at 1e-8, BPR.py:93)."""

    pools = (POOL_SUM, POOL_SUM, POOL_SUM)

    def __init__(self, features_M, n_user, n_item, hidden_factor, learning_rate, lamda_bilinear, optimizer_type,
                 random_seed=2016):
        self.n_user = n_user
        self.n_item = n_item
        self.learning_rate = learning_rate
        self.hidden_factor = hidden_factor
        self.features_M = features_M
        self.lamda_bilinear = lamda_bilinear
        self.optimizer_type = optimizer_type
        self.random_seed = random_seed
        self.train_rmse, self.valid_rmse, self.test_rmse = [], [], []
        self._init_graph()

    def _init_graph(self):
        self.Pos, self.Neg = Handle("Pos"), Handle("Neg")
        self.PositiveFeadback = Handle("PositiveFeadback")
        self.loss, self.optimizer = Handle("loss"), Handle("optimizer")
        self._setup(self.features_M, self.hidden_factor, self.random_seed, False, self.optimizer_type,
                    self.learning_rate, 1e-8, self.lamda_bilinear)

    def partial_fit(self, data):
        Y = np.asarray(data["Y"])
        return self._fit_records([np.asarray(data["X"])[:, :2], Y], 0, 0, Y.shape[1])

    def positive_feedback(self, X):
        return self._positive_feedback([np.asarray(X)[:, :2]], 0, 0)

    def score_device(self, idx):
        return self._positive_feedback_dev(idx, 0, 0)

    def topk(self, A, Topk):
        return self._topk(QUERY_USER, A, 0, 0, (0, 0, 0), None, Topk)

    def _run(self, fetches, feed):
        if fetches is self.PositiveFeadback:
            return self.positive_feedback(feed[self.Pos])
        if isinstance(fetches, (tuple, list)) and len(fetches) == 2 and fetches[0] is self.loss:
            return self.partial_fit({"X": feed[self.Pos], "Y": feed[self.Neg]}), None
        raise NotImplementedError("sess.run: unsupported fetch %r" % (fetches,))


# ====================================================================================================
class AFM(FM):
    """Attentional FM, Newcode/AFM.py:63-246.  hidden_factor = [attention size A, embedding size K] (AFM.py:39)."""

    _supports_sparse_dp = False

    def __init__(self, n_user, n_item, features_M, attention, hidden_factor, activation_function, learning_rate,
                 lamda_attention, keep, optimizer_type, decay, valid_dimension, random_seed=2016):
        self.n_user = n_user
        self.n_item = n_item
        self.learning_rate = learning_rate
        self.attention = attention
        self.hidden_factor = hidden_factor
        self.activation_function = activation_function      # unused by the reference graph too (relu is hard-coded, AFM.py:123)
        self.features_M = features_M
        self.valid_dimension = valid_dimension
        self.lamda_attention = lamda_attention
        self.keep = keep
        self.random_seed = random_seed
        self.optimizer_type = optimizer_type
        self.decay = decay
        self.u_f = valid_dimension - 1
        self._init_graph()

    def _init_graph(self):
        self.keep = [float(k) for k in self.keep]
        if len(self.keep) != 2 or not all(0.0 < k <= 1.0 for k in self.keep):
            raise ValueError("keep must be two values in (0, 1] (attention weights, pooled vector)")
        self.attention = 1 if self.attention else 0
        self.train_features = Handle("train_features_afm")
        self.train_labels = Handle("train_labels_afm")
        self.dropout_keep = Handle("dropout_keep_afm")
        self.train_phase = Handle("train_phase_afm")
        self.out = Handle("out_afm")
        self.loss = Handle("loss")
        self.optimizer = Handle("optimizer")
        A, K = int(self.hidden_factor[0]), int(self.hidden_factor[1])
        self._A = A
        self._setup(self.features_M, K, self.random_seed, True, self.optimizer_type, self.learning_rate, 0.1, 0.0)
        if K > 128 or A > 128 or (K + 31) // 32 != (A + 31) // 32:
            raise _lib.HhfmError("AFM kernels need K, A <= 128 in the same 32-tier (reference: A == K)")
        dev = self.device
        self._b0 = torch.zeros(1, dtype=torch.float32, device=dev)
        self.weights["bias"] = self._b0.view(())                                            # AFM.py:186
        rs = np.random.RandomState(self.random_seed)
        glorot = np.sqrt(2.0 / (A + K))                                                     # AFM.py:190
        self.weights["attention_W"] = torch.tensor(rs.normal(0, glorot, (K, A)), dtype=torch.float32, device=dev)
        self.weights["attention_b"] = torch.tensor(rs.normal(0, glorot, (1, A)), dtype=torch.float32, device=dev)
        self.weights["attention_p"] = torch.tensor(rs.normal(0, 1, (A,)), dtype=torch.float32, device=dev)
        self.weights["prediction"] = torch.ones(K, 1, dtype=torch.float32, device=dev)      # AFM.py:199
        self._gW = torch.zeros(K, A, dtype=torch.float32, device=dev)
        self._gbatt = torch.zeros(A, dtype=torch.float32, device=dev)
        self._gp = torch.zeros(A, dtype=torch.float32, device=dev)
        self._gwp = torch.zeros(K, dtype=torch.float32, device=dev)

    def _fused_segments(self):
        return None            # attention_W / b / p and the projection are dense variables outside the arena

    def _small(self):
        w = self.weights
        return ptr(w["attention_W"]), ptr(w["attention_b"]), ptr(w["attention_p"]), ptr(w["prediction"])

    def predict(self, X):
        X = np.asarray(X)
        idx = self._upload_rows(X)
        return self._predict_dev(idx).cpu().numpy().reshape(-1, 1)

    def score_device(self, idx):
        return self._predict_dev(idx)

    def _predict_dev(self, idx):
        """The forward with keep = [1, 1] (the reference evaluates without dropout)."""
        B, F = idx.shape
        out = torch.empty(B, dtype=torch.float32, device=self.device)
        W, batt, pv, wp = self._small()
        _lib.call("hhfm_afm_fwd_attn", ptr(idx), B, F, ptr(self.weights["feature_embeddings"]), ptr(self.weights["feature_bias"]),
                  ptr(self._b0), W, batt, pv, wp, self._M, self._K, self._A, self.attention, ptr(out), cur_stream())
        return out

    def _drop_args(self):
        """(keep_att, keep_vec, seed) of this step's dropout masks (AFM.py:126,134; training only).  The seed follows the
        scheme of FM / MF: a pure function of (random_seed, step)."""
        k0, k1 = self.keep
        if k0 >= 1.0 and k1 >= 1.0:
            return 1.0, 1.0, 0
        return k0, k1, self._drop_seed()

    def _sample_base(self, B):
        """Index of this rank's first row in the global batch, so that every rank draws the masks of its own rows: the
        ranks' batch sizes are exchanged (rank order) under data parallelism, 0 on one GPU."""
        if self._dp_group is None:
            return 0
        import torch.distributed as dist
        ws = dist.get_world_size(self._dp_group)
        sizes = [torch.zeros(1, dtype=torch.int64, device=self.device) for _ in range(ws)]
        dist.all_gather(sizes, torch.tensor([B], dtype=torch.int64, device=self.device), group=self._dp_group)
        rank = dist.get_rank(self._dp_group)
        return int(sum(int(t.item()) for t in sizes[:rank]))

    def partial_fit(self, data):
        """AFM.py:205-208.  V and feature_bias receive IndexedSlices (only touched rows move); attention_W carries the
        lamda_attention L2 term (AFM.py:146); attention_b/p, prediction and bias are small dense variables."""
        idx = self._upload_rows(data["X"])
        y = self._upload_f32(data["Y"])
        self.fit_device(idx, y)
        return self._read_loss()

    def fit_device(self, idx, y):
        B, F = idx.shape
        self._opt.begin_step()
        ts, stamp, tr, tc = self._touch_args(extra=True)
        hot = self._hot_plan(idx, True)
        W, batt, pv, wp = self._small()
        common = (ptr(idx), B, F, ptr(self.weights["feature_embeddings"]), ptr(self.weights["feature_bias"]), ptr(self._b0), W, batt,
                  pv, wp, self._M, self._K, self._A, ptr(y), None, ptr(self._gV), ptr(self._gb), ptr(self._gb0), ptr(self._gW),
                  ptr(self._gbatt), ptr(self._gp), ptr(self._gwp), ptr(self._loss_partials), ts, stamp, tr, tc,
                  *(hot.args(True) if hot else NO_HOT_BIAS))
        # K == A == 64, F <= 11: one fused tcgen05 kernel (csrc/afm_fused_tc.cu); other shapes: fp32 CUDA-core kernels
        k0, k1, dseed = self._drop_args()
        att = self.attention
        if att and k0 >= 1.0 and k1 >= 1.0:
            _lib.call("hhfm_afm_fwd_bwd_sqloss", *common, cur_stream())
        else:
            base = self._sample_base(B) if dseed else 0
            _lib.call("hhfm_afm_fwd_bwd_sqloss_dropout", *common, att, k0, k1, dseed, base, cur_stream())
        # attention=0: attention_W / b / p are not part of the graph (no gradient, no update, no regulariser: AFM.py:132)
        dense = (self._gW, self._gbatt, self._gp, self._gwp) if att else (self._gwp,)
        if hot:
            hot.fold(self._gV, self._gb)
        if self._dp_group is not None:
            import torch.distributed as dist
            self._allreduce_grads()
            for g in dense:
                dist.all_reduce(g, group=self._dp_group)
        self._apply_table(sparse_ok=True)                       # lamda on V is 0: rows (or the dense equivalent under DP)
        self._apply_bias()
        lam = float(self.lamda_attention) if att else 0.0
        o = self._opt
        if att:
            o.apply_dense("attention_W", self.weights["attention_W"], self._gW, lam, self._sq_partials if lam > 0 else None)
            o.apply_dense("attention_b", self.weights["attention_b"], self._gbatt, 0.0, None)
            o.apply_dense("attention_p", self.weights["attention_p"], self._gp, 0.0, None)
        o.apply_dense("prediction", self.weights["prediction"], self._gwp, 0.0, None)
        self._enqueue_loss(lam > 0, 0.5 * lam)

    def topk(self, A, tp):
        """AFM.topk (AFM.py:209-246) scores every item for each context row.  The reference restates `out` with an
        un-normalised exp attention and drops the per-row constants, which is rank-equivalent to scoring the full model.
        Covered shapes (K == A in {16, 32, 64}) go through the item-separable scorer (csrc/afm_topn.cu: the context-only
        pairs once per row, the F-1 item pairs per (row, item)); other shapes, and attention=0, send every (row, item) pair
        through the model's forward kernel.  Either way the exact selector (lowest-index ties) makes the lists."""
        A = np.asarray(A)
        A_dev, stride = self._topn.upload_rows(A, self._M)
        C_rows, F = A.shape
        N = self.n_item
        K, Adim = int(self.hidden_factor[1]), int(self._A)
        out_ids = torch.empty(C_rows, tp, dtype=torch.int32, device=self.device)
        separable = bool(_lib.load().hhfm_afm_topn_supported(F, K, Adim)) and os.environ.get("HHFM_AFM_TOPN_SEPARABLE", "1") != "0" \
            and self.attention == 1
        w = self.weights
        if separable:
            chunk = max(1, min(65535, (1 << 26) // max(N, 1)))
            stats = torch.empty(min(chunk, C_rows), 4, dtype=torch.float32, device=self.device)
            for c0 in range(0, C_rows, chunk):
                c1 = min(C_rows, c0 + chunk)
                sc = torch.empty(c1 - c0, N, dtype=torch.float32, device=self.device)
                _lib.call("hhfm_afm_topn_scores", ptr(A_dev[c0:c1]), stride, c1 - c0, F, 1, ptr(w["feature_embeddings"]),
                          ptr(w["feature_bias"]), ptr(w["bias"]), ptr(w["attention_W"]), ptr(w["attention_b"]),
                          ptr(w["attention_p"]), ptr(w["prediction"]), self._M, K, Adim, self.n_user, N, ptr(stats), ptr(sc),
                          cur_stream())
                _lib.call("hhfm_topn_select", ptr(sc), None, None, c1 - c0, N, N, tp, 0, None, ptr(out_ids[c0:c1]), cur_stream())
            return out_ids.cpu().numpy()
        items = torch.arange(self.n_user, self.n_user + N, dtype=torch.int32, device=self.device)
        chunk = max(1, (1 << 22) // max(N, 1))
        for c0 in range(0, C_rows, chunk):
            c1 = min(C_rows, c0 + chunk)
            rows = A_dev[c0:c1, :F].unsqueeze(1).repeat(1, N, 1)              # [c, N, F]
            rows[:, :, 1] = items.unsqueeze(0)
            sc = self._predict_dev(rows.reshape(-1, F).contiguous()).view(c1 - c0, N)
            _lib.call("hhfm_topn_select", ptr(sc), None, None, c1 - c0, N, N, tp, 0, None, ptr(out_ids[c0:c1]), cur_stream())
        return out_ids.cpu().numpy()


# ====================================================================================================
class DeepFM(_Base):
    """DeepFM, Newcode/DFM.py:50-232.  FM first/second-order parts + a relu MLP tower over the flattened embeddings,
    joined by `concat_projection`; Adagrad only (DFM.py:153); l2 on the projection and the layer matrices (:145-150).

    All dense variables live in ONE flat device buffer (layout: include/hhfm_sm100.h, K8); `weights[...]` are views."""

    def __init__(self, n_user, n_item, feature_size, field_size, embedding_size, deep_layers, deep_layers_activation,
                 learning_rate, verbose=True, l2_reg=0.0, random_seed=2016, use_fm=True, use_deep=True, loss_type="mse"):
        assert (use_fm or use_deep)
        assert loss_type in ["logloss", "mse"], \
            "loss_type can be either 'logloss' for classification task or 'mse' for regression task"
        self.n_user = n_user
        self.n_item = n_item
        self.feature_size = feature_size
        self.field_size = field_size
        self.embedding_size = embedding_size
        self.deep_layers = [int(d) for d in deep_layers]
        self.deep_layers_activation = deep_layers_activation
        self.use_fm = use_fm
        self.use_deep = use_deep
        self.l2_reg = l2_reg
        self.learning_rate = learning_rate
        self.verbose = verbose
        self.random_seed = random_seed
        self.loss_type = loss_type
        self._init_graph()

    def _init_graph(self):
        if not (self.use_fm and self.use_deep) or self.loss_type != "mse":
            raise NotImplementedError("only use_fm=use_deep=True, loss_type='mse' (what DFM.py:257-259 builds) is on the "
                                      "accelerated path")
        act = self.deep_layers_activation
        if not (act == "relu" or getattr(act, "__name__", "") == "relu"):
            raise NotImplementedError("deep_layers_activation must be relu (DFM.py:258 passes tf.nn.relu)")
        self.feat_index, self.label = Handle("feat_index"), Handle("label")
        self.dropout_keep_fm, self.dropout_keep_deep = Handle("dropout_keep_fm"), Handle("dropout_keep_deep")
        self.train_phase = Handle("train_phase")
        self.out, self.loss, self.optimizer = Handle("out"), Handle("loss"), Handle("optimizer")
        F, K, L = int(self.field_size), int(self.embedding_size), len(self.deep_layers)
        self._setup(self.feature_size, K, self.random_seed, True, "AdagradOptimizer", self.learning_rate, 0.1, 0.0)
        dev = self.device
        gen = torch.Generator(device="cpu")
        gen.manual_seed(int(self.random_seed) + 1)
        self.weights["feature_bias"].copy_(torch.empty(self._M, 1).uniform_(0.0, 1.0, generator=gen))   # DFM.py:180-181
        self._sizes = np.asarray(self.deep_layers, dtype=np.int32)
        lib = _lib.load()
        sp = self._sizes.ctypes.data
        n_par = int(lib.hhfm_dfm_param_count(F, K, L, sp))
        self._n_reg = int(lib.hhfm_dfm_reg_count(F, K, L, sp))
        if n_par < 0:
            raise _lib.HhfmError("DeepFM: %s" % lib.hhfm_last_error().decode())
        self._params = torch.zeros(n_par, dtype=torch.float32, device=dev)
        self._gparams = torch.zeros(n_par, dtype=torch.float32, device=dev)
        rs = np.random.RandomState(self.random_seed)
        dims = [F * K] + self.deep_layers
        off = 0
        for i in range(L):                                                                    # DFM.py:184-198
            glorot = np.sqrt(2.0 / (dims[i] + dims[i + 1]))
            n = dims[i] * dims[i + 1]
            self.weights["layer_%d" % i] = self._params[off:off + n].view(dims[i], dims[i + 1])
            self.weights["layer_%d" % i].copy_(torch.tensor(rs.normal(0, glorot, (dims[i], dims[i + 1])), dtype=torch.float32))
            off += n
        n_in = F + K + dims[-1]
        self.weights["concat_projection"] = self._params[off:off + n_in].view(n_in, 1)        # DFM.py:201-210
        self.weights["concat_projection"].copy_(torch.tensor(rs.normal(0, np.sqrt(2.0 / (n_in + 1)), (n_in, 1)), dtype=torch.float32))
        off = self._n_reg                      # the regularised block is zero-padded to a multiple of 4 elements
        for i in range(L):
            glorot = np.sqrt(2.0 / (dims[i] + dims[i + 1]))
            self.weights["bias_%d" % i] = self._params[off:off + dims[i + 1]].view(1, dims[i + 1])
            self.weights["bias_%d" % i].copy_(torch.tensor(rs.normal(0, glorot, (1, dims[i + 1])), dtype=torch.float32))
            off += dims[i + 1]
        self.weights["concat_bias"] = self._params[off:off + 1].view(())
        self.weights["concat_bias"].fill_(0.01)                                               # DFM.py:211
        self._ws = None

    def _workspace(self, B):
        need = int(_lib.load().hhfm_workspace_bytes_dfm(B, int(self.field_size), self._K, len(self.deep_layers),
                                                        self._sizes.ctypes.data)) // 4
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(max(need, 1), dtype=torch.float32, device=self.device)
        return self._ws

    def score_device(self, idx):
        return self._forward_dev(idx)

    def _forward_dev(self, idx):
        B, F = idx.shape
        out = torch.empty(B, dtype=torch.float32, device=self.device)
        _lib.call("hhfm_dfm_fwd", ptr(idx), B, F, ptr(self.weights["feature_embeddings"]), ptr(self.weights["feature_bias"]),
                  self._M, self._K, ptr(self._params), len(self.deep_layers), self._sizes.ctypes.data,
                  ptr(self._workspace(B)), ptr(out), cur_stream())
        return out

    def predict(self, X):
        X = np.asarray(X)
        idx = self._upload_rows(X)
        return self._forward_dev(idx).cpu().numpy().reshape(-1, 1)

    def partial_fit(self, data):
        """DFM.py:216-219: one Adagrad step on {'X': [B,F] ids, 'Y': [B,1] labels}; returns the loss."""
        idx = self._upload_rows(data["X"])
        y = self._upload_f32(data["Y"])
        self.fit_device(idx, y)
        return self._read_loss()

    def fit_device(self, idx, y):
        B, F = idx.shape
        if F != int(self.field_size):
            raise _lib.HhfmError("DeepFM: X has %d columns, field_size is %d" % (F, self.field_size))
        self._opt.begin_step()
        V, fb = self.weights["feature_embeddings"], self.weights["feature_bias"]
        hot = self._hot_plan(idx, True)
        _lib.call("hhfm_dfm_fwd_bwd_sqloss", ptr(idx), B, F, ptr(V), ptr(fb), self._M, self._K, ptr(self._params),
                  len(self.deep_layers), self._sizes.ctypes.data, ptr(y), ptr(self._workspace(B)), None, ptr(self._gV),
                  ptr(self._gb), ptr(self._gparams), ptr(self._loss_partials), *(hot.args(True) if hot else NO_HOT_BIAS),
                  cur_stream())
        if hot:
            hot.fold(self._gV, self._gb)
        if self._dp_group is not None:
            import torch.distributed as dist
            self._allreduce_grads()
            dist.all_reduce(self._gparams, group=self._dp_group)
        # V / feature_bias get IndexedSlices: Adagrad leaves rows with g = 0 untouched, so the dense kernel is exact
        o = self._opt
        self._apply_arena_dense("feature_embeddings", V, self._gV, 0.0, None)
        self._apply_arena_dense("feature_bias", fb, self._gb, 0.0, None)
        lam = float(self.l2_reg)
        nr = self._n_reg
        o.apply_dense("dense_reg", self._params[:nr], self._gparams[:nr], lam if lam > 0 else 0.0,
                      self._sq_partials if lam > 0 else None)
        o.apply_dense("dense_bias", self._params[nr:], self._gparams[nr:], 0.0, None)
        self._enqueue_loss(lam > 0, 0.5 * lam)

    def topk(self, A, tp):
        """DFM.py:220-231: every (row, item) pair scored by the forward graph, then top_k (lowest index first on ties).  The
        item-separable evaluator (hhfm_dfm_topn_scores) pays the first hidden layer once per row and once per item;
        HHFM_DFM_TOPN_SEPARABLE=0 sends every expanded row through hhfm_dfm_fwd instead (A/B runs, tests)."""
        A = np.asarray(A)
        A_dev, stride = self._topn.upload_rows(A, self._M)
        C_rows, F = A.shape
        N = self.n_item
        out_ids = torch.empty(C_rows, tp, dtype=torch.int32, device=self.device)
        chunk = max(1, (1 << 21) // max(N, 1))
        if os.environ.get("HHFM_DFM_TOPN_SEPARABLE", "1") != "0":
            L = len(self.deep_layers)
            need = int(_lib.load().hhfm_workspace_bytes_dfm_topn(min(chunk, C_rows), N, F, self._K, L, self._sizes.ctypes.data)) // 4
            if need < 0:
                raise _lib.HhfmError("hhfm_workspace_bytes_dfm_topn: bad shape")
            if self._ws is None or self._ws.numel() < need:
                self._ws = torch.empty(max(need, 1), dtype=torch.float32, device=self.device)
            for c0 in range(0, C_rows, chunk):
                c1 = min(C_rows, c0 + chunk)
                sc = torch.empty(c1 - c0, N, dtype=torch.float32, device=self.device)
                _lib.call("hhfm_dfm_topn_scores", ptr(A_dev[c0:c1]), stride, c1 - c0, F, 1, ptr(self.weights["feature_embeddings"]),
                          ptr(self.weights["feature_bias"]), self._M, self._K, ptr(self._params), L, self._sizes.ctypes.data,
                          self.n_user, N, ptr(self._ws), ptr(sc), cur_stream())
                _lib.call("hhfm_topn_select", ptr(sc), None, None, c1 - c0, N, N, tp, 0, None, ptr(out_ids[c0:c1]), cur_stream())
            return out_ids.cpu().numpy()
        items = torch.arange(self.n_user, self.n_user + N, dtype=torch.int32, device=self.device)
        for c0 in range(0, C_rows, chunk):
            c1 = min(C_rows, c0 + chunk)
            rows = A_dev[c0:c1, :F].unsqueeze(1).repeat(1, N, 1)
            rows[:, :, 1] = items.unsqueeze(0)
            sc = self._forward_dev(rows.reshape(-1, F).contiguous()).view(c1 - c0, N)
            _lib.call("hhfm_topn_select", ptr(sc), None, None, c1 - c0, N, N, tp, 0, None, ptr(out_ids[c0:c1]), cur_stream())
        return out_ids.cpu().numpy()

    def _run(self, fetches, feed):
        if fetches is self.out:
            return self.predict(feed[self.feat_index])
        if isinstance(fetches, (tuple, list)) and len(fetches) == 2 and fetches[0] is self.loss:
            return self.partial_fit({"X": feed[self.feat_index], "Y": feed[self.label]}), None
        raise NotImplementedError("sess.run: unsupported fetch %r" % (fetches,))


# ====================================================================================================
class WD(_Base):
    """Wide&Deep, Newcode/WDMF.py:51-126: `WD(feature_num, n_user, n_item)` wraps tf.contrib.learn's
    DNNLinearCombinedClassifier (hashed columns + all pairwise crossed columns -> linear model trained with FTRL; 128-d
    embedding columns -> DNN [1024, 512, 256] trained with Adagrad; sigmoid cross-entropy head).  Everything numeric in the
    reference happens inside TensorFlow, so this class follows TF's documented defaults with its own bucket functions
    (include/hhfm_sm100.h K11, oracle wd_*): PARITY UNPINNED against the reference, pinned against the oracle restatement.

      * single hashed columns: ONE table keyed by the loader's global feature id (ids must be < features_M, default 10^5 =
        the reference's hash_bucket_size).  A token that occurs in two columns shares its weight / embedding, as it shares its
        id in every other model of the reference; TF's per-column tables would keep them apart.  Crossed columns: splitmix64
        of the id pair mod 10^4, one table per column pair;
      * linear half: FTRL, learning rate min(0.2, 1/sqrt(#linear columns)), accumulators 0.1, l1 = l2 = 0, weights start at 0;
      * DNN half: Adagrad lr 0.05 (accumulators 0.1), Glorot-uniform kernels, zero biases, embeddings N(0, 1/sqrt(dim))
        truncated at 2 sigma, field order = column order;
      * `partial_fit(X, Y)` = `fit(steps=500)`: 500 full-batch steps; `predict(X)` = predict_proba rows [1-p, p]."""

    def __init__(self, feature_num, n_user, n_item, features_M=100000, hidden_units=(1024, 512, 256), embedding_dim=128,
                 cross_buckets=10000, steps=500, random_seed=2016):
        self.feature_num = int(feature_num)
        self.n_user = n_user
        self.n_item = n_item
        self.keys = ["Feature" + str(i) for i in range(self.feature_num)]
        self.hidden_units = [int(h) for h in hidden_units]
        self.steps = int(steps)
        self.cross_buckets = int(cross_buckets)
        self.random_seed = random_seed
        F, K, L = self.feature_num, int(embedding_dim), len(self.hidden_units)
        self.dnn_learning_rate = 0.05
        n_pairs = F * (F - 1) // 2
        self.linear_learning_rate = min(0.2, 1.0 / np.sqrt(F + n_pairs))
        self._setup(features_M, K, random_seed, False, "AdagradOptimizer", self.dnn_learning_rate, 0.1, 0.0)
        dev = self.device
        rs = np.random.RandomState(self.random_seed)
        emb = rs.normal(0, 1.0, (self._M, K))
        bad = np.abs(emb) > 2.0
        while bad.any():                                   # truncated normal: redraw beyond two sigma
            emb[bad] = rs.normal(0, 1.0, int(bad.sum()))
            bad = np.abs(emb) > 2.0
        self.weights["feature_embeddings"].copy_(torch.tensor(emb / np.sqrt(K), dtype=torch.float32))
        self._sizes = np.asarray(self.hidden_units, dtype=np.int32)
        lib = _lib.load()
        sp = self._sizes.ctypes.data
        n_par = int(lib.hhfm_dfm_param_count(F, K, L, sp))
        self._n_reg = int(lib.hhfm_dfm_reg_count(F, K, L, sp))
        if n_par < 0:
            raise _lib.HhfmError("WD: %s" % lib.hhfm_last_error().decode())
        self._params = torch.zeros(n_par, dtype=torch.float32, device=dev)
        self._gparams = torch.zeros(n_par, dtype=torch.float32, device=dev)
        dims = [F * K] + self.hidden_units
        off = 0
        for i in range(L):
            lim = np.sqrt(6.0 / (dims[i] + dims[i + 1]))                                      # Glorot uniform
            n = dims[i] * dims[i + 1]
            self.weights["layer_%d" % i] = self._params[off:off + n].view(dims[i], dims[i + 1])
            self.weights["layer_%d" % i].copy_(torch.tensor(rs.uniform(-lim, lim, (dims[i], dims[i + 1])), dtype=torch.float32))
            off += n
        off += F + K                                       # the FM slots of the DeepFM projection block: unused, zero
        lim = np.sqrt(6.0 / (dims[-1] + 1))
        self.weights["logits_w"] = self._params[off:off + dims[-1]].view(dims[-1], 1)
        self.weights["logits_w"].copy_(torch.tensor(rs.uniform(-lim, lim, (dims[-1], 1)), dtype=torch.float32))
        off = self._n_reg
        for i in range(L):
            self.weights["bias_%d" % i] = self._params[off:off + dims[i + 1]].view(1, dims[i + 1])
            off += dims[i + 1]
        self.weights["logits_b"] = self._params[off:off + 1].view(())
        # wide half: [w_lin (M) | w_cross (P x buckets) | bias (1)] in one block with its FTRL slots
        n_wide = self._M + n_pairs * self.cross_buckets + 1
        self._wide = torch.zeros(n_wide, dtype=torch.float32, device=dev)
        self._gwide = torch.zeros(n_wide, dtype=torch.float32, device=dev)
        self._ftrl_accum = torch.full((n_wide,), 0.1, dtype=torch.float32, device=dev)
        self._ftrl_linear = torch.zeros(n_wide, dtype=torch.float32, device=dev)
        self.weights["wide_linear"] = self._wide[:self._M]
        self.weights["wide_cross"] = self._wide[self._M:n_wide - 1].view(n_pairs, self.cross_buckets)
        self.weights["wide_bias"] = self._wide[n_wide - 1:].view(())
        self._n_pairs = n_pairs
        self._ws = None
        self._wide_logit = None
        self._gsample = None

    def _workspace(self, B):
        need = int(_lib.load().hhfm_workspace_bytes_dfm(B, self.feature_num, self._K, len(self.hidden_units),
                                                        self._sizes.ctypes.data)) // 4
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(max(need, 1), dtype=torch.float32, device=self.device)
        if self._wide_logit is None or self._wide_logit.numel() < B:
            self._wide_logit = torch.empty(B, dtype=torch.float32, device=self.device)
            self._gsample = torch.empty(B, dtype=torch.float32, device=self.device)
        return self._ws

    def _wide_fwd(self, idx):
        B, F = idx.shape
        _lib.call("hhfm_wd_wide_fwd", ptr(idx), B, F, ptr(self.weights["wide_linear"]), ptr(self.weights["wide_cross"]),
                  ptr(self.weights["wide_bias"]), self._M, self.cross_buckets, ptr(self._wide_logit), cur_stream())

    def score_device(self, idx):
        """Logits [B] (device) for device rows [B,F]; monotone in the probability the reference ranks by."""
        B, F = idx.shape
        if F != self.feature_num:
            raise _lib.HhfmError("WD: X has %d columns, feature_num is %d" % (F, self.feature_num))
        ws = self._workspace(B)
        self._wide_fwd(idx)
        out = torch.empty(B, dtype=torch.float32, device=self.device)
        _lib.call("hhfm_wd_deep_fwd", ptr(idx), B, F, ptr(self.weights["feature_embeddings"]), self._M, self._K,
                  ptr(self._params), len(self.hidden_units), self._sizes.ctypes.data, ptr(self._wide_logit), ptr(ws), ptr(out),
                  cur_stream())
        return out

    def predict(self, X):
        """model.predict_proba (WDMF.py:108-111): rows [P(label 0), P(label 1)]."""
        p = torch.sigmoid(self.score_device(self._upload_rows(np.asarray(X)))).cpu().numpy()
        return np.stack([1.0 - p, p], axis=1)

    def fit_device(self, idx, y):
        """One full-batch step of the estimator on device rows / labels: FTRL on the wide half, Adagrad on the DNN half."""
        B, F = idx.shape
        if F != self.feature_num:
            raise _lib.HhfmError("WD: X has %d columns, feature_num is %d" % (F, self.feature_num))
        if self._dp_group is not None:
            raise NotImplementedError("WD is single-process (the reference estimator is)")
        self._opt.begin_step()
        V = self.weights["feature_embeddings"]
        ws = self._workspace(B)
        hot = self._hot_plan(idx, False)
        self._wide_fwd(idx)
        _lib.call("hhfm_wd_deep_fwd_bwd_logloss", ptr(idx), B, F, ptr(V), self._M, self._K, ptr(self._params),
                  len(self.hidden_units), self._sizes.ctypes.data, ptr(y), ptr(self._wide_logit), ptr(ws), None, ptr(self._gV),
                  ptr(self._gparams), ptr(self._gsample), ptr(self._loss_partials), *(hot.args() if hot else NO_HOT), cur_stream())
        if hot:
            hot.fold(self._gV, None)
        n_wide = self._wide.numel()
        _lib.call("hhfm_wd_wide_bwd", ptr(idx), B, F, ptr(self._gsample), self._M, self.cross_buckets, ptr(self._gwide),
                  ptr(self._gwide[self._M:]), ptr(self._gwide[n_wide - 1:]), cur_stream())
        self._apply_arena_dense("feature_embeddings", V, self._gV, 0.0, None)      # rows with g = 0 do not move under Adagrad
        self._opt.apply_dense("dnn", self._params, self._gparams, 0.0, None)
        _lib.call("hhfm_opt_ftrl_dense", ptr(self._wide), ptr(self._ftrl_accum), ptr(self._ftrl_linear), ptr(self._gwide), n_wide,
                  float(self.linear_learning_rate), 0.0, 0.0, 1, cur_stream())
        self._enqueue_loss(False)

    def partial_fit(self, X, Y, steps=None):
        """WDMF.py:113-115 `model.fit(input_fn, steps=500)`: `steps` steps on the whole (X, Y); returns the last loss."""
        idx = self._upload_rows(np.asarray(X)).clone()
        y = self._upload_f32(np.asarray(Y, dtype=np.float32)).clone()
        for _ in range(self.steps if steps is None else int(steps)):
            self.fit_device(idx, y)
        return self._read_loss()

    def topk(self, feed_dict, tp):
        """WDMF.py:116-126: every (row, item) pair through predict_proba, then top_k (lowest index first on ties).  The
        ranking uses the logit (sigmoid is monotone; equal logits are equal probabilities)."""
        A = np.array(feed_dict, dtype=np.int64)
        A_dev, stride = self._topn.upload_rows(A, self._M)
        C_rows, F = A.shape
        N = self.n_item
        out_ids = torch.empty(C_rows, tp, dtype=torch.int32, device=self.device)
        items = torch.arange(self.n_user, self.n_user + N, dtype=torch.int32, device=self.device)
        chunk = max(1, (1 << 18) // max(N, 1))      # <= 2^18 expanded rows per pass: the tower's workspace is ~50 KB per row
        for c0 in range(0, C_rows, chunk):
            c1 = min(C_rows, c0 + chunk)
            rows = A_dev[c0:c1, :F].unsqueeze(1).repeat(1, N, 1)
            rows[:, :, 1] = items.unsqueeze(0)
            sc = self.score_device(rows.reshape(-1, F).contiguous()).view(c1 - c0, N)
            _lib.call("hhfm_topn_select", ptr(sc), None, None, c1 - c0, N, N, tp, 0, None, ptr(out_ids[c0:c1]), cur_stream())
        return out_ids.cpu().numpy()


# ====================================================================================================
class CARS2:
    """CARS2, Newcode/CARS2.py:45-187: the context-aware baseline of main.py:50-63.  One flat parameter block
    [UI | Context | W | Z | A | B] (layout: include/hhfm_sm100.h, K10); `weights[...]` are views."""

    def __init__(self, features_M, n_user, n_item, hidden_factor, learning_rate, lamda_bilinear, optimizer_type,
                 random_seed=2016):
        self.n_user = n_user
        self.n_item = n_item
        self.learning_rate = learning_rate
        self.D = int(hidden_factor)
        self.D_c = int(hidden_factor / 2.5)                  # CARS2.py:54-56
        self.D_p = int(hidden_factor / 5)
        self.D_q = int(hidden_factor / 2.5)
        self.features_M = features_M
        self.lamda_bilinear = lamda_bilinear
        self.optimizer_type = optimizer_type
        self.random_seed = random_seed
        self._init_graph()

    def _init_graph(self):
        self.device = require_cuda()
        if self.D > 128 or self.D_c < 1 or self.D_p < 1:
            raise _lib.HhfmError("CARS2: hidden_factor must be in [5, 128] (D_c = D/2.5, D_p = D/5 >= 1)")
        self.Pos, self.Fea, self.Neg = Handle("Pos"), Handle("Fea"), Handle("Neg")
        self.PositiveFeadback = Handle("PositiveFeadback")
        self.loss, self.optimizer = Handle("loss"), Handle("optimizer")
        lib = _lib.load()
        n_ui = self.n_user + self.n_item
        D, Dc, Dp, Dq, M = self.D, self.D_c, self.D_p, self.D_q, int(self.features_M)
        self._dims = (n_ui, M, D, Dp, Dq, Dc)
        n = int(lib.hhfm_cars2_param_count(*self._dims))
        self._params = torch.zeros(n + 4, dtype=torch.float32, device=self.device)[:n]
        self._gparams = torch.zeros(n + 4, dtype=torch.float32, device=self.device)[:n]
        gen = torch.Generator(device="cpu")
        gen.manual_seed(int(self.random_seed))
        self.weights = {}
        off = 0
        for name, shape, std in (("UI", (n_ui, D), 0.01), ("Context", (M, Dc), 0.01), ("W", (D, Dp, Dc), 0.01),
                                 ("Z", (D, Dq, Dc), 0.01), ("A", (Dp,), 0.0), ("B", (Dq,), 0.0)):       # CARS2.py:155-167
            cnt = int(np.prod(shape))
            self.weights[name] = self._params[off:off + cnt].view(*shape)
            if std > 0:
                self.weights[name].copy_(torch.empty(*shape).normal_(0.0, std, generator=gen))
            off += cnt
        P = _lib.partials_len()
        self._loss_partials = torch.zeros(P, dtype=torch.float32, device=self.device)
        self._sq_partials = torch.zeros(P, dtype=torch.float32, device=self.device)
        self._loss_dev = torch.zeros(1, dtype=torch.float32, device=self.device)
        self._opt = Optimizer(self.optimizer_type, self.learning_rate, initial_accumulator_value=0.1)
        self._uploader = RecordUploader(self.device)
        self._topn = TopN(self.device)
        self._M = max(n_ui, M)                 # id limit of the packed records (users/items and context-tuple ids)
        self._ws = None
        self._version = 0
        self.topn_method = "auto"
        self.sess = Session(self)

    def _workspace(self, B):
        need = int(_lib.load().hhfm_workspace_bytes_cars2(B, self.D, self.D_c)) // 4 + 4
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.float32, device=self.device)
        return self._ws

    def _forward(self, rec, mode):
        B, stride = rec.shape
        out = torch.empty(B if mode == 0 else (B, self.D), dtype=torch.float32, device=self.device)
        _lib.call("hhfm_cars2_fwd", ptr(rec), B, stride, ptr(self._params), *self._dims, mode, ptr(out),
                  ptr(self._workspace(B)), cur_stream())
        return out

    def score_device(self, rec):
        """PositiveFeadback [n] (device) for device records [n, >=3] = [user, item, context-tuple id]."""
        return self._forward(rec, 0)

    def positive_feedback(self, X, F1):
        rec, _ = self._uploader.upload([np.asarray(X)[:, :2], np.asarray(F1).reshape(-1, 1)], self._M)
        return self.score_device(rec).cpu().numpy().reshape(-1, 1)

    def partial_fit(self, data):
        """CARS2.py:168-171: data = {'X': [B,2], 'F1': [B] context-tuple ids, 'Y': [B,NG] negatives}; returns the loss."""
        Y = np.asarray(data["Y"])
        rec, _ = self._uploader.upload([np.asarray(data["X"])[:, :2], np.asarray(data["F1"]).reshape(-1, 1), Y], self._M)
        self.fit_device(rec, Y.shape[1])
        loss_host = self._loss_dev.cpu()
        return float(loss_host[0])

    def fit_device(self, rec, n_neg):
        B, stride = rec.shape
        self._opt.begin_step()
        _lib.call("hhfm_cars2_fwd_bwd", ptr(rec), B, stride, n_neg, ptr(self._params), *self._dims, ptr(self._gparams),
                  ptr(self._loss_partials), ptr(self._workspace(B)), cur_stream())
        lam = float(self.lamda_bilinear)
        if lam <= 0 and self._opt.kind == "momentum":
            # without the L2 term TF hands UI / Context IndexedSlices to SparseApplyMomentum (only touched rows move); the
            # dense kernel would keep moving untouched rows (accum *= mu; w -= lr * accum)
            raise NotImplementedError("CARS2: MomentumOptimizer with lamda == 0 needs the touched-row update, which is not "
                                      "implemented for the CARS2 parameter block; use lamda > 0 (reference default 0.001)")
        self._opt.apply_dense("params", self._params, self._gparams, lam if lam > 0 else 0.0,
                              self._sq_partials if lam > 0 else None)
        self._version += 1
        _lib.call("hhfm_loss_finalize", ptr(self._loss_partials), ptr(self._sq_partials) if lam > 0 else None, 0.5 * lam,
                  ptr(self._loss_dev), cur_stream())

    def topk(self, feed_dict, tp):
        """CARS2.py:171-187: feed_dict = {'X': user ids [C], 'F1': context-tuple ids [C]}.  score(c, item) = item . (u + T c)
        + a per-row constant, so the catalog is ranked by the dot product with that query vector (exact fp32 scorer or the
        tcgen05 filter + exact rescoring, lowest index first on ties)."""
        users = np.asarray(feed_dict["X"]).reshape(-1, 1)
        fea = np.asarray(feed_dict["F1"]).reshape(-1, 1)
        rec, _ = self._uploader.upload([users, np.zeros_like(users), fea], self._M)
        Q = self._forward(rec, 2)
        items = self.weights["UI"][self.n_user:self.n_user + self.n_item]
        return self._topn.topk_from_query(Q, items, tp, method=self.topn_method, version=self._version).cpu().numpy()

    def load_weights(self, weights):
        for k, v in weights.items():
            t = torch.as_tensor(np.asarray(v, dtype=np.float32)).reshape(self.weights[k].shape)
            self.weights[k].copy_(t.to(self.device))
        self._version += 1

    def get_weights(self):
        return {k: v.detach().cpu().numpy().copy() for k, v in self.weights.items()}

    def _run(self, fetches, feed):
        if fetches is self.PositiveFeadback:
            return self.positive_feedback(feed[self.Pos], feed[self.Fea])
        if isinstance(fetches, (tuple, list)) and len(fetches) == 2 and fetches[0] is self.loss:
            return self.partial_fit({"X": feed[self.Pos], "F1": feed[self.Fea], "Y": feed[self.Neg]}), None
        raise NotImplementedError("sess.run: unsupported fetch %r" % (fetches,))
