"""Host-side plumbing between the reference-shaped Python API and the C ABI (libhhfm_sm100.so).

PyTorch is used for device memory, streams and torch.distributed only; every arithmetic step of the hot path
is a hand-written sm_100a kernel behind `include/hhfm_sm100.h`.  Nothing here falls back to CPU math.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import weakref

import numpy as np
import torch

from . import _lib

POOL_SUM, POOL_MAX, POOL_MEAN = 0, 1, 2
QUERY_USER, QUERY_FM, QUERY_HHFM = 0, 1, 2


def _pack_threads():
    """Worker threads of the host packer.  One process per GPU: every rank of a box gets its share of the cores (and pins its
    pool to them) instead of a full-width pool per rank fighting over all cores.  HHFM_PACK_THREADS / HHFM_PACK_PIN_BASE
    override; 0 = hardware concurrency."""
    if "HHFM_PACK_THREADS" in os.environ:
        return int(os.environ["HHFM_PACK_THREADS"])
    lws = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1)
    if lws <= 1:
        return 0
    cores = os.cpu_count() or 1
    n = max(2, cores // lws)
    os.environ.setdefault("HHFM_PACK_PIN_BASE", str((int(os.environ.get("LOCAL_RANK", "0") or 0) * n) % cores))
    return n


_NTHREADS = _pack_threads()


def require_cuda():
    if not torch.cuda.is_available():
        raise _lib.HhfmError("hhfm_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    _lib.load()
    return torch.device("cuda", torch.cuda.current_device())


def ptr(t):
    """Device/host pointer of a tensor (or numpy array) as c_void_p; None -> NULL."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return C.c_void_p(t.ctypes.data)
    return C.c_void_p(t.data_ptr())


def cur_stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _round_up(x, m):
    return (x + m - 1) // m * m


# --------------------------------------------------------------------------------------------------
# K0: batch packing into pinned staging buffers
# --------------------------------------------------------------------------------------------------
class Staging:
    """Growable pinned-host + device buffer pair for one kind of batch record (int32 or float32)."""

    def __init__(self, dtype, device=None):
        self.dtype = dtype
        self.device = device
        self.host = None
        self.dev = None
        self._busy = None          # recorded after the last upload: the pinned buffer may be rewritten once it has passed

    def ensure(self, numel):
        if self._busy is not None:
            self._busy.synchronize()    # a step may still be in flight (partial_fit_async): its copy must have read the buffer
        if self.host is None or self.host.numel() < numel:
            cap = max(numel, 1024)
            pin = torch.cuda.is_available()
            self.host = torch.empty(cap, dtype=self.dtype, pin_memory=pin)
            if self.device is not None:
                self.dev = torch.empty(cap, dtype=self.dtype, device=self.device)
        return self.host[:numel]

    def upload(self, numel):
        """Asynchronous H2D of the first `numel` elements on the current stream."""
        self.dev[:numel].copy_(self.host[:numel], non_blocking=True)
        if self.host.is_pinned():
            if self._busy is None:
                self._busy = torch.cuda.Event()
            self._busy.record()
        return self.dev[:numel]


def _as_2d_ids(a):
    a = np.asarray(a)
    if a.ndim == 1:
        a = a.reshape(-1, 1)
    if a.dtype not in (np.int64, np.int32):
        if not np.issubdtype(a.dtype, np.integer):
            # the reference feeds float ndarrays holding integral ids in places (DataFrame.values)
            a = a.astype(np.int64)
        else:
            a = a.astype(np.int64)
    if a.strides[1] != a.itemsize:
        a = np.ascontiguousarray(a)
    return a


def pack_ids_into(dst_host, dst_stride, dst_col0, src, id_limit):
    """Narrow an [rows, cols] id array into columns [dst_col0, dst_col0+cols) of int32 records."""
    src = _as_2d_ids(src)
    rows, cols = src.shape
    if cols == 0:
        return 0
    fn = "hhfm_pack_ids_i64" if src.dtype == np.int64 else "hhfm_pack_ids_i32"
    _lib.call(fn, ptr(src), rows, cols, src.strides[0] // src.itemsize, ptr(dst_host), dst_stride, dst_col0,
              id_limit, _NTHREADS)
    return cols


def pack_records(parts, id_limit, staging: Staging, align=4):
    """Concatenate id blocks column-wise into one [B, stride] int32 record buffer (stride % align == 0, padding
    = -1).  Returns (host_view [B,stride], stride)."""
    parts = [_as_2d_ids(p) for p in parts if p is not None]
    B = parts[0].shape[0]
    for p in parts:
        if p.shape[0] != B:
            raise ValueError("pack_records: blocks disagree on the number of rows")
    width = sum(p.shape[1] for p in parts)
    stride = _round_up(max(width, 1), align)
    host = staging.ensure(B * stride)
    col = 0
    for p in parts:
        col += pack_ids_into(host, stride, col, p, id_limit)
    if stride > width:
        _lib.call("hhfm_pack_fill_i32", ptr(host), B, stride - width, stride, width, -1, _NTHREADS)
    return host.view(B, stride), stride


class PackPart(C.Structure):
    _fields_ = [("data", C.c_void_p), ("cols", C.c_int64), ("row_stride", C.c_int64), ("elem_bytes", C.c_int32),
                ("reserved", C.c_int32)]


class RecordUploader:
    """Host id blocks -> int32 device records through `hhfm_pack_upload_records`: a persistent host thread pool packs
    chunk i+1 while chunk i crosses PCIe; uint16 wire format when every id fits (id_limit <= 65535)."""

    def __init__(self, device):
        self.device = device
        self.host = None
        self.dev_stage = None
        self.dev = None
        self._busy = None          # event recorded after the last upload: the pinned staging is free once it has passed

    def upload(self, parts, id_limit, align=4, extra_cols=0):
        """`extra_cols` reserves columns after the packed ones (filled with the padding code -1 here, e.g. negatives that
        the device sampler writes afterwards).  The returned tensor is a VIEW of this uploader's device buffer: the next
        `upload` overwrites it (clone it to keep it)."""
        parts = [_as_2d_ids(p) for p in parts if p is not None]
        B = parts[0].shape[0]
        for p in parts:
            if p.shape[0] != B:
                raise ValueError("upload: blocks disagree on the number of rows")
        width = sum(p.shape[1] for p in parts)
        stride = _round_up(max(width + int(extra_cols), 1), align)
        lib = _lib.load()
        nbytes = int(lib.hhfm_pack_upload_staging_bytes(B, stride, id_limit))
        if self._busy is not None and (self.host is None or self.host.numel() < nbytes or self.dev is None
                                       or self.dev.numel() < B * stride):
            self._busy.synchronize()        # the previous upload's copies (issued by library threads) still use the old buffers
        if self.host is None or self.host.numel() < nbytes:
            cap = max(nbytes, 4096)
            self.host = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
            self.dev_stage = torch.empty(cap, dtype=torch.uint8, device=self.device)
        if self.dev is None or self.dev.numel() < B * stride:
            self.dev = torch.empty(max(B * stride, 1024), dtype=torch.int32, device=self.device)
        if B == 0:
            return self.dev[:0].view(0, stride), stride
        if self._busy is not None:
            self._busy.synchronize()
        arr = (PackPart * len(parts))()
        for i, p in enumerate(parts):
            arr[i].data = p.ctypes.data
            arr[i].cols = p.shape[1]
            arr[i].row_stride = p.strides[0] // p.itemsize
            arr[i].elem_bytes = p.itemsize
        _lib.call("hhfm_pack_upload_records", C.cast(arr, C.c_void_p), len(parts), B, stride, id_limit, ptr(self.host),
                  ptr(self.dev_stage), ptr(self.dev), _NTHREADS, cur_stream())
        if self._busy is None:
            self._busy = torch.cuda.Event()
        self._busy.record()
        return self.dev[:B * stride].view(B, stride), stride


class DeviceSampler:
    """`Train.sample_negative` (FM.py:284-294) on the device: uniform item draws with rejection against
    positive_feedback[key(row)], the membership test being a binary search in the loader's sorted (key_id, item) codes.
    Counter-based generator (csrc/sampler.cu): reproducible from `seed`, statistically the reference's sampler, not its
    numpy stream."""

    def __init__(self, loader, n_user, n_item, device, seed=2016):
        self.loader = loader
        self.n_user, self.n_item = int(n_user), int(n_item)
        self.device = device
        self.codes = torch.as_tensor(np.ascontiguousarray(loader._pf_codes, dtype=np.int64)).to(device)
        self.span = int(loader._span)
        self.seed = int(seed)
        self.calls = 0

    def key_ids(self, rows):
        """rows [n, F] host ids (label column removed) -> int32 device tensor of key ids (-1: key never trained)."""
        return torch.as_tensor(self.loader.key_ids(rows).astype(np.int32)).to(self.device)

    def next_seed(self):
        self.calls += 1
        return (self.seed * 0x9E3779B97F4A7C15 + self.calls) & 0xFFFFFFFFFFFFFFFF

    def sample(self, key_id_dev, num, out=None, out_stride=None, out_col0=0, seed=None):
        """Writes `num` negatives per row into out[:, out_col0:out_col0+num] (int32, row stride out_stride); allocates a
        dense [n, num] tensor when `out` is None."""
        n = int(key_id_dev.numel())
        if out is None:
            out = torch.empty(n, num, dtype=torch.int32, device=self.device)
            out_stride, out_col0 = num, 0
        _lib.call("hhfm_sample_negatives", ptr(key_id_dev), n, num, self.n_user, self.n_item, ptr(self.codes),
                  int(self.codes.numel()), self.span, self.next_seed() if seed is None else seed, ptr(out), out_stride,
                  out_col0, cur_stream())
        return out


def expand_rows(rows_dev, F, items_dev, out_stride=None):
    """[n, stride] records + [n, num] items -> [n*num, out_stride] rows with column 1 replaced (FM.py:303-305) and -1
    padding after column F, on the device."""
    n, stride = rows_dev.shape
    num = items_dev.shape[1]
    out_stride = F if out_stride is None else out_stride
    out = torch.empty(n * num, out_stride, dtype=torch.int32, device=rows_dev.device)
    _lib.call("hhfm_expand_rows", ptr(rows_dev), n, F, stride, ptr(items_dev), num, ptr(out), out_stride, cur_stream())
    return out


def auc_wins(pos_dev, neg_dev, num, wins_dev):
    _lib.call("hhfm_auc_count", ptr(pos_dev), ptr(neg_dev), int(pos_dev.numel()), num, ptr(wins_dev), cur_stream())


# --------------------------------------------------------------------------------------------------
# K5: optimizers with TF-1.x semantics
# --------------------------------------------------------------------------------------------------
class Optimizer:
    """tf.train.{Adagrad,Adam,Momentum,GradientDescent}Optimizer (FM.py:129-136) over device tensors."""

    KINDS = {"AdagradOptimizer": "adagrad", "AdamOptimizer": "adam", "MomentumOptimizer": "momentum",
             "GradientDescentOptimizer": "sgd"}

    def __init__(self, optimizer_type, learning_rate, initial_accumulator_value=0.1, momentum=0.95, beta1=0.9,
                 beta2=0.999, epsilon=1e-8):
        if optimizer_type not in self.KINDS:
            raise ValueError("unknown optimizer_type %r" % (optimizer_type,))
        self.kind = self.KINDS[optimizer_type]
        self.lr = float(learning_rate)
        self.acc0 = float(initial_accumulator_value)
        self.momentum = float(momentum)
        self.beta1, self.beta2, self.eps = float(beta1), float(beta2), float(epsilon)
        self.t = 0
        self.state = {}

    def slots(self, name, w):
        if name not in self.state:
            if self.kind == "adagrad":
                self.state[name] = (torch.full_like(w, self.acc0), None)
            elif self.kind == "adam":
                self.state[name] = (torch.zeros_like(w), torch.zeros_like(w))
            elif self.kind == "momentum":
                self.state[name] = (torch.zeros_like(w), None)
            else:
                self.state[name] = (None, None)
        return self.state[name]

    def begin_step(self):
        self.t += 1

    def _lr_t(self):
        return self.lr * math.sqrt(1.0 - self.beta2 ** self.t) / (1.0 - self.beta1 ** self.t)

    def apply_dense(self, name, w, g, lamda=0.0, sq_partials=None, zero_grad=True):
        """Dense update of every element with g_eff = g + lamda*w (aggregated dense gradient)."""
        s1, s2 = self.slots(name, w)
        n = w.numel()
        z = 1 if zero_grad else 0
        st = cur_stream()
        if self.kind == "adagrad":
            _lib.call("hhfm_opt_adagrad_dense_l2", ptr(w), ptr(s1), ptr(g), n, self.lr, lamda, z, ptr(sq_partials), st)
        elif self.kind == "adam":
            _lib.call("hhfm_opt_adam_dense_l2", ptr(w), ptr(s1), ptr(s2), ptr(g), n, self._lr_t(), self.beta1,
                      self.beta2, self.eps, lamda, z, ptr(sq_partials), st)
        elif self.kind == "momentum":
            _lib.call("hhfm_opt_momentum_dense_l2", ptr(w), ptr(s1), ptr(g), n, self.lr, self.momentum, lamda, z,
                      ptr(sq_partials), st)
        else:
            _lib.call("hhfm_opt_sgd_dense_l2", ptr(w), ptr(g), n, self.lr, lamda, z, ptr(sq_partials), st)

    KIND_ID = {"adagrad": 0, "adam": 1, "momentum": 2, "sgd": 3}

    def apply_rows(self, name, w, g, rows, n_rows_dev, K, zero_grad=True):
        """Sparse (IndexedSlices) update: only the touched rows move.  TF1's sparse Adam moves every row, so it
        maps to the dense kernel."""
        if self.kind == "adam":
            return self.apply_dense(name, w, g, 0.0, None, zero_grad)
        s1, _ = self.slots(name, w)
        z = 1 if zero_grad else 0
        st = cur_stream()
        max_rows = rows.numel()
        if self.kind == "adagrad":
            _lib.call("hhfm_opt_adagrad_rows", ptr(w), ptr(s1), ptr(g), ptr(rows), ptr(n_rows_dev), max_rows, K, self.lr, z, st)
        elif self.kind == "momentum":
            _lib.call("hhfm_opt_momentum_rows", ptr(w), ptr(s1), ptr(g), ptr(rows), ptr(n_rows_dev), max_rows, K, self.lr,
                      self.momentum, z, st)
        else:
            _lib.call("hhfm_opt_sgd_rows", ptr(w), ptr(g), ptr(rows), ptr(n_rows_dev), max_rows, K, self.lr, z, st)


class TouchTracker:
    """Per-step list of touched embedding rows, produced on the device by the scatter kernels."""

    def __init__(self, M, device):
        self.stamp_arr = torch.zeros(M, dtype=torch.int32, device=device)
        self.rows = torch.empty(M, dtype=torch.int32, device=device)
        self.count = torch.zeros(1, dtype=torch.int32, device=device)
        self.stamp = 0

    def begin_step(self):
        self.stamp += 1
        if self.stamp >= 2 ** 31 - 1:
            self.stamp_arr.zero_()
            self.stamp = 1
        self.count.zero_()


class HotRows:
    """Two-level scatter plan (see hhfm_sm100.h `hot_slot`): rows that many samples of a batch share get
    `n_rep` replicated accumulators so their vector reductions do not serialise on one L2 slice."""

    N_REP = int(os.environ.get("HHFM_HOT_REP", "64"))
    MAX_HOT = int(os.environ.get("HHFM_HOT_MAX", "1024"))
    MIN_COUNT = int(os.environ.get("HHFM_HOT_MIN_COUNT", "2048"))

    def __init__(self, hot_rows, M, K, device, with_bias=False, n_rep=None):
        hot_rows = torch.as_tensor(hot_rows, dtype=torch.int32, device=device).reshape(-1)
        self.n_hot = int(hot_rows.numel())
        self.n_rep = int(n_rep or self.N_REP)
        self.K = K
        self.rows = hot_rows.contiguous()
        self.slot = torch.full((M,), -1, dtype=torch.int32, device=device)
        self.slot[self.rows.long()] = torch.arange(self.n_hot, dtype=torch.int32, device=device)
        self.ghot = torch.zeros(self.n_rep, self.n_hot, K, dtype=torch.float32, device=device)
        self.ghot_bias = torch.zeros(self.n_rep, self.n_hot, dtype=torch.float32, device=device) if with_bias else None

    @classmethod
    def from_batch(cls, idx_dev, M, K, device, with_bias=False, exclude=None):
        """Pick the hot rows from the id histogram of one packed batch (one-time plumbing, not on the hot path):
        rows hit at least MIN_COUNT times, the MAX_HOT most frequent of them, never a row of `exclude` (the member rows
        of pooled context groups, which the scatter kernel does not reduce into).  Returns None if there are none."""
        flat = idx_dev.reshape(-1)
        flat = flat[flat >= 0].long()
        counts = torch.bincount(flat, minlength=M)
        if exclude is not None:
            counts[exclude.to(counts.device)] = 0
        hot = torch.nonzero(counts >= cls.MIN_COUNT).reshape(-1)
        if hot.numel() == 0:
            return None
        if hot.numel() > cls.MAX_HOT:
            hot = torch.topk(counts, cls.MAX_HOT).indices
        return cls(torch.sort(hot).values, M, K, device, with_bias)

    def args(self, with_bias=False):
        if with_bias:
            return (ptr(self.slot), ptr(self.ghot), ptr(self.ghot_bias), self.n_rep, self.n_hot)
        return (ptr(self.slot), ptr(self.ghot), self.n_rep, self.n_hot)

    def fold(self, gV, gbias=None):
        _lib.call("hhfm_hot_fold", ptr(self.ghot), ptr(self.ghot_bias) if gbias is not None else None, self.n_rep,
                  self.n_hot, self.K, ptr(self.rows), ptr(gV), ptr(gbias), cur_stream())


NO_HOT = (None, None, 0, 0)
NO_HOT_BIAS = (None, None, None, 0, 0)


# --------------------------------------------------------------------------------------------------
# K3: pooled context groups (include/hhfm_sm100.h hhfm_pool_groups_attach)
# --------------------------------------------------------------------------------------------------
POOL_GROUP_CAP = 1 << 15          # combinations of one group
POOL_GROUP_TOTAL_CAP = 1 << 16    # combinations of all groups: 2^16 rows x K = 128 x 4 B = 32 MB per table, L2-resident
POOL_GROUP_MAX_SLOTS = 4          # pooled rows per sample after grouping that the kernels are compiled for


def plan_pool_groups(lo, card, cap=POOL_GROUP_CAP, total_cap=POOL_GROUP_TOTAL_CAP, max_slots=POOL_GROUP_MAX_SLOTS):
    """Group assignment of the pooled columns with id ranges [lo[c], lo[c] + card[c]) (card[c] < 1: not groupable).

    Columns are packed smallest first, each onto the open group while its cardinality product stays <= cap and the
    combinations of all groups <= total_cap, otherwise the group is closed and a new one opened.  Columns whose range
    overlaps another groupable column's are not grouped (their member rows must be distinct), a group of one column is
    dissolved (it would remove nothing), and if the pooled rows per sample after grouping would exceed max_slots or not
    drop, nothing is grouped.  Returns a list: group number per column, -1 = ungrouped."""
    n = len(card)
    ok = [card[c] >= 1 and lo[c] >= 0 for c in range(n)]
    for a in range(n):
        for b in range(a + 1, n):
            if ok[a] and ok[b] and lo[a] < lo[b] + card[b] and lo[b] < lo[a] + card[a]:
                ok[a] = ok[b] = False
    groups, cur, prod, total = [], [], 1, 0
    for c in sorted((c for c in range(n) if ok[c]), key=lambda c: (card[c], c)):
        if cur and prod * card[c] <= cap and total + prod * card[c] <= total_cap:
            cur.append(c)
            prod *= card[c]
            continue
        if len(cur) >= 2:
            groups.append(cur)
            total += prod
        cur, prod = ([c], card[c]) if (card[c] <= cap and total + card[c] <= total_cap) else ([], 1)
    if len(cur) >= 2:
        groups.append(cur)
    out = [-1] * n
    for g, cols in enumerate(groups):
        for c in cols:
            out[c] = g
    n_slots = len(groups) + out.count(-1)
    if not groups or n_slots > max_slots or n_slots >= n:
        return [-1] * n
    return out


def pool_group_index(ids, lo, card, members):
    """Mixed-radix combination index of one group for rows of pooled ids [B, n_pool] (numpy): first member least
    significant, members in record order.  Returns (index [B], in_range [B]); out-of-range rows are the fallback samples."""
    ids = np.asarray(ids, dtype=np.int64)
    k = np.zeros(ids.shape[0], dtype=np.int64)
    ok = np.ones(ids.shape[0], dtype=bool)
    mult = 1
    for c in sorted(members):
        d = ids[:, c] - lo[c]
        ok &= (d >= 0) & (d < card[c])
        k += d * mult
        mult *= card[c]
    return k, ok


class PoolGroups:
    """Pooled context groups of one table (hhfm_pool_groups_attach), planned from the id ranges of one packed batch.
    The library owns the group tables; the plan is detached when this object goes away."""

    def __init__(self, V, n_pool, stride, lo, card, groups):
        self.V = V
        self.groups = list(groups)
        self.lo, self.card = list(lo), list(card)
        M, K = V.shape
        arr = lambda xs: np.ascontiguousarray(np.asarray(xs, dtype=np.int32))
        self._g, self._lo, self._card = arr(groups), arr(lo), arr(card)
        h = C.c_int64(0)
        _lib.call("hhfm_pool_groups_attach", ptr(V), M, K, n_pool, stride, ptr(self._g), ptr(self._lo), ptr(self._card),
                  C.byref(h))
        self.handle = h.value
        self._fin = weakref.finalize(self, PoolGroups._detach, V.data_ptr(), self.handle)
        self._fin.atexit = False

    @staticmethod
    def _detach(v_ptr, handle):
        _lib.load().hhfm_pool_groups_detach(C.c_void_p(v_ptr), handle)

    def member_rows(self):
        """Table rows covered by a group (int64 numpy)."""
        return np.concatenate([np.arange(self.lo[c], self.lo[c] + self.card[c]) for c in range(len(self.groups))
                               if self.groups[c] >= 0]).astype(np.int64)

    def tables(self):
        """(S, G): copies of the library's group tables, [rows, K] float32 on the table's device (tests, inspection)."""
        S, G, rows = C.c_void_p(), C.c_void_p(), C.c_int64()
        _lib.call("hhfm_pool_groups_tables", ptr(self.V), C.byref(S), C.byref(G), C.byref(rows))
        shape = (rows.value, self.V.shape[1])

        class _View:           # __cuda_array_interface__ of a library-owned buffer
            def __init__(self, p):
                self.__cuda_array_interface__ = {"shape": shape, "typestr": "<f4", "data": (p, False), "version": 2}

        with torch.cuda.device(self.V.device):
            return tuple(torch.as_tensor(_View(p.value), device=self.V.device).clone() for p in (S, G))

    @classmethod
    def from_batch(cls, V, idx_dev, n_pool):
        """Plan from the pooled columns [2, 2 + n_pool) of one packed batch: each column's range is [min, max].  Returns
        None when HHFM_POOL_GROUPS=0, the configuration is not covered, or no group forms."""
        if os.environ.get("HHFM_POOL_GROUPS") == "0" or n_pool not in (3, 8, 10) or V.shape[1] not in (32, 64, 128):
            return None
        cols = idx_dev[:, 2:2 + n_pool]
        lo = cols.min(0).values.cpu().numpy().astype(np.int64)
        hi = cols.max(0).values.cpu().numpy().astype(np.int64)
        card = [int(h - l + 1) if l >= 0 else 0 for l, h in zip(lo, hi)]
        groups = plan_pool_groups([int(x) for x in lo], card)
        if all(g < 0 for g in groups):
            return None
        return cls(V, n_pool, idx_dev.shape[1], [int(x) if g >= 0 else 0 for x, g in zip(lo, groups)],
                   [c if g >= 0 else 0 for c, g in zip(card, groups)], groups)


# --------------------------------------------------------------------------------------------------
# K6/K7: full-catalog top-N, exact path
# --------------------------------------------------------------------------------------------------
class TopN:
    """Full-catalog scorer + selector over an item shard [item_lo, item_hi) of the catalog.

    method="exact": fp32 SIMT scorer (canonical order) + radix select.
    method="tc":    tcgen05 bf16 GEMM filter with a fused group-max epilogue, exact rescoring of the survivors, select;
                    same lists bit for bit (see csrc/topn_tc.cu).
    method="auto":  "tc" when the configuration is supported and the problem is big enough to leave launch latency
                    behind (C*N >= 2^22 pairs), otherwise "exact".
    """

    def __init__(self, device, max_workspace_bytes=1 << 30):
        self.device = device
        self.stage = Staging(torch.int32, device)
        self.max_ws = max_workspace_bytes
        self._ws = None
        self._ws_bytes = None
        self._items = {}            # (kind, lo, hi) -> (version, operand, stats)
        self.last_method = None
        self.last_overflow_rows = 0

    def _workspace(self, numel):
        if self._ws is None or self._ws.numel() < numel:
            self._ws = torch.empty(numel, dtype=torch.float32, device=self.device)
        return self._ws[:numel]

    def _byte_workspace(self, nbytes):
        if self._ws_bytes is None or self._ws_bytes.numel() < nbytes:
            self._ws_bytes = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        return self._ws_bytes

    def upload_rows(self, A, id_limit):
        host, stride = pack_records([A], id_limit, self.stage)
        dev = self.stage.upload(host.numel()).view(host.shape[0], stride)
        return dev, stride

    def build_query(self, kind, A_dev, stride, n_ctx, n_time, pools, V):
        C_rows = A_dev.shape[0]
        M, K = V.shape
        Q = torch.empty(C_rows, K, dtype=torch.float32, device=self.device)
        Fc = torch.empty(C_rows, K, dtype=torch.float32, device=self.device) if kind == QUERY_FM else None
        _lib.call("hhfm_topn_build_query", kind, ptr(A_dev), C_rows, stride, n_ctx, n_time, pools[0], pools[1], pools[2],
                  ptr(V), M, K, ptr(Q), ptr(Fc), cur_stream())
        return Q, Fc

    def topk(self, kind, A_dev, stride, n_ctx, n_time, pools, V, bias, n_user, n_item, tp, item_lo=0, item_hi=None,
             return_scores=False, method="auto", version=None):
        """A_dev int32 [C,stride] on device.  Returns ids int32 [C,tp] relative to the item range (+ scores)."""
        item_hi = n_item if item_hi is None else item_hi
        N = item_hi - item_lo
        C_rows = A_dev.shape[0]
        K = V.shape[1]
        Q, Fc = self.build_query(kind, A_dev, stride, n_ctx, n_time, pools, V)
        items = V[n_user + item_lo:n_user + item_hi]
        ibias = bias.reshape(-1)[n_user + item_lo:n_user + item_hi] if (bias is not None and kind == QUERY_FM) else None
        lib = _lib.load()
        supported = bool(lib.hhfm_topn_tc_supported(kind, N, K, tp)) and N > 0
        if method == "tc" and not supported:
            raise _lib.HhfmError("tensor-core top-N does not cover kind=%d N=%d K=%d tp=%d" % (kind, N, K, tp))
        use_tc = supported and (method == "tc" or (method == "auto" and C_rows * N >= (1 << 22)))
        self.last_method = "tc" if use_tc else "exact"
        if use_tc:
            out_ids, out_sc = self._topk_tc(kind, Q, Fc, items, ibias, N, K, tp, item_lo, version)
        else:
            out_ids, out_sc = self._topk_exact(kind, Q, Fc, items, ibias, N, K, tp, item_lo)
        return (out_ids, out_sc) if return_scores else out_ids

    def topk_from_query(self, Q, items, tp, method="auto", version=None):
        """Top-tp items per row of a precomputed query matrix Q [C, K] under score = sum_k fl(q_k * v_nk) (the QUERY_USER
        scorer); ids are item offsets."""
        N, K = items.shape
        lib = _lib.load()
        supported = bool(lib.hhfm_topn_tc_supported(QUERY_USER, N, K, tp)) and N > 0
        use_tc = supported and (method == "tc" or (method == "auto" and Q.shape[0] * N >= (1 << 22)))
        self.last_method = "tc" if use_tc else "exact"
        Q = Q.contiguous()
        if use_tc:
            ids, _ = self._topk_tc(QUERY_USER, Q, None, items, None, N, K, tp, 0, version)
        else:
            ids, _ = self._topk_exact(QUERY_USER, Q, None, items, None, N, K, tp, 0)
        return ids

    def _topk_exact(self, kind, Q, Fc, items, ibias, N, K, tp, item_lo):
        C_rows = Q.shape[0]
        st = cur_stream()
        out_ids = torch.empty(C_rows, tp, dtype=torch.int32, device=self.device)
        out_sc = torch.empty(C_rows, tp, dtype=torch.float32, device=self.device)
        chunk = max(1, min(C_rows, self.max_ws // max(1, 4 * N), 65535 * 32))
        for c0 in range(0, C_rows, chunk):
            c1 = min(C_rows, c0 + chunk)
            ws = self._workspace((c1 - c0) * N).view(c1 - c0, N)
            _lib.call("hhfm_topn_score_exact", kind, ptr(Q[c0:c1]), ptr(Fc[c0:c1]) if Fc is not None else None, c1 - c0,
                      ptr(items), ptr(ibias), N, K, ptr(ws), N, st)
            _lib.call("hhfm_topn_select", ptr(ws), None, None, c1 - c0, N, N, tp, item_lo, ptr(out_sc[c0:c1]),
                      ptr(out_ids[c0:c1]), st)
        return out_ids, out_sc

    def _item_operand(self, kind, items, ibias, N, K, key, version):
        hit = self._items.get(key)
        if hit is not None and version is not None and hit[0] == version:
            return hit[1], hit[2]
        lib = _lib.load()
        nbytes = int(lib.hhfm_topn_tc_item_operand_bytes(kind, N, K))
        op = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        stats = torch.zeros(2, dtype=torch.float32, device=self.device)
        _lib.call("hhfm_topn_tc_prepare_items", kind, ptr(items), ptr(ibias), N, K, ptr(op), ptr(stats), cur_stream())
        self._items[key] = (version, op, stats)
        return op, stats

    def _topk_tc(self, kind, Q, Fc, items, ibias, N, K, tp, item_lo, version):
        lib = _lib.load()
        C_rows = Q.shape[0]
        st = cur_stream()
        op, stats = self._item_operand(kind, items, ibias, N, K, (kind, item_lo, item_lo + N), version)
        out_ids = torch.empty(C_rows, tp, dtype=torch.int32, device=self.device)
        out_sc = torch.empty(C_rows, tp, dtype=torch.float32, device=self.device)
        overflow = torch.zeros(C_rows, dtype=torch.int32, device=self.device)
        chunk = C_rows                 # largest context chunk whose workspace fits the budget
        while chunk > 128 and int(lib.hhfm_workspace_bytes_topn(kind, chunk, N, K, tp)) > self.max_ws:
            chunk = max(128, (chunk // 2 + 127) // 128 * 128)
        for c0 in range(0, C_rows, chunk):
            c1 = min(C_rows, c0 + chunk)
            nbytes = int(lib.hhfm_workspace_bytes_topn(kind, c1 - c0, N, K, tp))
            ws = self._byte_workspace(nbytes)
            fcp = ptr(Fc[c0:c1]) if Fc is not None else None
            _lib.call("hhfm_topn_score", kind, ptr(Q[c0:c1]), fcp, c1 - c0, ptr(op), N, K, tp, ptr(stats), ptr(ws), nbytes, st)
            _lib.call("hhfm_topn_rescore_merge", kind, ptr(Q[c0:c1]), fcp, c1 - c0, ptr(items), ptr(ibias), N, K,
                      tp, item_lo, ptr(ws), nbytes, ptr(out_sc[c0:c1]), ptr(out_ids[c0:c1]), ptr(overflow[c0:c1]), st)
        bad = torch.nonzero(overflow).reshape(-1)
        self.last_overflow_rows = int(bad.numel())
        if bad.numel() > 0:          # candidate buffer overflowed (tie-degenerate rows): redo those rows exactly
            Qb = Q[bad].contiguous()
            Fb = Fc[bad].contiguous() if Fc is not None else None
            ids_b, sc_b = self._topk_exact(kind, Qb, Fb, items, ibias, N, K, tp, item_lo)
            out_ids[bad] = ids_b
            out_sc[bad] = sc_b
        return out_ids, out_sc


def metrics_walk(pred_global, target, target_in_pf, TopK):
    """Device evaluate_TopK walk (FM.py:336-357).  Tensors on device; returns rank codes int32 [C]."""
    C_rows, tp = pred_global.shape
    code = torch.empty(C_rows, dtype=torch.int32, device=pred_global.device)
    _lib.call("hhfm_metrics_walk", ptr(pred_global), ptr(target), ptr(target_in_pf), C_rows, tp, TopK, ptr(code),
              cur_stream())
    return code


def metrics_from_codes(codes):
    """[mean HR, mean NDCG, mean reciprocal rank] exactly as FM.py:340-359 builds them from the walk: the
    per-row values are appended in row order and averaged with np.average; rows with code -2 append nothing."""
    res_map, res_ndcg, res_pre = [], [], []
    for n in np.asarray(codes).tolist():
        if n == -2:
            continue
        if n == -1:
            res_map.append(0); res_ndcg.append(0); res_pre.append(0)
        else:
            res_map.append(1)
            res_ndcg.append(np.log(2) / np.log(n + 2))
            res_pre.append(1 / (n + 1))
    return [np.average(res_map), np.average(res_ndcg), np.average(res_pre)]
