"""GPU: MomentumOptimizer under data parallelism.

- `hhfm_dp_step_touched` with n_ranks == 1 against the separate kernels (fold + hhfm_opt_momentum_dense_l2 +
  hhfm_opt_momentum_rows over the compacted stamps), bit for bit; and against `hhfm_dp_step` for the other optimizers.
- Emulated ranks: the scatter kernel on 2, 3 and 8 shards of one batch into separate arenas and stamp arrays, the arenas
  added in rank order, the union taken with the MAX of the stamps + `hhfm_touched_compact`, then both the NCCL-path
  kernels and `hhfm_dp_step_touched` -- against oracle/momentum_dp.py.  (N > 1 of the fused kernel needs that many GPUs:
  its ranks wait on each other's flags.)
- The models under an NCCL group of min(device_count, 2) ranks with every exchange: teacher-forced against the oracle,
  untouched rows unmoved, replicas bit-identical.
"""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch

from oracle import momentum_dp as MD

pytestmark = pytest.mark.gpu

LR, MU = 0.05, 0.95


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _segs(specs):
    from hhfm_b200 import dist as hd
    arr = (hd.DpSegment * len(specs))()
    for i, (w, s1, s2, off, n, lam) in enumerate(specs):
        arr[i].w, arr[i].s1, arr[i].s2 = w.data_ptr(), (s1.data_ptr() if s1 is not None else None), \
            (s2.data_ptr() if s2 is not None else None)
        arr[i].offset, arr[i].n, arr[i].lamda = int(off), int(n), float(lam)
    return arr


def _dyadic(rng, shape, scale=6):
    """Small multiples of 2^-scale: every sum the fold forms is exact, whatever its order."""
    return torch.tensor(rng.integers(-8, 9, shape) * 2.0 ** -scale, dtype=torch.float32)


class _Problem:
    """Arena [gV (M*K) | gbias (M) | gb0], touched-row stamps, optional hot replicas; V, feature_bias, bias + Momentum slots."""

    def __init__(self, M, K, hot, seed, lamda):
        from hhfm_b200 import _lib
        rng = np.random.default_rng(seed)
        dev = "cuda"
        self.M, self.K, self.lamda = M, K, lamda
        self.n_g = M * K + M + 1
        touched = rng.random(M) < 0.4
        touched[[0, M - 1]] = True                       # the first and the last row of the table
        zero_g = touched & (rng.random(M) < 0.2)          # touched rows whose gradient is exactly 0
        gV = _dyadic(rng, (M, K)) * torch.tensor(touched & ~zero_g, dtype=torch.float32)[:, None]
        gb = _dyadic(rng, (M,)) * torch.tensor(touched & ~zero_g, dtype=torch.float32)
        self.arena = torch.zeros((self.n_g + 3) // 4 * 4 + 4, dtype=torch.float32)
        self.arena[:M * K] = gV.reshape(-1); self.arena[M * K:M * K + M] = gb; self.arena[M * K + M] = 0.375
        self.arena = self.arena.to(dev)
        self.stamps = torch.where(torch.tensor(touched), 5, torch.tensor(rng.integers(0, 5, M))).to(torch.int32).to(dev)
        self.lp = _dyadic(rng, (_lib.partials_len(),), 8).to(dev)
        self.V = torch.tensor(rng.normal(0, 0.1, (M, K)), dtype=torch.float32, device=dev)
        self.fb = torch.tensor(rng.normal(0, 0.1, (M, 1)), dtype=torch.float32, device=dev)
        self.b0 = torch.tensor([0.125], dtype=torch.float32, device=dev)
        self.s = [torch.tensor(np.abs(rng.normal(0, 0.05, t.shape)), dtype=torch.float32, device=dev)
                  for t in (self.V, self.fb, self.b0)]
        self.s2 = [torch.tensor(np.abs(rng.normal(0, 0.05, t.shape)), dtype=torch.float32, device=dev)
                   for t in (self.V, self.fb, self.b0)]
        self.hot = None
        if hot:
            rows = np.flatnonzero(touched)[::3][:16]
            n_rep = 5
            slot = torch.full((M,), -1, dtype=torch.int32)
            slot[torch.tensor(rows)] = torch.arange(len(rows), dtype=torch.int32)
            ghot = _dyadic(rng, (n_rep, len(rows), K)); ghb = _dyadic(rng, (n_rep, len(rows)))
            self.hot = (ghot.to(dev), ghb.to(dev), n_rep, len(rows), torch.tensor(rows, dtype=torch.int32, device=dev),
                        slot.to(dev))

    def clone(self):
        import copy
        c = copy.copy(self)
        for k in ("arena", "stamps", "lp", "V", "fb", "b0"):
            setattr(c, k, getattr(self, k).clone())
        c.s = [t.clone() for t in self.s]; c.s2 = [t.clone() for t in self.s2]
        if self.hot is not None:
            c.hot = (self.hot[0].clone(), self.hot[1].clone()) + self.hot[2:]
        return c

    def seg_specs(self, kind):
        M, K = self.M, self.K
        s2 = self.s2 if kind == "adam" else [None] * 3
        s1 = self.s if kind != "sgd" else [None] * 3
        return [(self.V, s1[0], s2[0], 0, M * K, self.lamda), (self.fb, s1[1], s2[1], M * K, M, 0.0),
                (self.b0, s1[2], s2[2], M * K + M, 1, 0.0)]

    def hargs(self):
        if self.hot is None:
            return (None, None, 0, 0, self.K, self.M, None, self.M * self.K)
        ghot, ghb, n_rep, n_hot, _, slot = self.hot
        return (_ptr(ghot), _ptr(ghb), n_rep, n_hot, self.K, self.M, _ptr(slot), self.M * self.K)

    def fused(self, kind, widths, touched_entry=True, lr=LR, b1=MU):
        from hhfm_b200 import _lib
        from hhfm_b200.engine import Optimizer
        lib = _lib.load()
        x = torch.zeros(int(lib.hhfm_dp_exchange_floats_touched(self.n_g)), dtype=torch.float32, device="cuda")
        state = torch.zeros(4, dtype=torch.int32, device="cuda")
        reg = torch.zeros(512, dtype=torch.float32, device="cuda")
        loss = torch.zeros(1, dtype=torch.float32, device="cuda")
        segs = _segs(self.seg_specs(kind))
        tail = (_ptr(self.lp), _ptr(x), None, None, None, 0, 1, _ptr(state), lr, b1, 0.999, 1e-8, _ptr(reg), _ptr(loss), 5.0, _st())
        k = Optimizer.KIND_ID[kind]
        if touched_entry:
            w = (C.c_int32 * 3)(*widths)
            _lib.call("hhfm_dp_step_touched", k, C.cast(segs, C.c_void_p), 3, w, _ptr(self.stamps), 5, _ptr(self.arena), self.n_g,
                      *self.hargs(), *tail)
        else:
            _lib.call("hhfm_dp_step", k, C.cast(segs, C.c_void_p), 3, _ptr(self.arena), self.n_g, *self.hargs(), *tail)
        torch.cuda.synchronize()
        return float(loss.item())

    def separate(self, v_rows):
        """The NCCL-path kernels of a Momentum step: fold, rows of the stamp union, row / dense updates, loss."""
        from hhfm_b200 import _lib
        M, K = self.M, self.K
        gV = self.arena[:M * K]; gb = self.arena[M * K:M * K + M]; gb0 = self.arena[M * K + M:M * K + M + 1]
        if self.hot is not None:
            ghot, ghb, n_rep, n_hot, rows, _ = self.hot
            _lib.call("hhfm_hot_fold", _ptr(ghot), _ptr(ghb), n_rep, n_hot, K, _ptr(rows), _ptr(gV), _ptr(gb), _st())
        rows = torch.empty(M, dtype=torch.int32, device="cuda"); cnt = torch.full((1,), 77, dtype=torch.int32, device="cuda")
        _lib.call("hhfm_touched_compact", _ptr(self.stamps), 5, M, _ptr(rows), _ptr(cnt), _st())
        sq = torch.zeros(_lib.partials_len(), dtype=torch.float32, device="cuda")
        if v_rows:
            _lib.call("hhfm_opt_momentum_rows", _ptr(self.V), _ptr(self.s[0]), _ptr(gV), _ptr(rows), _ptr(cnt), M, K, LR, MU, 1, _st())
        else:
            _lib.call("hhfm_opt_momentum_dense_l2", _ptr(self.V), _ptr(self.s[0]), _ptr(gV), M * K, LR, MU, self.lamda, 1, _ptr(sq), _st())
        _lib.call("hhfm_opt_momentum_rows", _ptr(self.fb), _ptr(self.s[1]), _ptr(gb), _ptr(rows), _ptr(cnt), M, 1, LR, MU, 1, _st())
        _lib.call("hhfm_opt_momentum_dense_l2", _ptr(self.b0), _ptr(self.s[2]), _ptr(gb0), 1, LR, MU, 0.0, 1, None, _st())
        loss = torch.zeros(1, dtype=torch.float32, device="cuda")
        _lib.call("hhfm_loss_finalize", _ptr(self.lp), _ptr(sq) if not v_rows else None, 0.5 * self.lamda, _ptr(loss), _st())
        torch.cuda.synchronize()
        return float(loss.item()), int(cnt.item())

    def result(self):
        return [t.cpu().numpy() for t in (self.V, self.fb, self.b0, *self.s)]


@pytest.mark.parametrize("K", [32, 64, 128, 100])
@pytest.mark.parametrize("hot", [False, True])
@pytest.mark.parametrize("lamda", [0.0, 0.1])
def test_dp_step_touched_one_rank_is_bit_identical_to_the_separate_momentum_kernels(cuda, K, hot, lamda):
    M = 203                                              # odd: the scalar bias gradient is not float4-aligned
    base = _Problem(M, K, hot, seed=K + 7 * hot + int(lamda * 10), lamda=lamda)
    a, b = base.clone(), base.clone()
    v_rows = lamda == 0
    loss_f = a.fused("momentum", (K if v_rows else 0, 1, 0))
    loss_s, n_rows = b.separate(v_rows)
    assert n_rows == int((base.stamps == 5).sum())
    for x, y, name in zip(a.result(), b.result(), ("V", "feature_bias", "bias", "acc V", "acc feature_bias", "acc bias")):
        assert np.array_equal(x, y), name
    assert abs(loss_f - loss_s) <= 1e-5 * abs(loss_s)
    assert float(a.arena[:base.n_g].abs().max()) == 0.0                # the fused step clears the arena
    untouched = (base.stamps != 5).cpu().numpy()
    for x, y in ((a.result()[1], base.fb), (a.result()[4], base.s[1])):
        assert np.array_equal(x[untouched], y.cpu().numpy()[untouched])
    if v_rows:
        assert np.array_equal(a.result()[0][untouched], base.V.cpu().numpy()[untouched])
    moved = (base.stamps == 5).cpu().numpy()
    assert not np.array_equal(a.result()[4][moved], base.s[1].cpu().numpy()[moved])     # zero-gradient rows decay too


@pytest.mark.parametrize("kind", ["adagrad", "sgd", "adam"])
@pytest.mark.parametrize("hot", [False, True])
def test_dp_step_touched_equals_dp_step_for_the_other_optimizers(cuda, kind, hot):
    M, K = 150, 64
    base = _Problem(M, K, hot, seed=3, lamda=0.1)
    a, b = base.clone(), base.clone()
    la = a.fused(kind, (0, 0, 0), lr=0.1, b1=0.9)
    lb = b.fused(kind, (0, 0, 0), touched_entry=False, lr=0.1, b1=0.9)
    assert la == lb
    for x, y in zip(a.result(), b.result()):
        assert np.array_equal(x, y)
    if kind != "adam":                   # untouched rows carry g = 0: Adagrad and SGD leave them where they are
        base0 = _Problem(M, K, hot, seed=4, lamda=0.0)
        a, b = base0.clone(), base0.clone()
        a.fused(kind, (K, 1, 0), lr=0.1, b1=0.9)
        b.fused(kind, (0, 0, 0), touched_entry=False, lr=0.1, b1=0.9)
        for x, y in zip(a.result(), b.result()):
            assert np.array_equal(x, y)


# ---- emulated ranks: the NCCL path's union on one GPU ----------------------------------------------------------------
@pytest.mark.parametrize("n_ranks", [2, 3, 8])
@pytest.mark.parametrize("lamda", [0.0, 0.1])
def test_emulated_ranks_union_step_matches_the_global_batch_oracle(cuda, n_ranks, lamda):
    from hhfm_b200 import _lib
    from hhfm_b200 import dist as hd
    rng = np.random.default_rng(n_ranks)
    M, K, F, B = 300, 64, 5, 1200
    X = rng.integers(0, M - 41, (B, F)).astype(np.int32)          # rows M-40 .. M-1: touched by nobody
    X[hd.shard_range(B, n_ranks - 1, n_ranks)[0], 0] = M - 41     # row M-41: by the last rank alone
    Y = rng.choice([1.0, 0.0], B).astype(np.float32)
    P = _lib.partials_len()
    V = torch.tensor(rng.normal(0, 0.1, (M, K)), dtype=torch.float32, device="cuda")
    fb = torch.tensor(rng.normal(0, 0.1, (M, 1)), dtype=torch.float32, device="cuda")
    b0 = torch.tensor([0.1], dtype=torch.float32, device="cuda")
    n_g = M * K + M + 1
    arena = torch.zeros(n_g + 3 + P + 4, dtype=torch.float32, device="cuda")
    stamps = []
    for r in range(n_ranks):
        lo, hi = hd.shard_range(B, r, n_ranks)
        idx = torch.tensor(X[lo:hi], device="cuda"); y = torch.tensor(Y[lo:hi], device="cuda")
        a = torch.zeros_like(arena)
        st_r = torch.zeros(M, dtype=torch.int32, device="cuda")
        rows = torch.empty(M, dtype=torch.int32, device="cuda"); cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
        _lib.call("hhfm_fm_fwd_bwd_sqloss_dropout", None, _ptr(idx), None, hi - lo, F, _ptr(V), _ptr(fb), _ptr(b0), M, K, 0,
                  _ptr(y), None, _ptr(a[:M * K]), _ptr(a[M * K:M * K + M]), _ptr(a[M * K + M:]), _ptr(a[n_g + 3:n_g + 3 + P]),
                  _ptr(st_r), 5, _ptr(rows), _ptr(cnt), None, None, None, 0, 0, 1, 1.0, 0, _st())
        arena += a                                                   # rank order
        stamps.append(st_r)
    union = torch.stack(stamps).amax(0)                              # what the MAX all-reduce leaves on every rank
    w0 = {"feature_embeddings": V.cpu().numpy(), "feature_bias": fb.cpu().numpy(), "bias": np.float32(0.1)}
    acc0 = {k: np.zeros(np.shape(v), np.float32) for k, v in w0.items()}
    shards = [slice(*hd.shard_range(B, r, n_ranks)) for r in range(n_ranks)]
    loss_ref, w1, a1 = MD.fm_step([X[s] for s in shards], [Y[s].reshape(-1, 1) for s in shards], w0, acc0, LR, lamda)
    results = {}
    for how in ("separate", "fused"):
        pr = _Problem.__new__(_Problem)
        pr.M, pr.K, pr.lamda, pr.n_g, pr.hot = M, K, lamda, n_g, None
        pr.arena = arena[:n_g + 3].clone(); pr.stamps = union.clone(); pr.lp = arena[n_g + 3:n_g + 3 + P].clone()
        pr.V, pr.fb, pr.b0 = V.clone(), fb.clone(), b0.clone()
        pr.s = [torch.zeros_like(t) for t in (pr.V, pr.fb, pr.b0)]; pr.s2 = [None] * 3
        loss = pr.separate(lamda == 0)[0] if how == "separate" else pr.fused("momentum", (K if lamda == 0 else 0, 1, 0))
        got = pr.result()
        results[how] = got
        assert abs(loss - float(loss_ref)) <= 2e-5 * abs(float(loss_ref)), how
        for g, name, acc_name in ((got[0], "feature_embeddings", 3), (got[1], "feature_bias", 4)):
            ref, ref_a, prev = w1[name], a1[name], w0[name]
            upd = ref - prev
            tol = 1e-4 * np.maximum(np.abs(upd), np.sqrt(np.mean(upd ** 2)))
            assert np.all(np.abs(g - ref) <= tol), (how, name)
            assert np.all(np.abs(got[acc_name] - ref_a) <= 1e-4 * np.maximum(np.abs(ref_a), np.sqrt(np.mean(ref_a ** 2)))), (how, name)
        assert np.array_equal(got[1][M - 40:], w0["feature_bias"][M - 40:]) and not got[4][M - 40:].any(), how
        assert got[4][M - 41] != 0                                    # the last rank's own row moved everywhere
        if lamda == 0:
            assert np.array_equal(got[0][M - 40:], w0["feature_embeddings"][M - 40:]), how
    for x, y in zip(results["separate"], results["fused"]):
        assert np.array_equal(x, y)


# ---- the models under an NCCL group ----------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


MODES = [dict(fused="auto"), dict(fused=False), dict(sparse=True)]
CASES = ["fm_l2", "fm", "fm_hot", "fm_bn", "afm", "mf", "our", "bpr", "our_l2"]


def _slots(m):
    return {k: (m._opt.state[k][0].cpu().numpy().reshape(np.shape(v)) if k in m._opt.state else np.zeros(np.shape(v), np.float32))
            for k, v in m.get_weights().items()}


def _close(got, ref, prev, rtol=1e-4, floor=0.0):
    upd = np.asarray(ref, np.float64) - np.asarray(prev, np.float64)
    scale = max(float(np.sqrt(np.mean(upd ** 2))), 1e-12)
    return bool(np.all(np.abs(np.asarray(got, np.float64) - ref) <= rtol * np.maximum(np.abs(upd), scale) + floor))


# AFM: d attention_b / d attention_p sum d s_p over the pairs, which sums to zero per sample -- cancellation noise, floored
# at 1e-4 of the attention_W update as in the AFM dropout tests
AFM_NOISY = ("attention_b", "attention_p")


def _case(name, mode, dp=True):
    """Returns (model, [global batches], step(model, batch, lo, hi), oracle(w, acc, batch, shards) or None, untouched rows)."""
    from hhfm_b200.models import AFM, BPR, FM, MF, OUR
    rng = np.random.default_rng(17)
    n_user, n_item, K, B = 60, 140, 32, 512
    M = n_user + n_item + 60                                          # the last 20 rows: touched by nobody
    free = np.arange(M - 20, M)
    if name.startswith("fm") or name in ("afm", "mf"):
        F = 5
        batches = []
        for _ in range(3):
            X = np.concatenate([np.stack([rng.integers(0, n_user, B), n_user + rng.integers(0, n_item, B)], axis=1),
                                rng.integers(n_user + n_item, M - 20, (B, F - 2))], axis=1)
            batches.append((X, rng.choice([1.0, 0.0], (B, 1)).astype(np.float32)))
        lam = 0.1 if name == "fm_l2" else 0.0
        if name == "afm":
            m = AFM(n_user, n_item, M, 1, [16, 16], "relu", LR, 0.01, [1.0, 1.0], "MomentumOptimizer", 0.9, F)
        elif name == "mf":
            m = MF(M, n_user, n_item, K, LR, 0.0, 1.0, "MomentumOptimizer", 0, 0)
        else:
            m = FM(F, M, n_user, n_item, K, LR, lam, 1.0, "MomentumOptimizer", 1 if name == "fm_bn" else 0, 0)
        if name == "fm_hot":
            m.hot_rows = list(range(n_user + n_item, n_user + n_item + 8))     # context rows: ~100 hits each per batch
        else:
            m.hot_rows = None
        if dp:
            m.enable_data_parallel(**(dict(mode, sync_batch_norm=True) if name == "fm_bn" else mode))

        def step(model, bt, lo, hi):
            return model.partial_fit({"X": bt[0][lo:hi], "Y": bt[1][lo:hi]})

        if name == "fm_bn":
            oracle = None
        elif name == "afm":
            def oracle(w, acc, bt, sh):
                return MD.afm_step([bt[0][s] for s in sh], [bt[1][s] for s in sh], w, acc, LR, 0.01)
        else:
            def oracle(w, acc, bt, sh, lam=lam):
                return MD.fm_step([bt[0][s] for s in sh], [bt[1][s] for s in sh], w, acc, LR, lam,
                                  interaction=1 if name == "mf" else 0)
        return m, batches, step, oracle, free
    fc = 0 if name == "bpr" else 4
    batches = []
    for _ in range(3):
        X = np.stack([rng.integers(0, n_user, B), n_user + rng.integers(0, n_item, B)], axis=1)
        Fe = rng.integers(n_user + n_item, M - 20, (B, fc)) if fc else None
        batches.append((X, Fe, n_user + rng.integers(0, n_item, (B, 10))))
    lam = 0.01 if name == "our_l2" else 0.0
    m = BPR(M, n_user, n_item, K, LR, lam, "MomentumOptimizer") if name == "bpr" else \
        OUR(fc, 0, M, n_user, n_item, K, LR, lam, "MomentumOptimizer", True, False)
    m.hot_rows = None
    if dp:
        m.enable_data_parallel(**mode)

    def step(model, bt, lo, hi):
        d = {"X": bt[0][lo:hi], "Y": bt[2][lo:hi]}
        if bt[1] is not None:
            d["F1"] = bt[1][lo:hi]
        return model.partial_fit(d)

    def oracle(w, acc, bt, sh):
        return MD.pairrank_step([bt[0][s] for s in sh], [bt[2][s] for s in sh], None if bt[1] is None else [bt[1][s] for s in sh],
                                w, acc, LR, lam)
    return m, batches, step, oracle, free


def _model_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from hhfm_b200 import dist as hd
        out = {}
        for name in CASES:
            for mode in MODES:
                key = "%s/%s" % (name, ",".join("%s=%s" % kv for kv in mode.items()))
                m, batches, step, oracle, free = _case(name, mode)
                ok, fails = True, []
                if name == "fm_bn":              # against the single-GPU step on the global batch
                    ref = _case("fm_bn", mode, dp=False)[0]
                B = batches[0][0].shape[0]
                lo, hi = hd.shard_range(B, rank, world)
                sh = [slice(*hd.shard_range(B, r, world)) for r in range(world)]
                for bt in batches:
                    w0, a0 = m.get_weights(), _slots(m)
                    loss = step(m, bt, lo, hi)
                    w1, a1 = m.get_weights(), _slots(m)
                    if oracle is not None:
                        lr_, wr, ar = oracle(w0, a0, bt, sh)
                        ok = ok and abs(loss - float(lr_)) <= 2e-4 * abs(float(lr_))
                        for k in wr:
                            fw = fa = 0.0
                            if name == "afm" and k in AFM_NOISY:
                                fw = 1e-4 * float(np.abs(wr["attention_W"] - w0["attention_W"]).max())
                                fa = 1e-4 * float(np.abs(ar["attention_W"] - a0["attention_W"]).max())
                            good = _close(w1[k], wr[k], w0[k], floor=fw) and _close(a1[k], ar[k], a0[k], floor=fa)
                            if not good:
                                fails.append(k)
                            ok = ok and good
                    else:
                        lr_ = step(ref, bt, 0, B)
                        wr = ref.get_weights()
                        ok = ok and abs(loss - lr_) <= 2e-4 * abs(lr_)
                        for k in ("feature_embeddings", "feature_bias", "bias"):
                            ok = ok and _close(w1[k], wr[k], w0[k], 2e-3)
                    for k in ("feature_embeddings", "feature_bias"):
                        if k in w1 and not (k == "feature_embeddings" and name in ("fm_l2", "our_l2")):
                            ok = ok and np.array_equal(w1[k][free], w0[k][free]) and np.array_equal(a1[k][free], a0[k][free])
                same = True
                for k, w in m.weights.items():
                    g = [torch.empty_like(w) for _ in range(world)]
                    dist.all_gather(g, w.contiguous())
                    same = same and all(bool(torch.equal(g[0], x)) for x in g)
                out[key] = (bool(ok), same, m._use_fused_tail(), m._dp_sparse, sorted(set(fails)))
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def test_models_train_with_momentum_on_every_exchange(cuda):
    import torch.multiprocessing as mp
    world = min(torch.cuda.device_count(), 2)
    mgr = mp.Manager(); ret = mgr.dict()
    mp.spawn(_model_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    for r in range(world):
        res = ret[r]
        assert len(res) == len(CASES) * len(MODES)
        bad = {k: v for k, v in res.items() if not (v[0] and v[1])}
        assert not bad, (r, bad)
        if world > 1:                    # the exchange each mode picks
            assert res["fm/fused=auto"][2] and res["our_l2/fused=auto"][2]
            assert res["fm/sparse=True"][3] and not res["afm/fused=auto"][2]
