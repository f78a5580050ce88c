"""GPU: synchronised batch norm (FM batch_norm=1 under data parallelism) -- the three phase entry points of csrc/fm_bn.cu
with one rank against the single call, bit for bit; several ranks emulated on one GPU (one workspace and one layer state
per rank, the per-rank vectors stacked in rank order as the all-gather delivers them) against the oracle step on the
global batch; the empty global batch; and FM.enable_data_parallel(sync_batch_norm=True) over NCCL."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import fm_batchnorm as BN
from oracle import fm_batchnorm_sync as SB
from test_gpu_fm_batchnorm import _GKEY, _NAMES, _abs_terms, _check_pass, _problem, _train_call, _update, dev

pytestmark = pytest.mark.gpu

_LAYER = ("gamma", "beta", "mm", "mv")


def _sync_call(cuda, X, Y, w, sizes, keep, seed, hot, det=1):
    """One step through hhfm_fm_bn_sync_stats / _loss / _scatter for len(sizes) emulated ranks holding consecutive shards
    of X.  Every rank has its own workspace, layer state and gradient buffers; V, b and b0 are shared.  Returns one dict per
    rank in the shape of _train_call's (hot replicas folded)."""
    from hhfm_b200 import _lib
    from hhfm_b200.engine import HotRows, cur_stream, ptr
    lib = _lib.load()
    M, K = w["V"].shape
    F = X.shape[1]
    N = len(sizes)
    L = int(lib.hhfm_fm_bn_sync_len(K))
    cuts = np.cumsum([0] + list(sizes))
    stats_all = torch.full((N, L), np.nan, dtype=torch.float64, device=cuda)
    sums_all = torch.full((N, L), np.nan, dtype=torch.float64, device=cuda)
    shared = {k: dev(np.asarray(w[k]).reshape(-1) if k == "b0" else w[k], cuda) for k in ("V", "b", "b0")}
    st = cur_stream()
    ranks = []
    for r in range(N):
        B = int(sizes[r])
        R = dict(B=B, X=dev(X[cuts[r]:cuts[r + 1]], cuda, torch.int32), Y=dev(Y[cuts[r]:cuts[r + 1]], cuda))
        R.update({k: dev(w[k], cuda) for k in _LAYER})
        R.update(gV=torch.zeros(M, K, device=cuda), gb=torch.zeros(M, device=cuda), gb0=torch.zeros(1, device=cuda),
                 dgb=torch.full((2, K), 7.0, device=cuda), lp=torch.zeros(_lib.partials_len(), device=cuda),
                 out=torch.empty(B, device=cuda), lo=torch.zeros(1, device=cuda),
                 ws=torch.empty(int(lib.hhfm_workspace_bytes_fm_bn_sync(B, K)), dtype=torch.uint8, device=cuda))
        if hot:
            R["hp"] = HotRows(np.arange(0, 8), M, K, cuda, with_bias=True, n_rep=4)
            R["stamp"] = torch.zeros(M, dtype=torch.int32, device=cuda)
            R["rows"] = torch.zeros(M, dtype=torch.int32, device=cuda)
            R["cnt"] = torch.zeros(1, dtype=torch.int32, device=cuda)
            R["tail"] = (ptr(R["stamp"]), 3, ptr(R["rows"]), ptr(R["cnt"]), *R["hp"].args(True))
        else:
            R["tail"] = (None, 0, None, None, None, None, None, 0, 0)
        ranks.append(R)
    for r, R in enumerate(ranks):
        _lib.call("hhfm_fm_bn_sync_stats", ptr(R["X"]), R["B"], F, ptr(shared["V"]), ptr(shared["b"]), M, K, ptr(stats_all[r]),
                  ptr(R["ws"]), R["ws"].numel(), st)
    for r, R in enumerate(ranks):
        _lib.call("hhfm_fm_bn_sync_loss", R["B"], K, ptr(shared["b0"]), ptr(R["Y"]), ptr(R["out"]), ptr(R["gb0"]), ptr(R["lp"]),
                  keep, seed, ptr(R["gamma"]), ptr(R["beta"]), ptr(R["mm"]), ptr(R["mv"]), 1e-3, 0.9, ptr(stats_all), N, r,
                  ptr(sums_all[r]), ptr(R["ws"]), R["ws"].numel(), st)
    for r, R in enumerate(ranks):
        _lib.call("hhfm_fm_bn_sync_scatter", ptr(R["X"]), R["B"], F, ptr(shared["V"]), M, K, ptr(R["gV"]), ptr(R["gb"]), *R["tail"],
                  det, keep, seed, ptr(R["dgb"][0]), ptr(R["dgb"][1]), ptr(sums_all), N, ptr(R["ws"]), R["ws"].numel(), st)
    res = []
    for R in ranks:
        if hot:
            R["hp"].fold(R["gV"], R["gb"])
        _lib.call("hhfm_loss_finalize", ptr(R["lp"]), None, 0.0, ptr(R["lo"]), st)
        res.append(dict(out=R["out"].cpu().numpy(), loss=R["lo"].item(), V=R["gV"].cpu().numpy(), b=R["gb"].cpu().numpy(),
                        b0=R["gb0"].item(), gamma=R["dgb"][0].cpu().numpy(), beta=R["dgb"][1].cpu().numpy(),
                        mm=R["mm"].cpu().numpy(), mv=R["mv"].cpu().numpy()))
    return res


def _bits_equal(a, b):
    a = np.asarray(a, np.float32).reshape(-1); b = np.asarray(b, np.float32).reshape(-1)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _one_rank_cases():
    return [(B, K, keep, hot) for B in (1, 2, 5000, 1 << 17) for K in (8, 64, 100, 512) for keep in (1.0, 0.7)
            for hot in (False, True)]


@pytest.mark.parametrize("B,K,keep,hot", _one_rank_cases())
def test_one_rank_is_bit_identical_to_the_single_call(cuda, B, K, keep, hot):
    F = 3 if B > 5000 else 6
    w, X, Y = _problem(B, F, K, seed=B + K + 1)
    seed = 0x5DEECE66D + B * K
    want = _train_call(cuda, X, Y, w, keep, seed, hot, det=1)
    got, = _sync_call(cuda, X, Y, w, [B], keep, seed, hot, det=1)
    for k in ("out", "loss", "V", "b", "b0", "gamma", "beta", "mm", "mv"):
        assert _bits_equal(got[k], want[k]), k


def _shard_sizes(B, N, seed):
    rng = np.random.default_rng(seed)
    cut = np.sort(rng.choice(np.arange(1, B), N - 1, replace=False))
    sizes = np.diff(np.concatenate([[0], cut, [B]]))
    if N > 2:                                                    # one empty shard, its rows given to the next one
        sizes[N // 2 + 1] += sizes[N // 2]
        sizes[N // 2] = 0
    return [int(s) for s in sizes]


@pytest.mark.parametrize("N", [2, 3, 8])
@pytest.mark.parametrize("K,keep,hot", [(8, 1.0, False), (64, 0.7, True), (100, 0.7, False), (512, 1.0, True)])
def test_emulated_ranks_match_the_global_batch(cuda, N, K, keep, hot):
    B, F = 5003, 6
    w, X, Y = _problem(B, F, K, seed=17 * N + K)
    seed = 0xC0FFEE + N
    sizes = _shard_sizes(B, N, N + K)
    assert sum(sizes) == B and (N == 2 or 0 in sizes)
    res = _sync_call(cuda, X, Y, w, sizes, keep, seed, hot, det=0)
    for r in range(1, N):                                        # the layer's state and gradients agree bit for bit
        for k in ("gamma", "beta", "mm", "mv"):                    # d gamma, d beta, moving mean, moving variance
            assert _bits_equal(res[r][k], res[0][k]), (r, k)
    got = dict(out=np.concatenate([q["out"] for q in res]), loss=float(np.sum([q["loss"] for q in res], dtype=np.float64)),
               V=np.sum([q["V"] for q in res], axis=0, dtype=np.float64), b=np.sum([q["b"] for q in res], axis=0, dtype=np.float64),
               b0=float(np.sum([q["b0"] for q in res], dtype=np.float64)), gamma=res[0]["gamma"], beta=res[0]["beta"],
               mm=res[0]["mm"], mv=res[0]["mv"])
    _check_pass(got, X, Y, w, keep, seed, "N=%d sizes=%s K=%d keep=%g hot=%d" % (N, sizes, K, keep, hot))


def test_emulated_merge_matches_the_oracle_statistics(cuda):
    """The gathered per-rank vectors of phase 1 are the oracle's shard (n, mean, M2)."""
    from hhfm_b200 import _lib
    from hhfm_b200.engine import cur_stream, ptr
    lib = _lib.load()
    B, F, K = 4099, 5, 100
    w, X, _ = _problem(B, F, K, seed=3)
    sizes = _shard_sizes(B, 4, 1)
    cuts = np.cumsum([0] + sizes)
    V = dev(w["V"], cuda)
    parts = []
    for r in range(4):
        n = sizes[r]
        vec = torch.zeros(int(lib.hhfm_fm_bn_sync_len(K)), dtype=torch.float64, device=cuda)
        ws = torch.empty(int(lib.hhfm_workspace_bytes_fm_bn_sync(n, K)), dtype=torch.uint8, device=cuda)
        _lib.call("hhfm_fm_bn_sync_stats", ptr(dev(X[cuts[r]:cuts[r + 1]], cuda, torch.int32)), n, F, ptr(V), None, 300, K, ptr(vec),
                  ptr(ws), ws.numel(), cur_stream())
        v = vec.cpu().numpy()
        want = SB.shard_stats(X[cuts[r]:cuts[r + 1]], w["V"])
        assert v[0] == n
        if n:
            np.testing.assert_allclose(v[1:K + 1], want[1], rtol=1e-5, atol=1e-6 * np.abs(want[1]).max())
            np.testing.assert_allclose(v[K + 1:], want[2], rtol=1e-4)
        parts.append((v[0], v[1:K + 1], v[K + 1:]))
    n, mean, m2 = SB.merge_shard_stats(parts)
    _, _, x = BN._interaction(X, w["V"], np.float64)
    assert n == B
    np.testing.assert_allclose(mean, x.mean(0), rtol=1e-5, atol=1e-6 * np.abs(x.mean(0)).max())
    np.testing.assert_allclose(m2 / n, x.var(0), rtol=1e-4)


@pytest.mark.parametrize("N", [1, 3])
def test_empty_global_batch_leaves_the_layer_alone(cuda, N):
    K, F = 64, 4
    w, X, Y = _problem(0, F, K, seed=9)
    res = _sync_call(cuda, X, Y, w, [0] * N, 0.7, 5, hot=(N == 3), det=0)
    for q in res:
        assert _bits_equal(q["mm"], w["mm"]) and _bits_equal(q["mv"], w["mv"])
        assert not q["gamma"].any() and not q["beta"].any()
        assert q["loss"] == 0.0 and q["b0"] == 0.0 and not q["V"].any() and not q["b"].any()


def test_single_gpu_step_calls_only_the_single_entry(cuda):
    from hhfm_b200 import _lib
    from hhfm_b200.models import FM
    rng = np.random.default_rng(4)
    m = FM(5, 200, 40, 60, 32, 0.05, 0.1, 0.8, "AdagradOptimizer", 1, 0)
    X = rng.integers(0, 200, (1000, 5)); Y = rng.choice([1.0, 0.0], (1000, 1)).astype(np.float32)
    m.partial_fit({"X": X, "Y": Y})
    before = dict(_lib.CALLS)
    m.partial_fit({"X": X, "Y": Y})
    delta = {k: v - before.get(k, 0) for k, v in _lib.CALLS.items() if v != before.get(k, 0)}
    assert delta.get("hhfm_fm_bn_fwd_bwd_sqloss") == 1, delta
    assert not [k for k in delta if k.startswith("hhfm_fm_bn_sync")], delta


# ---- the model over a process group -----------------------------------------------------------------------------
def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _teacher_forced_ok(m, w, st, X, Y, keep, seed, lam, loss):
    """test_gpu_fm_batchnorm.test_model_steps_match_oracle's check of one Adagrad step on the global batch."""
    args = (X, Y, w["feature_embeddings"], w["feature_bias"], w["bias"], w["bn_fm/gamma"], w["bn_fm/beta"], w["bn_fm/moving_mean"],
            w["bn_fm/moving_variance"], keep, seed, lam)
    loss_ref, _, _, (mm, mv) = BN.fm_bn_loss_grads(*args)
    _, _, g64, _ = BN.fm_bn_loss_grads(*args, float64=True)
    terms = _abs_terms(X, Y, w["feature_embeddings"], w["feature_bias"], w["bias"], w["bn_fm/gamma"], w["bn_fm/beta"], keep, seed)
    bad = []
    if not abs(loss - loss_ref) <= 1e-5 * abs(loss_ref):
        bad.append(("loss", loss, float(loss_ref)))
    got = m.get_weights()
    for k, ref in (("bn_fm/moving_mean", mm), ("bn_fm/moving_variance", mv)):
        a = np.asarray(got[k], np.float64); b = np.asarray(ref, np.float64)
        if not (np.abs(a - b) <= 1e-5 * np.maximum(np.abs(b), np.sqrt(np.mean(b * b)))).all():
            bad.append(k)
    for k in _NAMES:
        g = np.asarray(g64[{"feature_embeddings": "feature_embeddings", "feature_bias": "feature_bias", "bias": "bias",
                            "bn_fm/gamma": "gamma", "bn_fm/beta": "beta"}[k]], np.float64).reshape(np.asarray(w[k]).shape)
        floor = 1e-5 * (np.abs(g) + np.asarray(terms[_GKEY[k]], np.float64).reshape(g.shape))
        if k == "feature_embeddings":
            floor = floor + 1e-5 * lam * np.abs(np.asarray(w[k], np.float64))
        s1, s2 = st[k]
        ref = _update("adagrad", w[k], s1, s2, g, m._opt.lr, m._opt.t)
        lo = _update("adagrad", w[k], s1, s2, g - floor, m._opt.lr, m._opt.t)
        hi = _update("adagrad", w[k], s1, s2, g + floor, m._opt.lr, m._opt.t)
        delta = ref - np.asarray(w[k], np.float64)
        rms = float(np.sqrt(np.mean(delta * delta)))
        tol = np.maximum(np.abs(hi - ref), np.abs(lo - ref)) + 1e-5 * np.maximum(np.abs(delta), rms) + \
            4 * 1.2e-7 * np.abs(np.asarray(w[k], np.float64))
        if not (np.abs(np.asarray(got[k], np.float64).reshape(ref.shape) - ref) <= tol).all():
            bad.append(k)
    return bad


def _worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from hhfm_b200 import _lib
        from hhfm_b200 import dist as hd
        from hhfm_b200.models import FM
        n_user, n_item, M, F, K, lr, B = 40, 60, 160, 5, 64, 0.05, 3000
        out = {}
        refused = FM(F, M, n_user, n_item, K, lr, 0.1, 1, "AdagradOptimizer", 1, 0)
        try:
            refused.enable_data_parallel()
            out["refusal"] = False
        except NotImplementedError as e:
            out["refusal"] = "sync_batch_norm" in str(e)
        for mode, lam, keep in (("auto", 0.1, 1.0), (False, 0.1, 0.8), ("sparse", 0.0, 1.0)):
            rng = np.random.default_rng(21)
            m = FM(F, M, n_user, n_item, K, lr, lam, keep, "AdagradOptimizer", 1, 0)
            if mode == "sparse":
                m.enable_data_parallel(sparse=True, sync_batch_norm=True)
                assert m._dp_sparse == (world > 1)
            else:
                m.enable_data_parallel(fused=mode, sync_batch_norm=True)
                if world > 1 and mode == "auto":
                    assert m._dpx is not None
            w = m.get_weights()
            st = {k: (np.full(np.asarray(w[k]).shape, 0.1), None) for k in _NAMES}
            X = np.concatenate([np.stack([rng.integers(0, n_user, B), n_user + rng.integers(0, n_item, B)], axis=1),
                                rng.integers(n_user + n_item, M, (B, F - 2))], axis=1)
            Y = rng.choice([1.0, 0.0], (B, 1)).astype(np.float32)
            lo, hi = hd.shard_range(B, rank, world)
            before = dict(_lib.CALLS)
            loss = m.partial_fit({"X": X[lo:hi], "Y": Y[lo:hi]})
            calls = {k: v - before.get(k, 0) for k, v in _lib.CALLS.items() if k.startswith("hhfm_fm_bn") and v != before.get(k, 0)}
            calls_ok = calls == {"hhfm_fm_bn_sync_stats": 1, "hhfm_fm_bn_sync_loss": 1, "hhfm_fm_bn_sync_scatter": 1}
            seed = m._last_drop_seed if keep < 1 else 0
            bad = _teacher_forced_ok(m, w, st, X, Y, keep, seed, lam, loss)
            for step in range(3):
                r2 = np.random.default_rng(300 + step)
                Bs = 2000 + 7 * step
                Xs = np.concatenate([np.stack([r2.integers(0, n_user, Bs), n_user + r2.integers(0, n_item, Bs)], axis=1),
                                     r2.integers(n_user + n_item, M, (Bs, F - 2))], axis=1)
                Ys = r2.choice([1.0, 0.0], (Bs, 1)).astype(np.float32)
                l2, h2 = hd.shard_range(Bs, rank, world)
                m.partial_fit({"X": Xs[l2:h2], "Y": Ys[l2:h2]})
            m.flush()
            same = True
            for k, t in m.weights.items():
                t = t.reshape(-1).contiguous()
                gathered = [torch.empty_like(t) for _ in range(world)]
                dist.all_gather(gathered, t)
                same = same and all(bool(torch.equal(gathered[0], g)) for g in gathered)
            out[str(mode)] = (bad, calls_ok, same)
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def test_data_parallel_sync_batch_norm(cuda):
    import torch.multiprocessing as mp
    world = min(torch.cuda.device_count(), 2)
    mgr = mp.Manager(); ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    for r in range(world):
        got = dict(ret[r])
        assert got.pop("refusal") is True, (r, ret[r])
        assert got == {m: ([], True, True) for m in ("auto", "False", "sparse")}, (r, got)
