"""CPU: MomentumOptimizer under data parallelism -- the oracle's sharded step (oracle/momentum_dp.py), the host logic that
builds the union of the ranks' touched rows (gloo), and the argument checks of the C ABI entries behind it."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch

from oracle import hhfm_oracle as O
from oracle import momentum_dp as MD


def _split(a, n):
    from hhfm_b200 import dist as hd
    return [a[slice(*hd.shard_range(len(a), r, n))] for r in range(n)]


def _close(a, b, rtol=2e-5):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    scale = max(float(np.sqrt(np.mean(b * b))), 1e-30)
    return bool(np.all(np.abs(a - b) <= rtol * np.maximum(np.abs(b), scale)))


def _fm_state(rng, M, K, with_acc=True):
    w = {"feature_embeddings": rng.normal(0, 0.1, (M, K)).astype(np.float32),
         "feature_bias": rng.normal(0, 0.1, (M, 1)).astype(np.float32), "bias": np.float32(0.05)}
    acc = {k: (np.abs(rng.normal(0, 0.1, np.shape(v))).astype(np.float32) if with_acc else np.zeros(np.shape(v), np.float32))
           for k, v in w.items()}
    return w, acc


@pytest.mark.parametrize("lamda", [0.0, 0.1])
@pytest.mark.parametrize("n_ranks", [2, 3, 8])
def test_fm_sharded_step_equals_the_single_shard_step(lamda, n_ranks):
    rng = np.random.default_rng(n_ranks)
    M, K, B, F = 90, 8, 64, 4
    X = rng.integers(0, M - 10, (B, F))                       # rows M-10 .. M-1: touched by nobody
    Y = rng.choice([1.0, 0.0], (B, 1)).astype(np.float32)
    w, acc = _fm_state(rng, M, K)
    l1, w1, a1 = MD.fm_step([X], [Y], w, acc, 0.05, lamda)
    ln, wn, an = MD.fm_step(_split(X, n_ranks), _split(Y, n_ranks), w, acc, 0.05, lamda)
    assert abs(float(ln) - float(l1)) <= 1e-5 * abs(float(l1))
    for k in w:
        assert _close(wn[k], w1[k]) and _close(an[k], a1[k]), k
    assert np.array_equal(wn["feature_bias"][M - 10:], w["feature_bias"][M - 10:])
    assert np.array_equal(an["feature_bias"][M - 10:], acc["feature_bias"][M - 10:])
    if lamda == 0:
        assert np.array_equal(wn["feature_embeddings"][M - 10:], w["feature_embeddings"][M - 10:])
    else:                                                      # the dense L2 step moves every row
        assert not np.array_equal(wn["feature_embeddings"][M - 10:], w["feature_embeddings"][M - 10:])


@pytest.mark.parametrize("n_ranks", [2, 3])
def test_pairrank_mf_and_afm_sharded_steps_equal_the_single_shard_steps(n_ranks):
    rng = np.random.default_rng(7)
    M, K, B = 120, 8, 48
    V = rng.normal(0, 0.1, (M, K)).astype(np.float32)
    w, acc = {"feature_embeddings": V}, {"feature_embeddings": np.full_like(V, 0.01)}
    Pos = np.stack([rng.integers(0, 30, B), 30 + rng.integers(0, 60, B)], axis=1)
    Neg = 30 + rng.integers(0, 60, (B, 5)); Fea = 90 + rng.integers(0, 20, (B, 3))
    for fea in (Fea, None):
        l1, w1, a1 = MD.pairrank_step([Pos], [Neg], None if fea is None else [fea], w, acc, 0.05, 0.0)
        ln, wn, an = MD.pairrank_step(_split(Pos, n_ranks), _split(Neg, n_ranks), None if fea is None else _split(fea, n_ranks),
                                      w, acc, 0.05, 0.0)
        assert abs(float(ln) - float(l1)) <= 1e-5 * abs(float(l1))
        assert _close(wn["feature_embeddings"], w1["feature_embeddings"]) and _close(an["feature_embeddings"], a1["feature_embeddings"])
    Y = rng.choice([1.0, 0.0], (B, 1)).astype(np.float32)
    l1, w1, _ = MD.fm_step([Pos], [Y], w, acc, 0.05, 0.0, interaction=1)
    ln, wn, _ = MD.fm_step(_split(Pos, n_ranks), _split(Y, n_ranks), w, acc, 0.05, 0.0, interaction=1)
    assert abs(float(ln) - float(l1)) <= 1e-5 * abs(float(l1)) and _close(wn["feature_embeddings"], w1["feature_embeddings"])
    A = K
    wa = {"feature_embeddings": V, "feature_bias": rng.normal(0, 0.1, (M, 1)).astype(np.float32), "bias": np.float32(0.1),
          "attention_W": rng.normal(0, 0.3, (K, A)).astype(np.float32), "attention_b": rng.normal(0, 0.3, (1, A)).astype(np.float32),
          "attention_p": rng.normal(0, 1, A).astype(np.float32), "prediction": np.ones((K, 1), np.float32)}
    aa = {k: np.zeros(np.shape(v), np.float32) for k, v in wa.items()}
    X = rng.integers(0, M, (B, 4))
    l1, w1, a1 = MD.afm_step([X], [Y], wa, aa, 0.05, 0.01)
    ln, wn, an = MD.afm_step(_split(X, n_ranks), _split(Y, n_ranks), wa, aa, 0.05, 0.01)
    assert abs(float(ln) - float(l1)) <= 1e-5 * abs(float(l1))
    for k in wa:
        assert _close(wn[k], w1[k], 1e-4), k


def test_union_moves_rows_of_other_ranks_and_zero_sum_rows_and_nothing_else():
    M, K, lr, mu = 12, 4, 0.1, 0.95
    rng = np.random.default_rng(1)
    w = rng.normal(0, 1, (M, K)).astype(np.float32)
    acc = rng.normal(0, 1, (M, K)).astype(np.float32)
    g0, g1, g2 = (np.zeros((M, K), np.float32) for _ in range(3))
    g0[3] = 0.25; g1[3] = -0.25                  # row 3: touched on ranks 0 and 1, summed gradient exactly 0
    g2[9] = 0.5                                  # row 9: touched on the last rank only
    g0[1] = 1.0                                  # row 1: rank 0 only
    touched = [np.array([1, 3, -1]), np.array([3]), np.array([9])]
    rows = MD.union_rows(touched)
    assert rows.tolist() == [1, 3, 9]
    w2, a2 = MD.momentum_step(w, acc, [g0, g1, g2], rows, lr, mu)
    for r in (1, 3, 9):
        assert not np.array_equal(w2[r], w[r]) and not np.array_equal(a2[r], acc[r]), r
    assert np.array_equal(a2[3], (acc[3] * np.float32(mu)).astype(np.float32))          # accum decays, w follows it
    assert np.array_equal(w2[3], (w[3] - np.float32(lr) * a2[3]).astype(np.float32))
    others = [r for r in range(M) if r not in (1, 3, 9)]
    assert np.array_equal(w2[others], w[others]) and np.array_equal(a2[others], acc[others])
    # the per-rank lists need not be disjoint or sorted, and an empty rank changes nothing
    assert MD.union_rows([np.array([9, 1]), np.array([], np.int64), np.array([3, 3])]).tolist() == [1, 3, 9]


# ---- host logic of the union on the NCCL path (dist.union_touched), gloo ---------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from hhfm_b200 import dist as hd
        M, stamp = 40, 7
        rng = np.random.default_rng(0)
        history = rng.integers(0, stamp, M).astype(np.int32)       # earlier steps: identical on every rank (last union)
        mine = {0: [2, 5, 11], 1: [5, 30], 2: [39]}.get(rank, [])   # the last rank alone touches row 39
        arr = torch.from_numpy(history.copy())
        arr[mine] = stamp
        out = hd.union_touched(arr)
        ret[rank] = (torch.nonzero(out == stamp).reshape(-1).tolist(), out.tolist())
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_union_of_touched_rows_is_one_max_allreduce_of_the_stamps(world):
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    want = sorted(set(x for r in range(world) for x in {0: [2, 5, 11], 1: [5, 30], 2: [39]}[r]))
    for r in range(world):
        assert ret[r][0] == want, (r, ret[r][0])
        assert ret[r][1] == ret[0][1]                                  # identical stamp arrays on every rank


# ---- argument checks of the new entry points (no launch, no GPU) ----------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from hhfm_b200 import _lib, build
    build.build()
    return _lib.load()


P16 = ctypes.c_void_p(16)


def _touched(widths=(8, 1), lamdas=(0.0, 0.0), stamps=P16, kind=2, n=(80, 10), M=10, K=8, seg_widths=True):
    from hhfm_b200 import dist as hd
    segs = (hd.DpSegment * len(n))()
    off = 0
    for i, ni in enumerate(n):
        segs[i].w, segs[i].s1, segs[i].s2 = 16, 16, 16
        segs[i].offset, segs[i].n, segs[i].lamda = off, ni, lamdas[i]
        off += ni
    wd = (ctypes.c_int32 * len(n))(*widths) if seg_widths else None
    return (kind, ctypes.cast(segs, ctypes.c_void_p), len(n), wd, stamps, 1, P16, off + 1, None, None, 0, 0, K, M, None, -1,
            P16, P16, None, None, None, 0, 1, P16, 0.1, 0.95, 0.0, 0.0, P16, P16, 1.0, None), segs


@pytest.mark.parametrize("kw,match", [
    (dict(seg_widths=False), "seg_widths is NULL"),
    (dict(widths=(-1, 1)), "negative row width"),
    (dict(stamps=None), "needs the stamp array"),
    (dict(widths=(3, 1)), "segment 0 is not"),
    (dict(widths=(8, 1), n=(80, 20), M=10), "segment 1 is not"),
    (dict(lamdas=(0.1, 0.0)), "takes no L2 term"),
    (dict(kind=7), "unknown optimizer kind 7"),
])
def test_dp_step_touched_argument_checks(lib, kw, match):
    from hhfm_b200 import _lib
    args, keep = _touched(**kw)
    with pytest.raises(_lib.HhfmError, match=match):
        _lib.call("hhfm_dp_step_touched", *args)


def test_touched_compact_argument_checks_and_exchange_size(lib):
    from hhfm_b200 import _lib
    for args in [(None, 1, 10, P16, P16, None), (P16, 1, 0, P16, P16, None), (P16, 1, 10, None, P16, None),
                 (P16, 1, 10, P16, None, None)]:
        with pytest.raises(_lib.HhfmError, match="touched_compact: bad argument"):
            _lib.call("hhfm_touched_compact", *args)
    for n in (1, 5, 127, 128, 129, 10 ** 6 + 3):
        total4 = (n + 3) // 4 + 1
        assert lib.hhfm_dp_exchange_floats_touched(n) == 4 * (total4 + (total4 + 31) // 32)
        assert lib.hhfm_dp_exchange_floats_touched(n) > lib.hhfm_dp_exchange_floats(n)
    assert lib.hhfm_dp_exchange_floats_touched(0) == -1
