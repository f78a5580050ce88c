"""CPU: synchronised batch norm -- the oracle's rank-order merge of shard statistics gives the statistics of the global
batch, the shards' global-index dropout masks concatenate to the mask of the global batch, and the argument checks of the
three phase entry points (include/hhfm_sm100.h hhfm_fm_bn_sync_*) run before any launch."""
import ctypes

import numpy as np
import pytest

from oracle import fm_batchnorm as BN
from oracle import fm_batchnorm_sync as SB
from oracle import hhfm_oracle as O


def _shards(B, sizes):
    cuts = np.cumsum([0] + list(sizes))
    assert cuts[-1] == B
    return [(int(cuts[r]), int(cuts[r + 1])) for r in range(len(sizes))]


@pytest.mark.parametrize("sizes", [(700,), (300, 400), (0, 250, 1, 449), (100, 0, 0, 200, 50, 250, 99, 1)])
def test_merged_shard_statistics_are_the_global_statistics(sizes):
    rng = np.random.default_rng(len(sizes))
    M, F, K, B = 120, 5, 12, sum(sizes)
    V = rng.normal(0, 0.3, (M, K)).astype(np.float32)
    X = rng.integers(0, M, (B, F))
    parts = [SB.shard_stats(X[lo:hi], V) for lo, hi in _shards(B, sizes)]
    assert [p[0] for p in parts] == list(sizes)
    n, mean, m2 = SB.merge_shard_stats(parts)
    _, _, x = BN._interaction(X, V, np.float64)
    assert n == B
    np.testing.assert_allclose(mean, x.mean(0), rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(m2 / n, x.var(0), rtol=1e-12, atol=1e-14)
    # one shard: the merge into the empty state reproduces it exactly
    one = SB.merge_shard_stats([SB.shard_stats(X, V)])
    full = SB.shard_stats(X, V)
    assert one[0] == full[0] and np.array_equal(one[1], full[1]) and np.array_equal(one[2], full[2])


def test_empty_global_batch_merges_to_nothing():
    V = np.ones((4, 8), np.float32)
    n, mean, m2 = SB.merge_shard_stats([SB.shard_stats(np.zeros((0, 3), np.int64), V)] * 3)
    assert n == 0 and not mean.any() and not m2.any()


@pytest.mark.parametrize("sizes", [(517,), (200, 317), (0, 17, 0, 500), (64, 64, 64, 64, 64, 64, 64, 69)])
@pytest.mark.parametrize("keep", [0.7, 0.5])
def test_global_index_masks_concatenate_to_the_batch_mask(sizes, keep):
    seed, K, B = 0x9E3779B97F4A7C15 * 7 & 0xFFFFFFFFFFFFFFFF, 100, sum(sizes)
    whole = O.dropout_mask_hashed(seed, B, K, keep)
    cat = np.concatenate([SB.dropout_mask_global(seed, lo, hi - lo, K, keep) for lo, hi in _shards(B, sizes)], axis=0)
    assert cat.shape == whole.shape and np.array_equal(cat, whole)
    assert np.array_equal(SB.dropout_mask_global(seed, 0, B, K, keep), whole)
    if len(sizes) > 1 and sizes[0] > 0:              # a rank-local index would draw the first shard's mask again
        lo, hi = _shards(B, sizes)[1]
        assert not np.array_equal(SB.dropout_mask_global(seed, 0, hi - lo, K, keep), whole[lo:hi])


# ---- argument checks of the phase entry points (no launch, no GPU) --------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from hhfm_b200 import _lib, build
    build.build()
    return _lib.load()


P16 = ctypes.c_void_p(16)


def _stats(**kw):
    a = dict(col=P16, B=8, F=3, V=P16, bias=None, M=10, K=8, stats=P16, ws=P16, wsb=1 << 30)
    a.update(kw)
    return (a["col"], a["B"], a["F"], a["V"], a["bias"], a["M"], a["K"], a["stats"], a["ws"], a["wsb"], None)


def _loss(**kw):
    a = dict(B=8, K=8, b0=None, labels=P16, out=None, gb0=None, lp=P16, keep=1.0, seed=0, gamma=P16, beta=P16, mm=P16, mv=P16,
             eps=1e-3, decay=0.9, all=P16, n_ranks=2, rank=1, sums=P16, ws=P16, wsb=1 << 30)
    a.update(kw)
    return (a["B"], a["K"], a["b0"], a["labels"], a["out"], a["gb0"], a["lp"], a["keep"], a["seed"], a["gamma"], a["beta"], a["mm"],
            a["mv"], a["eps"], a["decay"], a["all"], a["n_ranks"], a["rank"], a["sums"], a["ws"], a["wsb"], None)


def _scatter(**kw):
    a = dict(col=P16, B=8, F=3, V=P16, M=10, K=8, gV=P16, gb=None, keep=1.0, dg=P16, db=P16, all=P16, n_ranks=2, ws=P16,
             wsb=1 << 30, hot=(None, None, None, 0, 0))
    a.update(kw)
    return (a["col"], a["B"], a["F"], a["V"], a["M"], a["K"], a["gV"], a["gb"], None, 0, None, None, *a["hot"], 0, a["keep"], 0,
            a["dg"], a["db"], a["all"], a["n_ranks"], a["ws"], a["wsb"], None)


@pytest.mark.parametrize("name,args,match", [
    ("hhfm_fm_bn_sync_stats", _stats(K=6), "K=6"),
    ("hhfm_fm_bn_sync_stats", _stats(B=-1), "bad size"),
    ("hhfm_fm_bn_sync_stats", _stats(stats=None), "per-rank vector"),
    ("hhfm_fm_bn_sync_stats", _stats(wsb=64), "workspace of 64 bytes"),
    ("hhfm_fm_bn_sync_stats", _stats(ws=None), "workspace must be non-NULL"),
    ("hhfm_fm_bn_sync_stats", _stats(col=None), "col and V"),
    ("hhfm_fm_bn_sync_stats", _stats(F=0), "F=0"),
    ("hhfm_fm_bn_sync_stats", _stats(V=ctypes.c_void_p(20)), "V must be 16-byte aligned"),
    ("hhfm_fm_bn_sync_loss", _loss(n_ranks=0, rank=0), "n_ranks=0"),
    ("hhfm_fm_bn_sync_loss", _loss(rank=2), "rank=2 outside"),
    ("hhfm_fm_bn_sync_loss", _loss(rank=-1), "rank=-1 outside"),
    ("hhfm_fm_bn_sync_loss", _loss(all=None), "per-rank vector"),
    ("hhfm_fm_bn_sync_loss", _loss(sums=None), "sums must be non-NULL"),
    ("hhfm_fm_bn_sync_loss", _loss(gamma=None), "gamma, beta"),
    ("hhfm_fm_bn_sync_loss", _loss(eps=0.0), "eps must be > 0"),
    ("hhfm_fm_bn_sync_loss", _loss(keep=0.0), "keep must be in"),
    ("hhfm_fm_bn_sync_loss", _loss(decay=1.0), "decay must be in"),
    ("hhfm_fm_bn_sync_loss", _loss(labels=None), "labels and loss_partials"),
    ("hhfm_fm_bn_sync_loss", _loss(wsb=1024), "workspace of 1024 bytes"),
    ("hhfm_fm_bn_sync_scatter", _scatter(n_ranks=0), "n_ranks=0"),
    ("hhfm_fm_bn_sync_scatter", _scatter(all=None), "per-rank vector"),
    ("hhfm_fm_bn_sync_scatter", _scatter(dg=None), "dgamma and dbeta"),
    ("hhfm_fm_bn_sync_scatter", _scatter(gV=None), "gV is required"),
    ("hhfm_fm_bn_sync_scatter", _scatter(keep=1.5), "keep must be in"),
    ("hhfm_fm_bn_sync_scatter", _scatter(hot=(P16, None, None, 0, 0)), "hot_slot needs"),
    ("hhfm_fm_bn_sync_scatter", _scatter(K=516), "K=516"),
])
def test_phase_argument_checks_fail_before_any_launch(lib, name, args, match):
    from hhfm_b200 import _lib
    with pytest.raises(_lib.HhfmError, match=match):
        _lib.call(name, *args)


def test_sizes_of_the_phase_buffers(lib):
    for K in (4, 64, 100, 512):
        assert lib.hhfm_fm_bn_sync_len(K) == 2 * K + 1
        for B in (0, 1, 5000):
            assert lib.hhfm_workspace_bytes_fm_bn_sync(B, K) > lib.hhfm_workspace_bytes_fm_bn(B, K)
    assert lib.hhfm_fm_bn_sync_len(0) == -1 and lib.hhfm_fm_bn_sync_len(513) == -1
    assert lib.hhfm_workspace_bytes_fm_bn_sync(-1, 8) == -1
