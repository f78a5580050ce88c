"""CPU oracle for synchronised batch norm (FM batch_norm=1 under data parallelism)  --  TEST INFRASTRUCTURE ONLY.

The data-parallel step is `oracle.fm_batchnorm.fm_bn_loss_grads` on the global batch, the ranks' shards concatenated in rank
order.  This module restates the pieces the ranks compute on their own shards: `shard_stats` is one rank's (n, mean, M2),
`merge_shard_stats` the rank-order Chan merge of the gathered ones, and `dropout_mask_global` a shard's mask drawn at the
global sample indices (rows of `hhfm_oracle.dropout_mask_hashed` of the global batch).
"""
from __future__ import annotations

import numpy as np

from oracle.fm_batchnorm import _interaction
from oracle.hhfm_oracle import _splitmix64


def shard_stats(X, V):
    """One shard's (n, mean [K], M2 [K]) of the interaction vectors, in float64; M2 = sum over the shard of (x - mean)^2."""
    X = np.asarray(X)
    _, _, x = _interaction(X.reshape(-1, X.shape[-1]), V, np.float64)
    n = x.shape[0]
    if n == 0:
        return 0, np.zeros(x.shape[1]), np.zeros(x.shape[1])
    mean = x.mean(axis=0)
    return n, mean, ((x - mean) ** 2).sum(axis=0)


def merge_shard_stats(parts):
    """Chan's formula over [(n, mean, M2), ...] in rank order, in float64 -> (n, mean, M2) of the shards concatenated.
    Empty shards are skipped; the biased variance of the global batch is M2 / n."""
    n, mean, m2 = 0, None, None
    for nb, mb, m2b in parts:
        mb = np.asarray(mb, np.float64); m2b = np.asarray(m2b, np.float64)
        if mean is None:
            mean, m2 = np.zeros_like(mb), np.zeros_like(m2b)
        if nb == 0:
            continue
        nn = n + nb
        d = mb - mean
        mean = mean + d * (nb / nn)
        m2 = m2 + m2b + d * d * (n * nb / nn)
        n = nn
    return n, mean, m2


def dropout_mask_global(seed, base, B, K, keep):
    """The dropout mask of a shard of B samples whose first sample has global index `base`: rows base .. base + B - 1 of
    `dropout_mask_hashed(seed, ...)` of the global batch.  Float32 0/1 [B, K]."""
    with np.errstate(over="ignore"):
        s = (np.uint64(base) + np.arange(B, dtype=np.uint64))[:, None]
        k = np.arange(K, dtype=np.uint64)[None, :]
        h = _splitmix64(np.uint64(seed) ^ _splitmix64(s * np.uint64(0x100000001B3) + k))
    u = (h >> np.uint64(40)).astype(np.float32) * np.float32(1.0 / 16777216.0)
    return (u < np.float32(keep)).astype(np.float32)
