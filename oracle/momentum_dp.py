"""MomentumOptimizer under data parallelism: the TF1 single-GPU step on the global batch (the ranks' shards concatenated in
rank order), restated from per-rank shards.

Per rank, the gradient of its shard and the rows it touched; the gradients are added in rank order, then
  - dense variables (V with lamda > 0, the scalar bias, AFM's small dense variables): ApplyMomentum with g (+ lamda*w);
  - IndexedSlices variables (feature_bias; V with lamda == 0; V of AFM): SparseApplyMomentum over the UNION of the rows
    touched on any rank -- a row touched only on another rank moves, a touched row whose summed gradient is exactly 0 still
    moves (accum decays, w follows it), a row no rank touched keeps w and accum bit for bit.
The loss is the sum of the shards' losses (the reference loss is a sum over the batch), plus the regulariser once.
"""
from __future__ import annotations

import numpy as np

from . import hhfm_oracle as O

F32 = np.float32


def union_rows(touched):
    """Rows touched on any rank: the ids >= 0 of every rank's list, sorted and without duplicates."""
    ids = [np.asarray(t, dtype=np.int64).reshape(-1) for t in touched]
    ids = np.concatenate(ids) if ids else np.zeros(0, np.int64)
    return np.unique(ids[ids >= 0])


def sum_rank_order(per_rank):
    """fp32 sum of the ranks' gradients, rank 0 first."""
    acc = np.zeros_like(np.asarray(per_rank[0], dtype=F32))
    for g in per_rank:
        acc = (acc + np.asarray(g, dtype=F32)).astype(F32)
    return acc


def momentum_step(w, acc, grads, rows, lr, momentum=0.95, lamda=0.0):
    """One variable: `grads` is the list of per-rank gradients, `rows` the union (None: a dense variable, g + lamda*w)."""
    g = sum_rank_order(grads)
    if rows is None:
        if lamda > 0:
            g = (g + F32(lamda) * np.asarray(w, dtype=F32)).astype(F32)
        return O.momentum_dense(w, acc, g, lr, momentum)
    return O.momentum_rows(w, acc, g, rows, lr, momentum)


def fm_step(X_shards, Y_shards, w, acc, lr, lamda, momentum=0.95, interaction=0):
    """FM (interaction 0) or MF (interaction 1: columns 0, 1, no bias) on per-rank shards.  `w` / `acc`: dicts keyed like
    the model's weights / Momentum slots.  Returns (loss, w', acc')."""
    losses, gV, gb, gb0, touched = [], [], [], [], []
    for X, Y in zip(X_shards, Y_shards):
        X = np.asarray(X)
        if interaction:
            loss, _, dV = O.mf_loss_grads(X[:, :2], Y, w["feature_embeddings"], 0.0)
            touched.append(X[:, :2].reshape(-1))
        else:
            loss, _, dV, db, db0, rows = O.fm_loss_grads(X, Y, w["feature_embeddings"], w["feature_bias"], w["bias"], 0.0)
            gb.append(np.asarray(db).reshape(-1, 1)); gb0.append(np.asarray(db0, dtype=F32).reshape(()))
            touched.append(rows)
        losses.append(loss); gV.append(dV)
    return _finish(w, acc, losses, gV, gb, gb0, touched, lr, lamda, momentum)


def pairrank_step(Pos_shards, Neg_shards, Fea_shards, w, acc, lr, lamda, momentum=0.95):
    """HHFM (OUR) / BPR: pair-ranking loss on per-rank shards (Fea None: BPR).  V is the only trained variable."""
    losses, gV, touched = [], [], []
    for r, (Pos, Neg) in enumerate(zip(Pos_shards, Neg_shards)):
        Fea = Fea_shards[r] if Fea_shards is not None else None
        loss, _, neg, dV = O.pairrank_loss_grads(w["feature_embeddings"], Pos, Neg, Fea, None, (0, 0, 0), 0.0)
        losses.append(loss); gV.append(dV)
        # the rows the step touches: user, item, context, and the negatives at the maximum (the others get no gradient,
        # and the single-GPU path does not list them either)
        tie = np.asarray(Neg)[neg == neg.max(axis=1, keepdims=True)]
        touched.append(np.concatenate([np.asarray(a).reshape(-1) for a in (Pos, tie, Fea) if a is not None]))
    return _finish(w, acc, losses, gV, [], [], touched, lr, lamda, momentum)


def afm_step(X_shards, Y_shards, w, acc, lr, lamda_attention, momentum=0.95):
    """AFM with attention and keep = [1, 1]: V and feature_bias are IndexedSlices, the rest dense (attention_W with L2)."""
    losses, grads, touched = [], [], []
    for X, Y in zip(X_shards, Y_shards):
        loss, _, g = O.afm_loss_grads(np.asarray(X), Y, w, 0.0)
        losses.append(loss); grads.append(g); touched.append(np.asarray(X).reshape(-1))
    rows = union_rows(touched)
    w2, acc2 = dict(w), dict(acc)
    for name in ("feature_embeddings", "feature_bias", "bias", "attention_W", "attention_b", "attention_p", "prediction"):
        sparse = name in ("feature_embeddings", "feature_bias")
        lam = lamda_attention if name == "attention_W" else 0.0
        gs = [np.asarray(g[name], dtype=F32).reshape(np.shape(w[name])) for g in grads]
        w2[name], acc2[name] = momentum_step(w[name], acc[name], gs, rows if sparse else None, lr, momentum, lam)
    loss = sum_rank_order([np.asarray(l, dtype=F32).reshape(()) for l in losses])
    if lamda_attention > 0:
        W = np.asarray(w["attention_W"], dtype=F32)
        loss = F32(loss + F32(lamda_attention) * F32(0.5) * (W * W).astype(F32).sum(dtype=F32))
    return F32(loss), w2, acc2


def _finish(w, acc, losses, gV, gb, gb0, touched, lr, lamda, momentum):
    rows = union_rows(touched)
    w2, acc2 = dict(w), dict(acc)
    V = np.asarray(w["feature_embeddings"], dtype=F32)
    w2["feature_embeddings"], acc2["feature_embeddings"] = momentum_step(
        V, acc["feature_embeddings"], gV, rows if lamda <= 0 else None, lr, momentum, lamda)
    if gb:
        w2["feature_bias"], acc2["feature_bias"] = momentum_step(w["feature_bias"], acc["feature_bias"], gb, rows, lr, momentum)
        w2["bias"], acc2["bias"] = momentum_step(np.asarray(w["bias"], dtype=F32).reshape(()),
                                                 np.asarray(acc["bias"], dtype=F32).reshape(()), gb0, None, lr, momentum)
    loss = sum_rank_order([np.asarray(l, dtype=F32).reshape(()) for l in losses])
    if lamda > 0:
        loss = F32(loss + F32(lamda) * F32(0.5) * (V * V).astype(F32).sum(dtype=F32))
    return F32(loss), w2, acc2
