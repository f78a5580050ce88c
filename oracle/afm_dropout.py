"""CPU oracle for AFM training with dropout (AFM.py:126,134) and with attention=0 (AFM.py:132)  --  TEST INFRASTRUCTURE ONLY.

NumPy fp32 restatement beside `oracle/hhfm_oracle.py` (whose `afm_forward` / `afm_loss_grads` cover keep = [1, 1],
attention = 1), in the same conventions: every ufunc rounds to fp32, the masks are the device's counter-based hash
(csrc/common.cuh `dropout_keep01`, restated by `hhfm_oracle.dropout_mask_hashed`) and so compare bit-exactly.
`oracle/afm_dropout_torch.py` is the torch-CPU restatement that autograd checks this one against.
"""
from __future__ import annotations

import numpy as np

from oracle.hhfm_oracle import F32, _f32, _splitmix64, afm_forward as _afm_forward_attention, pair_index


def afm_forward(X, w, attention=1):
    """The AFM forward (no dropout: the reference evaluates with keep = [1, 1]) for either value of `attention`.
    attention=0 (AFM.py:132): afm = sum_p P_p = 0.5 (S^2 - sum_f E_f^2), S = sum_f E_f; the attention net is unused."""
    if attention:
        return _afm_forward_attention(X, w)
    V = _f32(w["feature_embeddings"])
    E = V[X]
    S = E.sum(axis=1, dtype=F32)
    afm = (F32(0.5) * ((S * S).astype(F32) - (E * E).astype(F32).sum(axis=1, dtype=F32))).astype(F32)
    wp = _f32(w["prediction"]).reshape(-1)
    bil = (afm * wp).astype(F32).sum(axis=1, dtype=F32)
    fb = _f32(w["feature_bias"]).reshape(-1)[X].sum(axis=1, dtype=F32)
    out = (bil + fb + F32(np.asarray(w["bias"]).reshape(()))).astype(F32)
    return out, dict(E=E, S=S, afm=afm)


def afm_dropout_masks(seed, B, P, K, keep, sample_base=0):
    """The two 0/1 dropout masks of an AFM training step (AFM.py:126 on the attention weights, :134 on the pooled vector):
    mask_att [B, P] from (seed, s, p) and mask_vec [B, K] from (splitmix64(seed), s, k), s = sample_base + row.
    Element (s, c) of a stream with seed sd is kept iff (splitmix64(sd ^ splitmix64(s * 0x100000001B3 + c)) >> 40) * 2^-24
    < keep -- the hash of the FM / MF masks."""
    def mask(sd, n, k):
        with np.errstate(over="ignore"):
            s = np.arange(sample_base, sample_base + B, dtype=np.uint64)[:, None]
            c = np.arange(n, dtype=np.uint64)[None, :]
            h = _splitmix64(np.uint64(sd) ^ _splitmix64(s * np.uint64(0x100000001B3) + c))
        return ((h >> np.uint64(40)).astype(np.float32) * F32(1.0 / 16777216.0) < F32(k)).astype(F32)
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    with np.errstate(over="ignore"):
        vseed = int(_splitmix64(np.uint64(seed)))
    return mask(seed, P, keep[0]), mask(vseed, K, keep[1])


def afm_dropout_loss_grads(X, Y, w, lamda_attention, keep, seed, attention=1, sample_base=0):
    """AFM.py:103-148 in training mode with dropout_keep = [k0, k1] and either value of `attention`.
    tf.nn.dropout(x, k) = x / k * mask: the attention weights are dropped per (sample, pair) (:126), the pooled vector
    per (sample, k) (:134); out = (afm / k1 * mask_vec) . prediction + sum_f b[x_f] + b0.
    attention=0 (:132): afm = sum_p P_p, k0 is unused, attention_W/b/p get zero gradients and the lamda_attention term
    is left out of the loss (the regulariser sits under `if attention` in the AFM authors' code).
    With keep = [1, 1] and attention = 1 every result is bit-identical to hhfm_oracle.afm_loss_grads."""
    Y = _f32(Y).reshape(-1)
    B, F = X.shape
    V = _f32(w["feature_embeddings"]); W = _f32(w["attention_W"])
    ap = _f32(w["attention_p"]).reshape(-1); wp = _f32(w["prediction"]).reshape(-1)
    K = V.shape[1]
    m_att, m_vec = afm_dropout_masks(seed, B, F * (F - 1) // 2, K, keep, sample_base)
    n = (m_vec / F32(keep[1])).astype(F32)                                # [B,K]
    E = V[X]
    if attention:
        pi = pair_index(F)
        I = np.array([p[0] for p in pi]); J = np.array([p[1] for p in pi])
        P = (E[:, I, :] * E[:, J, :]).astype(F32)
        Z = (P.reshape(-1, K) @ W).astype(F32).reshape(B, P.shape[1], -1) + _f32(w["attention_b"]).reshape(-1)
        H = np.maximum(Z, F32(0)).astype(F32)
        s = (H * ap).astype(F32).sum(axis=2, dtype=F32)
        ex = np.exp((s - s.max(axis=1, keepdims=True)).astype(F32)).astype(F32)
        a = (ex / ex.sum(axis=1, keepdims=True, dtype=F32)).astype(F32)
        m = (m_att / F32(keep[0])).astype(F32)                            # [B,P]
        am = ((a / F32(keep[0])).astype(F32) * m_att).astype(F32)         # tf.nn.dropout: x / keep * mask
        afm = (am[:, :, None] * P).astype(F32).sum(axis=1, dtype=F32)
    else:
        S = E.sum(axis=1, dtype=F32)
        afm = (F32(0.5) * ((S * S).astype(F32) - (E * E).astype(F32).sum(axis=1, dtype=F32))).astype(F32)
    afm_d = ((afm / F32(keep[1])).astype(F32) * m_vec).astype(F32)
    bil = (afm_d * wp).astype(F32).sum(axis=1, dtype=F32)
    fb = _f32(w["feature_bias"]).reshape(-1)[X].sum(axis=1, dtype=F32)
    out = (bil + fb + F32(np.asarray(w["bias"]).reshape(()))).astype(F32)
    diff = (Y - out).astype(F32)
    loss = F32(0.5) * (diff * diff).astype(F32).sum(dtype=F32)
    g = (-diff).astype(F32)
    d_afm = ((g[:, None] * wp[None, :]).astype(F32) * n).astype(F32)     # g w~, w~ = prediction * n
    d_wp = (g[:, None] * afm_d).astype(F32).sum(axis=0, dtype=F32)
    if attention:
        d_am = (P * d_afm[:, None, :]).astype(F32).sum(axis=2, dtype=F32)    # g u_p, u_p = w~ . P_p
        d_a = (d_am * m).astype(F32)
        dP = (am[:, :, None] * d_afm[:, None, :]).astype(F32)
        d_s = (a * (d_a - (a * d_a).astype(F32).sum(axis=1, keepdims=True, dtype=F32))).astype(F32)
        d_ap = (d_s[:, :, None] * H).astype(F32).sum(axis=(0, 1), dtype=F32)
        d_Z = (d_s[:, :, None] * ap[None, None, :] * (Z > 0)).astype(F32)
        d_ab = d_Z.sum(axis=(0, 1), dtype=F32)
        d_W = (P.reshape(-1, K).T @ d_Z.reshape(B * P.shape[1], -1)).astype(F32)
        dP = (dP + (d_Z.reshape(B * P.shape[1], -1) @ W.T).astype(F32).reshape(B, P.shape[1], K)).astype(F32)
        dE = np.zeros_like(E)
        np.add.at(dE, (slice(None), I), (dP * E[:, J, :]).astype(F32))
        np.add.at(dE, (slice(None), J), (dP * E[:, I, :]).astype(F32))
    else:
        dE = (d_afm[:, None, :] * (S[:, None, :] - E)).astype(F32)
        d_ap = np.zeros_like(ap)
        d_ab = np.zeros(W.shape[1], F32)
        d_W = np.zeros_like(W)
    dV = np.zeros_like(V)
    np.add.at(dV, X.reshape(-1), dE.reshape(-1, K))
    db = np.zeros(V.shape[0], F32)
    np.add.at(db, X.reshape(-1), np.broadcast_to(g[:, None], X.shape).reshape(-1))
    if attention and lamda_attention > 0:
        loss = F32(loss + F32(lamda_attention) * F32(0.5) * (W * W).astype(F32).sum(dtype=F32))
        d_W = (d_W + F32(lamda_attention) * W).astype(F32)
    grads = dict(feature_embeddings=dV, feature_bias=db.reshape(-1, 1), bias=g.sum(dtype=F32),
                 attention_W=d_W, attention_b=d_ab.reshape(1, -1), attention_p=d_ap, prediction=d_wp.reshape(-1, 1))
    return F32(loss), out, grads
