"""CPU oracle for FM training with batch normalisation of the interaction vector (FM.py:111-112, batch_norm=1)  --
TEST INFRASTRUCTURE ONLY.

NumPy restatement beside `oracle/hhfm_oracle.py` in the same conventions: in fp32 every ufunc rounds to fp32; with
`float64=True` the same graph is evaluated in float64 (the reference for the sums that cancel: d gamma, d beta and the
`- dbeta/B - xhat dgamma/B` term of dx).  The dropout mask is the device's counter-based hash
(`hhfm_oracle.dropout_mask_hashed`).  `oracle/fm_batchnorm_torch.py` is the torch restatement autograd checks this one
against.

The layer is tf.contrib.layers.batch_norm(x, decay=0.9, center=True, scale=True, updates_collections=None,
is_training=train_phase) on x = 0.5 (S^2 - sum_f e_f^2) [B, K], before the dropout of FM.py:114:
  training:    xhat = (x - mu) / sqrt(var + eps), mu / var (biased) over the batch; y = gamma xhat + beta;
               moving_mean -= (1 - decay) (moving_mean - mu); moving_var -= (1 - decay) (moving_var - var B / max(B - 1, 1))
  evaluation:  y = gamma (x - moving_mean) / sqrt(moving_var + eps) + beta, no dropout.
"""
from __future__ import annotations

import numpy as np

from oracle.hhfm_oracle import dropout_mask_hashed

EPS, DECAY = 1e-3, 0.9


def _colsum(a, T):
    """Sum over the batch (axis 0) with numpy's pairwise summation: a reduction along a non-contiguous axis is a running
    sum, whose fp32 rounding grows with B and would dominate the comparison at B = 2^17."""
    return np.ascontiguousarray(a.T).sum(axis=1, dtype=T).astype(T)


def _interaction(X, V, T):
    E = np.asarray(V, T)[X]
    S = E.sum(axis=1, dtype=T)
    x = (T(0.5) * ((S * S).astype(T) - (E * E).astype(T).sum(axis=1, dtype=T))).astype(T)
    return E, S, x


def fm_bn_forward(X, V, b, b0, gamma, beta, moving_mean, moving_var, eps=EPS, float64=False):
    """The evaluation forward (train_phase=False): out [B]."""
    T = np.float64 if float64 else np.float32
    _, _, x = _interaction(X, V, T)
    a = (np.asarray(gamma, T) / np.sqrt((np.asarray(moving_var, T) + T(eps)).astype(T))).astype(T)
    y = ((a * (x - np.asarray(moving_mean, T)).astype(T)).astype(T) + np.asarray(beta, T)).astype(T)
    out = y.sum(axis=1, dtype=T)
    out = (out + np.asarray(b, T).reshape(-1)[X].sum(axis=1, dtype=T)).astype(T)
    return (out + T(np.asarray(b0).reshape(()))).astype(T)


def fm_bn_loss_grads(X, Y, V, b, b0, gamma, beta, moving_mean, moving_var, keep=1.0, seed=0, lamda=0.0, eps=EPS, decay=DECAY,
                     float64=False):
    """One training step.  Returns loss, out [B], a dict of gradients (feature_embeddings [M,K] with + lamda V,
    feature_bias [M], bias, gamma [K], beta [K]) and the new (moving_mean, moving_var)."""
    T = np.float64 if float64 else np.float32
    X = np.asarray(X)
    B = X.shape[0]
    V = np.asarray(V, T)
    E, S, x = _interaction(X, V, T)
    K = V.shape[1]
    mu = (_colsum(x, T) / T(B)).astype(T)
    xc = (x - mu).astype(T)
    var = (_colsum((xc * xc).astype(T), T) / T(B)).astype(T)
    inv = (T(1) / np.sqrt((var + T(eps)).astype(T))).astype(T)
    xh = (xc * inv).astype(T)
    gamma = np.asarray(gamma, T); beta = np.asarray(beta, T)
    y = ((gamma * xh).astype(T) + beta).astype(T)
    m = dropout_mask_hashed(seed, B, K, keep).astype(T) if keep < 1.0 else np.ones((B, K), T)
    z = ((y / T(keep)).astype(T) * m).astype(T)
    out = z.sum(axis=1, dtype=T)
    out = (out + np.asarray(b, T).reshape(-1)[X].sum(axis=1, dtype=T)).astype(T)
    out = (out + T(np.asarray(b0).reshape(()))).astype(T)
    diff = (np.asarray(Y, T).reshape(-1) - out).astype(T)
    loss = T(0.5) * (diff * diff).astype(T).sum(dtype=T)
    g = (-diff).astype(T)
    d = (g[:, None] * (m / T(keep)).astype(T)).astype(T)                       # d loss / d y
    dbeta = _colsum(d, T)
    dgamma = _colsum((d * xh).astype(T), T)
    dx = ((gamma * inv).astype(T) * ((d - (dbeta / T(B)).astype(T)).astype(T) - (xh * (dgamma / T(B)).astype(T)).astype(T))).astype(T)
    dE = (dx[:, None, :] * (S[:, None, :] - E)).astype(T)
    dV = np.zeros_like(V)
    np.add.at(dV, X.reshape(-1), dE.reshape(-1, K))
    db = np.zeros(V.shape[0], T)
    np.add.at(db, X.reshape(-1), np.broadcast_to(g[:, None], X.shape).reshape(-1))
    if lamda > 0:
        loss = T(loss + T(lamda) * T(0.5) * (V * V).astype(T).sum(dtype=T))
        dV = (dV + T(lamda) * V).astype(T)
    f = T(1) - T(decay)
    var_u = (var * T(B / max(B - 1, 1))).astype(T)
    mm = np.asarray(moving_mean, T); mv = np.asarray(moving_var, T)
    mm1 = (mm - ((mm - mu).astype(T) * f).astype(T)).astype(T)
    mv1 = (mv - ((mv - var_u).astype(T) * f).astype(T)).astype(T)
    grads = dict(feature_embeddings=dV, feature_bias=db, bias=g.sum(dtype=T), gamma=dgamma, beta=dbeta)
    return T(loss), out, grads, (mm1, mv1)
