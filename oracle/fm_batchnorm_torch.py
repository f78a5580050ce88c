"""PyTorch-CPU restatement of FM training with batch normalisation of the interaction vector (FM.py:111-112)  --  TEST
INFRASTRUCTURE ONLY.

The graph of `oracle/fm_batchnorm.py` through `torch.nn.functional.batch_norm` (training mode; its running variance is
the Bessel-corrected one, as the moving variance here) and tf.nn.dropout with a given 0/1 mask; torch.autograd on it
checks the analytic gradients of the numpy oracle.  The product never imports this file.
"""
from __future__ import annotations

import torch
import torch.nn.functional as Fn


def fm_bn_loss(X, Y, w, keep, mask, lamda=0.0, eps=1e-3, decay=0.9):
    """w: feature_embeddings [M,K], feature_bias [M], bias [], gamma [K], beta [K], moving_mean [K], moving_variance [K].
    Returns loss, out [B], new moving mean, new moving variance."""
    E = w["feature_embeddings"][X]
    S = E.sum(1)
    x = 0.5 * (S * S - (E * E).sum(1))
    rm = w["moving_mean"].detach().clone()
    rv = w["moving_variance"].detach().clone()
    if x.shape[0] > 1:
        y = Fn.batch_norm(x, rm, rv, w["gamma"], w["beta"], training=True, momentum=1.0 - decay, eps=eps)
    else:
        # torch refuses training-mode batch norm on one sample; the layer maps it to beta, and the Bessel correction of the
        # moving variance takes B - 1 as 1 (so the batch variance, 0, is what the moving variance moves towards)
        xc = x - x.mean(0)
        y = w["gamma"] * xc / torch.sqrt((xc * xc).mean(0) + eps) + w["beta"]
        with torch.no_grad():
            rm = rm - (1.0 - decay) * (rm - x.mean(0))
            rv = rv - (1.0 - decay) * (rv - (xc * xc).mean(0))
    out = (y / keep * mask).sum(1) + w["feature_bias"][X].sum(1) + w["bias"]
    loss = 0.5 * (Y - out).square().sum()
    if lamda > 0:
        loss = loss + lamda * 0.5 * w["feature_embeddings"].square().sum()
    return loss, out, rm, rv
