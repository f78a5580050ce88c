"""PyTorch-CPU restatement of AFM training with dropout and with attention=0  --  TEST INFRASTRUCTURE ONLY.

The op-for-op graph of `oracle/torch_cpu.py::afm_loss` with tf.nn.dropout on the attention weights (AFM.py:126) and on
the pooled vector (:134), and the attention=0 variant (:132).  torch.autograd on it checks the analytic gradients of
`oracle/afm_dropout.py`; run in float64 it is also the reference for gradients whose fp32 sums are cancellation noise.
The product never imports this file.
"""
from __future__ import annotations

import torch


def afm_dropout_loss(X, Y, w, lamda_attention, keep, m_att, m_vec, attention=1):
    """tf.nn.dropout with the given 0/1 masks (m_att [B,P] on the attention weights, m_vec [B,K] on the pooled vector).
    attention=0: afm = sum_p P_p, no attention net and no lamda_attention term (the regulariser sits under `if attention`
    in the AFM authors' code)."""
    E = w["feature_embeddings"][X]
    F = X.shape[1]
    prods = [E[:, i, :] * E[:, j, :] for i in range(F) for j in range(i + 1, F)]
    P = torch.stack(prods).transpose(0, 1)                              # [B,P,K]
    if attention:
        K = P.shape[2]
        mul = (P.reshape(-1, K) @ w["attention_W"]).reshape(P.shape[0], P.shape[1], -1)
        s = (w["attention_p"] * torch.relu(mul + w["attention_b"])).sum(2, keepdim=True)
        a = torch.softmax(s, dim=1) / keep[0] * m_att.unsqueeze(2)
        afm = (a * P).sum(1)
    else:
        afm = P.sum(1)
    afm = afm / keep[1] * m_vec
    out = (afm @ w["prediction"]).sum(1, keepdim=True) + w["feature_bias"][X].sum(1) + w["bias"]
    loss = 0.5 * (Y - out).square().sum()
    if attention and lamda_attention > 0:
        loss = loss + lamda_attention * 0.5 * w["attention_W"].square().sum()
    return loss, out
