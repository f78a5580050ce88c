"""DeepFM with the reference's options (Newcode/DFM.py:50-152: use_fm, use_deep, loss_type), fp32 NumPy.

`dfm_forward` / `dfm_loss_grads` take the keyword arguments of the reference's constructor; with the defaults they give
bit for bit what `hhfm_oracle.dfm_forward` / `dfm_loss_grads` give.  The TF semantics restated here:
  * concat input [y_first_order | y_second_order | y_deep] (both parts), [F | K] (use_fm only) or [D] (use_deep only),
    times concat_projection (input_size, 1), plus concat_bias;
  * loss_type='logloss': out = sigmoid(logit); loss = tf.losses.log_loss(label, out) with epsilon 1e-7, reduced by
    SUM_BY_NONZERO_WEIGHTS (the mean over the batch); the gradient reaches the logit through TF's SigmoidGrad p (1 - p);
  * L2: l2_reg/2 ||concat_projection||^2, and l2_reg/2 ||layer_i||^2 only when the tower is in the graph.
"""
import numpy as np

from .hhfm_oracle import F32, _f32, _sigmoid

DFM_LOGLOSS_EPS = 1e-7          # tf.losses.log_loss's default epsilon


def dfm_forward(X, w, n_layers=3, use_fm=True, use_deep=True, loss_type="mse"):
    """DFM.py:104-143.  concat_projection is (input_size, 1) with input_size = F+K+D, F+K (use_deep=False) or D
    (use_fm=False); under loss_type='logloss' `out` is sigmoid(logit) (DFM.py:138-139)."""
    V = _f32(w["feature_embeddings"])
    E = V[X]                                                             # :104-105
    S = E.sum(axis=1, dtype=F32)
    parts = []
    if use_fm:
        y1 = _f32(w["feature_bias"]).reshape(-1)[X]                      # :109-110  [B,F]
        y2 = (F32(0.5) * (S * S - (E * E).astype(F32).sum(axis=1, dtype=F32))).astype(F32)   # :114-122
        parts += [y1, y2]
    h = E.reshape(E.shape[0], -1)                                        # :125
    acts = [h]
    if use_deep:
        for i in range(n_layers):                                        # :126-128
            h = np.maximum((h @ _f32(w["layer_%d" % i])).astype(F32) + _f32(w["bias_%d" % i]).reshape(1, -1), F32(0)).astype(F32)
            acts.append(h)
        parts.append(h)
    cat = np.concatenate(parts, axis=1)                                  # :131-136
    logit = ((cat @ _f32(w["concat_projection"])).astype(F32).reshape(-1) + F32(np.asarray(w["concat_bias"]).reshape(()))).astype(F32)  # :137
    out = logit
    if loss_type == "logloss":
        with np.errstate(over="ignore"):
            out = _sigmoid(logit)                                        # :138-139
    return out, dict(E=E, S=S, acts=acts, cat=cat, logit=logit)


def dfm_loss_grads(X, Y, w, l2_reg=0.0, n_layers=3, use_fm=True, use_deep=True, loss_type="mse", B_total=None):
    """DFM.py:139-152 and the gradient of every variable in the graph (TF autodiff restated; relu'(0) = 0).
      mse:     loss = 0.5*sum(y-out)^2
      logloss: loss = tf.losses.log_loss(y, out) = sum_s [-y log(out+eps) - (1-y) log((1-out)+eps)] / B_total (eps = 1e-7,
               SUM_BY_NONZERO_WEIGHTS: the mean over the batch; B_total = len(X) unless the batch is one rank's share),
               d/d logit = out (1-out) (-y/(out+eps) + (1-y)/((1-out)+eps)) / B_total.  Labels are used as given.
      + l2_reg/2*||concat_projection||^2, + l2_reg/2*sum_i ||layer_i||^2 when use_deep.
    Variables outside the graph (feature_bias when not use_fm, the layers and their biases when not use_deep) get no entry."""
    Y = _f32(Y).reshape(-1)
    out, c = dfm_forward(X, w, n_layers, use_fm, use_deep, loss_type)
    V = _f32(w["feature_embeddings"])
    B, F, K = c["E"].shape
    proj = _f32(w["concat_projection"]).reshape(-1)
    if loss_type == "logloss":
        eps = F32(DFM_LOGLOSS_EPS)
        inv = F32(1.0 / (B if B_total is None else B_total))
        q = (F32(1) - out).astype(F32)
        per = (-(Y * np.log((out + eps).astype(F32))).astype(F32) - ((F32(1) - Y) * np.log((q + eps).astype(F32))).astype(F32)).astype(F32)
        loss = F32((per * inv).astype(F32).sum(dtype=F32))
        dp = ((-Y / (out + eps)).astype(F32) + ((F32(1) - Y) / (q + eps)).astype(F32)).astype(F32)
        g = ((dp * inv).astype(F32) * out * q).astype(F32)               # d loss / d logit
    else:
        diff = (Y - out).astype(F32)
        loss = F32(0.5) * (diff * diff).astype(F32).sum(dtype=F32)
        g = (-diff).astype(F32)                                           # d loss / d out
    grads = {}
    grads["concat_projection"] = (c["cat"].T @ g).astype(F32).reshape(-1, 1)
    grads["concat_bias"] = g.sum(dtype=F32)
    d_cat = (g[:, None] * proj[None, :]).astype(F32)
    n_fm = F + K if use_fm else 0
    d_y1, d_y2, d_h = d_cat[:, :F], d_cat[:, F:F + K], d_cat[:, n_fm:]
    dE = np.zeros((B, F, K), F32)
    if use_deep:
        for i in reversed(range(n_layers)):
            h_out, h_in = c["acts"][i + 1], c["acts"][i]
            dZ = (d_h * (h_out > 0)).astype(F32)
            grads["layer_%d" % i] = (h_in.T @ dZ).astype(F32)
            grads["bias_%d" % i] = dZ.sum(axis=0, dtype=F32).reshape(1, -1)
            d_h = (dZ @ _f32(w["layer_%d" % i]).T).astype(F32)
        dE = d_h.reshape(B, F, K)
    if use_fm:
        dE = (dE + (d_y2[:, None, :] * (c["S"][:, None, :] - c["E"])).astype(F32)).astype(F32)
    dV = np.zeros_like(V)
    np.add.at(dV, X.reshape(-1), dE.reshape(-1, K))
    grads["feature_embeddings"] = dV
    if use_fm:
        db = np.zeros(V.shape[0], F32)
        np.add.at(db, X.reshape(-1), d_y1.reshape(-1))
        grads["feature_bias"] = db.reshape(-1, 1)
    if l2_reg > 0:
        for k in ["concat_projection"] + (["layer_%d" % i for i in range(n_layers)] if use_deep else []):
            wk = _f32(w[k])
            loss = F32(loss + F32(l2_reg) * F32(0.5) * (wk * wk).astype(F32).sum(dtype=F32))
            grads[k] = (grads[k] + F32(l2_reg) * wk.reshape(grads[k].shape)).astype(F32)
    return F32(loss), out, grads
