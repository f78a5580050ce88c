"""GPU: FM with batch normalisation of the interaction vector (FM.py:111-112, batch_norm=1) -- the training entry
(csrc/fm_bn.cu) against oracle/fm_batchnorm.py over batch sizes, factor sizes, dropout and hot rows; run-to-run
bit-identity of the reductions; the evaluation forward; FM(batch_norm=1) step by step with every optimizer; predict,
topk and the data-parallel refusal; the FM.py drop-in with --batch_norm 1; and the entry points of a batch_norm=0 step."""
import os
import re

import numpy as np
import pytest
import torch

from conftest import assert_close
from oracle import fm_batchnorm as BN
from oracle import hhfm_oracle as O

pytestmark = pytest.mark.gpu

_KEEP = []


def dev(a, cuda, dtype=torch.float32):
    t = torch.as_tensor(np.ascontiguousarray(a)).to(dtype).to(cuda)
    _KEEP.append(t)
    return t


def _problem(B, F, K, seed, M=300):
    rng = np.random.default_rng(seed)
    w = dict(V=rng.normal(0, 0.1, (M, K)).astype(np.float32), b=rng.normal(0, 0.1, M).astype(np.float32), b0=np.float32(0.05),
             gamma=rng.normal(1, 0.1, K).astype(np.float32), beta=rng.normal(0, 0.1, K).astype(np.float32),
             mm=rng.normal(0, 0.01, K).astype(np.float32), mv=rng.uniform(0.5, 1.5, K).astype(np.float32))
    X = rng.integers(0, M, (B, F))
    if F > 2:
        X[:, 2] = X[:, 1]
    Y = rng.choice([1.0, 0.0], B).astype(np.float32)
    return w, X, Y


def _train_call(cuda, X, Y, w, keep, seed, hot, det=0):
    """One pass through hhfm_fm_bn_fwd_bwd_sqloss; the device results as numpy (hot replicas folded)."""
    from hhfm_b200 import _lib
    from hhfm_b200.engine import HotRows, cur_stream, ptr
    B, F = X.shape
    M, K = w["V"].shape
    t = {k: dev(np.asarray(v).reshape(-1) if k == "b0" else v, cuda) for k, v in w.items()}
    gV = torch.zeros(M, K, device=cuda); gb = torch.zeros(M, device=cuda); gb0 = torch.zeros(1, device=cuda)
    dgb = torch.full((2, K), 7.0, device=cuda)                   # written, not accumulated
    lp = torch.zeros(_lib.partials_len(), device=cuda); o = torch.empty(B, device=cuda); lo = torch.zeros(1, device=cuda)
    ws = torch.empty(int(_lib.load().hhfm_workspace_bytes_fm_bn(B, K)), dtype=torch.uint8, device=cuda)
    if hot:
        hp = HotRows(np.arange(0, 8), M, K, cuda, with_bias=True, n_rep=4)
        stamp = torch.zeros(M, dtype=torch.int32, device=cuda); rows = torch.zeros(M, dtype=torch.int32, device=cuda)
        cnt = torch.zeros(1, dtype=torch.int32, device=cuda)
        tail = (ptr(stamp), 3, ptr(rows), ptr(cnt), *hp.args(True))
    else:
        tail = (None, 0, None, None, None, None, None, 0, 0)
    _lib.call("hhfm_fm_bn_fwd_bwd_sqloss", None, ptr(dev(X, cuda, torch.int32)), None, B, F, ptr(t["V"]), ptr(t["b"]), ptr(t["b0"]),
              M, K, 0, ptr(dev(Y, cuda)), ptr(o), ptr(gV), ptr(gb), ptr(gb0), ptr(lp), *tail, det, keep, seed, ptr(t["gamma"]),
              ptr(t["beta"]), ptr(t["mm"]), ptr(t["mv"]), ptr(dgb[0]), ptr(dgb[1]), 1e-3, 0.9, ptr(ws), ws.numel(), cur_stream())
    if hot:
        hp.fold(gV, gb)
        n = int(cnt.item())
        assert sorted(rows[:n].cpu().numpy().tolist()) == sorted(np.unique(X).tolist())
    _lib.call("hhfm_loss_finalize", ptr(lp), None, 0.0, ptr(lo), cur_stream())
    return dict(out=o.cpu().numpy(), loss=lo.item(), V=gV.cpu().numpy(), b=gb.cpu().numpy(), b0=gb0.item(),
                gamma=dgb[0].cpu().numpy(), beta=dgb[1].cpu().numpy(), mm=t["mm"].cpu().numpy(), mv=t["mv"].cpu().numpy())


def _abs_terms(X, Y, V, b, b0, gamma, beta, keep, seed):
    """Sums of the absolute values of the terms that make up each gradient, in float64: the scale of the rounding of a sum
    whose terms cancel (d gamma, d beta, and the - dbeta/B - xhat dgamma/B term of dx).  g = out - y is itself such a sum
    (out = sum_k z_k + sum_f b + b0), so its terms stand in for |g|."""
    T = np.float64
    B, K = X.shape[0], V.shape[1]
    E, S, x = BN._interaction(X, V, T)
    mu = x.mean(0); xc = x - mu; inv = 1 / np.sqrt((xc * xc).mean(0) + 1e-3); xh = xc * inv
    m = O.dropout_mask_hashed(seed, B, K, keep).astype(T) if keep < 1 else np.ones((B, K))
    y = np.asarray(gamma, T) * xh + np.asarray(beta, T)
    g = (np.abs(y / keep * m).sum(1) + np.abs(np.asarray(b, T).reshape(-1)[X]).sum(1) + abs(float(b0)) +
         np.abs(np.asarray(Y, T).reshape(-1)))
    d = g[:, None] * m / keep
    dbeta = np.abs(d).sum(0); dgamma = np.abs(d * xh).sum(0)
    dx = np.abs(np.asarray(gamma, T) * inv) * (np.abs(d) + dbeta / B + np.abs(xh) * dgamma / B)
    dV = np.zeros((V.shape[0], K))
    np.add.at(dV, X.reshape(-1), (dx[:, None, :] * np.abs(S[:, None, :] - E)).reshape(-1, K))
    db = np.zeros(V.shape[0])
    np.add.at(db, X.reshape(-1), np.broadcast_to(np.abs(g)[:, None], X.shape).reshape(-1))
    return dict(V=dV, b=db, b0=np.abs(g).sum(), gamma=dgamma, beta=dbeta)


def _close64(got, ref64, terms, what):
    """|got - ref| <= 1e-5 (|ref| + sum |terms|), ref the float64 evaluation of the same graph."""
    got = np.asarray(got, np.float64).reshape(-1); ref64 = np.asarray(ref64, np.float64).reshape(-1)
    tol = 1e-5 * (np.abs(ref64) + np.asarray(terms, np.float64).reshape(-1))
    err = np.abs(got - ref64)
    assert (err <= tol).all(), "%s: %d/%d off, worst err %.3e tol %.3e" % (what, int((err > tol).sum()), err.size, err.max(),
                                                                            tol[np.argmax(err - tol)])


def _check_pass(got, X, Y, w, keep, seed, what):
    args = (X, Y, w["V"], w["b"], w["b0"], w["gamma"], w["beta"], w["mm"], w["mv"], keep, seed)
    loss, out, g, (mm, mv) = BN.fm_bn_loss_grads(*args)
    _, _, g64, _ = BN.fm_bn_loss_grads(*args, float64=True)
    terms = _abs_terms(X, Y, w["V"], w["b"], w["b0"], w["gamma"], w["beta"], keep, seed)
    assert abs(got["loss"] - loss) <= 1e-5 * abs(loss), (what, got["loss"], loss)
    assert_close(got["out"], out, what=what + " out")
    assert_close(got["mm"], mm, what=what + " moving mean")
    assert_close(got["mv"], mv, what=what + " moving variance")
    for k, ok in (("V", "feature_embeddings"), ("b", "feature_bias"), ("b0", "bias"), ("gamma", "gamma"), ("beta", "beta")):
        _close64(got[k], g64[ok], terms[k], what + " d" + k)


def _cases():
    out = []
    for B in (1, 2, 5000, 1 << 17):
        for K in (8, 64, 100, 128, 512):
            for keep in (1.0, 0.7):
                hots = (False, True) if B == 5000 else ((keep < 1) ^ (K % 3 == 0),)
                out += [(B, K, keep, h) for h in hots]
    return out


@pytest.mark.parametrize("B,K,keep,hot", _cases())
def test_training_pass_matches_oracle(cuda, B, K, keep, hot):
    F = 3 if B > 5000 else 6
    w, X, Y = _problem(B, F, K, seed=B + K)
    seed = 0x5DEECE66D + B + K
    got = _train_call(cuda, X, Y, w, keep, seed, hot)
    _check_pass(got, X, Y, w, keep, seed, "B=%d K=%d keep=%g hot=%d" % (B, K, keep, hot))


@pytest.mark.parametrize("B,K", [(5000, 64), (1 << 17, 100)])
def test_reductions_are_bit_identical_run_to_run(cuda, B, K):
    w, X, Y = _problem(B, 5, K, seed=11)
    a = _train_call(cuda, X, Y, w, 0.7, 1234, True)
    b = _train_call(cuda, X, Y, w, 0.7, 1234, True)
    for k in ("loss", "out", "mm", "mv", "gamma", "beta", "b0"):
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k
    # deterministic = 1: the row scatter is one warp in program order, so the row gradients repeat too
    c = _train_call(cuda, X, Y, w, 0.7, 1234, False, det=1)
    d = _train_call(cuda, X, Y, w, 0.7, 1234, False, det=1)
    for k in c:
        assert np.array_equal(np.asarray(c[k]), np.asarray(d[k])), k
    for k in ("loss", "mm", "mv", "gamma", "beta"):
        assert np.array_equal(np.asarray(a[k]), np.asarray(c[k])), k
    _check_pass(c, X, Y, w, 0.7, 1234, "deterministic")


@pytest.mark.parametrize("K", [8, 64, 100, 512])
def test_inference_forward_matches_oracle(cuda, K):
    from hhfm_b200 import _lib
    from hhfm_b200.engine import cur_stream, ptr
    w, X, _ = _problem(3001, 7, K, seed=K)
    t = {k: dev(np.asarray(v).reshape(-1) if k == "b0" else v, cuda) for k, v in w.items()}
    o = torch.empty(len(X), device=cuda)
    _lib.call("hhfm_fm_bn_fwd", ptr(dev(X, cuda, torch.int32)), len(X), X.shape[1], ptr(t["V"]), ptr(t["b"]), ptr(t["b0"]), 300, K,
              ptr(t["gamma"]), ptr(t["beta"]), ptr(t["mm"]), ptr(t["mv"]), 1e-3, ptr(o), cur_stream())
    assert_close(o.cpu().numpy(), BN.fm_bn_forward(X, w["V"], w["b"], w["b0"], w["gamma"], w["beta"], w["mm"], w["mv"]),
                 what="evaluation forward")


# ---- the model ---------------------------------------------------------------------------------------------------
_NAMES = ("feature_embeddings", "feature_bias", "bias", "bn_fm/gamma", "bn_fm/beta")
_GKEY = {"feature_embeddings": "V", "feature_bias": "b", "bias": "b0", "bn_fm/gamma": "gamma", "bn_fm/beta": "beta"}


def _update(kind, w, s1, s2, g, lr, t, rows=None):
    """One TF1 optimizer step in float64 (Optimizer defaults: Momentum 0.95, Adam 0.9 / 0.999 / 1e-8)."""
    w = np.asarray(w, np.float64); g = np.asarray(g, np.float64).reshape(w.shape)
    if kind == "adagrad":
        return w - lr * g / np.sqrt(s1 + g * g)
    if kind == "sgd":
        return w - lr * g
    if kind == "momentum":
        new = w - lr * (0.95 * s1 + g)
        if rows is not None:                                     # SparseApplyMomentum: only the touched rows move
            keep = np.ones(w.shape[0], bool); keep[rows] = False
            new[keep] = w[keep]
        return new
    lr_t = lr * np.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t)
    m = 0.9 * s1 + 0.1 * g; v = 0.999 * s2 + 0.001 * g * g
    return w - lr_t * m / (np.sqrt(v) + 1e-8)


@pytest.mark.parametrize("opt", ["AdagradOptimizer", "AdamOptimizer", "GradientDescentOptimizer", "MomentumOptimizer"])
def test_model_steps_match_oracle(cuda, opt):
    """FM(batch_norm=1).partial_fit, teacher-forced: each step starts from the model's weights and optimizer slots, the
    oracle's gradients go through the optimizer, and the gradient parity floor (1e-5 of |ref| + sum |terms| against the
    float64 graph) is carried through the update by evaluating it at g -/+ the floor."""
    from hhfm_b200.models import FM
    rng = np.random.default_rng(5)
    n_user, n_item, M, F, K, lr, lam = 40, 60, 160, 5, 64, 0.05, 0.1
    keep = 0.8 if opt != "AdagradOptimizer" else 1.0
    m = FM(F, M, n_user, n_item, K, lr, lam, keep, opt, 1, 0)
    kind = m._opt.kind
    for step in range(3):
        w = m.get_weights()
        st = {}
        for k in _NAMES:
            s = m._opt.state.get(k)
            shape = np.asarray(w[k]).shape
            if s is None:
                s1 = np.full(shape, 0.1) if kind == "adagrad" else np.zeros(shape)
                s2 = np.zeros(shape)
            else:
                s1 = s[0].detach().cpu().numpy().reshape(shape).astype(np.float64) if s[0] is not None else None
                s2 = s[1].detach().cpu().numpy().reshape(shape).astype(np.float64) if s[1] is not None else None
            st[k] = (s1, s2)
        B = 3000 if step < 2 else 517
        X = np.concatenate([np.stack([rng.integers(0, n_user, B), n_user + rng.integers(0, n_item, B)], axis=1),
                            rng.integers(n_user + n_item, M, (B, F - 2))], axis=1)
        Y = rng.choice([1.0, 0.0], (B, 1)).astype(np.float32)
        loss = m.partial_fit({"X": X, "Y": Y})
        seed = m._last_drop_seed if keep < 1 else 0
        args = (X, Y, w["feature_embeddings"], w["feature_bias"], w["bias"], w["bn_fm/gamma"], w["bn_fm/beta"], w["bn_fm/moving_mean"],
                w["bn_fm/moving_variance"], keep, seed, lam)
        loss_ref, _, _, (mm, mv) = BN.fm_bn_loss_grads(*args)
        _, _, g64, _ = BN.fm_bn_loss_grads(*args, float64=True)
        terms = _abs_terms(X, Y, w["feature_embeddings"], w["feature_bias"], w["bias"], w["bn_fm/gamma"], w["bn_fm/beta"], keep, seed)
        assert abs(loss - loss_ref) <= 1e-5 * abs(loss_ref), (step, loss, loss_ref)
        got = m.get_weights()
        assert_close(got["bn_fm/moving_mean"], mm, what="moving mean step %d" % step)
        assert_close(got["bn_fm/moving_variance"], mv, what="moving variance step %d" % step)
        for k in _NAMES:
            g = np.asarray(g64[{"feature_embeddings": "feature_embeddings", "feature_bias": "feature_bias", "bias": "bias",
                                "bn_fm/gamma": "gamma", "bn_fm/beta": "beta"}[k]], np.float64).reshape(np.asarray(w[k]).shape)
            floor = 1e-5 * (np.abs(g) + np.asarray(terms[_GKEY[k]], np.float64).reshape(g.shape))
            if k == "feature_embeddings":
                floor = floor + 1e-5 * lam * np.abs(np.asarray(w[k], np.float64))
            rows = np.unique(X) if (kind == "momentum" and k == "feature_bias") else None
            s1, s2 = st[k]
            ref = _update(kind, w[k], s1, s2, g, lr, m._opt.t, rows)
            lo = _update(kind, w[k], s1, s2, g - floor, lr, m._opt.t, rows)
            hi = _update(kind, w[k], s1, s2, g + floor, lr, m._opt.t, rows)
            delta = ref - np.asarray(w[k], np.float64)
            rms = float(np.sqrt(np.mean(delta * delta)))
            ulp = 4 * 1.2e-7 * np.abs(np.asarray(w[k], np.float64))
            tol = np.maximum(np.abs(hi - ref), np.abs(lo - ref)) + 1e-5 * np.maximum(np.abs(delta), rms) + ulp
            err = np.abs(np.asarray(got[k], np.float64).reshape(ref.shape) - ref)
            assert (err <= tol).all(), (opt, step, k, float(err.max()), float(tol.reshape(-1)[np.argmax(err - tol)]))


def _trained_bn_model(steps=3):
    from hhfm_b200.models import FM
    rng = np.random.default_rng(8)
    n_user, n_item, M, F, K = 50, 120, 200, 4, 32
    m = FM(F, M, n_user, n_item, K, 0.05, 0.1, 1, "AdagradOptimizer", 1, 0)
    for _ in range(steps):
        X = np.concatenate([np.stack([rng.integers(0, n_user, 2000), n_user + rng.integers(0, n_item, 2000)], axis=1),
                            rng.integers(n_user + n_item, M, (2000, F - 2))], axis=1)
        m.partial_fit({"X": X, "Y": rng.choice([1.0, 0.0], (2000, 1)).astype(np.float32)})
    return m, X, (n_user, n_item, M, F, K)


def test_predict_uses_the_moving_statistics_and_topk_ignores_the_layer(cuda):
    from hhfm_b200.models import FM
    m, X, (n_user, n_item, M, F, K) = _trained_bn_model()
    w = m.get_weights()
    assert not np.allclose(w["bn_fm/moving_mean"], 0) and not np.allclose(w["bn_fm/moving_variance"], 1)
    out = m.predict(X[:500])[:, 0]
    want = BN.fm_bn_forward(X[:500], w["feature_embeddings"], w["feature_bias"], w["bias"], w["bn_fm/gamma"], w["bn_fm/beta"],
                            w["bn_fm/moving_mean"], w["bn_fm/moving_variance"])
    assert_close(out, want, what="predict")
    init = BN.fm_bn_forward(X[:500], w["feature_embeddings"], w["feature_bias"], w["bias"], w["bn_fm/gamma"], w["bn_fm/beta"],
                            np.zeros(K), np.ones(K))
    assert np.abs(out - init).max() > 1e-3 * np.abs(init).max()
    # topk scores b[n] + (u_c + F_c) . (v_n + F_c) from the embeddings (FM.py:174-185), as without the layer
    plain = FM(F, M, n_user, n_item, K, 0.05, 0.1, 1, "AdagradOptimizer", 0, 0)
    plain.load_weights({k: w[k] for k in ("feature_embeddings", "feature_bias", "bias")})
    A = X[:64]
    assert np.array_equal(m.topk(A, 20), plain.topk(A, 20))


def test_data_parallel_is_refused(cuda):
    m, _, _ = _trained_bn_model(steps=1)
    with pytest.raises(NotImplementedError, match="batch_norm"):
        m.enable_data_parallel()


def test_batch_norm_0_step_calls_the_parent_entry_points(cuda):
    from hhfm_b200 import _lib
    from hhfm_b200.models import FM
    rng = np.random.default_rng(2)
    M, B = 300, 4096
    for keep, opt, want in ((1, "AdagradOptimizer", {"hhfm_fm_fwd_bwd_sqloss_st": 1, "hhfm_dp_step": 1}),
                            (0.8, "AdagradOptimizer", {"hhfm_fm_fwd_bwd_sqloss_st": 1, "hhfm_dp_step": 1}),
                            (1, "MomentumOptimizer", {"hhfm_fm_fwd_bwd_sqloss_st": 1, "hhfm_opt_momentum_dense_l2": 2,
                                                      "hhfm_opt_momentum_rows": 1, "hhfm_loss_finalize": 1})):
        m = FM(6, M, 50, 100, 64, 0.05, 0.1, keep, opt, 0, 0)
        idx = dev(rng.integers(0, M, (B, 6)), cuda, torch.int32)
        y = dev(rng.choice([1.0, 0.0], B), cuda)
        m.fit_device(idx, y)                                     # first step plans the hot rows
        before = dict(_lib.CALLS)
        m.fit_device(idx, y)
        torch.cuda.synchronize()
        delta = {k: v - before.get(k, 0) for k, v in _lib.CALLS.items() if v != before.get(k, 0)}
        assert delta == want, (keep, opt, delta)


@pytest.mark.parametrize("flags", [["--batch_norm", "1"], ["--batch_norm", "1", "--keep", "0.8"]])
def test_fm_main_with_batch_norm(cuda, flags, tmp_path, monkeypatch):
    rng = np.random.default_rng(3)
    name, rows, n_user, n_item = "frappe", 4000, 60, 120
    os.makedirs(os.path.join(str(tmp_path), name))
    u = rng.integers(0, n_user, rows); it = rng.integers(0, n_item, rows)
    day = rng.integers(0, 7, rows); wk = rng.integers(0, 2, rows); hw = rng.integers(0, 3, rows)
    with open(os.path.join(str(tmp_path), name, name + ".libfm"), "w") as f:
        for r in range(rows):
            f.write("1 u%d i%d d%d w%d h%d\n" % (u[r], it[r], day[r], wk[r], hw[r]))
    result = os.path.join(str(tmp_path), "result.txt")
    monkeypatch.setenv("HHFM_RESULT_FILE", result)
    from hhfm_b200 import trainer
    from hhfm_b200.Newcode.FM import FM_main
    monkeypatch.setattr(trainer.BaseTrain, "device_sampler", False)
    np.random.seed(7)
    session = FM_main(name, 32, 5, argv=["--path", os.path.join(str(tmp_path), ""), "--epoch", "3", "--batch_size", "2000",
                                        "--verbose", "1"] + flags)
    assert session.model._bn
    losses = [float(x) for x in session.loss_epoch]
    assert losses and all(np.isfinite(losses))
    text = open(result).read()
    m = re.findall(r"AUC:([0-9.naninf]+);test=AUC:([0-9.naninf]+),HR:([0-9.naninf]+),NDCG:([0-9.naninf]+)", text)
    assert m and all(np.isfinite(float(v)) for row in m for v in row), text


def test_lazy_l2_takes_the_dense_steps(cuda, monkeypatch):
    """HHFM_LAZY_L2=1 (rows brought up to date when gathered, flushed when read): the same weights and layer state as the
    dense update of every row."""
    from hhfm_b200.models import FM
    rng = np.random.default_rng(12)
    M, F, B = 160, 5, 3000
    batches = [{"X": rng.integers(0, M, (B, F)), "Y": rng.choice([1.0, 0.0], (B, 1)).astype(np.float32)} for _ in range(3)]
    res = {}
    for lazy in ("0", "1"):
        monkeypatch.setenv("HHFM_LAZY_L2", lazy)
        m = FM(F, M, 40, 60, 64, 0.05, 0.1, 1, "AdagradOptimizer", 1, 0)
        m.deterministic = True
        assert m._lazy() == (lazy == "1")
        for b in batches:
            m.partial_fit(b)
        res[lazy] = m.get_weights()
    for k in res["0"]:
        assert np.allclose(res["1"][k], res["0"][k], rtol=1e-5, atol=1e-7), k
