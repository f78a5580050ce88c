"""GPU: AFM training with dropout (keep < 1, AFM.py:126,134) and with attention=0 (AFM.py:132) on every kernel that runs
it -- the fused tcgen05 pass (afm_fused_tc.cu, DROP instantiation), the two fp32 CUDA-core layouts (afm.cu) and the
attention=0 kernel -- against oracle/afm_dropout.py (afm_dropout_loss_grads) with the same masks; then the model (partial_fit + TF1
Adagrad, predict, topk) and the AFM.py drop-in with --keep / --attention 0."""
import os

import numpy as np
import pytest
import torch

from conftest import assert_close, assert_update_close
from oracle import afm_dropout as AD
from oracle import hhfm_oracle as O

pytestmark = pytest.mark.gpu

_KEEP = []


def dev(a, cuda, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    t = t.to(cuda)
    _KEEP.append(t)
    return t


def _weights(rng, M, K, A):
    return dict(feature_embeddings=rng.normal(0, 0.1, (M, K)).astype(np.float32), feature_bias=rng.normal(0, 0.1, (M, 1)).astype(np.float32),
                bias=np.float32(0.05), attention_W=rng.normal(0, 0.2, (K, A)).astype(np.float32),
                attention_b=rng.normal(0, 0.2, (1, A)).astype(np.float32), attention_p=rng.normal(0, 1, (A,)).astype(np.float32),
                prediction=rng.normal(1, 0.1, (K, 1)).astype(np.float32))


def _train_call(cuda, X, Y, w, attention, keep, seed, sample_base, extras, entry="hhfm_afm_fwd_bwd_sqloss_dropout"):
    """One training pass through the C entry; returns the device results as numpy (hot replicas folded)."""
    from hhfm_b200 import _lib
    from hhfm_b200.engine import HotRows, cur_stream, ptr
    B, F = X.shape
    M, K = w["feature_embeddings"].shape
    A = w["attention_W"].shape[1]
    tw = {k: dev(np.asarray(v, np.float32).reshape(-1) if k == "bias" else v, cuda) for k, v in w.items()}
    gV = torch.zeros(M, K, device=cuda); gb = torch.zeros(M, device=cuda); gb0 = torch.zeros(1, device=cuda)
    gW = torch.zeros(K, A, device=cuda); gba = torch.zeros(A, device=cuda); gp = torch.zeros(A, device=cuda); gwp = torch.zeros(K, device=cuda)
    lp = torch.zeros(_lib.partials_len(), device=cuda); o = torch.empty(B, device=cuda); lo = torch.zeros(1, device=cuda)
    tX = dev(X, cuda, torch.int32)
    if extras:
        hot = HotRows(np.arange(0, 8), M, K, cuda, with_bias=True, n_rep=4)
        stamp = torch.zeros(M, dtype=torch.int32, device=cuda); rows = torch.zeros(M, dtype=torch.int32, device=cuda)
        cnt = torch.zeros(1, dtype=torch.int32, device=cuda)
        tail = (ptr(stamp), 3, ptr(rows), ptr(cnt), *hot.args(True))
    else:
        tail = (None, 0, None, None, None, None, None, 0, 0)
    args = (ptr(tX), B, F, ptr(tw["feature_embeddings"]), ptr(tw["feature_bias"]), ptr(tw["bias"]), ptr(tw["attention_W"]),
            ptr(tw["attention_b"]), ptr(tw["attention_p"]), ptr(tw["prediction"]), M, K, A, ptr(dev(Y.reshape(-1), cuda)), ptr(o),
            ptr(gV), ptr(gb), ptr(gb0), ptr(gW), ptr(gba), ptr(gp), ptr(gwp), ptr(lp), *tail)
    if entry == "hhfm_afm_fwd_bwd_sqloss":
        _lib.call(entry, *args, cur_stream())
    else:
        _lib.call(entry, *args, attention, keep[0], keep[1], seed, sample_base, cur_stream())
    if extras:
        hot.fold(gV, gb)
        n = int(cnt.item())
        assert sorted(rows[:n].cpu().numpy().tolist()) == sorted(np.unique(X).tolist())
    _lib.call("hhfm_loss_finalize", ptr(lp), None, 0.0, ptr(lo), cur_stream())
    return dict(out=o.cpu().numpy(), loss=lo.item(), feature_embeddings=gV.cpu().numpy(), feature_bias=gb.cpu().numpy(),
                bias=gb0.item(), attention_W=gW.cpu().numpy(), attention_b=gba.cpu().numpy(), attention_p=gp.cpu().numpy(),
                prediction=gwp.cpu().numpy())


def _grads64(X, Y, w, lam, keep, seed, attention, sample_base=0):
    """The gradients of the same graph and masks in float64 (torch autograd on oracle/afm_dropout_torch.py).  d attention_b and
    d attention_p are sums of B*P terms that cancel (the softmax gradients sum to zero over the pairs); with dropout their
    fp32 rounding in the oracle alone reaches the tolerance, so those two are compared with this evaluation instead."""
    from oracle import afm_dropout_torch as TD
    B, F = X.shape
    m_att, m_vec = AD.afm_dropout_masks(seed, B, F * (F - 1) // 2, w["prediction"].shape[0], keep, sample_base)
    tw = {k: torch.tensor(np.asarray(v, np.float64), requires_grad=True) for k, v in w.items()}
    loss, _ = TD.afm_dropout_loss(torch.tensor(X), torch.tensor(Y, dtype=torch.float64), tw, lam, keep,
                                 torch.tensor(m_att, dtype=torch.float64), torch.tensor(m_vec, dtype=torch.float64), attention)
    loss.backward()
    return {k: (t.grad.numpy() if t.grad is not None else np.zeros(t.shape)) for k, t in tw.items()}


def _check(got, loss, out, g, attention, B, what, g64=None):
    assert_close(got["out"], out, what=what + " out"); assert_close(got["loss"], loss, what=what + " loss")
    assert_close(got["feature_embeddings"], g["feature_embeddings"], rtol=2e-5, what=what + " gV")
    assert_close(got["feature_bias"], g["feature_bias"].reshape(-1), what=what + " gbias")
    assert_close(got["bias"], g["bias"], what=what + " gb0")
    assert_close(got["prediction"], g["prediction"].reshape(-1), rtol=2e-5, what=what + " gw_pred")
    if attention:
        assert_close(got["attention_W"], g["attention_W"], rtol=2e-5, what=what + " gW")
        # d attention_b / p sum d s_p over the pairs, which sums to zero per sample: cancellation noise, floored at 1e-5 of
        # the attention_W gradient's scale as in the keep = [1, 1] tests
        noise = 2e-5 if B < 2000 else 1e-4
        floor = 1e-5 * float(np.abs(g["attention_W"]).max())
        ref = g64 if g64 is not None else g
        assert_close(got["attention_b"], ref["attention_b"].reshape(-1), rtol=noise, atol=floor, what=what + " gb_att")
        assert_close(got["attention_p"], ref["attention_p"].reshape(-1), rtol=noise, atol=floor, what=what + " gp")
    else:
        for k in ("attention_W", "attention_b", "attention_p"):
            assert not got[k].any(), what + " " + k + " must not be written under attention=0"


def _problem(B, F, K, seed):
    rng = np.random.default_rng(seed)
    M = 300
    w = _weights(rng, M, K, K)
    X = rng.integers(0, M, (B, F)); X[:, 1] = rng.integers(0, 4, B)
    if F > 3:
        X[:, 3] = X[:, 2]
    Y = rng.choice([1.0, -1.0], (B, 1)).astype(np.float32)
    return w, X, Y


# (kernel, B, F, K): "tc4" / "tc2" the fused tcgen05 pass (16 / 8 warps), "afm2" pair-per-lane, "afm1" column-per-lane
CASES = [("tc4", 1001, 10, 64), ("tc4", 64, 11, 64), ("tc4", 77, 3, 64), ("tc4", 517, 6, 64), ("tc2", 1001, 10, 64), ("tc2", 130, 6, 64),
         ("afm2", 1001, 10, 64), ("afm2", 130, 6, 32), ("afm2", 37, 7, 16),
         ("afm1", 1001, 10, 64), ("afm1", 77, 12, 128), ("afm1", 130, 6, 32), ("afm1", 50, 3, 16)]
ENV = {"tc4": dict(HHFM_AFM_TC=None, HHFM_AFM_V1=None), "tc2": dict(HHFM_AFM_TC="2", HHFM_AFM_V1=None),
       "afm2": dict(HHFM_AFM_TC="0", HHFM_AFM_V1="0"), "afm1": dict(HHFM_AFM_TC="0", HHFM_AFM_V1="1")}


def _env(monkeypatch, kernel):
    for k, v in ENV[kernel].items():
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, v)


@pytest.mark.parametrize("kernel,B,F,K", CASES)
@pytest.mark.parametrize("keep,extras", [((0.7, 0.5), False), ((0.5, 1.0), True), ((1.0, 0.5), True)])
def test_afm_dropout_pass_matches_oracle(cuda, kernel, B, F, K, keep, extras, monkeypatch):
    _env(monkeypatch, kernel)
    w, X, Y = _problem(B, F, K, B + F + K)
    seed, base = 0x5DEECE66D + B, 1000 * F
    loss, out, g = AD.afm_dropout_loss_grads(X, Y, w, 0.0, keep, seed, 1, sample_base=base)
    got = _train_call(cuda, X, Y, w, 1, keep, seed, base, extras)
    _check(got, loss, out, g, 1, B, "%s keep=%s" % (kernel, keep), _grads64(X, Y, w, 0.0, keep, seed, 1, base))


@pytest.mark.parametrize("K", [32, 64, 128])
@pytest.mark.parametrize("keep,extras", [((1.0, 1.0), False), ((0.3, 0.5), True)])
def test_afm_attention0_pass_matches_oracle(cuda, K, keep, extras):
    B, F = 1001, 10
    w, X, Y = _problem(B, F, K, K + 5)
    seed, base = 77, 5
    loss, out, g = AD.afm_dropout_loss_grads(X, Y, w, 0.0, keep, seed, 0, sample_base=base)
    got = _train_call(cuda, X, Y, w, 0, keep, seed, base, extras)
    _check(got, loss, out, g, 0, B, "attention=0 K=%d" % K)
    from hhfm_b200 import _lib
    from hhfm_b200.engine import cur_stream, ptr
    tw = {k: dev(np.asarray(v, np.float32).reshape(-1) if k == "bias" else v, cuda) for k, v in w.items()}
    o = torch.empty(B, device=cuda)
    _lib.call("hhfm_afm_fwd_attn", ptr(dev(X, cuda, torch.int32)), B, F, ptr(tw["feature_embeddings"]), ptr(tw["feature_bias"]),
              ptr(tw["bias"]), ptr(tw["attention_W"]), ptr(tw["attention_b"]), ptr(tw["attention_p"]), ptr(tw["prediction"]), 300, K, K,
              0, ptr(o), cur_stream())
    assert_close(o.cpu().numpy(), AD.afm_forward(X, w, attention=0)[0], what="attention=0 forward")


@pytest.mark.parametrize("kernel", ["tc4", "afm2", "afm1"])
def test_no_dropout_through_the_new_entry_is_the_existing_pass(cuda, kernel, monkeypatch):
    """keep = [1, 1], attention = 1 runs the kernels of hhfm_afm_fwd_bwd_sqloss: out and the loss are bit-identical; the
    gradients are added with float atomics, whose order differs from launch to launch, so they are held to 1e-5."""
    _env(monkeypatch, kernel)
    w, X, Y = _problem(1001, 10, 64, 3)
    a = _train_call(cuda, X, Y, w, 1, (1.0, 1.0), 123, 9, True)
    b = _train_call(cuda, X, Y, w, 1, (1.0, 1.0), 0, 0, True, entry="hhfm_afm_fwd_bwd_sqloss")
    assert np.array_equal(a["out"], b["out"]) and a["loss"] == b["loss"]
    for k in ("feature_embeddings", "feature_bias", "bias", "attention_W", "prediction"):
        assert_close(a[k], b[k], rtol=1e-5, what=k)


def _frappe_like(rng, B, n_user, n_item, ctx=(7, 2, 3, 9)):
    cols = [rng.integers(0, n_user, B), n_user + rng.integers(0, n_item, B)]
    base = n_user + n_item
    for c in ctx:
        cols.append(base + rng.integers(0, c, B))
        base += c
    return np.stack(cols, axis=1), base


@pytest.mark.parametrize("attention,keep", [(1, [0.7, 0.5]), (0, [1, 1]), (0, [1, 0.5])])
def test_afm_dropout_steps_match_oracle(cuda, attention, keep):
    """AFM.partial_fit with dropout / attention=0, teacher-forced against the oracle (mask seed from the model) + TF1 Adagrad;
    predict and topk score without dropout."""
    from hhfm_b200.models import AFM
    rng = np.random.default_rng(17)
    n_user, n_item = 60, 200
    X0, M = _frappe_like(rng, 10, n_user, n_item)
    K, lr, lam = 64, 0.1, 100.0
    F = X0.shape[1]
    model = AFM(n_user, n_item, M, attention, [K, K], 'relu', lr, lam, keep, 'AdagradOptimizer', 0.999, F)
    names = ["feature_embeddings", "feature_bias", "bias", "attention_W", "attention_b", "attention_p", "prediction"]
    w_init = model.get_weights()
    for step in range(4):
        w = model.get_weights()
        acc = {k: (model._opt.state[k][0].detach().cpu().numpy().reshape(np.asarray(w[k]).shape).copy() if k in model._opt.state
                   else np.full(np.asarray(w[k]).shape, 0.1, np.float32)) for k in names}
        X, _ = _frappe_like(rng, 3000 if step < 3 else 517, n_user, n_item)
        Y = rng.choice([1.0, -1.0], (len(X), 1)).astype(np.float32)
        loss = model.partial_fit({"X": X, "Y": Y})
        seed = model._last_drop_seed if min(keep) < 1 else 0
        loss_ref, _, g = AD.afm_dropout_loss_grads(X, Y, w, lam, keep, seed, attention)
        g64 = _grads64(X, Y, w, lam, keep, seed, attention)
        g = dict(g, attention_b=g64["attention_b"].astype(np.float32), attention_p=g64["attention_p"].astype(np.float32))
        assert_close(loss, loss_ref, what="loss step %d" % step)
        got = model.get_weights()
        for k in names:
            if not attention and k in ("attention_W", "attention_b", "attention_p"):
                assert np.array_equal(got[k], w_init[k]), "%s moved under attention=0" % k
                continue
            gk = np.asarray(g[k], np.float32).reshape(np.asarray(w[k]).shape)
            w1, _ = O.adagrad_dense(np.asarray(w[k], np.float32), acc[k], gk, lr)
            if k in ("feature_embeddings", "feature_bias"):
                assert_update_close(got[k], w1, w[k], gk, acc[k], lr, rtol=3e-5, what="%s step %d" % (k, step))
            else:
                # small dense variables: compared norm-wise, as in test_afm_steps_and_topk_match_oracle
                d_ref = np.asarray(w1, np.float64) - np.asarray(w[k], np.float64)
                d_got = np.asarray(got[k], np.float64).reshape(d_ref.shape) - np.asarray(w[k], np.float64)
                ulp = 4 * 1.2e-7 * float(np.abs(np.asarray(w[k], np.float64)).max())
                tol = 1e-4 * np.abs(d_ref).max() + 1e-8 + ulp
                if k in ("attention_b", "attention_p"):
                    # sums over B*P terms that cancel exactly once the relus of most pairs are off (max |g| ~ 1e-15 here):
                    # the kernels' parity floor for them, 1e-5 of the attention_W data gradient (DESIGN 2), carried
                    # through the Adagrad step lr * g / sqrt(acc)
                    g_w_data = np.asarray(g["attention_W"], np.float64) - lam * np.asarray(w["attention_W"], np.float64)
                    tol += lr * 1e-5 * float(np.abs(g_w_data).max()) / float(np.sqrt(np.asarray(acc[k], np.float64).min()))
                assert np.abs(d_got - d_ref).max() <= tol, \
                    (k, step, np.abs(d_got - d_ref).max(), np.abs(d_ref).max(), np.abs(gk).max(), tol)
    w = model.get_weights()
    out = model.predict(X[:300])[:, 0]
    assert_close(out, AD.afm_forward(X[:300], w, attention)[0], what="predict (no dropout)")
    A = X[:20]
    ids = model.topk(A, 20)
    rows = np.repeat(A[:, None, :], n_item, 1); rows[:, :, 1] = n_user + np.arange(n_item)[None, :]
    ref = AD.afm_forward(rows.reshape(-1, F), w, attention)[0].reshape(20, n_item)
    want = O.topk_lowest_index(ref, 20)
    for r in range(len(A)):
        if (ids[r] == want[r]).all():
            continue
        kth = ref[r, want[r, -1]]
        tol = 2e-5 * max(abs(kth), float(np.sqrt(np.mean(ref[r] ** 2))))
        for a_, b_ in zip(ids[r], want[r]):
            assert abs(ref[r, a_] - ref[r, b_]) <= tol, (r, a_, b_)


@pytest.mark.parametrize("flags", [["--keep", "[0.5,0.5]"], ["--attention", "0"]])
def test_afm_main_with_dropout_and_attention0(cuda, flags, tmp_path, monkeypatch):
    rng = np.random.default_rng(3)
    name, rows, n_user, n_item = "frappe", 4000, 60, 120
    os.makedirs(os.path.join(str(tmp_path), name))
    u = rng.integers(0, n_user, rows); it = rng.integers(0, n_item, rows)
    day = rng.integers(0, 7, rows); wk = rng.integers(0, 2, rows); hw = rng.integers(0, 3, rows)
    with open(os.path.join(str(tmp_path), name, name + ".libfm"), "w") as f:
        for r in range(rows):
            f.write("1 u%d i%d d%d w%d h%d\n" % (u[r], it[r], day[r], wk[r], hw[r]))
    monkeypatch.setenv("HHFM_RESULT_FILE", os.path.join(str(tmp_path), "result.txt"))
    from hhfm_b200 import trainer
    from hhfm_b200.Newcode.AFM import AFM_main
    monkeypatch.setattr(trainer.BaseTrain, "device_sampler", False)
    np.random.seed(7)
    session = AFM_main(name, 32, 5, argv=["--path", os.path.join(str(tmp_path), ""), "--epoch", "3", "--batch_size", "2000",
                                         "--verbose", "1"] + flags)
    losses = [float(x) for x in session.loss_epoch]
    assert losses and all(np.isfinite(losses))
    text = open(os.path.join(str(tmp_path), "result.txt")).read()
    import re
    m = re.findall(r"AUC:([0-9.naninf]+)", text)
    assert m and all(np.isfinite(float(x)) for x in m), text
