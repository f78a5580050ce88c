"""CPU: FM with batch normalisation of the interaction vector (FM.py:111-112, batch_norm=1) -- the numpy oracle against
torch.autograd through torch.nn.functional.batch_norm, its evaluation forward, and the argument checks of the C entry
points (which run before any launch)."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import assert_close
from oracle import fm_batchnorm as BN
from oracle import fm_batchnorm_torch as TB
from oracle import hhfm_oracle as O


def _problem(B, F, K, seed=0, M=60):
    rng = np.random.default_rng(seed)
    V = rng.normal(0, 0.3, (M, K))
    w = dict(feature_embeddings=V, feature_bias=rng.normal(0, 0.1, M), bias=0.1, gamma=rng.normal(1, 0.2, K),
             beta=rng.normal(0, 0.2, K), moving_mean=rng.normal(0, 0.1, K), moving_variance=rng.uniform(0.5, 2, K))
    X = rng.integers(0, M, (B, F))
    if F > 2:
        X[:, 2] = X[:, 1]                                # a repeated id inside a row
    Y = rng.choice([1.0, 0.0], B)
    return w, X, Y


@pytest.mark.parametrize("B,F,K,keep", [(1, 3, 8, 1.0), (2, 4, 8, 0.7), (2, 1, 12, 1.0), (37, 5, 16, 0.6), (200, 10, 64, 1.0),
                                        (129, 7, 100, 0.8)])
def test_oracle_matches_autograd_in_float64(B, F, K, keep):
    w, X, Y = _problem(B, F, K, seed=B + K)
    seed = 0xC0FFEE + B
    loss, out, g, (mm, mv) = BN.fm_bn_loss_grads(X, Y, w["feature_embeddings"], w["feature_bias"], w["bias"], w["gamma"], w["beta"],
                                                 w["moving_mean"], w["moving_variance"], keep, seed, lamda=0.1, float64=True)
    mask = O.dropout_mask_hashed(seed, B, K, keep) if keep < 1 else np.ones((B, K), np.float32)
    tw = {k: torch.tensor(np.asarray(v, np.float64), requires_grad=k not in ("moving_mean", "moving_variance")) for k, v in w.items()}
    l, o, rm, rv = TB.fm_bn_loss(torch.tensor(X), torch.tensor(Y), tw, keep, torch.tensor(mask, dtype=torch.float64), lamda=0.1)
    l.backward()
    assert abs(loss - l.item()) <= 1e-12 * abs(l.item())
    assert np.allclose(out, o.detach().numpy(), rtol=1e-12, atol=1e-12)
    assert np.allclose(mm, rm.numpy(), rtol=1e-12, atol=1e-14)
    assert np.allclose(mv, rv.numpy(), rtol=1e-12, atol=1e-14)
    for ours, theirs in (("feature_embeddings", "feature_embeddings"), ("feature_bias", "feature_bias"), ("bias", "bias"),
                         ("gamma", "gamma"), ("beta", "beta")):
        ref = tw[theirs].grad.numpy()
        scale = max(float(np.abs(ref).max()), 1e-300)
        assert np.abs(np.asarray(g[ours]) - ref).max() <= 1e-10 * scale, ours


def test_float32_oracle_is_the_same_graph():
    w, X, Y = _problem(500, 8, 32, seed=4)
    args = (X, Y, w["feature_embeddings"], w["feature_bias"], w["bias"], w["gamma"], w["beta"], w["moving_mean"], w["moving_variance"],
            0.8, 99)
    l32, o32, g32, s32 = BN.fm_bn_loss_grads(*args)
    l64, o64, g64, s64 = BN.fm_bn_loss_grads(*args, float64=True)
    assert o32.dtype == np.float32 and g32["gamma"].dtype == np.float32
    assert abs(l32 - l64) <= 1e-5 * abs(l64)
    assert_close(o32, o64, what="out")
    assert_close(s32[0], s64[0], what="moving mean"); assert_close(s32[1], s64[1], what="moving variance")
    assert_close(g32["feature_embeddings"], g64["feature_embeddings"], rtol=1e-4, what="dV")


def test_evaluation_forward_with_the_batch_statistics_is_the_training_output():
    """With moving_mean / moving_var set to the batch's mean and biased variance, and no dropout, the evaluation forward
    and the training forward compute the same thing."""
    w, X, Y = _problem(300, 6, 16, seed=7)
    V = w["feature_embeddings"]
    _, _, x = BN._interaction(X, V, np.float64)
    _, out, _, _ = BN.fm_bn_loss_grads(X, Y, V, w["feature_bias"], w["bias"], w["gamma"], w["beta"], w["moving_mean"],
                                       w["moving_variance"], float64=True)
    ev = BN.fm_bn_forward(X, V, w["feature_bias"], w["bias"], w["gamma"], w["beta"], x.mean(0), x.var(0), float64=True)
    assert np.allclose(ev, out, rtol=1e-12, atol=1e-12)


def test_unit_batch_is_normalised_to_beta():
    w, X, Y = _problem(1, 4, 8, seed=2)
    loss, out, g, (mm, mv) = BN.fm_bn_loss_grads(X, Y, w["feature_embeddings"], w["feature_bias"], w["bias"], w["gamma"], w["beta"],
                                                 w["moving_mean"], w["moving_variance"], float64=True)
    want = w["beta"].sum() + w["feature_bias"][X].sum() + w["bias"]
    assert abs(out[0] - want) <= 1e-12
    assert not np.asarray(g["feature_embeddings"]).any() and not np.asarray(g["gamma"]).any()
    assert np.allclose(mv, 0.9 * w["moving_variance"])


def _p(n=16):
    return ctypes.c_void_p(n)


def _train_args(**over):
    p = _p()
    a = dict(row_ptr=None, col=p, val=None, B=4, F=3, V=p, bias=p, b0=p, M=100, K=64, interaction=0, labels=p, out=None, gV=p,
             gbias=p, gb0=p, lp=p, ts=None, stamp=0, tr=None, tc=None, hs=None, gh=None, ghb=None, n_rep=0, n_hot=0, det=0, keep=1.0,
             seed=0, gamma=p, beta=p, mm=p, mv=p, dgamma=p, dbeta=p, eps=1e-3, decay=0.9, ws=p, ws_bytes=1 << 40, stream=None)
    a.update(over)
    return list(a.values())


@pytest.mark.parametrize("over,what", [
    (dict(K=6), "K=6"), (dict(K=516), "K=516"), (dict(F=0), "F=0"), (dict(col=None), "col and V"),
    (dict(gamma=None), "gamma, beta"), (dict(mv=None), "moving_var"), (dict(dbeta=None), "dgamma and dbeta"),
    (dict(mm=_p(20)), "16-byte aligned"), (dict(eps=0.0), "eps"), (dict(eps=-1e-3), "eps"), (dict(eps=float("nan")), "eps"),
    (dict(decay=1.0), "decay"), (dict(decay=-0.1), "decay"), (dict(decay=float("nan")), "decay"), (dict(keep=0.0), "keep"),
    (dict(keep=1.5), "keep"), (dict(ws=None), "workspace"), (dict(ws=_p(24)), "workspace"), (dict(ws_bytes=1000), "workspace of 1000"),
    (dict(row_ptr=_p()), "fixed-width"), (dict(val=_p()), "fixed-width"), (dict(interaction=1), "interaction"),
    (dict(labels=None), "labels"), (dict(B=0), "empty batch"), (dict(hs=_p()), "hot_slot"), (dict(ts=_p()), "touch_stamp")])
def test_training_entry_rejects_bad_arguments_without_a_gpu(over, what):
    from hhfm_b200 import build, _lib
    build.build()
    with pytest.raises(_lib.HhfmError, match=what):
        _lib.call("hhfm_fm_bn_fwd_bwd_sqloss", *_train_args(**over))


def test_forward_entry_and_workspace_query_without_a_gpu():
    from hhfm_b200 import build, _lib
    build.build()
    lib = _lib.load()
    p = _p()
    assert lib.hhfm_workspace_bytes_fm_bn(1 << 20, 64) >= (1 << 20) * 64 * 4 + 2 * (1 << 20) * 4
    assert lib.hhfm_workspace_bytes_fm_bn(-1, 64) == -1 and lib.hhfm_workspace_bytes_fm_bn(8, 6 * 100) == -1
    for args, what in (((p, 4, 3, p, p, p, 100, 64, p, p, p, p, 0.0, p, None), "eps"),
                       ((p, 4, 3, p, p, p, 100, 64, None, p, p, p, 1e-3, p, None), "gamma"),
                       ((p, 4, 3, p, p, p, 100, 60 + 2, p, p, p, p, 1e-3, p, None), "K=62"),
                       ((p, 4, 3, p, p, p, 100, 64, p, p, p, p, 1e-3, None, None), "out")):
        with pytest.raises(_lib.HhfmError, match=what):
            _lib.call("hhfm_fm_bn_fwd", *args)
