"""CPU: the AFM training pass with dropout (keep < 1, AFM.py:126,134) and the attention=0 variant (AFM.py:132) --
the oracle against torch.autograd on the same masks, its reductions to the existing oracles, the mask streams, and
the argument checks of the C entry points (which run before any launch)."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import assert_close
from oracle import afm_dropout as AD
from oracle import hhfm_oracle as O
from oracle import afm_dropout_torch as TD


def _problem(seed=0, M=200, K=16, A=16, B=64, F=6):
    rng = np.random.default_rng(seed)
    w = dict(feature_embeddings=rng.normal(0, 0.1, (M, K)).astype(np.float32),
             feature_bias=rng.normal(0, 0.1, (M, 1)).astype(np.float32), bias=np.float32(0.1),
             attention_W=rng.normal(0, 0.2, (K, A)).astype(np.float32),
             attention_b=rng.normal(0, 0.2, (1, A)).astype(np.float32),
             attention_p=rng.normal(0, 1, (A,)).astype(np.float32),
             prediction=rng.normal(1, 0.1, (K, 1)).astype(np.float32))
    X = rng.integers(0, M, (B, F)); X[:, 3] = X[:, 2]
    Y = rng.choice([1.0, -1.0], (B, 1)).astype(np.float32)
    return w, X, Y


@pytest.mark.parametrize("attention", [1, 0])
@pytest.mark.parametrize("keep", [(1.0, 1.0), (0.7, 0.5), (0.5, 1.0)])
def test_afm_dropout_gradients_agree_with_autograd(attention, keep):
    w, X, Y = _problem()
    seed, base = 0x1234567890ABCDEF, 17
    loss, out, g = AD.afm_dropout_loss_grads(X, Y, w, 100.0, keep, seed, attention, sample_base=base)
    B, F = X.shape
    m_att, m_vec = AD.afm_dropout_masks(seed, B, F * (F - 1) // 2, w["prediction"].shape[0], keep, base)
    tw = {k: torch.tensor(v, requires_grad=True) for k, v in w.items()}
    l, o = TD.afm_dropout_loss(torch.tensor(X), torch.tensor(Y), tw, 100.0, keep, torch.tensor(m_att), torch.tensor(m_vec),
                              attention)
    l.backward()
    assert_close(loss, l.item(), what="loss")
    assert_close(out, o.detach().numpy()[:, 0], what="out")
    assert len(g) == 7
    for k in g:
        ref = tw[k].grad
        ref = np.zeros(tw[k].shape, np.float32) if ref is None else ref.numpy()
        assert_close(np.asarray(g[k]).reshape(-1), ref.reshape(-1), rtol=2e-5, what="grad " + k)
    if not attention:
        for k in ("attention_W", "attention_b", "attention_p"):
            assert not np.asarray(g[k]).any(), k


def test_no_dropout_is_bit_identical_to_afm_loss_grads():
    w, X, Y = _problem(1)
    loss0, out0, g0 = O.afm_loss_grads(X, Y, w, 100.0)
    loss1, out1, g1 = AD.afm_dropout_loss_grads(X, Y, w, 100.0, (1.0, 1.0), 99, 1, sample_base=5)
    assert loss0 == loss1 and (out0 == out1).all()
    for k in g0:
        assert np.array_equal(np.asarray(g0[k]), np.asarray(g1[k])), k
    assert (O.afm_forward(X, w)[0] == AD.afm_forward(X, w, attention=1)[0]).all()


def test_attention0_with_unit_projection_is_the_fm_bilinear_term():
    """attention=0 and prediction = ones: out is FM's dropped interaction under the same mask (FM.py:109-114)."""
    w, X, Y = _problem(2)
    w["prediction"] = np.ones_like(w["prediction"])
    seed, keep = 4242, (0.3, 0.6)
    loss, out, g = AD.afm_dropout_loss_grads(X, Y, w, 100.0, keep, seed, attention=0)
    vseed = int(O._splitmix64(np.uint64(seed)))
    floss, fout, dV, db, db0 = O.fm_dropout_loss_grads(X, Y, w["feature_embeddings"], w["feature_bias"], w["bias"], keep[1], vseed)
    assert (out == fout).all() and loss == floss
    assert_close(g["feature_embeddings"], dV, rtol=1e-6, what="dV")
    assert_close(g["feature_bias"].reshape(-1), db, what="db"); assert_close(g["bias"], db0, what="db0")
    # and without dropout, the forward with attention=0 is the same sum
    assert (AD.afm_forward(X, w, attention=0)[0] == AD.afm_dropout_loss_grads(X, Y, w, 0.0, (1, 1), 0, attention=0)[1]).all()


def test_mask_streams():
    B, P, K, seed = 4096, 45, 64, 0xDEADBEEF
    for keep in ((0.7, 0.5), (0.5, 0.9), (0.1, 0.3)):
        m_att, m_vec = AD.afm_dropout_masks(seed, B, P, K, keep)
        for m, k in ((m_att, keep[0]), (m_vec, keep[1])):
            n = m.size
            sigma = np.sqrt(n * k * (1 - k))
            assert abs(m.sum() - n * k) <= 5 * sigma, (m.sum(), n * k)
    m_att, m_vec = AD.afm_dropout_masks(seed, B, K, K, (0.5, 0.5))
    assert (m_att == O.dropout_mask_hashed(seed, B, K, 0.5)).all()          # the FM / MF mask hash (csrc/common.cuh)
    assert (m_att != m_vec).mean() > 0.4                          # independent streams, not one mask twice
    a1, v1 = AD.afm_dropout_masks(seed, B, P, K, (0.5, 0.5), sample_base=0)
    a2, v2 = AD.afm_dropout_masks(seed, B - 100, P, K, (0.5, 0.5), sample_base=100)
    assert (a1[100:] == a2).all() and (v1[100:] == v2).all()
    assert (a1[:-100] != a2).any()
    ones = AD.afm_dropout_masks(seed, 64, P, K, (1.0, 1.0))
    assert all(m.all() for m in ones)


def _p(n=16):
    return ctypes.c_void_p(n)


def test_dropout_entry_rejects_bad_keep_and_attention_without_a_gpu():
    from hhfm_b200 import build, _lib
    build.build()
    p = _p()
    head = (p, 4, 10, p, p, p, p, p, p, p, 100, 64, 64, p, None, p, p, p, p, p, p, p, p, None, 0, None, None, None, None, None, 0, 0)
    for att, k0, k1, what in ((1, 0.0, 1.0, "keep"), (1, 1.0, 1.5, "keep"), (0, 1.0, -0.5, "keep"), (1, float("nan"), 1.0, "keep"),
                              (2, 1.0, 1.0, "attention"), (-1, 0.5, 0.5, "attention")):
        with pytest.raises(_lib.HhfmError, match=what):
            _lib.call("hhfm_afm_fwd_bwd_sqloss_dropout", *head, att, k0, k1, 7, 0, None)
    with pytest.raises(_lib.HhfmError, match="sample_base"):
        _lib.call("hhfm_afm_fwd_bwd_sqloss_dropout", *head, 1, 0.5, 0.5, 7, -1, None)
    with pytest.raises(_lib.HhfmError, match="attention"):
        _lib.call("hhfm_afm_fwd_attn", p, 4, 10, p, p, p, p, p, p, p, 100, 64, 64, 3, p, None)
