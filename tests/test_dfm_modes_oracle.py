"""CPU: DeepFM with the reference's options (use_fm, use_deep, loss_type).  The fp32 oracle (oracle/dfm_modes.py) against a
float64 torch-autograd restatement of the TF graph, its defaults against the existing DeepFM oracle, and the mode checks
of the C ABI (no GPU needed)."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import assert_close
from oracle import dfm_modes as D
from oracle import hhfm_oracle as O

MODES = [(True, True), (True, False), (False, True)]


def _weights(rng, M, F, K, layers, use_fm, use_deep, scale=1.0):
    dims = [F * K] + list(layers)
    n_in = (F + K if use_fm else 0) + (dims[-1] if use_deep else 0)
    w = dict(feature_embeddings=rng.normal(0, 0.3, (M, K)).astype(np.float32),
             feature_bias=rng.uniform(0, 1, (M, 1)).astype(np.float32),
             concat_projection=(scale * rng.normal(0, np.sqrt(2.0 / (n_in + 1)), (n_in, 1))).astype(np.float32),
             concat_bias=np.float32(0.01))
    for i in range(len(layers)):
        gl = np.sqrt(2.0 / (dims[i] + dims[i + 1]))
        w["layer_%d" % i] = rng.normal(0, gl, (dims[i], dims[i + 1])).astype(np.float32)
        w["bias_%d" % i] = rng.normal(0, gl, (1, dims[i + 1])).astype(np.float32)
    return w


class _Sigmoid32(torch.autograd.Function):
    """tf.sigmoid in an fp32 graph: the output is an fp32 value (1.0 exactly once saturated) and SigmoidGrad is
    dy * y * (1 - y) on that output, so a saturated sample passes no gradient."""

    @staticmethod
    def forward(ctx, z):
        y = torch.sigmoid(z.float()).double()
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        return dy * y * (1 - y)


def _torch_graph(X, Y, w, l2_reg, n_layers, use_fm, use_deep, loss_type, B_total):
    """DFM.py:104-152 in float64 with autograd: returns loss, out and the gradient of every variable in the graph."""
    tw = {k: torch.tensor(np.asarray(v, np.float64), requires_grad=True) for k, v in w.items()}
    Xt = torch.as_tensor(X)
    E = tw["feature_embeddings"][Xt]
    parts = []
    if use_fm:
        parts.append(tw["feature_bias"].reshape(-1)[Xt])
        S = E.sum(1)
        parts.append(0.5 * (S * S - (E * E).sum(1)))
    if use_deep:
        h = E.reshape(E.shape[0], -1)
        for i in range(n_layers):
            h = torch.relu(h @ tw["layer_%d" % i] + tw["bias_%d" % i])
        parts.append(h)
    out = (torch.cat(parts, 1) @ tw["concat_projection"]).reshape(-1) + tw["concat_bias"]
    y = torch.tensor(np.asarray(Y, np.float64).reshape(-1))
    if loss_type == "logloss":
        out = _Sigmoid32.apply(out)
        eps = 1e-7
        loss = (-(y * torch.log(out + eps)) - (1 - y) * torch.log((1 - out) + eps)).sum() / B_total
    else:
        loss = 0.5 * ((y - out) ** 2).sum()
    if l2_reg > 0:
        loss = loss + l2_reg * 0.5 * (tw["concat_projection"] ** 2).sum()
        if use_deep:
            for i in range(n_layers):
                loss = loss + l2_reg * 0.5 * (tw["layer_%d" % i] ** 2).sum()
    loss.backward()
    return loss.item(), out.detach().numpy(), {k: (t.grad.numpy() if t.grad is not None else None) for k, t in tw.items()}


@pytest.mark.parametrize("use_fm,use_deep", MODES)
@pytest.mark.parametrize("loss_type,cbias", [("mse", 0.01), ("logloss", 0.01), ("logloss", 30.0), ("logloss", -30.0)])
@pytest.mark.parametrize("labels", ["01", "pm1"])
@pytest.mark.parametrize("l2_reg", [0.0, 0.01])
def test_oracle_matches_float64_autograd(use_fm, use_deep, loss_type, labels, l2_reg, cbias):
    """Every (use_fm, use_deep, loss_type) against the float64 graph.  cbias = +-30 pushes every logit far enough out that
    the fp32 sigmoid saturates (1.0f: log_loss then sees log(eps) and passes no gradient)."""
    rng = np.random.default_rng(hash((use_fm, use_deep, loss_type, labels, l2_reg, cbias)) % 2 ** 32)
    M, F, K, layers, B = 40, 4, 8, [12, 6], 64
    w = _weights(rng, M, F, K, layers, use_fm, use_deep)
    w["concat_bias"] = np.float32(cbias)
    X = rng.integers(0, M, (B, F))
    X[:, 3] = X[:, 2]                                       # one token in two columns shares its row
    Y = (rng.choice([1.0, 0.0], (B, 1)) if labels == "01" else rng.choice([1.0, -1.0], (B, 1))).astype(np.float32)
    B_total = B if labels == "01" else 3 * B                # the logloss mean over a larger (data-parallel) batch
    loss, out, g = D.dfm_loss_grads(X, Y, w, l2_reg, n_layers=len(layers), use_fm=use_fm, use_deep=use_deep,
                                    loss_type=loss_type, B_total=B_total)
    L, o, tg = _torch_graph(X, Y, w, l2_reg, len(layers), use_fm, use_deep, loss_type, B_total)
    assert_close(out, o, what="out")
    if loss_type == "logloss":              # terms of both signs under labels -1 can cancel: scale by the sum of |terms|
        y = Y.reshape(-1).astype(np.float64)
        per = -y * np.log(o + 1e-7) - (1 - y) * np.log((1 - o) + 1e-7)
        assert_close(loss, L, atol=1e-5 * np.abs(per).sum() / B_total, what="loss")
    else:
        assert_close(loss, L, what="loss")
    if loss_type == "logloss":
        assert ((out >= 0) & (out <= 1)).all()
        if cbias > 20:
            assert (out == 1.0).all()
        elif cbias < -20:
            assert (out < 1e-6).all()
    trained = {"feature_embeddings", "concat_projection", "concat_bias"}
    trained |= {"feature_bias"} if use_fm else set()
    trained |= {"%s_%d" % (k, i) for k in ("layer", "bias") for i in range(len(layers))} if use_deep else set()
    assert set(g) == trained
    for k in w:
        if k not in trained:
            assert tg[k] is None or not np.any(tg[k]), k
            continue
        ref = tg[k].reshape(-1)
        got = np.asarray(g[k], np.float64).reshape(-1)
        if not np.any(ref):
            assert not np.any(got), k
        else:
            assert_close(got, ref, rtol=2e-5, what="grad " + k)
    if loss_type == "logloss" and cbias > 20 and l2_reg == 0:
        assert all(not np.any(g[k]) for k in g), "a saturated sigmoid passes no gradient"


def test_defaults_reproduce_the_deepfm_oracle_bit_for_bit():
    rng = np.random.default_rng(7)
    M, F, K, layers = 60, 5, 8, [10, 7, 3]
    w = _weights(rng, M, F, K, layers, True, True)
    X = rng.integers(0, M, (200, F))
    Y = rng.choice([1.0, -1.0], (200, 1)).astype(np.float32)
    for lam in (0.0, 0.01):
        a = O.dfm_loss_grads(X, Y, w, lam, n_layers=3)
        b = D.dfm_loss_grads(X, Y, w, lam, n_layers=3)
        assert a[0] == b[0] and np.array_equal(a[1], b[1])
        assert sorted(a[2]) == sorted(b[2])
        for k in a[2]:
            assert np.array_equal(np.asarray(a[2][k]), np.asarray(b[2][k])), k
    assert np.array_equal(O.dfm_forward(X, w)[0], D.dfm_forward(X, w)[0])


# ----------------------------------------------------------------------------------------------------
# C ABI: mode checks and layouts (argument validation runs before any launch)
# ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from hhfm_b200 import build, _lib
    build.build()
    return _lib


def test_bad_modes_are_refused(lib):
    L = lib.load()
    sizes = np.asarray([150, 200, 150], np.int32)
    sp = sizes.ctypes.data
    for bad, msg in ((3, b"neither"), (8, b"unknown mode"), (-1, b"unknown mode"), (1 << 8, b"unknown mode")):
        assert L.hhfm_dfm_param_count_mode(10, 64, 3, sp, bad) == -1
        assert msg in L.hhfm_last_error(), (bad, L.hhfm_last_error())
        assert L.hhfm_dfm_reg_count_mode(10, 64, 3, sp, bad) == -1
        assert L.hhfm_workspace_bytes_dfm_mode(100, 10, 64, 3, sp, bad) == -1
        assert L.hhfm_workspace_bytes_dfm_topn_mode(4, 100, 10, 64, 3, sp, bad) == -1
        p16 = ctypes.c_void_p(16)
        with pytest.raises(lib.HhfmError, match=msg.decode()):
            lib.call("hhfm_dfm_fwd_mode", p16, 4, 10, p16, p16, 100, 64, p16, 3, sp, bad, p16, p16, None)
        with pytest.raises(lib.HhfmError, match=msg.decode()):
            lib.call("hhfm_dfm_fwd_bwd_mode", p16, 4, 10, p16, p16, 100, 64, p16, 3, sp, bad, 4, p16, p16, None, p16, p16, p16,
                     p16, None, None, None, 0, 0, None)
        with pytest.raises(lib.HhfmError, match=msg.decode()):
            lib.call("hhfm_dfm_topn_scores_mode", p16, 10, 4, 10, 1, p16, p16, 100, 64, p16, 3, sp, bad, 0, 50, p16, p16, None)
    p16 = ctypes.c_void_p(16)
    with pytest.raises(lib.HhfmError, match="B_total"):
        lib.call("hhfm_dfm_fwd_bwd_mode", p16, 4, 10, p16, p16, 100, 64, p16, 3, sp, 4, 3, p16, p16, None, p16, p16, p16,
                 p16, None, None, None, 0, 0, None)
    with pytest.raises(lib.HhfmError, match="NULL"):        # the FM part reads feature_bias
        lib.call("hhfm_dfm_fwd_bwd_mode", p16, 4, 10, p16, None, 100, 64, p16, 3, sp, 2, 4, p16, p16, None, p16, p16, p16,
                 p16, None, None, None, 0, 0, None)


def test_layout_per_mode(lib):
    """Mode 0 and NO_FM keep the DeepFM layout; NO_DEEP starts the projection on a multiple of 4 elements.  Workspaces:
    none without the tower; the FM-only top-N scorer holds no per-(row, item) activations."""
    L = lib.load()
    for F, K, layers in ((10, 64, [150, 200, 150]), (3, 4, [7]), (5, 8, [3, 5])):
        sizes = np.asarray(layers, np.int32)
        sp = sizes.ctypes.data
        n = len(layers)
        dims = [F * K] + layers
        n_w = sum(dims[i] * dims[i + 1] for i in range(n))
        n0, r0 = L.hhfm_dfm_param_count(F, K, n, sp), L.hhfm_dfm_reg_count(F, K, n, sp)
        for mode in (0, 1, 4, 5):
            assert L.hhfm_dfm_param_count_mode(F, K, n, sp, mode) == n0
            assert L.hhfm_dfm_reg_count_mode(F, K, n, sp, mode) == r0
            assert L.hhfm_workspace_bytes_dfm_mode(100, F, K, n, sp, mode) == L.hhfm_workspace_bytes_dfm(100, F, K, n, sp)
        proj = (n_w + 3) // 4 * 4
        reg = (proj + F + K + dims[-1] + 3) // 4 * 4
        for mode in (2, 6):
            assert L.hhfm_dfm_reg_count_mode(F, K, n, sp, mode) == reg
            assert L.hhfm_dfm_param_count_mode(F, K, n, sp, mode) == reg + sum(layers) + 1
            assert L.hhfm_workspace_bytes_dfm_mode(100, F, K, n, sp, mode) == 0
            C, N = 16, 1000
            assert L.hhfm_workspace_bytes_dfm_topn_mode(C, N, F, K, n, sp, mode) == 4 * (C * 2 * K + (C + 3) // 4 * 4)
        assert L.hhfm_workspace_bytes_dfm_topn_mode(16, 1000, F, K, n, sp, 0) == L.hhfm_workspace_bytes_dfm_topn(16, 1000, F, K, n, sp)
