"""GPU: DeepFM with the reference's options (use_fm, use_deep, loss_type) -- the mode entry points of K8 and the model
class -- against the fp32 oracle (oracle/dfm_modes.py)."""
import os
import socket

import numpy as np
import pytest
import torch

from conftest import assert_close, assert_update_close
from oracle import dfm_modes as D
from oracle import hhfm_oracle as O

pytestmark = pytest.mark.gpu

NO_FM, NO_DEEP, LOGLOSS = 1, 2, 4
MODES = [0, NO_FM, NO_DEEP, LOGLOSS, NO_FM | LOGLOSS, NO_DEEP | LOGLOSS]

_KEEP = []


@pytest.fixture(autouse=True)
def _release_device_tensors():
    yield
    torch.cuda.synchronize()
    _KEEP.clear()


def dev(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a))
    t = (t.to(dtype) if dtype is not None else t).cuda()
    _KEEP.append(t)
    return t


def opts(mode):
    return dict(use_fm=not (mode & NO_FM), use_deep=not (mode & NO_DEEP), loss_type="logloss" if mode & LOGLOSS else "mse")


def _lib_ptr():
    from hhfm_b200 import _lib
    from hhfm_b200.engine import cur_stream, ptr
    return _lib, ptr, cur_stream


def _weights(rng, M, F, K, layers, mode, proj_scale=1.0):
    o = opts(mode)
    dims = [F * K] + list(layers)
    n_in = (F + K if o["use_fm"] else 0) + (dims[-1] if o["use_deep"] else 0)
    w = dict(feature_embeddings=rng.normal(0, 0.1, (M, K)).astype(np.float32),
             feature_bias=rng.uniform(0, 1, (M, 1)).astype(np.float32),
             concat_projection=(proj_scale * rng.normal(0, np.sqrt(2.0 / (n_in + 1)), (n_in, 1))).astype(np.float32),
             concat_bias=np.float32(0.01))
    for i in range(len(layers)):
        gl = np.sqrt(2.0 / (dims[i] + dims[i + 1]))
        w["layer_%d" % i] = rng.normal(0, gl, (dims[i], dims[i + 1])).astype(np.float32)
        w["bias_%d" % i] = rng.normal(0, gl, (1, dims[i + 1])).astype(np.float32)
    return w


def _flat(w, F, K, layers, mode, lib):
    """The K8 parameter block of `mode`: slots name -> (offset, size); the projection slot is the slice the mode uses."""
    o = opts(mode)
    sizes = np.asarray(layers, np.int32)
    n = int(lib.load().hhfm_dfm_param_count_mode(F, K, len(layers), sizes.ctypes.data, mode))
    nr = int(lib.load().hhfm_dfm_reg_count_mode(F, K, len(layers), sizes.ctypes.data, mode))
    flat = np.zeros(n, np.float32)
    slots, off = {}, 0
    for i in range(len(layers)):
        a = w["layer_%d" % i].reshape(-1); flat[off:off + a.size] = a; slots["layer_%d" % i] = (off, a.size); off += a.size
    proj_off = off if o["use_deep"] else (off + 3) // 4 * 4
    assert proj_off % 4 == 0 or o["use_deep"]
    p0 = proj_off + (0 if o["use_fm"] else F + K)
    a = w["concat_projection"].reshape(-1); flat[p0:p0 + a.size] = a; slots["concat_projection"] = (p0, a.size)
    off = nr
    for i in range(len(layers)):
        a = w["bias_%d" % i].reshape(-1); flat[off:off + a.size] = a; slots["bias_%d" % i] = (off, a.size); off += a.size
    flat[off] = w["concat_bias"]; slots["concat_bias"] = (off, 1)
    assert off + 1 == n
    return flat, slots, sizes


def _trained(mode, n_layers):
    o = opts(mode)
    t = {"feature_embeddings", "concat_projection", "concat_bias"}
    if o["use_fm"]:
        t.add("feature_bias")
    if o["use_deep"]:
        t |= {"%s_%d" % (k, i) for k in ("layer", "bias") for i in range(n_layers)}
    return t


def _fwd_bwd(X, Y, w, F, K, layers, mode, M, hot_ids=None, B_total=None, parts=None):
    """One hhfm_dfm_fwd_bwd_mode pass (or one per row range of `parts`, accumulating) -> out, loss, gV, gbias, gparams."""
    lib, ptr, st = _lib_ptr()
    from hhfm_b200.engine import HotRows
    fm = opts(mode)["use_fm"]
    B = len(X)
    flat, slots, sizes = _flat(w, F, K, layers, mode, lib)
    L = len(layers)
    tV = dev(w["feature_embeddings"]); tb = dev(w["feature_bias"]); tp = dev(flat)
    gV = torch.zeros(M, K, device="cuda"); gb = torch.zeros(M, device="cuda"); gp = torch.zeros(flat.size, device="cuda")
    out = torch.empty(B, device="cuda")
    hot = HotRows(torch.as_tensor(hot_ids, dtype=torch.int32), M, K, torch.device("cuda"), fm) if hot_ids is not None else None
    loss = 0.0
    for r0, r1 in (parts or [(0, B)]):
        b = r1 - r0
        ws = dev(np.zeros(max(1, int(lib.load().hhfm_workspace_bytes_dfm_mode(b, F, K, L, sizes.ctypes.data, mode)) // 4), np.float32))
        lp = torch.zeros(lib.partials_len(), device="cuda"); lo = torch.zeros(1, device="cuda")
        if hot is None:
            hargs = (None, None, None, 0, 0)
        elif fm:
            hargs = hot.args(True)
        else:
            s_, g_, r_, n_ = hot.args()
            hargs = (s_, g_, None, r_, n_)
        tX = dev(X[r0:r1], torch.int32); tY = dev(Y.reshape(-1)[r0:r1])
        lib.call("hhfm_dfm_fwd_bwd_mode", ptr(tX), b, F, ptr(tV), ptr(tb) if fm else None, M, K, ptr(tp), L, sizes.ctypes.data, mode,
                 B if B_total is None else B_total, ptr(tY), ptr(ws), ptr(out[r0:r1]), ptr(gV), ptr(gb) if fm else None, ptr(gp),
                 ptr(lp), *hargs, st())
        lib.call("hhfm_loss_finalize", ptr(lp), None, 0.0, ptr(lo), st())
        loss += lo.item()
    if hot is not None:
        hot.fold(gV, gb if fm else None)
    return out.cpu().numpy(), loss, gV.cpu().numpy(), gb.cpu().numpy(), gp.cpu().numpy(), slots


def _check_grads(mode, layers, g, gV, gb, gp, slots, what):
    o = opts(mode)
    assert_close(gV, g["feature_embeddings"], rtol=2e-5, what=what + " gV")
    if o["use_fm"]:
        assert_close(gb, g["feature_bias"].reshape(-1), rtol=2e-5, what=what + " gbias")
    else:
        assert not gb.any(), what + ": feature_bias is outside the graph"
    used = np.zeros(gp.size, bool)
    for k, (off, n) in slots.items():
        if k in g:
            assert_close(gp[off:off + n], np.asarray(g[k], np.float32).reshape(-1), rtol=2e-5, what=what + " g " + k)
            used[off:off + n] = True
    assert not gp[~used].any(), what + ": gradient outside the mode's variables"


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("K", [64, 256, 512])          # kv = K/4 selects the head instance VPL = 1 / 2 / 4
@pytest.mark.parametrize("tc", ["1", "0"])
def test_mode_pass_matches_oracle(cuda, monkeypatch, mode, K, tc):
    """hhfm_dfm_fwd_mode / hhfm_dfm_fwd_bwd_mode against the oracle on both GEMM paths, with and without hot rows."""
    monkeypatch.setenv("HHFM_DFM_TC", tc)
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(mode * 100 + K + int(tc))
    M, F, B, layers = 300, 4, 333, (40, 24)
    w = _weights(rng, M, F, K, layers, mode)
    X = rng.integers(0, M, (B, F)); X[:, 1] = rng.integers(0, 4, B); X[:, 3] = X[:, 2]
    Y = rng.choice([1.0, -1.0], (B, 1)).astype(np.float32)
    loss, out, g = D.dfm_loss_grads(X, Y, w, 0.0, n_layers=len(layers), **opts(mode))
    flat, _, sizes = _flat(w, F, K, layers, mode, lib)
    ws = dev(np.zeros(max(1, int(lib.load().hhfm_workspace_bytes_dfm_mode(B, F, K, 2, sizes.ctypes.data, mode)) // 4), np.float32))
    o = torch.empty(B, device=cuda)
    fb = dev(w["feature_bias"]) if opts(mode)["use_fm"] else None
    lib.call("hhfm_dfm_fwd_mode", ptr(dev(X, torch.int32)), B, F, ptr(dev(w["feature_embeddings"])), ptr(fb) if fb is not None else None,
             M, K, ptr(dev(flat)), 2, sizes.ctypes.data, mode, ptr(ws), ptr(o), st())
    assert_close(o.cpu().numpy(), out, what="fwd out")
    for hot_ids in (None, [0, 1, 2, 3]):
        o2, lo, gV, gb, gp, slots = _fwd_bwd(X, Y, w, F, K, layers, mode, M, hot_ids)
        what = "mode %d K %d tc %s hot %s" % (mode, K, tc, hot_ids is not None)
        assert_close(o2, out, what=what + " out")
        assert_close(lo, loss, what=what + " loss")
        _check_grads(mode, layers, g, gV, gb, gp, slots, what)


@pytest.mark.parametrize("mode", [LOGLOSS, NO_FM | LOGLOSS, NO_DEEP | LOGLOSS])
def test_split_batch_with_b_total_accumulates_the_full_batch(cuda, mode):
    """Two half-batch passes with B_total = B give the full batch's mean loss and gradients: the data-parallel normaliser."""
    rng = np.random.default_rng(40 + mode)
    M, F, K, B, layers = 300, 5, 64, 1000, (64, 32)
    w = _weights(rng, M, F, K, layers, mode)
    X = rng.integers(0, M, (B, F))
    Y = rng.choice([1.0, -1.0], (B, 1)).astype(np.float32)
    loss, out, g = D.dfm_loss_grads(X, Y, w, 0.0, n_layers=2, **opts(mode))
    o, lo, gV, gb, gp, slots = _fwd_bwd(X, Y, w, F, K, layers, mode, M, parts=[(0, 437), (437, B)])
    assert_close(o, out, what="split out")
    assert_close(lo, loss, what="split loss")
    _check_grads(mode, layers, g, gV, gb, gp, slots, "split")
    # and a half batch alone with B_total = B is half of the normaliser's batch, not its own
    _, lo_half, _, _, _, _ = _fwd_bwd(X[:500], Y[:500], w, F, K, layers, mode, M, B_total=B)
    ref_half, _, _ = D.dfm_loss_grads(X[:500], Y[:500], w, 0.0, n_layers=2, B_total=B, **opts(mode))
    assert_close(lo_half, ref_half, what="half loss over B_total")


def frappe_like(rng, B, n_user=60, n_item=200, ctx=(7, 2, 3, 9)):
    cols = [rng.integers(0, n_user, B), n_user + rng.integers(0, n_item, B)]
    base = n_user + n_item
    for c in ctx:
        cols.append(base + rng.integers(0, c, B))
        base += c
    return np.stack(cols, axis=1), base


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("lam", [0.0, 0.01])
def test_model_steps_match_oracle(cuda, mode, lam):
    """DeepFM.partial_fit teacher-forced against the oracle + TF1 Adagrad for four steps (the last one ragged): the trained
    variables follow the oracle; the variables outside the mode's graph and their optimizer state do not move at all."""
    from hhfm_b200.models import DeepFM
    rng = np.random.default_rng(11 + mode + int(lam * 1000))
    n_user, n_item = 60, 200
    X0, M = frappe_like(rng, 10)
    K, lr = 64, 0.01
    F = X0.shape[1]
    layers = [64, 48, 32]
    model = DeepFM(n_user, n_item, M, F, K, layers, 'relu', lr, 0, lam, **opts(mode))
    trained = _trained(mode, len(layers))
    w_init = model.get_weights()
    assert set(w_init) == set(model.weights)
    n_in = (F + K if opts(mode)["use_fm"] else 0) + (layers[-1] if opts(mode)["use_deep"] else 0)
    assert w_init["concat_projection"].shape == (n_in, 1)
    deep = opts(mode)["use_deep"]
    r0 = 0 if deep else model._proj_off
    b0 = model._n_reg if deep else model._cbias_off
    base = model._params.data_ptr()

    def acc_of(k, wk, state):
        if k in ("feature_embeddings", "feature_bias"):
            return state[k].copy() if k in state else np.full(wk.shape, 0.1, np.float32)
        off = (model.weights[k].data_ptr() - base) // 4
        name, start = ("dense_reg", r0) if off < model._n_reg else ("dense_bias", b0)
        if name not in state:
            return np.full(wk.shape, 0.1, np.float32)
        return state[name][off - start:off - start + wk.size].reshape(wk.shape)

    for step in range(4):
        w = model.get_weights()
        state = {k: v[0].cpu().numpy().copy() for k, v in model._opt.state.items()}
        X, _ = frappe_like(rng, 3000 if step < 3 else 517)
        Y = rng.choice([1.0, -1.0], (len(X), 1)).astype(np.float32)
        loss_ref, _, g = D.dfm_loss_grads(X, Y, w, lam, n_layers=len(layers), **opts(mode))
        loss = model.partial_fit({"X": X, "Y": Y})
        assert_close(loss, loss_ref, what="loss step %d" % step)
        got = model.get_weights()
        for k in model.weights:
            wk = np.asarray(w[k], np.float32)
            if k not in trained:
                assert np.array_equal(got[k], w_init[k]), "%s moved (mode %d)" % (k, mode)
                continue
            gk = np.asarray(g[k], np.float32).reshape(wk.shape)
            acc = acc_of(k, wk, state)
            w1, _ = O.adagrad_dense(wk, acc, gk, lr)
            assert_update_close(np.asarray(got[k]).reshape(wk.shape), w1, wk, gk, acc, lr, rtol=3e-5,
                                atol=4 * 1.2e-7 * float(np.abs(wk).max()), what="%s step %d" % (k, step))
    # optimizer state only for what the mode trains
    st = model._opt.state
    assert ("feature_bias" in st) == opts(mode)["use_fm"]
    assert st["dense_reg"][0].numel() == model._n_reg - r0
    assert st["dense_bias"][0].numel() == model._params.numel() - b0
    # the projection entries the mode does not use stay zero in the block
    p = model._params.cpu().numpy()
    used = np.zeros(p.size, bool)
    for k in model.weights:
        if k in ("feature_embeddings", "feature_bias"):
            continue
        off = (model.weights[k].data_ptr() - base) // 4
        used[off:off + model.weights[k].numel()] = True
    assert not p[~used].any()
    # sess.run(model.out) / predict: the sigmoid under logloss
    w = model.get_weights()
    out = model.sess.run(model.out, feed_dict={model.feat_index: X[:300], model.label: [[1]] * 300})
    ref = D.dfm_forward(X[:300], w, len(layers), **opts(mode))[0]
    assert_close(out[:, 0], ref, rtol=2e-5, what="predict")
    if mode & LOGLOSS:
        assert ((out >= 0) & (out <= 1)).all()
        logit = D.dfm_forward(X[:300], w, len(layers), use_fm=opts(mode)["use_fm"], use_deep=deep)[0]
        assert_close(out[:, 0], 1.0 / (1.0 + np.exp(-logit.astype(np.float64))), what="predict is the sigmoid")


def _check_lists(ids, want, ref, what):
    for r in range(len(want)):
        if (ids[r] == want[r]).all():
            continue
        kth = ref[r, want[r, -1]]
        tol = 2e-5 * max(abs(kth), float(np.sqrt(np.mean(ref[r] ** 2))))
        for a_, b_ in zip(ids[r], want[r]):
            assert abs(ref[r, a_] - ref[r, b_]) <= tol, (what, r, a_, b_, ref[r, a_], ref[r, b_])


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("saturate", [False, True])
def test_topk_matches_oracle(cuda, monkeypatch, mode, saturate):
    """DeepFM.topk on both evaluator paths and both GEMM paths against the oracle's lists.  saturate: projection weights
    x3 and concat_bias 60 push the logits past the point where the fp32 sigmoid is exactly 1.0: under logloss the items
    tie and the lowest index wins.  Where no item up to the last listed one has a logit near that point (10..30), the list
    must be exactly the oracle's."""
    from hhfm_b200.models import DeepFM
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(70 + mode)
    n_user, n_item = 60, 500
    X, M = frappe_like(rng, 40, n_item=n_item)
    K, F, layers = 64, X.shape[1], [64, 32]
    model = DeepFM(n_user, n_item, M, F, K, layers, 'relu', 0.01, 0, 0.0, **opts(mode))
    w = _weights(rng, M, F, K, layers, mode, 3.0 if saturate else 1.0)
    if saturate:
        w["concat_bias"] = np.float32(60.0)
    model.load_weights(w)
    w = model.get_weights()
    A = X[:40]
    rows = np.repeat(A[:, None, :], n_item, axis=1); rows[:, :, 1] = n_user + np.arange(n_item)[None, :]
    ref = D.dfm_forward(rows.reshape(-1, F), w, len(layers), **opts(mode))[0].reshape(len(A), n_item)
    want = O.topk_lowest_index(ref, 20)
    if saturate and mode & LOGLOSS:
        logit = D.dfm_forward(rows.reshape(-1, F), w, len(layers), use_fm=opts(mode)["use_fm"],
                              use_deep=opts(mode)["use_deep"])[0].reshape(len(A), n_item)
        amb = (logit > 10) & (logit < 30)
        sure = np.array([(ref[r] == 1.0).sum() >= 20 and not amb[r, :want[r, -1] + 1].any() for r in range(len(A))])
        assert sure.sum() >= 10, "the saturated case should saturate"
        assert not all((want[r] == np.argsort(-logit[r], kind="stable")[:20]).all() for r in np.nonzero(sure)[0])
    for tc in ("1", "0"):
        monkeypatch.setenv("HHFM_DFM_TC", tc)
        for sep in ("1", "0"):
            monkeypatch.setenv("HHFM_DFM_TOPN_SEPARABLE", sep)
            ids = model.topk(A, 20)
            _check_lists(ids, want, ref, "mode %d tc %s sep %s" % (mode, tc, sep))
            if saturate and mode & LOGLOSS:
                assert (ids[sure] == want[sure]).all(), "saturated items: lowest index first"
        # the separable scorer's scores themselves
        A_dev, stride = model._topn.upload_rows(A, model._M)
        need = int(lib.load().hhfm_workspace_bytes_dfm_topn_mode(len(A), n_item, F, K, 2, model._sizes.ctypes.data, mode)) // 4
        ws = torch.empty(max(need, 1), device=cuda); sc = torch.full((len(A), n_item), float("nan"), device=cuda)
        lib.call("hhfm_dfm_topn_scores_mode", ptr(A_dev), stride, len(A), F, 1, ptr(model.weights["feature_embeddings"]),
                 model._fbias_arg(), model._M, K, ptr(model._params), 2, model._sizes.ctypes.data, mode, n_user, n_item, ptr(ws),
                 ptr(sc), cur_stream_())
        assert_close(sc.cpu().numpy(), ref, rtol=2e-5, what="separable scores mode %d tc %s" % (mode, tc))


def cur_stream_():
    from hhfm_b200.engine import cur_stream
    return cur_stream()


def test_mode_zero_is_the_existing_path(cuda):
    """hhfm_dfm_fwd_mode / hhfm_dfm_topn_scores_mode with mode 0 give bit-identical scores to hhfm_dfm_fwd /
    hhfm_dfm_topn_scores on both GEMM paths."""
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(3)
    M, F, K, B, layers = 400, 10, 64, 2000, (150, 200, 150)
    w = _weights(rng, M, F, K, layers, 0)
    flat, _, sizes = _flat(w, F, K, layers, 0, lib)
    X = rng.integers(0, M, (B, F))
    tX, tV, tb, tp = dev(X, torch.int32), dev(w["feature_embeddings"]), dev(w["feature_bias"]), dev(flat)
    for tc in ("1", "0"):
        os.environ["HHFM_DFM_TC"] = tc
        try:
            ws = torch.zeros(int(lib.load().hhfm_workspace_bytes_dfm(B, F, K, 3, sizes.ctypes.data)) // 4, device=cuda)
            a = torch.empty(B, device=cuda); b = torch.empty(B, device=cuda)
            lib.call("hhfm_dfm_fwd", ptr(tX), B, F, ptr(tV), ptr(tb), M, K, ptr(tp), 3, sizes.ctypes.data, ptr(ws), ptr(a), st())
            lib.call("hhfm_dfm_fwd_mode", ptr(tX), B, F, ptr(tV), ptr(tb), M, K, ptr(tp), 3, sizes.ctypes.data, 0, ptr(ws), ptr(b), st())
            assert torch.equal(a, b), tc
            C, N = 16, 300
            rows = dev(X[:C], torch.int32)
            need = int(lib.load().hhfm_workspace_bytes_dfm_topn(C, N, F, K, 3, sizes.ctypes.data)) // 4
            ws2 = torch.zeros(need, device=cuda)
            s1 = torch.empty(C, N, device=cuda); s2 = torch.empty(C, N, device=cuda)
            lib.call("hhfm_dfm_topn_scores", ptr(rows), F, C, F, 1, ptr(tV), ptr(tb), M, K, ptr(tp), 3, sizes.ctypes.data, 50, N,
                     ptr(ws2), ptr(s1), st())
            lib.call("hhfm_dfm_topn_scores_mode", ptr(rows), F, C, F, 1, ptr(tV), ptr(tb), M, K, ptr(tp), 3, sizes.ctypes.data, 0, 50,
                     N, ptr(ws2), ptr(s2), st())
            assert torch.equal(s1, s2), tc
        finally:
            del os.environ["HHFM_DFM_TC"]


# ----------------------------------------------------------------------------------------------------
# two ranks: the logloss mean over the global batch
# ----------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _dp_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from hhfm_b200 import dist as hd
        from hhfm_b200.models import DeepFM
        rng = np.random.default_rng(9)
        X, M = frappe_like(rng, 3001)
        Y = rng.choice([1.0, -1.0], (len(X), 1)).astype(np.float32)
        F = X.shape[1]
        args = (60, 200, M, F, 64, [64, 32], 'relu', 0.01, 0, 0.01)
        single = DeepFM(*args, loss_type="logloss")
        loss_1 = single.partial_fit({"X": X, "Y": Y})
        model = DeepFM(*args, loss_type="logloss")
        model.enable_data_parallel()
        lo, hi = hd.shard_range(len(X), rank, world)
        loss_dp = model.partial_fit({"X": X[lo:hi], "Y": Y[lo:hi]})
        ok = abs(loss_dp - loss_1) <= 2e-5 * abs(loss_1)
        a, b = single.get_weights(), model.get_weights()
        for k in a:
            d = np.abs(a[k] - b[k])
            ok = ok and bool(np.all(d <= 1e-5 * np.maximum(np.abs(a[k]), np.sqrt(np.mean(a[k] ** 2))) + 1e-9))
        ret[rank] = ok
    finally:
        dist.destroy_process_group()


def test_two_rank_logloss_step_matches_one_gpu(cuda):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mgr = mp.Manager(); ret = mgr.dict()
    mp.spawn(_dp_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    assert ret[0] and ret[1], dict(ret)
