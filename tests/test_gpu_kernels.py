"""GPU parity tests: every C-ABI kernel against the CPU oracle on the same seeded inputs.

Bar (BASELINE.json north_star): scores / losses / gradients within 1e-5 relative in fp32 (assert_close: element
tolerance 1e-5 * max(|ref|, rms(ref))); top-K index lists, exact scores and HR/NDCG codes bit-exact.
"""
import numpy as np
import pytest
import torch

from conftest import assert_close
from oracle import hhfm_oracle as O

pytestmark = pytest.mark.gpu


_KEEP = []


def dev(a, cuda, dtype=None):
    """Host array -> device tensor.  The tensor is kept alive until the end of the test: the C ABI takes raw
    pointers, so a temporary freed right after `ptr(...)` could be recycled by the caching allocator."""
    t = torch.as_tensor(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    t = t.to(cuda)
    _KEEP.append(t)
    return t


@pytest.fixture(autouse=True)
def _release_device_tensors():
    yield
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    _KEEP.clear()


def _lib_ptr():
    from hhfm_b200 import _lib
    from hhfm_b200.engine import cur_stream, ptr
    return _lib, ptr, cur_stream


def make_table(rng, M, K, scale=0.1):
    return rng.normal(0, scale, (M, K)).astype(np.float32)


# ----------------------------------------------------------------------------------------------------
# K1 FM
# ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,F,K", [(64, 10, 64), (5000, 10, 64), (333, 6, 128), (257, 13, 8), (100, 3, 16),
                                   (65, 10, 32), (40, 5, 256), (31, 7, 100), (1, 1, 4), (70, 10, 512)])
def test_fm_forward_matches_oracle(cuda, B, F, K):
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(B * 1000 + K)
    M = 500
    V = make_table(rng, M, K); b = rng.normal(0, 0.1, (M, 1)).astype(np.float32); b0 = np.float32(0.25)
    X = rng.integers(0, M, (B, F))
    if F > 3:
        X[:, 3] = X[:, 2]                                   # the same token in two columns shares one row
    ref, _, _ = O.fm_forward(X, V, b, b0)
    out = torch.empty(B, device=cuda)
    tV, tb, tb0, tX = dev(V, cuda), dev(b, cuda), dev(np.array([b0]), cuda), dev(X, cuda, torch.int32)
    lib.call("hhfm_fm_fwd", None, ptr(tX), None, B, F, ptr(tV), ptr(tb), ptr(tb0), M, K, 0, ptr(out), st())
    assert_close(out.cpu().numpy(), ref, what="fm out")


def test_fm_forward_csr_ragged_with_values(cuda):
    """General CSR (variable row length incl. empty rows, explicit feature values)."""
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(7)
    M, K, B = 300, 64, 200
    V = make_table(rng, M, K); b = rng.normal(0, 0.1, (M, 1)).astype(np.float32)
    lens = rng.integers(0, 12, B); lens[0] = 0; lens[-1] = 0
    row_ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    col = rng.integers(0, M, row_ptr[-1]).astype(np.int32)
    val = rng.uniform(0.5, 2.0, row_ptr[-1]).astype(np.float32)
    ref = np.zeros(B, np.float32)
    for s in range(B):
        if lens[s] == 0:
            ref[s] = 0.0
            continue
        sl = slice(row_ptr[s], row_ptr[s + 1])
        ref[s] = O.fm_forward(col[sl][None, :], V, b, 0.0, val[sl][None, :])[0][0]
    out = torch.empty(B, device=cuda)
    lib.call("hhfm_fm_fwd", ptr(dev(row_ptr, cuda)), ptr(dev(col, cuda)), ptr(dev(val, cuda)), B, 0, ptr(dev(V, cuda)),
             ptr(dev(b, cuda)), None, M, K, 0, ptr(out), st())
    assert_close(out.cpu().numpy(), ref, what="fm csr out")


def _fm_train_call(cuda, X, Y, V, b, b0, interaction=0, deterministic=0, track=True, val=None, hot_rows=None):
    lib, ptr, st = _lib_ptr()
    from hhfm_b200.engine import NO_HOT_BIAS, HotRows
    B, F = X.shape
    M, K = V.shape
    hot = HotRows(hot_rows, M, K, cuda, with_bias=True, n_rep=4) if hot_rows is not None else None
    P = lib.partials_len()
    tV = dev(V, cuda); tb = dev(b, cuda) if b is not None else None
    tb0 = dev(np.array([b0], np.float32), cuda) if b0 is not None else None
    gV = torch.zeros(M, K, device=cuda); gb = torch.zeros(M, device=cuda); gb0 = torch.zeros(1, device=cuda)
    lp = torch.full((P,), 123.0, device=cuda); out = torch.empty(B, device=cuda); loss = torch.zeros(1, device=cuda)
    stamp = torch.zeros(M, dtype=torch.int32, device=cuda); rows = torch.full((M,), -1, dtype=torch.int32, device=cuda)
    cnt = torch.zeros(1, dtype=torch.int32, device=cuda)
    tval = dev(val, cuda) if val is not None else None
    lib.call("hhfm_fm_fwd_bwd_sqloss", None, ptr(dev(X, cuda, torch.int32)), ptr(tval), B, F, ptr(tV), ptr(tb), ptr(tb0), M, K,
             interaction, ptr(dev(Y.reshape(-1), cuda)), ptr(out), ptr(gV), ptr(gb) if b is not None else None,
             ptr(gb0) if b0 is not None else None, ptr(lp), ptr(stamp) if track else None, 1, ptr(rows) if track else None,
             ptr(cnt) if track else None, *(hot.args(True) if hot is not None else NO_HOT_BIAS), deterministic, st())
    if hot is not None:
        hot.fold(gV, gb if b is not None else None)
    lib.call("hhfm_loss_finalize", ptr(lp), None, 0.0, ptr(loss), st())
    n = int(cnt.item())
    return dict(loss=float(loss.item()), out=out.cpu().numpy(), gV=gV.cpu().numpy(), gb=gb.cpu().numpy(),
                gb0=float(gb0.item()), touched=np.sort(rows.cpu().numpy()[:n]))


@pytest.mark.parametrize("B,F,K", [(64, 10, 64), (5000, 10, 64), (999, 6, 128), (130, 12, 16), (77, 10, 256)])
def test_fm_fused_train_pass_matches_oracle(cuda, B, F, K):
    rng = np.random.default_rng(B + K)
    M = 400
    V = make_table(rng, M, K); b = rng.normal(0, 0.1, (M, 1)).astype(np.float32); b0 = np.float32(-0.1)
    X = rng.integers(0, M, (B, F)); X[:, 1] = rng.integers(0, 3, B)      # heavy duplicates across rows
    if F > 4:
        X[:, 4] = X[:, 0]                                                # duplicate inside a row
    Y = rng.choice([1.0, 0.0], (B, 1)).astype(np.float32)
    loss, out, dV, db, db0, touched = O.fm_loss_grads(X, Y, V, b, b0, lamda=0.0)
    got = _fm_train_call(cuda, X, Y, V, b, b0)
    assert_close(got["out"], out, what="out")
    assert_close(got["loss"], loss, what="loss")
    assert_close(got["gV"], dV, what="gV")
    assert_close(got["gb"], db, what="gbias")
    assert_close(got["gb0"], db0, what="gb0")
    assert (got["touched"] == touched).all()


def test_fm_train_pass_with_feature_values(cuda):
    rng = np.random.default_rng(3)
    M, K, B, F = 200, 32, 300, 7
    V = make_table(rng, M, K); b = rng.normal(0, 0.1, (M, 1)).astype(np.float32)
    X = rng.integers(0, M, (B, F)); Y = rng.normal(0, 1, (B, 1)).astype(np.float32)
    val = rng.uniform(0.5, 1.5, (B, F)).astype(np.float32)
    loss, out, dV, db, db0, _ = O.fm_loss_grads(X, Y, V, b, 0.0, 0.0, val=val)
    got = _fm_train_call(cuda, X, Y, V, b, 0.0, val=val)
    assert_close(got["loss"], loss, what="loss"); assert_close(got["gV"], dV, what="gV"); assert_close(got["gb"], db, what="gb")


def test_fm_deterministic_mode_is_bit_reproducible(cuda):
    rng = np.random.default_rng(11)
    M, K, B, F = 50, 64, 2000, 10
    V = make_table(rng, M, K); b = np.zeros((M, 1), np.float32)
    X = rng.integers(0, M, (B, F)); Y = rng.choice([1.0, -1.0], (B, 1)).astype(np.float32)
    a = _fm_train_call(cuda, X, Y, V, b, 0.0, deterministic=1)
    c = _fm_train_call(cuda, X, Y, V, b, 0.0, deterministic=1)
    assert (a["gV"].view(np.int32) == c["gV"].view(np.int32)).all() and a["loss"] == c["loss"]
    ref = O.fm_loss_grads(X, Y, V, b, 0.0, 0.0)
    assert_close(a["gV"], ref[2], what="det gV")


def test_mf_interaction_matches_oracle(cuda):
    rng = np.random.default_rng(5)
    M, K, B = 300, 64, 1000
    V = make_table(rng, M, K)
    X = rng.integers(0, M, (B, 2)); Y = rng.choice([1.0, -1.0], (B, 1)).astype(np.float32)
    loss, out, dV = O.mf_loss_grads(X, Y, V, 0.0)
    got = _fm_train_call(cuda, X, Y, V, None, None, interaction=1)
    assert_close(got["out"], out, what="mf out"); assert_close(got["loss"], loss, what="mf loss")
    assert_close(got["gV"], dV, what="mf gV")


def test_fm_backward_entry_point(cuda):
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(9)
    M, K, B, F = 120, 64, 500, 10
    V = make_table(rng, M, K); X = rng.integers(0, M, (B, F)); gout = rng.normal(0, 1, B).astype(np.float32)
    E = V[X]; S = E.sum(1)
    dV = np.zeros_like(V); np.add.at(dV, X.reshape(-1), (gout[:, None, None] * (S[:, None, :] - E)).reshape(-1, K))
    db = np.zeros(M, np.float32); np.add.at(db, X.reshape(-1), np.repeat(gout, F))
    gV = torch.zeros(M, K, device=cuda); gb = torch.zeros(M, device=cuda); gb0 = torch.zeros(1, device=cuda)
    lib.call("hhfm_fm_bwd", None, ptr(dev(X, cuda, torch.int32)), None, B, F, ptr(dev(V, cuda)), M, K, 0, ptr(dev(gout, cuda)),
             ptr(gV), ptr(gb), ptr(gb0), 0, st())
    assert_close(gV.cpu().numpy(), dV, what="bwd gV"); assert_close(gb.cpu().numpy(), db, what="bwd gb")
    assert_close(gb0.item(), gout.sum(), what="bwd gb0")


# ----------------------------------------------------------------------------------------------------
# K3 HHFM / BPR
# ----------------------------------------------------------------------------------------------------
def _records(Pos, Fea, Tim, Neg):
    parts = [Pos] + [p for p in (Fea, Tim, Neg) if p is not None and p.shape[1] > 0]
    w = sum(p.shape[1] for p in parts)
    stride = (w + 3) // 4 * 4
    rec = np.full((Pos.shape[0], stride), -1, np.int32)
    rec[:, :w] = np.concatenate(parts, axis=1)
    return rec, stride


def _pairrank_train(cuda, V, Pos, Fea, Tim, Neg, pools, deterministic=0, hot_rows=None):
    lib, ptr, st = _lib_ptr()
    from hhfm_b200.engine import NO_HOT, HotRows
    M, K = V.shape
    hot = HotRows(hot_rows, M, K, cuda, n_rep=8) if hot_rows is not None else None
    hot_args = hot.args() if hot is not None else NO_HOT
    rec, stride = _records(Pos, Fea, Tim, Neg)
    B = rec.shape[0]
    nc = 0 if Fea is None else Fea.shape[1]; nt = 0 if Tim is None else Tim.shape[1]; ng = Neg.shape[1]
    P = lib.partials_len()
    gV = torch.zeros(M, K, device=cuda); lp = torch.full((P,), -5.0, device=cuda); loss = torch.zeros(1, device=cuda)
    pos = torch.empty(B, device=cuda); neg = torch.empty(B, ng, device=cuda)
    stamp = torch.zeros(M, dtype=torch.int32, device=cuda); rows = torch.zeros(M, dtype=torch.int32, device=cuda)
    cnt = torch.zeros(1, dtype=torch.int32, device=cuda)
    lib.call("hhfm_pairrank_fwd_bwd", ptr(dev(rec, cuda)), B, stride, nc, nt, ng, pools[0], pools[1], pools[2],
             ptr(dev(V, cuda)), M, K, ptr(pos), ptr(neg), ptr(gV), ptr(lp), ptr(stamp), 3, ptr(rows), ptr(cnt),
             *hot_args, deterministic, st())
    if hot is not None:
        hot.fold(gV, None)
    lib.call("hhfm_loss_finalize", ptr(lp), None, 0.0, ptr(loss), st())
    return dict(loss=float(loss.item()), pos=pos.cpu().numpy(), neg=neg.cpu().numpy(), gV=gV.cpu().numpy(),
                touched=np.sort(rows.cpu().numpy()[:int(cnt.item())]))


@pytest.mark.parametrize("pools", [(0, 0, 0), (1, 1, 1), (2, 2, 2), (1, 0, 2), (0, 2, 1)])
@pytest.mark.parametrize("B,K,fc,ft", [(64, 64, 8, 0), (5000, 64, 8, 0), (700, 128, 5, 5), (300, 16, 3, 3), (200, 32, 0, 3)])
def test_hhfm_fused_pass_matches_oracle(cuda, pools, B, K, fc, ft):
    rng = np.random.default_rng(B + K + fc)
    M, NG = 600, 10
    V = make_table(rng, M, K)
    Pos = rng.integers(0, M, (B, 2))
    Fea = rng.integers(0, M, (B, fc)) if fc else None
    Tim = rng.integers(0, M, (B, ft)) if ft else None
    if fc > 1:
        Fea[:, 1] = Fea[:, 0]                       # same token twice in the group -> exact max-pool ties
    if ft > 2:
        Tim[:, 2] = Tim[:, 0]
    Neg = rng.integers(0, M, (B, NG)); Neg[:, 3] = Neg[:, 2]; Neg[::7] = Neg[::7, :1]   # duplicate / all-same negatives
    loss, pos, neg, dV = O.pairrank_loss_grads(V, Pos, Neg, Fea, Tim, pools, 0.0)
    got = _pairrank_train(cuda, V, Pos, Fea, Tim, Neg, pools)
    assert_close(got["pos"], pos, what="pos"); assert_close(got["neg"], neg, what="neg")
    assert_close(got["loss"], loss, what="loss")
    assert_close(got["gV"], dV, what="gV")
    assert set(got["touched"].tolist()) <= set(np.unique(np.concatenate([a.reshape(-1) for a in (Pos, Fea, Tim, Neg) if a is not None])).tolist())
    assert set(np.unique(Pos).tolist()) <= set(got["touched"].tolist())


def test_hot_row_replicas_fold_to_the_same_gradient(cuda):
    """Two-level scatter: rows flagged hot accumulate in replicated buffers; after hhfm_hot_fold the gradient equals
    the single-level result (and the oracle)."""
    rng = np.random.default_rng(77)
    M, K, B = 300, 64, 4000
    V = make_table(rng, M, K)
    Pos = np.stack([rng.integers(0, 5, B), rng.integers(100, 200, B)], axis=1)       # 5 very hot users
    Fea = np.stack([250 + rng.integers(0, 2, B), 260 + rng.integers(0, 3, B), 270 + rng.integers(0, 7, B)], axis=1)
    Neg = rng.integers(100, 200, (B, 10))
    hot_rows = np.concatenate([np.arange(5), 250 + np.arange(2), 260 + np.arange(3), 270 + np.arange(7), [150]])
    loss, pos, neg, dV = O.pairrank_loss_grads(V, Pos, Neg, Fea, None, (0, 0, 0), 0.0)
    got = _pairrank_train(cuda, V, Pos, Fea, None, Neg, (0, 0, 0), hot_rows=hot_rows)
    assert_close(got["loss"], loss, what="loss"); assert_close(got["gV"], dV, what="gV with hot replicas")


def test_fm_hot_row_replicas_with_bias(cuda):
    lib, ptr, st = _lib_ptr()
    from hhfm_b200.engine import HotRows
    rng = np.random.default_rng(78)
    M, K, B, F = 200, 32, 3000, 6
    V = make_table(rng, M, K); b = rng.normal(0, 0.1, (M, 1)).astype(np.float32)
    X = np.stack([rng.integers(0, 100, B), rng.integers(100, 180, B), 190 + rng.integers(0, 2, B), 192 + rng.integers(0, 3, B),
                  195 + rng.integers(0, 5, B), rng.integers(0, 3, B)], axis=1)
    Y = rng.choice([1.0, 0.0], (B, 1)).astype(np.float32)
    loss, out, dV, db, db0, _ = O.fm_loss_grads(X, Y, V, b, 0.0, 0.0)
    hot = HotRows(np.concatenate([np.arange(3), np.arange(190, 200)]), M, K, cuda, with_bias=True, n_rep=4)
    P = lib.partials_len()
    gV = torch.zeros(M, K, device=cuda); gb = torch.zeros(M, device=cuda); gb0 = torch.zeros(1, device=cuda)
    lp = torch.zeros(P, device=cuda)
    lib.call("hhfm_fm_fwd_bwd_sqloss", None, ptr(dev(X, cuda, torch.int32)), None, B, F, ptr(dev(V, cuda)), ptr(dev(b, cuda)), None,
             M, K, 0, ptr(dev(Y.reshape(-1), cuda)), None, ptr(gV), ptr(gb), ptr(gb0), ptr(lp), None, 0, None, None,
             *hot.args(True), 0, st())
    hot.fold(gV, gb)
    assert_close(gV.cpu().numpy(), dV, what="fm gV hot"); assert_close(gb.cpu().numpy(), db, what="fm gb hot")
    assert float(hot.ghot.abs().max()) == 0.0 and float(hot.ghot_bias.abs().max()) == 0.0, "fold must clear the replicas"


@pytest.mark.parametrize("K,fc,ft", [(64, 8, 0), (128, 5, 5), (32, 0, 0), (64, 3, 0), (128, 5, 3), (64, 0, 0)])
@pytest.mark.parametrize("use_hot", [False, True])
def test_specialised_sum_pooling_kernel_matches_oracle_and_generic(cuda, K, fc, ft, use_hot):
    """The unrolled fast path (all pools = sum, NG = 10, K in {32,64,128}) against the oracle and the generic kernel."""
    import os
    lib, ptr, st = _lib_ptr()
    from hhfm_b200.engine import NO_HOT, HotRows
    rng = np.random.default_rng(K + fc + ft)
    M, B, NG = 700, 3001, 10
    V = make_table(rng, M, K)
    Pos = np.stack([rng.integers(0, 6, B), rng.integers(100, 400, B)], axis=1)
    Fea = np.stack([600 + 3 * c + rng.integers(0, 3, B) for c in range(fc)], axis=1) if fc else None
    Tim = rng.integers(100, 400, (B, ft)) if ft else None
    Neg = rng.integers(100, 400, (B, NG)); Neg[::9] = Neg[::9, :1]; Neg[:, 5] = Neg[:, 4]
    loss, pos, neg, dV = O.pairrank_loss_grads(V, Pos, Neg, Fea, Tim, (0, 0, 0), 0.0)
    rec, stride = _records(Pos, Fea, Tim, Neg)
    P = lib.partials_len()
    results = {}
    for mode in ("fast", "generic"):
        os.environ["HHFM_NO_FAST"] = "1" if mode == "generic" else "0"
        hot = HotRows(np.concatenate([np.arange(6), np.arange(600, 600 + 3 * fc)]), M, K, cuda, n_rep=8) if use_hot else None
        gV = torch.zeros(M, K, device=cuda); lp = torch.zeros(P, device=cuda); out = torch.zeros(1, device=cuda)
        lib.call("hhfm_pairrank_fwd_bwd", ptr(dev(rec, cuda)), B, stride, fc, ft, NG, 0, 0, 0, ptr(dev(V, cuda)), M, K, None, None,
                 ptr(gV), ptr(lp), None, 0, None, None, *(hot.args() if hot else NO_HOT), 0, st())
        if hot:
            hot.fold(gV, None)
        lib.call("hhfm_loss_finalize", ptr(lp), None, 0.0, ptr(out), st())
        results[mode] = (gV.cpu().numpy(), float(out.item()))
    os.environ.pop("HHFM_NO_FAST", None)
    for mode, (gV, l) in results.items():
        assert_close(l, loss, what=mode + " loss"); assert_close(gV, dV, what=mode + " gV")


def test_bpr_is_the_no_context_special_case(cuda):
    rng = np.random.default_rng(21)
    M, K, B = 400, 128, 3000
    V = make_table(rng, M, K); Pos = rng.integers(0, M, (B, 2)); Neg = rng.integers(0, M, (B, 10))
    loss, pos, neg, dV = O.pairrank_loss_grads(V, Pos, Neg, None, None, (0, 0, 0), 0.0)
    got = _pairrank_train(cuda, V, Pos, None, None, Neg, (0, 0, 0))
    assert_close(got["loss"], loss, what="bpr loss"); assert_close(got["gV"], dV, what="bpr gV")


def test_pairrank_forward_and_backward_entry_points(cuda):
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(22)
    M, K, B, NG = 300, 64, 400, 6
    V = make_table(rng, M, K); Pos = rng.integers(0, M, (B, 2)); Fea = rng.integers(0, M, (B, 4)); Neg = rng.integers(0, M, (B, NG))
    rec, stride = _records(Pos, Fea, None, Neg)
    pos = torch.empty(B, device=cuda); neg = torch.empty(B, NG, device=cuda)
    tV, trec = dev(V, cuda), dev(rec, cuda)
    lib.call("hhfm_pairrank_fwd", ptr(trec), B, stride, 4, 0, NG, 0, 0, 0, ptr(tV), M, K, ptr(pos), ptr(neg), st())
    rp, rn, hyb, _ = O.pairrank_scores(V, Pos, Neg, Fea, None, (0, 0, 0))
    assert_close(pos.cpu().numpy(), rp, what="pos"); assert_close(neg.cpu().numpy(), rn, what="neg")
    dpos = rng.normal(0, 1, B).astype(np.float32); dneg = rng.normal(0, 1, (B, NG)).astype(np.float32)
    tVg = torch.tensor(V, requires_grad=True)
    h = tVg[Pos[:, 0]] + tVg[Fea].sum(1)
    ((h * tVg[Pos[:, 1]]).sum(1) * torch.tensor(dpos)).sum().add(((h[:, None, :] * tVg[Neg]).sum(2) * torch.tensor(dneg)).sum()).backward()
    gV = torch.zeros(M, K, device=cuda)
    lib.call("hhfm_pairrank_bwd", ptr(trec), B, stride, 4, 0, NG, 0, 0, 0, ptr(tV), M, K, ptr(dev(dpos, cuda)), ptr(dev(dneg, cuda)),
             ptr(gV), 0, st())
    assert_close(gV.cpu().numpy(), tVg.grad.numpy(), what="pairrank bwd gV")


# ----------------------------------------------------------------------------------------------------
# K4/K5 scatter + optimizers
# ----------------------------------------------------------------------------------------------------
def test_scatter_add_rows_sums_duplicates(cuda):
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(1)
    M, K, n = 100, 64, 5000
    rows = rng.integers(0, 5, n).astype(np.int32); src = rng.normal(0, 1, (n, K)).astype(np.float32)
    ref = np.zeros((M, K), np.float32); np.add.at(ref, rows, src)
    dst = torch.zeros(M, K, device=cuda)
    lib.call("hhfm_scatter_add_rows", ptr(dev(rows, cuda)), ptr(dev(src, cuda)), n, K, ptr(dst), M, st())
    assert_close(dst.cpu().numpy(), ref, rtol=2e-5, what="scatter")


@pytest.mark.parametrize("n", [4096, 4099, 3, 1])
def test_dense_optimizers_match_tf1_semantics(cuda, n):
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(n)
    w0 = rng.normal(0, 0.1, n).astype(np.float32); g0 = rng.normal(0, 1, n).astype(np.float32)
    lam, lr = 0.1, 0.05
    P = lib.partials_len()
    # adagrad
    w, acc, g = dev(w0, cuda), torch.full((n,), 0.1, device=cuda), dev(g0, cuda)
    sq = torch.zeros(P, device=cuda)
    lib.call("hhfm_opt_adagrad_dense_l2", ptr(w), ptr(acc), ptr(g), n, lr, lam, 1, ptr(sq), st())
    rw, racc = O.adagrad_dense(w0, np.full(n, 0.1, np.float32), g0 + np.float32(lam) * w0, lr)
    assert_close(w.cpu().numpy(), rw, what="adagrad w"); assert_close(acc.cpu().numpy(), racc, what="adagrad acc")
    assert (g.cpu().numpy() == 0).all()
    assert_close(sq.sum().item(), (w0.astype(np.float64) ** 2).sum(), what="sum w^2")
    # adam (t = 3)
    w, m, v, g = dev(w0, cuda), dev(g0 * 0.1, cuda), dev(g0 * g0 * 0.01, cuda), dev(g0, cuda)
    import math
    lr_t = lr * math.sqrt(1 - 0.999 ** 3) / (1 - 0.9 ** 3)
    lib.call("hhfm_opt_adam_dense_l2", ptr(w), ptr(m), ptr(v), ptr(g), n, lr_t, 0.9, 0.999, 1e-8, 0.0, 0, None, st())
    rw, rm, rv = O.adam_dense(w0, g0 * 0.1, g0 * g0 * 0.01, g0, lr, 3)
    assert_close(w.cpu().numpy(), rw, what="adam w"); assert_close(m.cpu().numpy(), rm, what="adam m"); assert_close(v.cpu().numpy(), rv, what="adam v")
    assert (g.cpu().numpy() == g0).all()
    # momentum
    w, a, g = dev(w0, cuda), dev(g0 * 0.5, cuda), dev(g0, cuda)
    lib.call("hhfm_opt_momentum_dense_l2", ptr(w), ptr(a), ptr(g), n, lr, 0.95, 0.0, 1, None, st())
    rw, ra = O.momentum_dense(w0, g0 * 0.5, g0, lr)
    assert_close(w.cpu().numpy(), rw, what="momentum w"); assert_close(a.cpu().numpy(), ra, what="momentum acc")
    # sgd
    w, g = dev(w0, cuda), dev(g0, cuda)
    lib.call("hhfm_opt_sgd_dense_l2", ptr(w), ptr(g), n, lr, 0.0, 1, None, st())
    assert_close(w.cpu().numpy(), O.sgd_dense(w0, g0, lr), what="sgd w")


def test_row_optimizers_move_only_touched_rows(cuda):
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(2)
    M, K = 300, 64
    w0 = make_table(rng, M, K); g0 = np.zeros((M, K), np.float32)
    touched = np.sort(rng.choice(M, 40, replace=False)).astype(np.int32)
    g0[touched] = rng.normal(0, 1, (40, K)).astype(np.float32)
    rows = np.full(M, -1, np.int32); rows[:40] = rng.permutation(touched)
    cnt = dev(np.array([40], np.int32), cuda)
    w, acc, g = dev(w0, cuda), torch.full((M, K), 1e-8, device=cuda), dev(g0, cuda)
    lib.call("hhfm_opt_adagrad_rows", ptr(w), ptr(acc), ptr(g), ptr(dev(rows, cuda)), ptr(cnt), M, K, 0.01, 1, st())
    rw, racc = O.adagrad_rows(w0, np.full((M, K), 1e-8, np.float32), g0, touched, 0.01)
    assert_close(w.cpu().numpy(), rw, what="rows w"); assert_close(acc.cpu().numpy(), racc, what="rows acc")
    assert (g.cpu().numpy() == 0).all()
    untouched = np.setdiff1d(np.arange(M), touched)
    assert (w.cpu().numpy()[untouched] == w0[untouched]).all()
    w, a, g = dev(w0, cuda), dev(g0 * 0 + 0.5, cuda), dev(g0, cuda)
    lib.call("hhfm_opt_momentum_rows", ptr(w), ptr(a), ptr(g), ptr(dev(rows, cuda)), ptr(cnt), M, K, 0.1, 0.95, 0, st())
    rw, ra = O.momentum_rows(w0, np.full((M, K), 0.5, np.float32), g0, touched, 0.1)
    assert_close(w.cpu().numpy(), rw, what="mom rows w"); assert (a.cpu().numpy()[untouched] == 0.5).all()
    # K == 1 (feature_bias vector)
    b0 = rng.normal(0, 0.1, M).astype(np.float32); gb = np.zeros(M, np.float32); gb[touched] = 1.5
    b, accb, g = dev(b0, cuda), torch.full((M,), 0.1, device=cuda), dev(gb, cuda)
    lib.call("hhfm_opt_adagrad_rows", ptr(b), ptr(accb), ptr(g), ptr(dev(rows, cuda)), ptr(cnt), M, 1, 0.1, 1, st())
    rb, _ = O.adagrad_rows(b0, np.full(M, 0.1, np.float32), gb, touched, 0.1)
    assert_close(b.cpu().numpy(), rb, what="bias rows")


# ----------------------------------------------------------------------------------------------------
# K6 / K7 exact top-N and the metric walk
# ----------------------------------------------------------------------------------------------------
def _topn(cuda, kind, A, V, bias, n_user, n_item, tp, n_ctx, n_time, pools=(0, 0, 0), lo=0, hi=None, method="exact", info=None):
    from hhfm_b200.engine import TopN
    t = TopN(cuda)
    A_dev, stride = t.upload_rows(A, V.shape[0])
    tb = dev(bias, cuda) if bias is not None else None
    ids, sc = t.topk(kind, A_dev, stride, n_ctx, n_time, pools, dev(V, cuda), tb, n_user, n_item, tp, lo, hi, return_scores=True,
                     method=method)
    if info is not None:
        info["method"] = t.last_method; info["overflow_rows"] = t.last_overflow_rows
    return ids.cpu().numpy(), sc.cpu().numpy()


@pytest.mark.parametrize("C,N,K,tp,F", [(300, 4082, 64, 20, 10), (37, 580, 128, 20, 12), (5, 24, 16, 20, 10), (64, 1000, 256, 100, 4),
                                        (3, 10, 8, 20, 2)])
def test_fm_topk_lists_are_bit_exact(cuda, C, N, K, tp, F):
    rng = np.random.default_rng(C + N)
    n_user = 50; M = n_user + N + 40
    V = make_table(rng, M, K); b = rng.normal(0, 0.01, (M, 1)).astype(np.float32)
    A = np.concatenate([rng.integers(0, n_user, (C, 1)), rng.integers(n_user, n_user + N, (C, 1)),
                        rng.integers(n_user + N, M, (C, F - 2))], axis=1)
    ref = O.fm_topk_scores(A, V, b, n_user, N)
    ids, sc = _topn(cuda, 1, A, V, b, n_user, N, tp, F - 2, 0)
    want = O.topk_lowest_index(ref, tp)
    k = min(tp, N)
    assert (ids[:, :k] == want[:, :k]).all()
    assert (ids[:, k:] == -1).all()
    got_sc = np.take_along_axis(ref, want[:, :k], axis=1)
    assert (sc[:, :k].view(np.int32) == got_sc.view(np.int32)).all(), "exact scores must be bit-identical to the oracle"


def test_topk_tie_break_is_lowest_index(cuda):
    """Quantised weights make many exactly equal scores; tf.nn.top_k keeps the lower index first."""
    rng = np.random.default_rng(4)
    n_user, N, K, C = 10, 500, 16, 40
    M = n_user + N
    V = rng.integers(-2, 3, (M, K)).astype(np.float32) * 0.25
    V[n_user + 100:n_user + 200] = V[n_user:n_user + 100]          # duplicated items -> guaranteed ties
    A = np.stack([rng.integers(0, n_user, C), rng.integers(n_user, M, C)], axis=1)
    ref = O.dot_topk_scores(V[A[:, 0]], V, n_user, N)
    ids, sc = _topn(cuda, 0, A, V, None, n_user, N, 50, 0, 0)
    assert (ids == O.topk_lowest_index(ref, 50)).all()
    # +0.0 and -0.0 compare equal
    V2 = V.copy(); V2[0] = 0.0; V2[n_user:n_user + N:2] *= -1.0
    A2 = np.stack([np.zeros(C, int), rng.integers(n_user, M, C)], axis=1)
    ids2, _ = _topn(cuda, 0, A2, V2, None, n_user, N, 30, 0, 0)
    assert (ids2 == np.arange(30)[None, :]).all()


@pytest.mark.parametrize("pools", [(0, 0, 0), (1, 1, 1), (2, 2, 2)])
def test_hhfm_topk_bit_exact(cuda, pools):
    rng = np.random.default_rng(6)
    n_user, N, K, C, fc, ft = 30, 777, 64, 100, 5, 5
    M = n_user + N + 60
    V = make_table(rng, M, K)
    A = np.concatenate([rng.integers(0, n_user, (C, 1)), rng.integers(n_user, n_user + N, (C, 1)),
                        rng.integers(n_user + N, M, (C, fc + ft))], axis=1)
    ref = O.hhfm_topk_scores(A, V, n_user, N, fc, ft, pools)
    ids, sc = _topn(cuda, 2, A, V, None, n_user, N, 20, fc, ft, pools)
    want = O.topk_lowest_index(ref, 20)
    assert (ids == want).all()
    assert (sc.view(np.int32) == np.take_along_axis(ref, want, axis=1).view(np.int32)).all()


@pytest.mark.parametrize("kind,C,N,K,tp,F", [(1, 300, 4082, 64, 20, 10), (0, 200, 5000, 128, 100, 2), (2, 130, 3001, 64, 20, 10),
                                              (1, 257, 2500, 128, 20, 6), (0, 64, 1111, 32, 20, 2), (0, 50, 9000, 200, 100, 2),
                                              (1, 17, 700, 16, 20, 4), (0, 1000, 20000, 64, 100, 2)])
def test_tensor_core_topk_is_bit_identical_to_the_exact_path(cuda, kind, C, N, K, tp, F):
    """tcgen05 GEMM filter + exact rescoring must return the oracle's lists and score bits."""
    rng = np.random.default_rng(kind * 100 + C + K)
    n_user = 40; M = n_user + N + 50
    V = make_table(rng, M, K, scale=0.05); b = rng.normal(0, 0.02, (M, 1)).astype(np.float32)
    V[n_user + 7] *= 8.0                                     # one large-norm item stresses the max-norm error bound
    A = np.concatenate([rng.integers(0, n_user, (C, 1)), rng.integers(n_user, n_user + N, (C, 1)),
                        rng.integers(n_user + N, M, (C, F - 2))], axis=1)
    n_ctx = F - 2 if kind != 0 else 0
    info = {}
    ids, sc = _topn(cuda, kind, A, V, b if kind == 1 else None, n_user, N, tp, n_ctx, 0, method="tc", info=info)
    assert info["method"] == "tc"
    if kind == 1:
        ref = O.fm_topk_scores(A, V, b, n_user, N)
    elif kind == 2:
        ref = O.hhfm_topk_scores(A, V, n_user, N, n_ctx, 0)
    else:
        ref = O.dot_topk_scores(V[A[:, 0]], V, n_user, N)
    want = O.topk_lowest_index(ref, tp)
    assert (ids == want).all(), "tensor-core path changed a top-%d list (%d rows differ)" % (tp, int((ids != want).any(axis=1).sum()))
    assert (sc.view(np.int32) == np.take_along_axis(ref, want, axis=1).view(np.int32)).all()


def test_tensor_core_topk_survives_degenerate_ties_and_shards(cuda):
    """Quantised weights: thousands of exactly tied scores overflow the candidate buffer of some rows -> those rows are
    redone by the exact path; sharded calls carry the shard offset.  Lists must still equal the exact path."""
    rng = np.random.default_rng(41)
    n_user, N, K, C, tp = 16, 6000, 64, 96, 20
    M = n_user + N
    V = (rng.integers(-1, 2, (M, K)) * 0.25).astype(np.float32)
    A = np.stack([rng.integers(0, n_user, C), rng.integers(n_user, M, C)], axis=1)
    info = {}
    ids, sc = _topn(cuda, 0, A, V, None, n_user, N, tp, 0, 0, method="tc", info=info)
    ref = O.dot_topk_scores(V[A[:, 0]], V, n_user, N)
    assert (ids == O.topk_lowest_index(ref, tp)).all()
    lo, hi = 1500, 5200
    ids2, _ = _topn(cuda, 0, A, V, None, n_user, N, tp, 0, 0, lo=lo, hi=hi, method="tc")
    assert (ids2 == O.topk_lowest_index(ref[:, lo:hi], tp) + lo).all()


def test_item_sharded_topk_merges_to_the_single_shard_answer(cuda):
    """SURVEY 8e: shard items, local top-tp with global offsets, concatenate, re-select: identical lists."""
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(8)
    n_user, N, K, C, tp = 20, 1003, 32, 50, 20
    M = n_user + N
    V = rng.integers(-3, 4, (M, K)).astype(np.float32) * 0.125          # tie-heavy
    A = np.stack([rng.integers(0, n_user, C), rng.integers(n_user, M, C)], axis=1)
    full, _ = _topn(cuda, 0, A, V, None, n_user, N, tp, 0, 0)
    G = 4
    bounds = [N * g // G for g in range(G + 1)]
    parts = [_topn(cuda, 0, A, V, None, n_user, N, tp, 0, 0, lo=bounds[g], hi=bounds[g + 1]) for g in range(G)]
    cat_ids = dev(np.concatenate([p[0] for p in parts], axis=1), cuda)
    cat_sc = dev(np.concatenate([p[1] for p in parts], axis=1), cuda)
    out_ids = torch.empty(C, tp, dtype=torch.int32, device=cuda); out_sc = torch.empty(C, tp, device=cuda)
    lib.call("hhfm_topn_select", ptr(cat_sc), ptr(cat_ids), None, C, G * tp, G * tp, tp, 0, ptr(out_sc), ptr(out_ids), st())
    assert (out_ids.cpu().numpy() == full).all()


def test_metrics_walk_matches_the_reference_walk(cuda):
    from hhfm_b200 import engine
    from collections import defaultdict
    rng = np.random.default_rng(12)
    C, tp, n_user, N = 500, 20, 40, 60
    rows = np.concatenate([rng.integers(0, n_user, (C, 1)), rng.integers(n_user, n_user + N, (C, 1)), rng.integers(100, 104, (C, 2))], axis=1)
    pred = np.stack([rng.permutation(N)[:tp] + n_user for _ in range(C)])
    pf = defaultdict(set)
    for r in rows[::3]:
        pf[(r[0], r[2], r[3])].add(r[1])                 # rows whose target item is in positive_feedback[key]
    in_pf = np.array([r[1] in pf[(r[0], r[2], r[3])] for r in rows], np.uint8)
    for TopK in (1, 5, 10, 20, 25):
        m, n, p = O.evaluate_topk_walk(pred, rows, pf, TopK)
        codes = engine.metrics_walk(dev(pred, cuda, torch.int32), dev(rows[:, 1], cuda, torch.int32), dev(in_pf, cuda), TopK).cpu().numpy()
        got = engine.metrics_from_codes(codes)
        assert got[0] == np.average(m) and got[1] == np.average(n) and got[2] == np.average(p)
        assert (codes != -2).sum() == len(m)


# ----------------------------------------------------------------------------------------------------
# committed golden fixtures (tests/golden/): the oracle's vectors and the reference's own metric walk
# ----------------------------------------------------------------------------------------------------
import os as _os

_GOLD = _os.path.join(_os.path.dirname(_os.path.abspath(__file__)), "golden")


def test_device_matches_committed_oracle_vectors(cuda):
    g = np.load(_os.path.join(_GOLD, "oracle_vectors.npz"))
    n_user, n_item, M, K, B, F, NG = [int(x) for x in g["dims"]]
    V, b, X, Y, Neg = g["V"], g["b"], g["X"], g["Y"], g["Neg"]
    got = _fm_train_call(cuda, X, Y, V, b, np.float32(0.05))
    assert_close(got["out"], g["fm_out"], what="golden fm out")
    assert_close(got["gV"] + np.float32(0.1) * V, g["fm_dV"], what="golden fm dV (+lamda*V)")
    assert_close(got["gb"], g["fm_db"], what="golden fm db"); assert_close(got["gb0"], g["fm_db0"], what="golden fm db0")
    ids, _ = _topn(cuda, 1, X[:16], V, b, n_user, n_item, 20, F - 2, 0)
    assert (ids == g["fm_top20"]).all()
    for tag, pools in (("sum", (0, 0, 0)), ("max", (1, 1, 1)), ("mean", (2, 2, 2))):
        r = _pairrank_train(cuda, V, X[:, :2], X[:, 2:4], X[:, 4:6], Neg, pools)
        assert_close(r["pos"], g["hhfm_%s_pos" % tag], what="golden pos " + tag)
        assert_close(r["neg"], g["hhfm_%s_neg" % tag], what="golden neg " + tag)
        assert_close(r["gV"] + np.float32(0.01) * V, g["hhfm_%s_dV" % tag], what="golden hhfm dV " + tag)
        ids, _ = _topn(cuda, 2, X[:16], V, None, n_user, n_item, 20, 2, 2, pools)
        assert (ids == g["hhfm_%s_top20" % tag]).all()
    r = _pairrank_train(cuda, V, X[:, :2], None, None, Neg, (0, 0, 0))
    assert_close(r["gV"] + np.float32(0.1) * V, g["bpr_dV"], what="golden bpr dV")
    r = _fm_train_call(cuda, X[:, :2], Y * 2 - 1, V, None, None, interaction=1)
    assert_close(r["out"], g["mf_out"], what="golden mf out"); assert_close(r["gV"] + np.float32(0.01) * V, g["mf_dV"], what="golden mf dV")


@pytest.mark.parametrize("name", ["frappe", "resturant"])
def test_device_metric_walk_reproduces_the_reference_run(cuda, name, tmp_path):
    """Rows + predictions recorded while the reference's own Train.evaluate_TopK (FM.py:325-359) ran; the device walk
    must return exactly its [HR, NDCG, reciprocal-rank] triple."""
    from hhfm_b200 import engine
    from hhfm_b200.Newcode.NewLoadData import LoadData
    g = np.load(_os.path.join(_GOLD, "reference_host_logic.npz"))
    d = tmp_path / name
    d.mkdir()
    (d / (name + ".libfm")).write_text(str(g["libfm_" + name]))
    np.random.seed(11)
    ld = LoadData(str(tmp_path) + "/", name)
    for TopK in (1, 5, 10, 20):
        rows = g["%s_walk%d_rows" % (name, TopK)]; pred = g["%s_walk%d_pred" % (name, TopK)] + ld.n_user
        codes = engine.metrics_walk(dev(pred, cuda, torch.int32), dev(rows[:, 1], cuda, torch.int32),
                                    dev(ld.in_positive_feedback(rows).astype(np.uint8), cuda), TopK).cpu().numpy()
        assert engine.metrics_from_codes(codes) == g["%s_walk%d_result" % (name, TopK)].tolist()


# ----------------------------------------------------------------------------------------------------
# K2 AFM
# ----------------------------------------------------------------------------------------------------
def _afm_weights(rng, M, K, A):
    return dict(feature_embeddings=rng.normal(0, 0.1, (M, K)).astype(np.float32), feature_bias=rng.normal(0, 0.1, (M, 1)).astype(np.float32),
                bias=np.float32(0.05), attention_W=rng.normal(0, 0.2, (K, A)).astype(np.float32),
                attention_b=rng.normal(0, 0.2, (1, A)).astype(np.float32), attention_p=rng.normal(0, 1, (A,)).astype(np.float32),
                prediction=rng.normal(1, 0.1, (K, 1)).astype(np.float32))


@pytest.mark.parametrize("C,N,F,K", [(7, 700, 10, 64), (3, 37, 6, 32), (5, 1100, 3, 16), (4, 513, 2, 64), (2, 90, 12, 32)])
def test_afm_item_separable_scorer_matches_forward(cuda, C, N, F, K):
    """hhfm_afm_topn_scores (afm_topn.cu): context-only pairs once per row + the F-1 item pairs per (row, item) must equal the
    op-by-op AFM forward (AFM.py:103-148) of every expanded row."""
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(C * 1000 + N + F + K)
    n_user = 23
    M = n_user + N + 40
    w = _afm_weights(rng, M, K, K)
    rows = rng.integers(n_user + N, M, (C, F)); rows[:, 0] = rng.integers(0, n_user, C); rows[:, 1] = -7      # column 1 is ignored
    X = np.repeat(rows[:, None, :], N, axis=1); X[:, :, 1] = n_user + np.arange(N)[None, :]
    ref = O.afm_forward(X.reshape(-1, F), w)[0].reshape(C, N)
    assert lib.load().hhfm_afm_topn_supported(F, K, K) == 1
    stats = torch.empty(C, 4, device=cuda); sc = torch.full((C, N), float("nan"), device=cuda)
    stride = F + 2
    rows_dev = torch.full((C, stride), -1, dtype=torch.int32, device=cuda); rows_dev[:, :F] = torch.from_numpy(rows.astype(np.int32)).to(cuda)
    lib.call("hhfm_afm_topn_scores", ptr(rows_dev), stride, C, F, 1, ptr(dev(w["feature_embeddings"], cuda)), ptr(dev(w["feature_bias"].reshape(-1), cuda)),
             ptr(dev(np.array([w["bias"]], np.float32), cuda)), ptr(dev(w["attention_W"], cuda)), ptr(dev(w["attention_b"].reshape(-1), cuda)),
             ptr(dev(w["attention_p"], cuda)), ptr(dev(w["prediction"].reshape(-1), cuda)), M, K, K, n_user, N, ptr(stats), ptr(sc), st())
    assert_close(sc.cpu().numpy(), ref, what="afm separable scores")
    assert lib.load().hhfm_afm_topn_supported(F, 128, 128) == 0 and lib.load().hhfm_afm_topn_supported(F, 64, 32) == 0


@pytest.mark.parametrize("layout", ["pair-per-lane", "column-per-lane"])
@pytest.mark.parametrize("B,F,K", [(64, 10, 64), (1001, 10, 64), (130, 6, 32), (77, 12, 128), (50, 3, 16), (33, 2, 64), (45, 9, 32), (40, 11, 32), (70, 8, 64), (37, 7, 16)])
def test_afm_fused_pass_matches_oracle(cuda, B, F, K, layout, monkeypatch):
    """Both layouts of the fused kernel (afm.cu: afm2_kernel covers K == A in {16, 32, 64}; afm_kernel everything else)."""
    monkeypatch.setenv("HHFM_AFM_V1", "1" if layout == "column-per-lane" else "0")
    monkeypatch.setenv("HHFM_AFM_TC", "0")          # the fp32 CUDA-core kernels (K = A = 64 would take the tcgen05 kernel)
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(B + F + K)
    M, A = 300, K
    w = _afm_weights(rng, M, K, A)
    X = rng.integers(0, M, (B, F)); X[:, 1] = rng.integers(0, 4, B)
    if F > 3:
        X[:, 3] = X[:, 2]
    Y = rng.choice([1.0, -1.0], (B, 1)).astype(np.float32)
    loss, out, g = O.afm_loss_grads(X, Y, w, 0.0)
    tw = {k: dev(np.asarray(v, np.float32).reshape(-1) if k == "bias" else v, cuda) for k, v in w.items()}
    P = lib.partials_len()
    gV = torch.zeros(M, K, device=cuda); gb = torch.zeros(M, device=cuda); gb0 = torch.zeros(1, device=cuda)
    gW = torch.zeros(K, A, device=cuda); gba = torch.zeros(A, device=cuda); gp = torch.zeros(A, device=cuda); gwp = torch.zeros(K, device=cuda)
    lp = torch.zeros(P, device=cuda); o = torch.empty(B, device=cuda); lo = torch.zeros(1, device=cuda)
    tX = dev(X, cuda, torch.int32)
    args = (ptr(tX), B, F, ptr(tw["feature_embeddings"]), ptr(tw["feature_bias"]), ptr(tw["bias"]), ptr(tw["attention_W"]),
            ptr(tw["attention_b"]), ptr(tw["attention_p"]), ptr(tw["prediction"]), M, K, A)
    o2 = torch.empty(B, device=cuda)
    lib.call("hhfm_afm_fwd", *args, ptr(o2), st())
    assert_close(o2.cpu().numpy(), out, what="afm fwd out")
    lib.call("hhfm_afm_fwd_bwd_sqloss", *args, ptr(dev(Y.reshape(-1), cuda)), ptr(o), ptr(gV), ptr(gb), ptr(gb0), ptr(gW), ptr(gba),
             ptr(gp), ptr(gwp), ptr(lp), None, 0, None, None, None, None, None, 0, 0, st())
    lib.call("hhfm_loss_finalize", ptr(lp), None, 0.0, ptr(lo), st())
    assert_close(o.cpu().numpy(), out, what="afm out"); assert_close(lo.item(), loss, what="afm loss")
    assert_close(gV.cpu().numpy(), g["feature_embeddings"], rtol=2e-5, what="afm gV")
    assert_close(gb.cpu().numpy(), g["feature_bias"].reshape(-1), what="afm gbias")
    assert_close(gb0.item(), g["bias"], what="afm gb0")
    assert_close(gW.cpu().numpy(), g["attention_W"], rtol=2e-5, what="afm gW")
    # d attention_b sums d s_p over the pairs, and the softmax makes those sum to zero per sample: what is left is
    # cancellation noise with no scale of its own, so it is held to 1e-5 of the attention_W gradient's scale
    floor = 1e-5 * float(np.abs(g["attention_W"]).max())
    assert_close(gba.cpu().numpy(), g["attention_b"].reshape(-1), rtol=2e-5, atol=floor, what="afm gb_att")
    assert_close(gp.cpu().numpy(), g["attention_p"], rtol=2e-5, atol=floor, what="afm gp")
    assert_close(gwp.cpu().numpy(), g["prediction"].reshape(-1), rtol=2e-5, what="afm gw_pred")


# ----------------------------------------------------------------------------------------------------
# K8 DeepFM
# ----------------------------------------------------------------------------------------------------
def _dfm_weights(rng, M, F, K, layers):
    dims = [F * K] + list(layers)
    w = dict(feature_embeddings=rng.normal(0, 0.1, (M, K)).astype(np.float32),
             feature_bias=rng.uniform(0, 1, (M, 1)).astype(np.float32),
             concat_projection=rng.normal(0, np.sqrt(2.0 / (F + K + dims[-1] + 1)), (F + K + dims[-1], 1)).astype(np.float32),
             concat_bias=np.float32(0.01))
    for i in range(len(layers)):
        gl = np.sqrt(2.0 / (dims[i] + dims[i + 1]))
        w["layer_%d" % i] = rng.normal(0, gl, (dims[i], dims[i + 1])).astype(np.float32)
        w["bias_%d" % i] = rng.normal(0, gl, (1, dims[i + 1])).astype(np.float32)
    return w


def _dfm_flat(w, F, K, layers, lib):
    sizes = np.asarray(layers, np.int32)
    n = int(lib.load().hhfm_dfm_param_count(F, K, len(layers), sizes.ctypes.data))
    nr = int(lib.load().hhfm_dfm_reg_count(F, K, len(layers), sizes.ctypes.data))
    flat = np.zeros(n, np.float32)
    off = 0
    slots = {}
    for i in range(len(layers)):
        a = w["layer_%d" % i].reshape(-1); flat[off:off + a.size] = a; slots["layer_%d" % i] = (off, w["layer_%d" % i].shape); off += a.size
    a = w["concat_projection"].reshape(-1); flat[off:off + a.size] = a; slots["concat_projection"] = (off, w["concat_projection"].shape)
    off = nr
    for i in range(len(layers)):
        a = w["bias_%d" % i].reshape(-1); flat[off:off + a.size] = a; slots["bias_%d" % i] = (off, w["bias_%d" % i].shape); off += a.size
    flat[off] = w["concat_bias"]; slots["concat_bias"] = (off, ())
    assert off + 1 == n
    return flat, slots, sizes


@pytest.mark.parametrize("B,F,K,layers", [(64, 10, 64, (150, 200, 150)), (1001, 10, 64, (150, 200, 150)), (300, 6, 32, (40, 24)),
                                          (77, 12, 128, (150, 200, 150)), (50, 3, 16, (7,)), (129, 2, 8, (33, 65, 17, 5))])
def test_dfm_fused_pass_matches_oracle(cuda, B, F, K, layers):
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(B + F + K)
    M = 300
    w = _dfm_weights(rng, M, F, K, layers)
    X = rng.integers(0, M, (B, F)); X[:, 1] = rng.integers(0, 4, B)
    if F > 3:
        X[:, 3] = X[:, 2]
    Y = rng.choice([1.0, -1.0], (B, 1)).astype(np.float32)
    loss, out, g = O.dfm_loss_grads(X, Y, w, 0.0, n_layers=len(layers))
    flat, slots, sizes = _dfm_flat(w, F, K, layers, lib)
    L = len(layers)
    tV = dev(w["feature_embeddings"], cuda); tb = dev(w["feature_bias"], cuda); tp = dev(flat, cuda)
    tX = dev(X, cuda, torch.int32)
    ws = torch.empty(int(lib.load().hhfm_workspace_bytes_dfm(B, F, K, L, sizes.ctypes.data)) // 4 + 1, device=cuda)
    o = torch.empty(B, device=cuda)
    lib.call("hhfm_dfm_fwd", ptr(tX), B, F, ptr(tV), ptr(tb), M, K, ptr(tp), L, sizes.ctypes.data, ptr(ws), ptr(o), st())
    assert_close(o.cpu().numpy(), out, what="dfm fwd out")
    gV = torch.zeros(M, K, device=cuda); gb = torch.zeros(M, device=cuda); gp = torch.zeros(flat.size, device=cuda)
    lp = torch.zeros(lib.partials_len(), device=cuda); lo = torch.zeros(1, device=cuda); o2 = torch.empty(B, device=cuda)
    lib.call("hhfm_dfm_fwd_bwd_sqloss", ptr(tX), B, F, ptr(tV), ptr(tb), M, K, ptr(tp), L, sizes.ctypes.data,
             ptr(dev(Y.reshape(-1), cuda)), ptr(ws), ptr(o2), ptr(gV), ptr(gb), ptr(gp), ptr(lp), None, None, None, 0, 0, st())
    lib.call("hhfm_loss_finalize", ptr(lp), None, 0.0, ptr(lo), st())
    assert_close(o2.cpu().numpy(), out, what="dfm out"); assert_close(lo.item(), loss, what="dfm loss")
    assert_close(gV.cpu().numpy(), g["feature_embeddings"], rtol=2e-5, what="dfm gV")
    assert_close(gb.cpu().numpy(), g["feature_bias"].reshape(-1), rtol=2e-5, what="dfm gbias")
    gp = gp.cpu().numpy()
    for k, (off, shape) in slots.items():
        ref = np.asarray(g[k], np.float32).reshape(-1)
        assert_close(gp[off:off + ref.size], ref, rtol=2e-5, what="dfm g %s" % k)


# ----------------------------------------------------------------------------------------------------
# K1 variants: the TMA-staged pipeline (large tables) against the oracle and the register kernels
# ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,F,K", [(64, 10, 64), (5000, 10, 128), (999, 6, 128), (3, 16, 64), (777, 10, 256), (2049, 1, 512),
                                   (1500, 12, 100)])
def test_fm_staged_pipeline_matches_oracle(cuda, B, F, K, monkeypatch):
    """fm_train_staged_kernel (cp.async.bulk row staging + mbarriers; chosen automatically when the table exceeds L2)
    forced on small inputs: out / loss / gradients / touched-row set against the oracle."""
    monkeypatch.setenv("HHFM_FM_STAGED", "1")
    rng = np.random.default_rng(B + K + F)
    M = 400
    V = make_table(rng, M, K); b = rng.normal(0, 0.1, (M, 1)).astype(np.float32); b0 = np.float32(-0.1)
    X = rng.integers(0, M, (B, F))
    if F > 1:
        X[:, 1] = rng.integers(0, 3, B)
    if F > 4:
        X[:, 4] = X[:, 0]
    Y = rng.choice([1.0, 0.0], (B, 1)).astype(np.float32)
    from test_kernel_instances import launched_kernels
    loss, out, dV, db, db0, touched = O.fm_loss_grads(X, Y, V, b, b0, lamda=0.0)
    names, got = launched_kernels(lambda: _fm_train_call(cuda, X, Y, V, b, b0))
    assert len(names) == 1 and names.pop().startswith("fm_train_staged_kernel<")
    assert_close(got["out"], out, what="out")
    assert_close(got["loss"], loss, what="loss")
    assert_close(got["gV"], dV, what="gV")
    assert_close(got["gb"], db, what="gbias")
    assert_close(got["gb0"], db0, what="gb0")
    assert (got["touched"] == touched).all()
    names, got2 = launched_kernels(lambda: _fm_train_call(cuda, X, Y, V, None, None, track=False))   # no bias, no tracking
    assert len(names) == 1 and names.pop().startswith("fm_train_staged_kernel<")
    monkeypatch.setenv("HHFM_FM_STAGED", "0")
    names, ref2 = launched_kernels(lambda: _fm_train_call(cuda, X, Y, V, None, None, track=False))
    assert len(names) == 1 and not names.pop().startswith("fm_train_staged_kernel<")
    assert_close(got2["out"], ref2["out"], what="staged vs register out"); assert_close(got2["gV"], ref2["gV"], what="staged vs register gV")


def test_fm_staged_pipeline_with_hot_rows(cuda, monkeypatch):
    lib, ptr, st = _lib_ptr()
    from hhfm_b200.engine import HotRows
    monkeypatch.setenv("HHFM_FM_STAGED", "1")
    rng = np.random.default_rng(79)
    M, K, B, F = 200, 128, 3000, 6
    V = make_table(rng, M, K); b = rng.normal(0, 0.1, (M, 1)).astype(np.float32)
    X = np.stack([rng.integers(0, 100, B), rng.integers(100, 180, B), 190 + rng.integers(0, 2, B), 192 + rng.integers(0, 3, B),
                  195 + rng.integers(0, 5, B), rng.integers(0, 3, B)], axis=1)
    Y = rng.choice([1.0, 0.0], (B, 1)).astype(np.float32)
    loss, out, dV, db, db0, _ = O.fm_loss_grads(X, Y, V, b, 0.0, 0.0)
    hot = HotRows(np.concatenate([np.arange(3), np.arange(190, 200)]), M, K, cuda, with_bias=True, n_rep=4)
    gV = torch.zeros(M, K, device=cuda); gb = torch.zeros(M, device=cuda); gb0 = torch.zeros(1, device=cuda)
    lp = torch.zeros(lib.partials_len(), device=cuda)
    lib.call("hhfm_fm_fwd_bwd_sqloss", None, ptr(dev(X, cuda, torch.int32)), None, B, F, ptr(dev(V, cuda)), ptr(dev(b, cuda)), None,
             M, K, 0, ptr(dev(Y.reshape(-1), cuda)), None, ptr(gV), ptr(gb), ptr(gb0), ptr(lp), None, 0, None, None,
             *hot.args(True), 0, st())
    hot.fold(gV, gb)
    assert_close(gV.cpu().numpy(), dV, what="fm gV hot staged"); assert_close(gb.cpu().numpy(), db, what="fm gb hot staged")


@pytest.mark.parametrize("K,fc,ft,NG,B", [(128, 8, 0, 10, 5000), (64, 8, 0, 10, 3001), (128, 5, 5, 10, 999), (256, 3, 0, 4, 777),
                                          (128, 0, 0, 10, 2049), (512, 2, 1, 1, 65), (64, 10, 10, 10, 1500)])
@pytest.mark.parametrize("use_hot", [False, True])
def test_pairrank_staged_pipeline_matches_oracle(cuda, K, fc, ft, NG, B, use_hot, monkeypatch):
    """pairrank_sum_train_staged_kernel (cp.async.bulk row staging + mbarriers; chosen automatically when the table exceeds
    L2, the scaled c5 shape) forced on small inputs: loss / gradient / touched-row set against the oracle, and against the
    register kernel."""
    lib, ptr, st = _lib_ptr()
    from hhfm_b200.engine import NO_HOT, HotRows
    from test_kernel_instances import launched_kernels
    if (K, 2 + fc + ft + NG) in ((128, 22), (512, 6)):
        monkeypatch.setenv("HHFM_PR_WARPS", "9")       # two stages of 10 warps exceed the 224 KB of shared memory
    rng = np.random.default_rng(K + fc + ft + NG)
    M = 700
    V = make_table(rng, M, K)
    Pos = np.stack([rng.integers(0, 6, B), rng.integers(100, 400, B)], axis=1)
    Fea = np.stack([600 + 3 * c + rng.integers(0, 3, B) for c in range(fc)], axis=1) if fc else None
    Tim = rng.integers(100, 400, (B, ft)) if ft else None
    Neg = rng.integers(100, 400, (B, NG)); Neg[::9] = Neg[::9, :1]
    if NG > 5:
        Neg[:, 5] = Neg[:, 4]
    loss, pos, neg, dV = O.pairrank_loss_grads(V, Pos, Neg, Fea, Tim, (0, 0, 0), 0.0)
    rec, stride = _records(Pos, Fea, Tim, Neg)
    P = lib.partials_len()
    res = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("HHFM_PR_STAGED", mode)
        hot = HotRows(np.concatenate([np.arange(6), np.arange(600, 600 + 3 * fc)]), M, K, cuda, n_rep=8) if use_hot else None
        gV = torch.zeros(M, K, device=cuda); lp = torch.zeros(P, device=cuda); out = torch.zeros(1, device=cuda)
        stamp = torch.zeros(M, dtype=torch.int32, device=cuda); rows = torch.zeros(M, dtype=torch.int32, device=cuda)
        cnt = torch.zeros(1, dtype=torch.int32, device=cuda)
        names, _ = launched_kernels(lambda: lib.call(
            "hhfm_pairrank_fwd_bwd", ptr(dev(rec, cuda)), B, stride, fc, ft, NG, 0, 0, 0, ptr(dev(V, cuda)), M, K, None, None,
            ptr(gV), ptr(lp), ptr(stamp), 5, ptr(rows), ptr(cnt), *(hot.args() if hot else NO_HOT), 0, st()))
        assert len(names) == 1
        kernel = names.pop()
        assert kernel.startswith("pairrank_sum_train_staged_kernel<" if mode == "1" else "pairrank_kernel<"), (mode, kernel)
        if hot:
            hot.fold(gV, None)
        lib.call("hhfm_loss_finalize", ptr(lp), None, 0.0, ptr(out), st())
        n = int(cnt.item())
        res[mode] = (gV.cpu().numpy(), float(out.item()), np.sort(rows[:n].cpu().numpy()))
    for mode, (gV, l, touched) in res.items():
        assert_close(l, loss, what="staged=%s loss" % mode); assert_close(gV, dV, what="staged=%s gV" % mode)
        assert len(set(touched.tolist())) == len(touched)
        nz = np.flatnonzero(np.abs(dV).sum(1) > 0)
        assert set(nz.tolist()) <= set(touched.tolist())
    assert (res["1"][2] == res["0"][2]).all(), "the staged and the register kernel disagree on the touched rows"


# ----------------------------------------------------------------------------------------------------
# K6 tensor-core path, sampled cut (large catalogs): the cut is a rank statistic of every 8th item tile, proven per row
# after rescoring; rows that cannot be proven are redone exactly.  Lists must stay bit-identical.
# ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,C,N,K,tp", [(0, 130, 120000, 64, 100), (1, 70, 100003, 64, 20), (0, 40, 150000, 128, 100)])
def test_tensor_core_sampled_cut_is_bit_identical(cuda, kind, C, N, K, tp, monkeypatch):
    rng = np.random.default_rng(kind + C + K)
    n_user = 40; M = n_user + N + 50
    V = make_table(rng, M, K, scale=0.05); b = rng.normal(0, 0.02, (M, 1)).astype(np.float32)
    F = 4 if kind == 1 else 2
    A = np.concatenate([rng.integers(0, n_user, (C, 1)), rng.integers(n_user, n_user + N, (C, 1)),
                        rng.integers(n_user + N, M, (C, F - 2))], axis=1)
    info = {}
    ids, sc = _topn(cuda, kind, A, V, b if kind == 1 else None, n_user, N, tp, F - 2 if kind == 1 else 0, 0, method="tc", info=info)
    assert info["method"] == "tc"
    ref = O.fm_topk_scores(A, V, b, n_user, N) if kind == 1 else O.dot_topk_scores(V[A[:, 0]], V, n_user, N)
    want = O.topk_lowest_index(ref, tp)
    assert (ids == want).all(), "sampled cut changed a top-%d list (%d rows differ)" % (tp, int((ids != want).any(axis=1).sum()))
    assert (sc.view(np.int32) == np.take_along_axis(ref, want, axis=1).view(np.int32)).all()
    assert info["overflow_rows"] <= max(2, C // 20), "the sampled cut should be provable for almost every row"
    monkeypatch.setenv("HHFM_TOPN_SAMPLE", "1")                      # two full passes, guaranteed cut
    ids1, sc1 = _topn(cuda, kind, A, V, b if kind == 1 else None, n_user, N, tp, F - 2 if kind == 1 else 0, 0, method="tc")
    assert (ids1 == ids).all() and (sc1.view(np.int32) == sc.view(np.int32)).all()


@pytest.mark.parametrize("where", ["sampled_tiles", "unsampled_tiles"])
def test_tensor_core_sampled_cut_unrepresentative_sample(cuda, where):
    """Adversarial catalog order: every high-scoring item sits in the sampled tiles (cut too high: too few survivors, the
    rows are flagged and redone exactly) or in none of them (cut too low: more survivors / overflow).  Same lists."""
    rng = np.random.default_rng(5)
    n_user, N, K, C, tp = 16, 131072, 64, 48, 50
    M = n_user + N
    V = make_table(rng, M, K, scale=0.02)
    tile = (np.arange(N) // 256)
    boost = (tile % 8 == 0) if where == "sampled_tiles" else (tile % 8 == 3)
    V[n_user:][boost] *= 6.0
    A = np.stack([rng.integers(0, n_user, C), rng.integers(n_user, M, C)], axis=1)
    info = {}
    ids, sc = _topn(cuda, 0, A, V, None, n_user, N, tp, 0, 0, method="tc", info=info)
    ref = O.dot_topk_scores(V[A[:, 0]], V, n_user, N)
    want = O.topk_lowest_index(ref, tp)
    assert (ids == want).all()
    assert (sc.view(np.int32) == np.take_along_axis(ref, want, axis=1).view(np.int32)).all()


# ----------------------------------------------------------------------------------------------------
# K0 pipelined pack + upload (uint16 wire format when every id fits, int32 otherwise)
# ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("id_limit,rows", [(5382, 200001), (65535, 70000), (65536, 70000), (10_000_000, 150000), (300, 5), (300, 0)])
def test_pack_upload_records_matches_the_host_packer(cuda, id_limit, rows):
    from hhfm_b200.engine import RecordUploader, Staging, pack_records
    from hhfm_b200 import _lib
    rng = np.random.default_rng(rows + id_limit)
    X = rng.integers(0, id_limit, (rows, 2)).astype(np.int64)
    F1 = rng.integers(0, id_limit, (rows, 8)).astype(np.int32)                 # int32 block
    Y = np.ascontiguousarray(rng.integers(0, id_limit, (rows, 13)).astype(np.int64))[:, :10]   # strided view
    if rows:
        X[-1, 1] = id_limit - 1
    up = RecordUploader(cuda)
    recs, stride = up.upload([X, F1, Y], id_limit)
    if rows == 0:
        assert stride == 20 and recs.shape == (0, 20)
        return
    host, stride2 = pack_records([X, F1, Y], id_limit, Staging(torch.int32))
    assert stride == stride2 == 20 and recs.shape == (rows, 20)
    assert (recs.cpu().numpy() == host.numpy().reshape(rows, 20)).all()
    recs3, stride3 = up.upload([X[:, :1], F1[:, :2]], id_limit)               # width 3 -> stride 4, one padding column
    if rows:
        got = recs3.cpu().numpy()
        assert stride3 == 4 and (got[:, 3] == -1).all() and (got[:, 0] == X[:, 0]).all() and (got[:, 1:3] == F1[:, :2]).all()
        Xbad = X.copy(); Xbad[rows // 2, 0] = id_limit
        with pytest.raises(_lib.HhfmError, match="out of range"):
            up.upload([Xbad, F1, Y], id_limit)
        # int64-only parts: the 16-bit wire format takes the vectorised packer (8 ids per instruction + masked tails)
        Z = rng.integers(0, id_limit, (rows, 17)).astype(np.int64)
        recs4, stride4 = up.upload([X, Y, Z], id_limit)
        host4, _ = pack_records([X, Y, Z], id_limit, Staging(torch.int32))
        assert (recs4.cpu().numpy() == host4.numpy().reshape(rows, stride4)).all()
        for badval in (id_limit, -1, -(1 << 40), 1 << 40):
            Zbad = Z.copy(); Zbad[rows - 1, 16] = badval
            with pytest.raises(_lib.HhfmError, match="out of range"):
                up.upload([X, Y, Zbad], id_limit)


# ----------------------------------------------------------------------------------------------------
# K9 device negative sampler / AUC plumbing (integer work: bit-exact against the oracle restatement)
# ----------------------------------------------------------------------------------------------------
def test_device_negative_sampler_matches_oracle_and_rejects_positives(cuda):
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(21)
    n_user, n_item, n_keys, n, num = 50, 40, 30, 3000, 10
    span = n_user + n_item
    # every key owns 0..35 of the 40 items: heavy rejection for some rows
    pf = []
    for k in range(n_keys):
        own = rng.choice(n_item, size=int(rng.integers(0, 36)), replace=False)
        pf += [k * span + n_user + int(i) for i in own]
    codes = np.unique(np.asarray(pf, dtype=np.int64))
    key_id = rng.integers(-1, n_keys, n).astype(np.int32)               # -1: key never trained
    seed = 0x1234ABCD5678
    out = torch.full((n, 16), -7, dtype=torch.int32, device=cuda)
    lib.call("hhfm_sample_negatives", ptr(dev(key_id, cuda)), n, num, n_user, n_item, ptr(dev(codes, cuda)), len(codes), span, seed,
             ptr(out), 16, 3, st())
    got = out.cpu().numpy()
    want = O.sample_negative_hashed(key_id, num, n_user, n_item, codes, span, seed)
    assert (got[:, 3:13] == want).all(), "device sampler differs from the oracle restatement"
    assert (got[:, :3] == -7).all() and (got[:, 13:] == -7).all()
    assert got[:, 3:13].min() >= n_user and got[:, 3:13].max() < n_user + n_item
    cset = set(codes.tolist())
    bad = sum((int(k) * span + int(it)) in cset for k, row in zip(key_id, got[:, 3:13]) if k >= 0 for it in row)
    assert bad == 0, "a sampled negative is in positive_feedback[key]"
    # rows without constraints are uniform over the catalog (chi-square, 39 dof: 99.9 % quantile ~ 72)
    free = got[key_id < 0][:, 3:13].reshape(-1) - n_user
    cnt = np.bincount(free, minlength=n_item); e = free.size / n_item
    assert ((cnt - e) ** 2 / e).sum() < 80.0


def test_expand_rows_and_auc_count(cuda):
    lib, ptr, st = _lib_ptr()
    from hhfm_b200 import engine
    rng = np.random.default_rng(22)
    n, F, num = 700, 6, 50
    rows = rng.integers(0, 1000, (n, 8)).astype(np.int32)
    items = rng.integers(1000, 2000, (n, num)).astype(np.int32)
    out = engine.expand_rows(dev(rows, cuda), F, dev(items, cuda), 8).cpu().numpy()
    ref = np.repeat(rows[:, None, :], num, axis=1); ref[:, :, 1] = items; ref[:, :, F:] = -1
    assert (out == ref.reshape(-1, 8)).all()
    pos = rng.normal(size=n).astype(np.float32); neg = rng.normal(size=n * num).astype(np.float32)
    neg[::7] = np.repeat(pos, num)[::7]                                   # ties count as losses (strict >, FM.py:321)
    wins = torch.zeros(1, dtype=torch.int64, device=cuda)
    engine.auc_wins(dev(pos, cuda), dev(neg, cuda), num, wins)
    assert int(wins.item()) == int((np.repeat(pos, num) > neg).sum())


# ----------------------------------------------------------------------------------------------------
# 3xTF32 tensor-core GEMM (building block of the DeepFM tower): fp32-grade accuracy against float64
# ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,K", [(128, 160, 32), (300, 150, 640), (5000, 200, 150), (1000, 640, 150), (640, 150, 4096),
                                   (129, 16, 8), (4096, 256, 256), (77, 300, 100)])
def test_tf32x3_gemm_is_fp32_accurate(cuda, M, N, K):
    lib, ptr, st = _lib_ptr()
    rng = np.random.default_rng(M + N + K)
    lda = (K + 3) // 4 * 4 + 4; ldb = (K + 3) // 4 * 4; ldc = (N + 3) // 4 * 4
    A = np.zeros((M, lda), np.float32); B = np.zeros((N, ldb), np.float32)
    A[:, :K] = rng.normal(0, 1, (M, K)); B[:, :K] = rng.normal(0, 1, (N, K))
    A[:, K:] = 7.0; B[:, K:] = -3.0                                  # padding must never be read
    tA = dev(A, cuda); tB = dev(B, cuda)
    C = torch.full((M, ldc), 99.0, device=cuda)
    ws = torch.empty(M * lda + N * ldb, device=cuda)
    lib.call("hhfm_gemm_tn_tf32x3", ptr(tA), lda, ptr(tB), ldb, M, N, K, ptr(C), ldc, ptr(ws), st())
    got = C.cpu().numpy()
    ref = A[:, :K].astype(np.float64) @ B[:, :K].astype(np.float64).T
    scale = np.sqrt(K)                                                # typical magnitude of a dot product of K N(0,1) terms
    err = np.abs(got[:, :N] - ref).max() / scale
    assert err < 4e-6, "3xTF32 GEMM error %.3e (relative to sqrt(K)); plain tf32 would be ~5e-4" % err
    assert (got[:, N:] == 99.0).all()


@pytest.mark.parametrize("B,F", [(64, 10), (5001, 10), (1, 10), (2, 10), (333, 11), (130, 6), (77, 3), (33, 2), (1000, 7)])
@pytest.mark.parametrize("extras", [False, True])
@pytest.mark.parametrize("groups", [4, 2])
def test_afm_fused_tensor_core_pass_matches_oracle(cuda, B, F, extras, groups, monkeypatch):
    """K2 as ONE tcgen05 kernel (afm_fused_tc.cu, K = A = 64, F <= 11): P W, dZ W^T and P^T dZ as 3xTF32 products with the
    operands built in shared memory; selected by hhfm_afm_fwd_bwd_sqloss from the shape.  `extras`: hot-row replicas and
    touched-row tracking.  Odd B exercises the half-empty last tile.  `groups`: 16 columns per thread / 16 warps (the default)
    or 32 columns per thread / 8 warps (HHFM_AFM_TC=2)."""
    if groups == 4:
        monkeypatch.delenv("HHFM_AFM_TC", raising=False)
    else:
        monkeypatch.setenv("HHFM_AFM_TC", "2")
    lib, ptr, st = _lib_ptr()
    from hhfm_b200.engine import HotRows
    rng = np.random.default_rng(B + F + 64 + 1)
    M, K, A = 300, 64, 64
    w = _afm_weights(rng, M, K, A)
    X = rng.integers(0, M, (B, F)); X[:, 1] = rng.integers(0, 4, B)
    if F > 3:
        X[:, 3] = X[:, 2]
    Y = rng.choice([1.0, -1.0], (B, 1)).astype(np.float32)
    loss, out, g = O.afm_loss_grads(X, Y, w, 0.0)
    tw = {k: dev(np.asarray(v, np.float32).reshape(-1) if k == "bias" else v, cuda) for k, v in w.items()}
    P = lib.partials_len()
    gV = torch.zeros(M, K, device=cuda); gb = torch.zeros(M, device=cuda); gb0 = torch.zeros(1, device=cuda)
    gW = torch.zeros(K, A, device=cuda); gba = torch.zeros(A, device=cuda); gp = torch.zeros(A, device=cuda); gwp = torch.zeros(K, device=cuda)
    lp = torch.zeros(P, device=cuda); o = torch.empty(B, device=cuda); lo = torch.zeros(1, device=cuda)
    tX = dev(X, cuda, torch.int32)
    args = (ptr(tX), B, F, ptr(tw["feature_embeddings"]), ptr(tw["feature_bias"]), ptr(tw["bias"]), ptr(tw["attention_W"]),
            ptr(tw["attention_b"]), ptr(tw["attention_p"]), ptr(tw["prediction"]), M, K, A)
    if extras:
        hot = HotRows(np.arange(0, 8), M, K, cuda, with_bias=True, n_rep=4)
        stamp = torch.zeros(M, dtype=torch.int32, device=cuda); rows = torch.zeros(M, dtype=torch.int32, device=cuda)
        cnt = torch.zeros(1, dtype=torch.int32, device=cuda)
        tail = (ptr(stamp), 3, ptr(rows), ptr(cnt), *hot.args(True))
    else:
        tail = (None, 0, None, None, None, None, None, 0, 0)
    lib.call("hhfm_afm_fwd_bwd_sqloss", *args, ptr(dev(Y.reshape(-1), cuda)), ptr(o), ptr(gV), ptr(gb), ptr(gb0), ptr(gW), ptr(gba),
             ptr(gp), ptr(gwp), ptr(lp), *tail, st())
    if extras:
        hot.fold(gV, gb)
        n = int(cnt.item())
        assert sorted(rows[:n].cpu().numpy().tolist()) == sorted(np.unique(X).tolist())
    lib.call("hhfm_loss_finalize", ptr(lp), None, 0.0, ptr(lo), st())
    assert_close(o.cpu().numpy(), out, what="afm tc out"); assert_close(lo.item(), loss, what="afm tc loss")
    assert_close(gV.cpu().numpy(), g["feature_embeddings"], rtol=2e-5, what="afm tc gV")
    assert_close(gb.cpu().numpy(), g["feature_bias"].reshape(-1), what="afm tc gbias")
    assert_close(gb0.item(), g["bias"], what="afm tc gb0")
    assert_close(gW.cpu().numpy(), g["attention_W"], rtol=2e-5, what="afm tc gW")
    # d attention_b / d attention_p are sums over B*P terms that largely cancel (softmax gradients sum to zero over the pairs):
    # their fp32 rounding noise grows with B in the oracle and on the device alike
    noise = 2e-5 if B < 2000 else 1e-4
    floor = 1e-5 * float(np.abs(g["attention_W"]).max())       # a tensor that is ALL cancellation noise has no scale of its own
    assert_close(gba.cpu().numpy(), g["attention_b"].reshape(-1), rtol=noise, atol=floor, what="afm tc gb_att")
    assert_close(gp.cpu().numpy(), g["attention_p"], rtol=noise, atol=floor, what="afm tc gp")
    assert_close(gwp.cpu().numpy(), g["prediction"].reshape(-1), rtol=2e-5, what="afm tc gw_pred")
