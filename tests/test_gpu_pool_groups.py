"""GPU: pooled context groups of the sum-pooling training pass (hhfm_pool_groups_attach) against the oracle and against the
generic kernel (HHFM_NO_FAST=1), at the existing 1e-5 tolerances."""
import numpy as np
import pytest
import torch

from conftest import assert_close, assert_update_close
from oracle import hhfm_oracle as O

pytestmark = pytest.mark.gpu

_KEEP = []
NG = 10


def dev(a, cuda):
    t = torch.as_tensor(np.ascontiguousarray(a)).to(cuda)
    _KEEP.append(t)
    return t


def records(Pos, Fea, Tim, Neg):
    parts = [Pos] + [p for p in (Fea, Tim, Neg) if p is not None and p.shape[1] > 0]
    w = sum(p.shape[1] for p in parts)
    stride = (w + 3) // 4 * 4
    rec = np.full((Pos.shape[0], stride), -1, np.int32)
    rec[:, :w] = np.concatenate(parts, axis=1)
    return rec, stride


def layout(cards, n_user=50, n_item=300):
    """Column id ranges after users and items: (lo per column, M)."""
    lo, base = [], n_user + n_item
    for c in cards:
        lo.append(base)
        base += c
    return lo, base


def batch(rng, B, lo, cards, fc, n_user=50, n_item=300, spill=None):
    """Pos, Fea, Tim, Neg; `spill` = (fraction, columns): that share of samples takes, in those columns, the id just past the
    planned range (the first id of the next column or of the table's tail)."""
    Pos = np.stack([rng.integers(0, n_user, B), n_user + rng.integers(0, n_item, B)], axis=1)
    cols = np.stack([lo[c] + rng.integers(0, cards[c], B) for c in range(len(cards))], axis=1)
    if spill is not None:
        frac, which = spill
        rows = rng.random(B) < frac
        for c in which:
            cols[rows, c] = lo[c] + cards[c]
    Neg = n_user + rng.integers(0, n_item, (B, NG))
    Neg[::9] = Neg[::9, :1]
    Neg[:, 5] = Neg[:, 4]
    return Pos, (cols[:, :fc] if fc else None), (cols[:, fc:] if len(cards) > fc else None), Neg


def run_pass(cuda, V_dev, M, K, rec, stride, fc, ft, hot=None):
    from hhfm_b200 import _lib
    from hhfm_b200.engine import NO_HOT, cur_stream, ptr
    B = rec.shape[0]
    gV = torch.zeros(M, K, device=cuda)
    lp = torch.zeros(_lib.partials_len(), device=cuda)
    out = torch.zeros(1, device=cuda)
    _lib.call("hhfm_pairrank_fwd_bwd", ptr(dev(rec, cuda)), B, stride, fc, ft, NG, 0, 0, 0, ptr(V_dev), M, K, None, None,
              ptr(gV), ptr(lp), None, 0, None, None, *(hot.args() if hot else NO_HOT), 0, cur_stream())
    if hot:
        hot.fold(gV, None)
    _lib.call("hhfm_loss_finalize", ptr(lp), None, 0.0, ptr(out), cur_stream())
    return gV.cpu().numpy(), float(out.item())


# bench-like context columns; a mix with two columns too wide for the group cap (cap = 64 here) and time columns; NP = 3
CASES = {
    "frappe8": ((7, 2, 3, 2, 9, 80, 233, 7), 8, None),
    "mixed_ctx5_time3": ((3, 2, 300, 4, 5, 2, 257, 3), 5, 64),
    "ctx2_time1": ((5, 4, 3), 2, None),
}


def plan(V_dev, n_pool, stride, lo, cards, cap):
    from hhfm_b200.engine import PoolGroups, plan_pool_groups
    groups = plan_pool_groups(lo, list(cards), **({"cap": cap} if cap else {}))
    assert any(g >= 0 for g in groups)
    return PoolGroups(V_dev, n_pool, stride, [l if g >= 0 else 0 for l, g in zip(lo, groups)],
                      [c if g >= 0 else 0 for c, g in zip(cards, groups)], groups)


@pytest.mark.parametrize("K", [32, 64, 128])
@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("use_hot", [False, True])
def test_grouped_pass_matches_oracle_and_generic(cuda, K, case, use_hot, monkeypatch):
    from hhfm_b200.engine import HotRows
    cards, fc, cap = CASES[case]
    ft = len(cards) - fc
    rng = np.random.default_rng(K + len(cards) + fc)
    lo, M = layout(cards)
    B = 3001
    V = rng.normal(0, 0.1, (M, K)).astype(np.float32)
    V_dev = dev(V, cuda)
    Pos, Fea, Tim, Neg = batch(rng, B, lo, cards, fc)
    rec, stride = records(Pos, Fea, Tim, Neg)
    pg = plan(V_dev, len(cards), stride, lo, cards, cap)
    hot = HotRows(np.arange(6), M, K, cuda, n_rep=8) if use_hot else None
    loss, _, _, dV = O.pairrank_loss_grads(V, Pos, Neg, Fea, Tim, (0, 0, 0), 0.0)
    gV, l = run_pass(cuda, V_dev, M, K, rec, stride, fc, ft, hot)
    assert_close(l, loss, what="grouped loss"); assert_close(gV, dV, what="grouped gV")
    S, G = pg.tables()
    assert float(G.abs().max()) == 0.0, "G must be zero after the pass"
    assert float(S.abs().max()) > 0.0
    monkeypatch.setenv("HHFM_NO_FAST", "1")
    gV_g, l_g = run_pass(cuda, V_dev, M, K, rec, stride, fc, ft, hot)
    assert_close(l, l_g, what="grouped vs generic loss"); assert_close(gV, gV_g, what="grouped vs generic gV")


@pytest.mark.parametrize("K", [32, 64, 128])
@pytest.mark.parametrize("use_hot", [False, True])
def test_fallback_samples_outside_the_planned_range(cuda, K, use_hot):
    """Plan from one batch, then a batch where 3 % of the samples carry an id just past a column's planned range."""
    from hhfm_b200.engine import HotRows
    cards, fc, cap = CASES["mixed_ctx5_time3"]
    ft = len(cards) - fc
    rng = np.random.default_rng(100 + K)
    lo, M = layout(cards)
    M += 1                                    # the id past the last column exists
    V = rng.normal(0, 0.1, (M, K)).astype(np.float32)
    V_dev = dev(V, cuda)
    rec0, stride = records(*batch(rng, 2000, lo, cards, fc))
    pg = plan(V_dev, len(cards), stride, lo, cards, cap)
    grouped = [c for c in range(len(cards)) if pg.groups[c] >= 0]
    Pos, Fea, Tim, Neg = batch(rng, 3001, lo, cards, fc, spill=(0.03, [grouped[0], grouped[-1]]))
    rec, stride = records(Pos, Fea, Tim, Neg)
    hot = HotRows(np.arange(6), M, K, cuda, n_rep=8) if use_hot else None
    loss, _, _, dV = O.pairrank_loss_grads(V, Pos, Neg, Fea, Tim, (0, 0, 0), 0.0)
    gV, l = run_pass(cuda, V_dev, M, K, rec, stride, fc, ft, hot)
    assert_close(l, loss, what="fallback loss"); assert_close(gV, dV, what="fallback gV")
    assert float(pg.tables()[1].abs().max()) == 0.0


def test_two_consecutive_steps_follow_the_table(cuda):
    """The pre-sum reads the table of each call: step 2 runs on V updated from step 1's gradient."""
    cards, fc, cap = CASES["frappe8"]
    rng = np.random.default_rng(5)
    lo, M = layout(cards)
    K = 64
    V = rng.normal(0, 0.1, (M, K)).astype(np.float32)
    V_dev = dev(V, cuda)
    pg = None
    for step in range(2):
        Pos, Fea, Tim, Neg = batch(rng, 3001, lo, cards, fc)
        rec, stride = records(Pos, Fea, Tim, Neg)
        if pg is None:
            pg = plan(V_dev, len(cards), stride, lo, cards, cap)
        loss, _, _, dV = O.pairrank_loss_grads(V, Pos, Neg, Fea, Tim, (0, 0, 0), 0.0)
        gV, l = run_pass(cuda, V_dev, M, K, rec, stride, fc, 0)
        assert_close(l, loss, what="step %d loss" % step); assert_close(gV, dV, what="step %d gV" % step)
        V = (V - 0.05 * dV / np.abs(dV).max()).astype(np.float32)
        V_dev.copy_(torch.from_numpy(V))


def test_fit_device_with_the_plan_from_hot_plan(cuda):
    """OUR.fit_device: the plan is built with the hot-row plan from the first batch, member rows are not hot, and the
    post-step weights (Adagrad, dense L2) match the oracle."""
    from hhfm_b200.models import OUR
    cards, fc, _ = CASES["frappe8"]
    n_user, n_item, K, B = 40, 300, 64, 20000
    lo, M = layout(cards, n_user, n_item)
    rng = np.random.default_rng(9)
    model = OUR(fc, 0, M, n_user, n_item, K, 0.1, 0.01, "AdagradOptimizer", True, False)
    V0 = model.get_weights()["feature_embeddings"].copy()
    Pos, Fea, _, Neg = batch(rng, B, lo, cards, fc, n_user, n_item)
    Pos[:, 0] = rng.integers(0, 4, B)                     # a few users hot enough for the hot-row plan
    rec, stride = records(Pos, Fea, None, Neg)
    rec_dev = dev(rec, cuda)
    model.fit_device(rec_dev, fc, 0, NG)
    loss = model._read_loss()
    assert model._pool_groups is not None and model._hot is not None
    members = set(model._pool_groups.member_rows().tolist())
    assert members and not members & set(model._hot.rows.cpu().numpy().tolist()), "member rows must not be hot"
    loss_ref, _, _, dV = O.pairrank_loss_grads(V0, Pos, Neg, Fea, None, (0, 0, 0), 0.01)
    V_ref, _ = O.adagrad_dense(V0, np.full_like(V0, 0.1), dV, 0.1)
    assert abs(loss - loss_ref) <= 1e-5 * abs(loss_ref), (loss, loss_ref)
    got = model.get_weights()["feature_embeddings"]
    assert_update_close(got, V_ref, V0, dV, np.full_like(V0, 0.1), 0.1, what="fit_device weights")
