"""CPU: the pooled-context-group planner (engine.plan_pool_groups), the mixed-radix index and fallback predicate, and an
oracle restatement showing that grouped pooling and the expanded group gradient equal the per-row computation."""
import numpy as np

from conftest import assert_close
from hhfm_b200.engine import plan_pool_groups, pool_group_index
from oracle import hhfm_oracle as O

BENCH_CARDS = (7, 2, 3, 2, 9, 80, 233, 7)


def bench_lo(cards=BENCH_CARDS, base=957 + 4082):
    lo = []
    for c in cards:
        lo.append(base)
        base += c
    return lo


def test_bench_columns_form_two_groups():
    g = plan_pool_groups(bench_lo(), list(BENCH_CARDS))
    small = {c for c in range(8) if g[c] == g[1]}
    assert small == {0, 1, 2, 3, 4, 7}
    assert g[5] == g[6] != g[1] and g[5] >= 0
    assert np.prod([BENCH_CARDS[c] for c in small]) == 5292 and 80 * 233 == 18640


def test_greedy_packing_respects_the_caps():
    cards = [3, 2, 300, 4, 5, 2, 257, 3]
    lo = bench_lo(cards)
    g = plan_pool_groups(lo, cards, cap=64)
    for gid in set(g) - {-1}:
        assert np.prod([cards[c] for c in range(8) if g[c] == gid]) <= 64
    assert g[2] == -1 and g[6] == -1                     # wider than the cap: stay per-row columns
    assert sum(1 for x in g if x >= 0) == 6
    # the total cap closes the second group early; a lone column is not a group
    g2 = plan_pool_groups(lo, cards, cap=64, total_cap=40)
    assert sum(np.prod([cards[c] for c in range(8) if g2[c] == gid]) for gid in set(g2) - {-1}) <= 40
    assert all(sum(1 for x in g2 if x == gid) >= 2 for gid in set(g2) - {-1})


def test_planner_declines_overlaps_bad_ranges_and_too_many_rows():
    lo = [100, 105, 200]
    assert plan_pool_groups(lo, [10, 3, 4]) == [-1, -1, -1]          # 100..109 overlaps 105..107: only one column left
    assert plan_pool_groups([100, 103, 200], [3, 0, 4]) == [0, -1, 0]  # card 0: not groupable
    # 8 wide columns + 2 small ones: 9 pooled rows after grouping exceed the compiled slot counts
    lo = bench_lo([50000] * 8 + [2, 2])
    assert plan_pool_groups(lo, [50000] * 8 + [2, 2]) == [-1] * 10


def test_mixed_radix_index_and_fallback_predicate():
    lo = [10, 20, 30]
    card = [3, 4, 5]
    ids = np.array([[10, 20, 30], [12, 23, 34], [11, 20, 33], [13, 20, 30], [10, 19, 30]])
    k, ok = pool_group_index(ids, lo, card, [0, 2])
    assert ok.tolist() == [True, True, True, False, True]
    assert k[:3].tolist() == [0, 2 + 3 * 4, 1 + 3 * 3]
    k, ok = pool_group_index(ids, lo, card, [1])
    assert ok.tolist() == [True, True, True, True, False]
    # every combination index is hit exactly once by the full grid of digits
    grid = np.array(np.meshgrid(*[np.arange(c) + l for l, c in zip(lo, card)], indexing="ij")).reshape(3, -1).T
    k, ok = pool_group_index(grid, lo, card, [0, 1, 2])
    assert ok.all() and sorted(k.tolist()) == list(range(60))


def _grouped_restatement(V, Pos, Neg, Fea, lo, card, groups):
    """The grouped formulation in NumPy: pre-sum tables, pooled rows per group, group gradients, expansion."""
    F32 = np.float32
    V = V.astype(F32)
    B, n_pool = Fea.shape
    hyb = V[Pos[:, 0]].copy()
    slots, grads = [], []
    for gid in sorted(set(groups) - {-1}, key=lambda g: groups.index(g)):
        members = [c for c in range(n_pool) if groups[c] == gid]
        P = int(np.prod([card[c] for c in members]))
        S = np.zeros((P, V.shape[1]), F32)
        kk = np.arange(P)
        for i, c in enumerate(members):                      # members in record order, first least significant
            S = V[lo[c] + kk % card[c]] if i == 0 else (S + V[lo[c] + kk % card[c]]).astype(F32)
            kk = kk // card[c]
        k, ok = pool_group_index(Fea, lo, card, members)
        assert ok.all()
        slots.append((members, P, k, S))
    for c in range(n_pool):
        if groups[c] < 0:
            hyb = (hyb + V[Fea[:, c]]).astype(F32)
    for members, P, k, S in slots:
        hyb = (hyb + S[k]).astype(F32)
    vp, vn = V[Pos[:, 1]], V[Neg]
    pos = (hyb * vp).sum(1, dtype=F32)
    neg = np.einsum("bk,bjk->bj", hyb, vn).astype(F32)
    m = neg.max(1)
    sg = (1.0 / (1.0 + np.exp(-(pos - m)))).astype(F32)
    loss = -np.log(sg).astype(F32).sum(dtype=F32)
    gp = (sg - 1).astype(F32)
    tie = (neg == m[:, None]).astype(F32)
    gn = (-gp[:, None] * tie / tie.sum(1, keepdims=True)).astype(F32)
    dh = (gp[:, None] * vp + np.einsum("bj,bjk->bk", gn, vn)).astype(F32)
    dV = np.zeros_like(V)
    np.add.at(dV, Pos[:, 1], gp[:, None] * hyb)
    np.add.at(dV, Neg.reshape(-1), (gn[:, :, None] * hyb[:, None, :]).reshape(-1, V.shape[1]))
    np.add.at(dV, Pos[:, 0], dh)
    for c in range(n_pool):
        if groups[c] < 0:
            np.add.at(dV, Fea[:, c], dh)
    for members, P, k, S in slots:
        G = np.zeros((P, V.shape[1]), F32)
        np.add.at(G, k, dh)                                  # one row per group per positive
        kk = np.arange(P)
        for c in members:                                    # expansion: every combination holding the row
            np.add.at(dV, lo[c] + kk % card[c], G)
            kk = kk // card[c]
    return loss, dV


def test_grouped_pooling_and_expanded_gradient_equal_the_per_row_computation():
    rng = np.random.default_rng(3)
    cards = [3, 2, 300, 4, 5, 2, 257, 3]
    lo = bench_lo(cards, base=60)
    M = lo[-1] + cards[-1]
    K, B = 16, 4000
    V = rng.normal(0, 0.1, (M, K)).astype(np.float32)
    Pos = np.stack([rng.integers(0, 20, B), 20 + rng.integers(0, 40, B)], 1)
    Fea = np.stack([lo[c] + rng.integers(0, cards[c], B) for c in range(8)], 1)
    Neg = 20 + rng.integers(0, 40, (B, 10))
    groups = plan_pool_groups(lo, cards, cap=64)
    loss, dV = _grouped_restatement(V, Pos, Neg, Fea, lo, cards, groups)
    loss_ref, _, _, dV_ref = O.pairrank_loss_grads(V, Pos, Neg, Fea, None, (0, 0, 0), 0.0)
    assert_close(loss, loss_ref, what="grouped loss")
    assert_close(dV, dV_ref, rtol=2e-5, what="expanded gradient")
