"""Every FM / HHFM training-kernel instance the dispatchers can launch, each reached by one case of INSTANCES.

The training entry points pick one template instance from the shape, the table size and a few environment knobs, so a
test that checks outputs without checking which kernel ran can pass on a different instance than the one it was written
for.  Here:
  * INSTANCES maps each instance to the case that reaches it; a CPU test asserts that its keys are exactly the instances
    compiled into the library (cuobjdump + cu++filt), so an instance added without a case, or a case left behind by a
    deleted instance, fails;
  * a GPU test runs each case once under torch.profiler, asserts that exactly the expected training kernel launched, and
    compares loss, outputs, gradients and touched rows with a float64 restatement of the same graph;
  * the staged (TMA pipeline) instances run at steady state: B is derived from the SM count and the instance's warps per
    CTA so that every full warp range holds 25 samples (the id ring of 2*NS-1 slots turns at least three times), one range
    is partial and one is empty.

Tolerance: per element |got - ref| <= 1e-5 (|ref| + sum |terms|), ref the float64 graph, sum |terms| the same graph on
absolute values (the scale of the fp32 rounding of a sum whose terms cancel); loss within 1e-5 relative.  Ids are drawn so
that no row outside a small hot set takes more than about 200 contributions, so one missing or doubled sample is far
above the tolerance (test_reference_sees_one_sample).  HHFM tables are quantised to multiples of 2^-7 so that every score
is exact in fp32 and float64 alike: the max negative and its ties are then the same in the kernel and the reference.
"""
from __future__ import annotations

import os
import re
import subprocess

import numpy as np
import pytest
import torch

# ----------------------------------------------------------------------------------------------------
# instance names
# ----------------------------------------------------------------------------------------------------
FAMILIES = ("fm_train_fixed_kernel", "fm_train_staged_kernel", "pairrank_sum_train_kernel",
            "pairrank_sum_train_staged_kernel", "fm_kernel", "pairrank_kernel")
_NAME = re.compile(r"(?<![\w])(%s)<([^<>]*)>" % "|".join(sorted(FAMILIES, key=len, reverse=True)))


def normalise(name):
    """'void hhfm::fm_kernel<(int)16, (int)1, (int)1, (bool)0>(hhfm::FmArgs)' (cu++filt), '... <16, 1, 1, false> ...'
    (c++filt, profiler) -> 'fm_kernel<16,1,1,false>'; None for a kernel outside FAMILIES."""
    s = re.sub(r"\s+", "", name).replace("(int)", "").replace("(bool)0", "false").replace("(bool)1", "true")
    m = _NAME.search(s)
    return None if m is None else "%s<%s>" % m.groups()


def is_training_instance(n):
    """The instances of the ledger: the specialised training kernels, fm_kernel with MODE = FM_TRAIN and DROP = false,
    pairrank_kernel with MODE = PR_TRAIN."""
    fam, args = n[:-1].split("<")
    a = args.split(",")
    if fam == "fm_kernel":
        return a[2] == "1" and a[3] == "false"
    if fam == "pairrank_kernel":
        return a[2] == "1"
    return True


def library_instances(lib_path):
    """Training-kernel instances compiled into the library: kernel sections of `cuobjdump -elf`, demangled by cu++filt."""
    bindir = os.path.dirname(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"))
    mangled = set()
    with subprocess.Popen([os.path.join(bindir, "cuobjdump"), "-elf", lib_path], stdout=subprocess.PIPE, text=True) as p:
        for line in p.stdout:
            mangled.update(re.findall(r"\.text\.(_Z\w+)", line))
    assert p.returncode == 0, "cuobjdump failed"
    dem = subprocess.run([os.path.join(bindir, "cu++filt")], input="\n".join(sorted(mangled)), capture_output=True, text=True,
                         check=True).stdout.splitlines()
    return {n for n in map(normalise, dem) if n is not None and is_training_instance(n)}


def launched_kernels(fn):
    """Run fn() under torch.profiler (CUDA activity); returns (normalised names of the FAMILIES kernels it launched, result)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = {normalise(e.name) for e in prof.events()}
    names.discard(None)
    return names, res


# ----------------------------------------------------------------------------------------------------
# the ledger
# ----------------------------------------------------------------------------------------------------
STEADY = "steady"      # B from the SM count and the instance's warps per CTA (steady_batch)


def _fm(*shapes, env=None, hot=0, M=None):
    """FM training pass (hhfm_fm_fwd_bwd_sqloss): (B, F, K) shapes run one after another, bias and b0 on, touched rows on;
    hot = number of hot rows (with bias replicas) drawn into field 1."""
    return dict(kind="fm", shapes=list(shapes), env=dict(env or {}), hot=hot, M=M)


def _pr(K, nc, nt, ng, B=3001, env=None, hot=False, groups=None, M=None):
    """Sum-pooling HHFM training pass without scores or touched rows (the register fast path and the pooled-group
    path accept no others); staged instances run with touched rows.  groups: explicit col_group of the pooled columns."""
    return dict(kind="pr", K=K, nc=nc, nt=nt, ng=ng, B=B, env=dict(env or {}), hot=hot, groups=groups, M=M)


def _prg(K, nc, nt, ng, pools, B=1999):
    """Generic HHFM kernel (pairrank_kernel) through the scoring + touched-rows entry (_pairrank_train)."""
    return dict(kind="prg", K=K, nc=nc, nt=nt, ng=ng, B=B, pools=pools, env={"HHFM_NO_FAST": "1"})


_FS = {"HHFM_FM_STAGED": "1"}
_PS = {"HHFM_PR_STAGED": "1"}


def _fs(ns, nw):
    return dict(_FS, HHFM_FM_STAGES=str(ns), HHFM_FM_WARPS=str(nw))


def _ps(ns, nw):
    return dict(_PS, HHFM_PR_STAGES=str(ns), HHFM_PR_WARPS=str(nw))


_NO_FS = {"HHFM_FM_STAGED": "0"}
_NO_PS = {"HHFM_PR_STAGED": "0"}

INSTANCES = {
    # ---- fm_train_fixed_kernel<LPS = K/4, NF>: F at each NF boundary (F <= K/4) ----
    "fm_train_fixed_kernel<8,8>": _fm((3001, 1, 32), (2999, 8, 32), env=_NO_FS, hot=16),
    "fm_train_fixed_kernel<16,8>": _fm((3001, 1, 64), (2999, 8, 64), env=_NO_FS),
    "fm_train_fixed_kernel<16,12>": _fm((3001, 9, 64), (2999, 12, 64), env=_NO_FS, hot=16),
    "fm_train_fixed_kernel<16,16>": _fm((3001, 13, 64), (2999, 16, 64), env=_NO_FS),
    "fm_train_fixed_kernel<32,8>": _fm((3001, 1, 128), (2999, 8, 128), env=_NO_FS, hot=16),
    "fm_train_fixed_kernel<32,12>": _fm((3001, 9, 128), (2999, 12, 128), env=_NO_FS),
    "fm_train_fixed_kernel<32,16>": _fm((3001, 13, 128), (2999, 16, 128), env=_NO_FS, hot=16),
    # ---- fm_train_staged_kernel<NS, NW> ----
    "fm_train_staged_kernel<4,10>": _fm((STEADY, 12, 100), env=_FS, hot=64),
    # no env knob: a table of 100 MB selects the staged kernel, and F = 10, K = 128 (the c5 shape) eleven warps x 3 stages
    "fm_train_staged_kernel<3,11>": _fm((STEADY, 10, 128), M=200_000),
    "fm_train_staged_kernel<2,10>": _fm((STEADY, 12, 196), env=_FS),
    "fm_train_staged_kernel<3,10>": _fm((STEADY, 16, 64), env=_fs(3, 10), hot=64),
    "fm_train_staged_kernel<2,11>": _fm((STEADY, 8, 256), env=_fs(2, 11)),
    "fm_train_staged_kernel<3,12>": _fm((STEADY, 6, 200), env=_fs(3, 12)),
    "fm_train_staged_kernel<2,12>": _fm((STEADY, 13, 128), env=_fs(2, 12), hot=64),
    "fm_train_staged_kernel<3,13>": _fm((STEADY, 9, 96), env=_fs(3, 13)),
    "fm_train_staged_kernel<2,13>": _fm((STEADY, 16, 128), env=_fs(2, 13)),
    "fm_train_staged_kernel<3,14>": _fm((STEADY, 11, 64), env=_fs(3, 14), hot=64),
    "fm_train_staged_kernel<2,14>": _fm((STEADY, 1, 512), env=_fs(2, 14)),
    "fm_train_staged_kernel<2,16>": _fm((STEADY, 14, 100), env=_fs(2, 16), hot=64),
    # ---- fm_kernel<LPS, VPL, FM_TRAIN, false>: one per HHFM_DISPATCH_K bucket, shapes the specialised kernels reject ----
    "fm_kernel<2,1,1,false>": _fm((2001, 10, 8), env=_NO_FS),
    "fm_kernel<4,1,1,false>": _fm((2001, 7, 16), env=_NO_FS),
    "fm_kernel<8,1,1,false>": _fm((2001, 9, 32), env=_NO_FS),
    "fm_kernel<16,1,1,false>": _fm((2001, 17, 64), env=_NO_FS),
    "fm_kernel<32,1,1,false>": _fm((2001, 17, 128), env=_NO_FS),
    "fm_kernel<32,2,1,false>": _fm((2001, 10, 256), env=_NO_FS),
    "fm_kernel<32,4,1,false>": _fm((2001, 5, 512), env=_NO_FS),
    # ---- pairrank_sum_train_kernel<LPS, NP, 10, NS>, ungrouped (NS = NP) ----
    **{"pairrank_sum_train_kernel<%d,%d,10,%d>" % (K // 4, np_, np_): _pr(K, nc, np_ - nc, 10, env=_NO_PS, hot=(np_ % 2 == 0))
       for K in (32, 64, 128) for np_, nc in ((0, 0), (3, 2), (8, 8), (10, 7))},
    # ---- grouped (explicit col_group, NS < NP; -1 = an ungrouped column, a slot of its own) ----
    **{"pairrank_sum_train_kernel<%d,%d,10,%d>" % (K // 4, len(g), ns): _pr(K, nc, len(g) - nc, 10, env=_NO_PS, groups=g)
       for K in (32, 64, 128)
       for g, ns, nc in (([0, 0, 0], 1, 3), ([0, -1, 0], 2, 2),
                         ([0] * 8, 1, 8), ([0, 0, 0, 0, 1, 1, 1, 1], 2, 8), ([0, 0, 0, -1, 1, 1, 1, 1], 3, 6),
                         ([0, 0, -1, 1, 1, 1, -1, 1], 4, 8),
                         ([0] * 10, 1, 7), ([0] * 5 + [-1] + [0] * 4, 2, 10), ([0, 0, 0, 1, 1, 1, 2, 2, 2, 2], 3, 7),
                         ([0, 0, 0, -1, 1, 1, 1, 2, 2, 2], 4, 10))},
    # ---- pairrank_sum_train_staged_kernel<NS, NW> ----
    "pairrank_sum_train_staged_kernel<2,7>": _pr(64, 0, 0, 30, B=STEADY, env=_ps(2, 7)),            # W = 32
    "pairrank_sum_train_staged_kernel<3,7>": _pr(64, 8, 0, 10, B=STEADY, env=_ps(3, 7), hot=True),
    "pairrank_sum_train_staged_kernel<4,7>": _pr(128, 2, 1, 1, B=STEADY, env=_ps(4, 7)),             # n_neg = 1
    "pairrank_sum_train_staged_kernel<2,8>": _pr(256, 3, 2, 6, B=STEADY, env=_ps(2, 8), hot=True),
    "pairrank_sum_train_staged_kernel<3,8>": _pr(64, 5, 5, 10, B=STEADY, env=_ps(3, 8)),
    "pairrank_sum_train_staged_kernel<4,8>": _pr(128, 0, 0, 10, B=STEADY, env=_ps(4, 8), hot=True),
    "pairrank_sum_train_staged_kernel<2,9>": _pr(128, 8, 0, 10, B=STEADY, env=_ps(2, 9)),
    "pairrank_sum_train_staged_kernel<3,9>": _pr(96, 3, 0, 4, B=STEADY, env=_ps(3, 9), hot=True),
    "pairrank_sum_train_staged_kernel<4,9>": _pr(192, 1, 1, 2, B=STEADY, env=_ps(4, 9)),
    # no env knob: the hhfm_c5 width (8 context columns, 10 negatives, W = 20) with a 100 MB table: ten warps x 2 stages
    "pairrank_sum_train_staged_kernel<2,10>": _pr(128, 8, 0, 10, B=STEADY, M=200_000, hot=True),
    "pairrank_sum_train_staged_kernel<3,10>": _pr(128, 1, 0, 3, B=STEADY, env=_ps(3, 10)),
    "pairrank_sum_train_staged_kernel<4,10>": _pr(64, 4, 0, 10, B=STEADY, env=_ps(4, 10), hot=True),
    # ---- pairrank_kernel<LPS, VPL, PR_TRAIN, ANYMAX>: every HHFM_DISPATCH_K bucket, sum and max pooling ----
    **{"pairrank_kernel<%d,%d,1,false>" % lv: _prg(K, 3, 2, 10, (0, 0, 0)) for K, lv in
       ((8, (2, 1)), (16, (4, 1)), (32, (8, 1)), (64, (16, 1)), (128, (32, 1)), (256, (32, 2)), (512, (32, 4)))},
    **{"pairrank_kernel<%d,%d,1,true>" % lv: _prg(K, 3, 2, 7, pools) for K, lv, pools in
       ((8, (2, 1), (1, 1, 1)), (16, (4, 1), (1, 0, 1)), (32, (8, 1), (0, 1, 0)), (64, (16, 1), (1, 1, 1)),
        (128, (32, 1), (0, 0, 1)), (256, (32, 2), (1, 1, 0)), (512, (32, 4), (1, 1, 1)))},
}


def staged_warps(name):
    """Warps per CTA of a staged instance (its second template argument)."""
    return int(name[:-1].split(",")[1])


def steady_batch(n_sm, nw, per=25):
    """B over n_sm CTAs x nw warps with ceil(B / warps) = per: full ranges of `per` samples, one partial (per - 7), one
    empty."""
    n_warps = n_sm * nw
    B = (n_warps - 1) * per - 7
    assert -(-B // n_warps) == per and B % per != 0
    return B


# ----------------------------------------------------------------------------------------------------
# float64 reference
# ----------------------------------------------------------------------------------------------------
def _t(a, dtype=torch.float64):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dtype)


def fm_reference(X, Y, V, b, b0, weight=None, chunk=1 << 13):
    """FM squared loss (FM.py:99-126) in float64, in chunks of samples: out, loss, dV, db, db0, and for each gradient the
    sum of |terms| (the same graph on absolute values: |g| -> |y| + sum of |out terms|, S - e_f -> sum |e| + |e_f|).
    weight[s] scales sample s's loss and gradient contributions (self-checks)."""
    M, K = V.shape
    X = _t(X, torch.int64)
    B, F = X.shape
    V64, b64, y = _t(V), _t(b.reshape(-1)), _t(Y.reshape(-1))
    w = torch.ones(B, dtype=torch.float64) if weight is None else _t(weight)
    r = dict(out=torch.zeros(B, dtype=torch.float64), out_t=torch.zeros(B, dtype=torch.float64), loss=0.0,
             V=torch.zeros(M, K, dtype=torch.float64), V_t=torch.zeros(M, K, dtype=torch.float64),
             b=torch.zeros(M, dtype=torch.float64), b_t=torch.zeros(M, dtype=torch.float64), b0=0.0, b0_t=0.0)
    for s0 in range(0, B, chunk):
        x, ys, ws = X[s0:s0 + chunk], y[s0:s0 + chunk], w[s0:s0 + chunk]
        E = V64[x]
        Ea = E.abs()
        S, Sa = E.sum(1), Ea.sum(1)
        out = 0.5 * (S * S - (E * E).sum(1)).sum(1) + b64[x].sum(1) + float(b0)
        out_t = 0.5 * (Sa * Sa + (E * E).sum(1)).sum(1) + b64[x].abs().sum(1) + abs(float(b0))
        g, g_t = (out - ys) * ws, (out_t + ys.abs()) * ws
        r["out"][s0:s0 + chunk], r["out_t"][s0:s0 + chunk] = out, out_t
        r["loss"] += float((0.5 * ws * (out - ys) ** 2).sum())
        idx = x.reshape(-1)
        r["V"].index_add_(0, idx, (g[:, None, None] * (S[:, None, :] - E)).reshape(-1, K))
        r["V_t"].index_add_(0, idx, (g_t[:, None, None] * (Sa[:, None, :] + Ea)).reshape(-1, K))
        r["b"].index_add_(0, idx, g.repeat_interleave(F))
        r["b_t"].index_add_(0, idx, g_t.repeat_interleave(F))
        r["b0"] += float(g.sum())
        r["b0_t"] += float(g_t.sum())
    r["touched"] = np.unique(X.numpy())
    return r


def hhfm_reference(V, Pos, Fea, Tim, Neg, pools=(0, 0, 0), weight=None, chunk=None):
    """HHFM training graph (OurModel7.py:105-184) in float64: pooling of the context and time groups (0 = sum, 1 = max,
    ties share the gradient equally), Pooling1F over [user, C, T] (sum or max), positive and negative scores, the max
    negative with ties split equally, -log sigmoid(pos - max).  Returns loss, pos, neg, dV, dV's sum of |terms| and the
    touched rows (user, item, pooled rows, the tied max negatives).  weight as in fm_reference."""
    M, K = V.shape
    B = Pos.shape[0]
    groups = [(g, m) for g, m in ((Fea, pools[0]), (Tim, pools[1])) if g is not None and g.shape[1] > 0]
    W = 2 + sum(g.shape[1] for g, _ in groups) + Neg.shape[1]
    chunk = chunk or max(64, (1 << 22) // (W * K))
    V64 = _t(V)
    Va = V64.abs()
    w = torch.ones(B, dtype=torch.float64) if weight is None else _t(weight)
    r = dict(loss=0.0, pos=np.zeros(B), neg=np.zeros(Neg.shape), V=torch.zeros(M, K, dtype=torch.float64),
             V_t=torch.zeros(M, K, dtype=torch.float64))
    touched = [np.unique(Pos)] + [np.unique(g) for g, _ in groups]
    for s0 in range(0, B, chunk):
        sl = slice(s0, s0 + chunk)
        pu, pi, ng = _t(Pos[sl, 0], torch.int64), _t(Pos[sl, 1], torch.int64), _t(Neg[sl], torch.int64)
        ws = w[sl]
        parts, parts_t, routes = [V64[pu]], [Va[pu]], []
        for g, mode in groups:
            ids = _t(g[sl], torch.int64)
            E = V64[ids]
            if mode == 0:
                P, Pt, rw = E.sum(1), E.abs().sum(1), torch.ones_like(E)
            else:
                P = E.max(1).values
                eq = (E == P[:, None, :]).double()
                rw, Pt = eq / eq.sum(1, keepdim=True), P.abs()
            parts.append(P); parts_t.append(Pt); routes.append((ids, rw))
        stack = torch.stack(parts, 1)
        if pools[2] == 0 or len(parts) == 1:
            hyb, sw = stack.sum(1), torch.ones_like(stack)
        else:
            hyb = stack.max(1).values
            eq = (stack == hyb[:, None, :]).double()
            sw = eq / eq.sum(1, keepdim=True)
        hyb_t = torch.stack(parts_t, 1).sum(1)
        Ei, En = V64[pi], V64[ng]
        pos = (hyb * Ei).sum(1)
        neg = (hyb[:, None, :] * En).sum(2)
        m = neg.max(1).values
        tie = (neg == m[:, None]).double()
        nt = tie.sum(1)
        x = pos - m
        sg = torch.sigmoid(x)
        r["loss"] += float((ws * torch.nn.functional.softplus(-x)).sum())
        r["pos"][sl], r["neg"][sl] = pos.numpy(), neg.numpy()
        gp, gpt = (sg - 1) * ws, (1 + sg) * ws
        cn, cnt = (-gp / nt)[:, None] * tie, (gpt / nt)[:, None] * tie
        for acc, hy, a, c, Vi, Vn in ((r["V"], hyb, gp, cn, Ei, En), (r["V_t"], hyb_t, gpt, cnt, Ei.abs(), En.abs())):
            acc.index_add_(0, pi, a[:, None] * hy)
            acc.index_add_(0, ng.reshape(-1), (c[:, :, None] * hy[:, None, :]).reshape(-1, K))
            dh = a[:, None] * Vi + (c[:, :, None] * Vn).sum(1)
            acc.index_add_(0, pu, dh * sw[:, 0])
            for q, (ids, rw) in enumerate(routes):
                acc.index_add_(0, ids.reshape(-1), ((dh * sw[:, 1 + q])[:, None, :] * rw).reshape(-1, K))
        touched.append(Neg[sl][tie.numpy() > 0])
    r["touched"] = np.unique(np.concatenate([t.reshape(-1) for t in touched]))
    return r


def close64(got, ref, terms, what):
    """|got - ref| <= 1e-5 (|ref| + sum |terms|), element-wise."""
    got = np.asarray(got, np.float64).reshape(-1)
    ref = np.asarray(ref, np.float64).reshape(-1)
    tol = 1e-5 * (np.abs(ref) + np.asarray(terms, np.float64).reshape(-1))
    err = np.abs(got - ref)
    bad = err > tol
    assert not bad.any(), "%s: %d/%d elements off, worst err %.3e (tol %.3e) at %d" % (
        what, int(bad.sum()), err.size, float(err.max()), float(tol[np.argmax(err - tol)]), int(np.argmax(err - tol)))


def close_loss(got, ref, what="loss"):
    assert abs(got - ref) <= 1e-5 * abs(ref), "%s: %.9g vs %.9g" % (what, got, ref)


def check_fm(got, ref):
    close64(got["out"], ref["out"], ref["out_t"], "out")
    close_loss(got["loss"], ref["loss"])
    close64(got["gV"], ref["V"], ref["V_t"], "gV")
    close64(got["gb"], ref["b"], ref["b_t"], "gbias")
    close64(got["gb0"], ref["b0"], ref["b0_t"], "gb0")


def check_hhfm(got, ref):
    close_loss(got["loss"], ref["loss"])
    close64(got["gV"], ref["V"], ref["V_t"], "gV")
    if "pos" in got:             # scores are exact on the quantised tables
        close64(got["pos"], ref["pos"], 0.0, "pos")
        close64(got["neg"], ref["neg"], 0.0, "neg")


# ----------------------------------------------------------------------------------------------------
# inputs
# ----------------------------------------------------------------------------------------------------
def qtable(rng, M, K):
    """Multiples of 2^-7 in [-1/8, 1/8]: sums of up to 12 rows and their dot products over K <= 512 are exact in fp32."""
    return (rng.integers(-16, 17, (M, K)) * (1.0 / 128)).astype(np.float32)


def fm_inputs(rng, B, F, K, n_hot, M=None):
    """ids: hot rows [0, n_hot) in field 1, every other field drawn from a range sized for about 50 contributions per row;
    every other sample repeats its field 0 in its last field."""
    M = M or n_hot + max(256, B * F // 50)
    X = rng.integers(n_hot, M, (B, F))
    if n_hot and F > 1:
        X[:, 1] = rng.integers(0, n_hot, B)
    if F > 1:
        X[::2, F - 1] = X[::2, 0]
    V = rng.normal(0, 0.1, (M, K)).astype(np.float32)
    b = rng.normal(0, 0.1, (M, 1)).astype(np.float32)
    Y = rng.choice([1.0, 0.0], (B, 1)).astype(np.float32)
    return X, Y, V, b, np.float32(-0.1)


def pr_inputs(rng, B, K, nc, nt, ng, groups=None, M=None):
    """Records of the HHFM pass.  Users from 6 hot rows; items and negatives from a range sized for about 25 positives per
    row; every 9th sample has all negatives equal (an ng-way tie) and negative 5 repeats negative 4.  Pooled columns:
    grouped ones from small disjoint ranges [lo, lo + card) with 3 % of the samples one past the range (the fallback of
    the pooled-group kernel), ungrouped ones from a wide range.  Returns V, Pos, Fea, Tim, Neg, (lo, card) of each column."""
    n_pool = nc + nt
    n_items = max(400, B // 12)
    lo, card = [0] * n_pool, [0] * n_pool
    base = 6 + n_items
    for c in range(n_pool):
        if groups is not None and groups[c] >= 0:
            lo[c], card[c] = base, 2 + (c % 2)
            base += card[c] + 1                      # a spare row after each range: the out-of-range id
    wide = max(300, B * max(n_pool, 1) // 50)
    M = max(M or 0, base + wide)
    Pos = np.stack([rng.integers(0, 6, B), rng.integers(6, 6 + n_items, B)], axis=1)
    Neg = rng.integers(6, 6 + n_items, (B, ng))
    Neg[::9] = Neg[::9, :1]
    if ng > 5:
        Neg[:, 5] = Neg[:, 4]
    P = np.zeros((B, n_pool), np.int64)
    for c in range(n_pool):
        if card[c]:
            P[:, c] = lo[c] + rng.integers(0, card[c], B)
            P[rng.random(B) < 0.03, c] = lo[c] + card[c]
        else:
            P[:, c] = rng.integers(base, base + wide, B)
    if n_pool > 1 and groups is None:
        P[::3, 1] = P[::3, 0]                      # the same token in two pooled columns
    Fea = P[:, :nc] if nc else None
    Tim = P[:, nc:] if nt else None
    return qtable(rng, M, K), Pos, Fea, Tim, Neg, (lo, card)


# ----------------------------------------------------------------------------------------------------
# CPU tests
# ----------------------------------------------------------------------------------------------------
def test_ledger_matches_the_library():
    """INSTANCES names exactly the training-kernel instances compiled into the library."""
    from hhfm_b200 import build
    compiled = library_instances(build.build())
    assert compiled, "no training kernels found in the library"
    missing = sorted(compiled - set(INSTANCES))
    stale = sorted(set(INSTANCES) - compiled)
    assert not missing and not stale, "compiled but without a case: %s; a case but not compiled: %s" % (missing, stale)


def test_name_normalisation():
    assert normalise("void hhfm::fm_kernel<(int)16, (int)1, (int)1, (bool)0>(hhfm::FmArgs)") == "fm_kernel<16,1,1,false>"
    assert normalise("void hhfm::pairrank_kernel<8, 1, 1, true>(hhfm::PrArgs)") == "pairrank_kernel<8,1,1,true>"
    assert normalise("void hhfm::afm_kernel<(int)1, (int)1, (int)2, (bool)0, (bool)0>(hhfm::AfmArgs)") is None
    assert normalise("void hhfm::pairrank_sum_train_kernel<16, 8, 10, 2>(hhfm::PrArgs, hhfm::PoolGroups)") == \
        "pairrank_sum_train_kernel<16,8,10,2>"
    assert normalise("hhfm::pairrank_sum_train_staged_kernel<(int)2, (int)10>") == "pairrank_sum_train_staged_kernel<2,10>"


def test_float64_reference_matches_the_oracle():
    """The float64 restatements agree with the fp32 oracle (oracle/hhfm_oracle.py) on small inputs."""
    from conftest import assert_close
    from oracle import hhfm_oracle as O
    rng = np.random.default_rng(0)
    X, Y, V, b, b0 = fm_inputs(rng, 300, 6, 16, 4)
    loss, out, dV, db, db0, touched = O.fm_loss_grads(X, Y, V, b, b0, lamda=0.0)
    r = fm_reference(X, Y, V, b, b0, chunk=100)
    assert_close(r["out"].numpy(), out, what="out"); assert_close(r["loss"], loss, what="loss")
    assert_close(r["V"].numpy(), dV, what="dV"); assert_close(r["b"].numpy(), db.reshape(-1), what="db")
    assert_close(r["b0"], db0, what="db0"); assert (r["touched"] == touched).all()
    for pools in ((0, 0, 0), (1, 1, 1), (1, 0, 1), (0, 1, 0)):
        V, Pos, Fea, Tim, Neg, _ = pr_inputs(rng, 200, 16, 3, 2, 7)
        Fea[:, 1] = Fea[:, 0]
        loss, pos, neg, dV = O.pairrank_loss_grads(V, Pos, Neg, Fea, Tim, pools, 0.0)
        r = hhfm_reference(V, Pos, Fea, Tim, Neg, pools, chunk=70)
        assert_close(r["loss"], loss, what="loss %s" % (pools,)); assert_close(r["pos"], pos, what="pos")
        assert_close(r["neg"], neg, what="neg"); assert_close(r["V"].numpy(), dV, what="dV %s" % (pools,))


# ----------------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------------
@pytest.fixture
def kernels_module():
    import test_gpu_kernels as T
    yield T
    torch.cuda.synchronize()
    T._KEEP.clear()


def _fm_case(cuda, T, case, B, F, K, seed):
    rng = np.random.default_rng(seed)
    X, Y, V, b, b0 = fm_inputs(rng, B, F, K, case["hot"], case["M"])
    hot = np.arange(case["hot"]) if case["hot"] else None
    names, got = launched_kernels(lambda: T._fm_train_call(cuda, X, Y, V, b, b0, hot_rows=hot))
    return names, got, (X, Y, V, b, b0)


def _pr_entry(cuda, T, V, Pos, Fea, Tim, Neg, track, hot, groups, lo, card):
    """hhfm_pairrank_fwd_bwd without scores (sum pooling everywhere), touched rows when `track`, a pooled-group plan when
    `groups`."""
    from hhfm_b200 import _lib
    from hhfm_b200.engine import NO_HOT, HotRows, PoolGroups, cur_stream, ptr
    rec, stride = T._records(Pos, Fea, Tim, Neg)
    M, K = V.shape
    B = rec.shape[0]
    nc = 0 if Fea is None else Fea.shape[1]
    nt = 0 if Tim is None else Tim.shape[1]
    tV = T.dev(V, cuda)
    pg = PoolGroups(tV, nc + nt, stride, lo, card, groups) if groups is not None else None
    h = HotRows(np.arange(6), M, K, cuda, n_rep=8) if hot else None
    gV = torch.zeros(M, K, device=cuda)
    lp = torch.zeros(_lib.partials_len(), device=cuda)
    loss = torch.zeros(1, device=cuda)
    stamp = torch.zeros(M, dtype=torch.int32, device=cuda)
    rows = torch.full((M,), -1, dtype=torch.int32, device=cuda)
    cnt = torch.zeros(1, dtype=torch.int32, device=cuda)
    _lib.call("hhfm_pairrank_fwd_bwd", ptr(T.dev(rec, cuda)), B, stride, nc, nt, Neg.shape[1], 0, 0, 0, ptr(tV), M, K, None, None,
              ptr(gV), ptr(lp), ptr(stamp) if track else None, 7, ptr(rows) if track else None, ptr(cnt) if track else None,
              *(h.args() if h else NO_HOT), 0, cur_stream())
    if h:
        h.fold(gV, None)
    _lib.call("hhfm_loss_finalize", ptr(lp), None, 0.0, ptr(loss), cur_stream())
    out = dict(loss=float(loss.item()), gV=gV.cpu().numpy())
    if track:
        out["touched"] = np.sort(rows[:int(cnt.item())].cpu().numpy())
    if pg is not None:
        out["G_max"] = float(pg.tables()[1].abs().max())
        pg._fin()
    return out


def _pr_case(cuda, T, name, case, seed, n_sm):
    rng = np.random.default_rng(seed)
    B = steady_batch(n_sm, staged_warps(name)) if case["B"] == STEADY else case["B"]
    pools = case.get("pools", (0, 0, 0))
    V, Pos, Fea, Tim, Neg, (lo, card) = pr_inputs(rng, B, case["K"], case["nc"], case["nt"], case["ng"], case.get("groups"),
                                                  case.get("M"))
    if case["kind"] == "prg":
        if Fea is not None and Fea.shape[1] > 1:
            Fea[::2, 1] = Fea[::2, 0]                                  # exact max-pool ties
        names, got = launched_kernels(lambda: T._pairrank_train(cuda, V, Pos, Fea, Tim, Neg, pools))
    else:
        track = name.startswith("pairrank_sum_train_staged_kernel")
        names, got = launched_kernels(lambda: _pr_entry(cuda, T, V, Pos, Fea, Tim, Neg, track, case["hot"], case["groups"],
                                                        lo, card))
    return names, got, (V, Pos, Fea, Tim, Neg, pools)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(INSTANCES))
def test_instance_launches_and_matches_reference(cuda, kernels_module, monkeypatch, name):
    case = INSTANCES[name]
    for k in ("HHFM_FM_STAGED", "HHFM_FM_STAGES", "HHFM_FM_WARPS", "HHFM_PR_STAGED", "HHFM_PR_STAGES", "HHFM_PR_WARPS",
              "HHFM_NO_FAST", "HHFM_POOL_GROUPS"):
        monkeypatch.delenv(k, raising=False)
    for k, v in case["env"].items():
        monkeypatch.setenv(k, v)
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    seed = sum(map(ord, name))
    if case["kind"] == "fm":
        for i, (B, F, K) in enumerate(case["shapes"]):
            if B == STEADY:
                B = steady_batch(n_sm, staged_warps(name))
            names, got, inputs = _fm_case(cuda, kernels_module, case, B, F, K, seed + i)
            assert names == {name}, "B=%d F=%d K=%d launched %s" % (B, F, K, sorted(names))
            ref = fm_reference(*inputs)
            check_fm(got, ref)
            assert np.array_equal(got["touched"], ref["touched"]), "touched rows (B=%d F=%d K=%d)" % (B, F, K)
    else:
        names, got, inputs = _pr_case(cuda, kernels_module, name, case, seed, n_sm)
        assert names == {name}, "launched %s" % sorted(names)
        ref = hhfm_reference(*inputs)
        check_hhfm(got, ref)
        if "touched" in got:
            assert np.array_equal(got["touched"], ref["touched"]), "touched rows: %d listed, %d expected" % (
                len(got["touched"]), len(ref["touched"]))
        if "G_max" in got:
            assert got["G_max"] == 0.0, "the group gradient table must be clear after the pass"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fm_train_fixed_kernel<16,12>", "fm_train_staged_kernel<2,16>",
                                  "pairrank_sum_train_kernel<16,8,10,3>", "pairrank_sum_train_staged_kernel<3,9>"])
@pytest.mark.parametrize("change", [0.0, 2.0])
def test_reference_sees_one_sample(cuda, kernels_module, monkeypatch, name, change):
    """The gradient comparison fails against a reference with one sample left out (weight 0) or counted twice (weight 2).
    (The loss, a sum over up to 6e4 samples held to 1e-5 relative, cannot see every single sample.)"""
    case = INSTANCES[name]
    for k, v in case["env"].items():
        monkeypatch.setenv(k, v)
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    seed = sum(map(ord, name))
    if case["kind"] == "fm":
        B, F, K = case["shapes"][0]
        B = steady_batch(n_sm, staged_warps(name)) if B == STEADY else B
        _, got, inputs = _fm_case(cuda, kernels_module, case, B, F, K, seed)
        check_fm(got, fm_reference(*inputs))
        reference = fm_reference
    else:
        _, got, inputs = _pr_case(cuda, kernels_module, name, case, seed, n_sm)
        check_hhfm(got, hhfm_reference(*inputs))
        B = inputs[1].shape[0]
        reference = hhfm_reference
    w = np.ones(B)
    w[B // 2] = change
    ref = reference(*inputs, weight=w)
    with pytest.raises(AssertionError):
        close64(got["gV"], ref["V"], ref["V_t"], "gV")


# ----------------------------------------------------------------------------------------------------
# touched-row compaction through hhfm_mark_rows
# ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("tail", [0, 1, 2, 3])
def test_mark_rows_compacts_every_marked_row(cuda, aligned, tail):
    """M >= 2.5 rounds of touched_compact_kernel (sm_count x 8 CTAs x 256 threads x 4 rows per round) with M % 4 = tail;
    a stamp array that starts one element into its buffer selects touched_compact_scalar_kernel.  Ids include 0, M-1,
    M-2, M-3, padding -1 and duplicates; the stamp array holds stale stamps (stamp - 1, stamp + 1) in other rows."""
    from hhfm_b200 import _lib
    from hhfm_b200.engine import cur_stream, ptr
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    per_round = n_sm * 8 * 256 * 4
    M = (5 * per_round // 2) // 4 * 4 + 4 + tail
    rng = np.random.default_rng(M)
    stamp = 77
    ids = np.concatenate([[0, M - 1, M - 2, M - 3, -1, 0, M - 1], rng.integers(0, M, 200_000), np.full(1000, -1),
                          rng.integers(0, M, 5000).repeat(3)]).astype(np.int32)
    rng.shuffle(ids)
    init = rng.choice(np.array([0, stamp - 1, stamp + 1], np.int32), M)
    buf = torch.zeros(M + 4, dtype=torch.int32, device=cuda)
    st_arr = buf[:M] if aligned else buf[1:M + 1]
    assert (st_arr.data_ptr() % 16 == 0) == aligned
    st_arr.copy_(torch.from_numpy(init))
    rows = torch.full((M,), -7, dtype=torch.int32, device=cuda)
    cnt = torch.zeros(1, dtype=torch.int32, device=cuda)
    ids_dev = torch.from_numpy(ids).to(cuda)
    _lib.call("hhfm_mark_rows", ptr(ids_dev), ids.size, ptr(st_arr), stamp, M, ptr(rows), ptr(cnt), cur_stream())
    want = np.unique(ids[ids >= 0])
    n = int(cnt.item())
    assert n == want.size
    got = rows[:n].cpu().numpy()
    assert np.array_equal(np.sort(got), want)
    assert (rows[n:].cpu().numpy() == -7).all(), "nothing is written past the count"
    after = st_arr.cpu().numpy()
    assert (after[want] == stamp).all() and np.array_equal(np.delete(after, want), np.delete(init, want))
