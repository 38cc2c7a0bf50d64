"""The bounded sweep (csrc/bounded.cuh) at its window, candidate and batch-size edges, against an FP64 oracle.

A ragged batch holds pairs in all three prefix-window regimes of bounded_prefix_groups (the whole pair is the prefix;
stage A already covers the prefix, so stage B has nothing to do; stage B extends stage A), pairs with H = 0, 1 and H on
both sides of 256 and 512, a pair whose every count is 0, NaN rows, runs of duplicated hypotheses that put the K-th
largest prefix count inside a tie group, and two planted pairs where the first maximum is a hypothesis that only stage B
can keep alive.  A second batch holds more than 256 tiny pairs in one pass.

The oracle scores the call's own hypotheses (F_all of a bounded call) with oracle.f_path in FP64, so the comparison
isolates the sweep's selection logic from the 8-point solver: winner, count and mask must equal the oracle's, and F must
equal the full sweep's (option 12 = 0) bit for bit, for every combination of scoring mode, tie rule, prefix stage
(options 15 / 16), candidate count (option 14) and pass schedule (options 6 / 10)."""
import numpy as np
import pytest

from oracle import f_path as orc

pytestmark = pytest.mark.gpu
SEED = 20261022
THR = 1.5
KSUB = 8
RHO, RHO0 = 450, 380                         # defaults of options 13 and 16
DEFAULTS = {2: 0, 6: 0, 10: 1, 12: 1, 14: 512, 15: 1, 16: RHO0}
PREFIX = {"exact": (0, RHO0), "exact_rho0_1000": (0, 1000), "one_step": (1, 1000), "two_step": (1, RHO0)}


# ---- the prefix windows: a restatement of bounded_prefix_groups and f_plan (csrc/plan.cuh) ----
def prefix_groups(G, rho_milli):
    g = (G * rho_milli + 999) // 1000
    return min(G, (g + 31) // 32 * 32)


def windows(n, bound_prefix=True, rho0=RHO0):
    """(G, gA0, gA): groups of the pair, end of stage A, end of the prefix."""
    G = (n + KSUB - 1) // KSUB
    gA = prefix_groups(G, RHO)
    gA0 = min(gA, prefix_groups(G, rho0)) if bound_prefix else gA
    return G, gA0, gA


def regime(n):
    G, gA0, gA = windows(n)
    return "gA == G" if gA == G else ("gA0 == gA < G" if gA0 == gA else "gA0 < gA < G")


# ---- batches ----
class Batch:
    def __init__(self, pts, idx, names):
        self.pts, self.idx, self.names = pts, idx, names
        self.N = [len(p) for p in pts]
        self.H = [len(i) for i in idx]
        self.P = len(pts)
        self._oracle = {}

    def split(self, p):
        return self.pts[p][:, :2].T.copy(), self.pts[p][:, 2:].T.copy()


def _rot(t):
    return np.array([[np.cos(t), -np.sin(t)], [np.sin(t), np.cos(t)]])


def planted_pair(rg, seed, a_c, s_w):
    """600 correspondences, exact for one of two geometries w and c (image 2 of c is that of w turned by 0.02 rad), with
    k0 = 256 (end of stage A) and k = 512 (end of the prefix).  Hypothesis 0 is an exact sample of w, hypothesis 1 one of
    c, the other six are degenerate.  Every distance to w or c is below 1 px or above 2.5 px, so the bound-only counts of
    both equal their exact counts.  Points [0, 256) hold a_c outliers of w (inliers of c), points [512, 600) s_w outliers
    of c (inliers of w), all others are inliers of both: full(w) = 600 - a_c, full(c) = 600 - s_w, and c wins stage A.
    With K = 1, c is the only candidate, L = full(c), and w survives only through stage B (its stage-A count plus the 88
    points after the prefix stays below L); with a_c == s_w it then ties L exactly."""
    syn = rg.synth
    Ps = syn.dino()["Ps"]
    rng = np.random.default_rng(seed)
    X = rng.uniform(syn.DINO_BBOX[:, 0], syn.DINO_BBOX[:, 1], size=(4000, 3))
    x = syn.project(Ps[0], X)
    y = syn.project(Ps[2], X)
    ctr = y.mean(axis=0)
    yc = (y - ctr) @ _rot(0.02).T + ctr
    w_rows = np.hstack([x[:2000], y[:2000]])                  # exact for w
    c_rows = np.hstack([x[2000:], yc[2000:]])                 # exact for c
    Fw = orc.fmatrix_stls(w_rows[:40, :2].T, w_rows[:40, 2:].T)
    Fc = orc.fmatrix_stls(c_rows[:40, :2].T, c_rows[:40, 2:].T)
    d_c = orc.distance(Fc, w_rows[:, :2].T, w_rows[:, 2:].T)
    d_w = orc.distance(Fw, c_rows[:, :2].T, c_rows[:, 2:].T)
    w_both, w_only = w_rows[d_c < 1.0], w_rows[d_c > 2.5]
    c_both, c_only = c_rows[d_w < 1.0], c_rows[d_w > 2.5]
    both = np.empty((600, 4))
    both[0::2], both[1::2] = w_both[:300], c_both[:300]
    A = np.vstack([c_only[:a_c], both[:256 - a_c]])
    B = both[256 - a_c:512 - a_c]                              # B[0::2] are w's rows, B[1::2] c's (256 - a_c is even)
    S = np.vstack([w_only[:s_w], both[512 - a_c:600 - a_c - s_w]])
    A, S = A[rng.permutation(len(A))], S[rng.permutation(len(S))]
    pts = np.ascontiguousarray(np.vstack([A, B, S]))
    assert pts.shape == (600, 4) and (256 - a_c) % 2 == 0
    w_sample = 256 + 2 * np.arange(8) * 15                     # spread over B
    idx = np.vstack([w_sample, w_sample + 1] + [np.full(8, 7 * j + 3) for j in range(6)]).astype(np.int32)
    return pts, idx


def _triples(rg, n, h, seed):
    """h hypotheses, each distinct sample three times in a row: every group of equal counts has a multiple of 3 members."""
    return np.ascontiguousarray(np.repeat(rg.sampling.fast(n, (h + 2) // 3, 8, seed=seed), 3, axis=0)[:h])


def _ragged(rg):
    two_view = rg.synth.two_view
    fast = rg.sampling.fast
    pts, idx, names = [], [], []

    def add(name, p, i):
        names.append(name)
        pts.append(np.ascontiguousarray(p))
        idx.append(np.ascontiguousarray(i, dtype=np.int32))

    add("8193 x 4097", two_view(8193, seed=101)[0], fast(8193, 4097, 8, seed=1))
    add("8 x 1", two_view(8, seed=102, outlier_frac=0.0)[0], fast(8, 1, 8, seed=2))
    add("255 x 0", two_view(255, seed=103)[0], np.zeros((0, 8), np.int32))
    add("2049 x 999 triples", two_view(2049, seed=104)[0], _triples(rg, 2049, 999, 4))
    add("9 x 255", two_view(9, seed=105, outlier_frac=0.0)[0], fast(9, 255, 8, seed=5))
    add("256 x 513 clean", two_view(256, seed=106, outlier_frac=0.0)[0], fast(256, 513, 8, seed=6))
    add("257 x 511 all NaN", np.full((257, 4), np.nan), fast(257, 511, 8, seed=7))
    p = two_view(400, seed=108)[0]
    p[np.random.default_rng(8).choice(400, 40, replace=False)] = np.nan
    add("400 x 512 NaN rows", p, fast(400, 512, 8, seed=8))
    add("568 x 257 triples", two_view(568, seed=109)[0], _triples(rg, 568, 257, 9))
    add("569 x 256 all outliers", two_view(569, seed=110, outlier_frac=1.0)[0], fast(569, 256, 8, seed=10))
    add("600 x 8 planted tie", *planted_pair(rg, 111, 20, 20))
    add("600 x 8 planted gap", *planted_pair(rg, 112, 10, 20))
    return Batch(pts, idx, names)


TIE_PAIR, PLANTED = 3, (10, 11)
# evaluations per pass (option 6): passes [0], [1, 2], [3], [4 .. 7], [8 .. 11] — a large pass ahead of small ones, so
# the workspace sets are reused by passes of other shapes
PASS_EVALS = 600_000


@pytest.fixture(scope="module")
def rt(rg):
    return rg.runtime


@pytest.fixture(scope="module")
def ragged(rg):
    return _ragged(rg)


@pytest.fixture(scope="module")
def tiny(rg):
    """320 pairs of 16 .. 300 correspondences and 8 .. 600 hypotheses (every 40th without any), 0 .. 100 % outliers."""
    rng = np.random.default_rng(SEED)
    pts, idx, names = [], [], []
    for p in range(320):
        n, h = int(rng.integers(16, 301)), int(rng.integers(8, 601))
        h = 0 if p % 40 == 17 else h
        pts.append(rg.synth.two_view(n, seed=5000 + p, outlier_frac=(0.0, 0.3, 0.6, 1.0)[p % 4])[0])
        idx.append(rg.sampling.fast(n, h, 8, seed=p) if h else np.zeros((0, 8), np.int32))
        names.append(f"tiny {p}")
    return Batch(pts, idx, names)


def _call(rt, batch, mode, tie_mode, opts, **kw):
    """One host-entry call with the options `opts` set; every option is restored to its default afterwards."""
    try:
        for k, v in opts.items():
            rt.set_option(k, v)
        r = rt.f_ransac_batched(batch.pts, batch.idx, thr=THR, mode=mode, tie_mode=tie_mode, **kw)
        return r, rt.bounded_stats(), rt.last_stats()
    finally:
        for k in opts:
            rt.set_option(k, DEFAULTS[k])


def oracle(rt, batch, mode):
    """Per tie rule the expected winner, count and mask of every pair: FP64 counts of the hypotheses the bounded sweep
    itself solved (want_F_all keeps the bounded path), first maximum (tie_mode 0) or the reference's rule (tie_mode 1)."""
    if mode in batch._oracle:
        return batch._oracle[mode]
    r, s, _ = _call(rt, batch, mode, 0, {2: 1}, want_F_all=True)
    assert s["K"] == DEFAULTS[14]
    F_all = r["F_all"]
    out = {"F_all": F_all, "counts": []}
    for tie_mode in (0, 1):
        out[tie_mode] = []
    for p in range(batch.P):
        p1, p2 = batch.split(p)
        counts = orc.score_hypotheses(F_all[p], p1, p2, THR, mode)
        out["counts"].append(counts)
        for tie_mode in (0, 1):
            if tie_mode == 0:
                best = orc.select_first_max(counts)
            else:
                best = orc.select_reference_rule(counts, F_all[p], p1, p2, mode)
            mask = np.zeros(batch.N[p], np.uint8)
            if best >= 0:
                mask[orc.inliers(F_all[p][best], p1, p2, THR, mode)] = 1
            out[tie_mode].append((best, int(counts.max()) if len(counts) else 0, mask))
    batch._oracle[mode] = out
    return out


def _check(batch, r, ref, tie_mode, full, what):
    for p in range(batch.P):
        best, count, mask = ref[tie_mode][p]
        where = (what, batch.names[p])
        assert int(r["best_idx"][p]) == best, where
        assert int(r["best_count"][p]) == count, where
        assert np.array_equal(r["mask"][p], mask), where
        if best >= 0:
            assert np.array_equal(r["F"][p].view(np.uint64), ref["F_all"][p][best].view(np.uint64)), where
    if full is not None:
        assert np.array_equal(r["F"].view(np.uint64), full["F"].view(np.uint64)), what


def _check_stats(batch, s, K, bound_prefix, rho0):
    """Statistics of a bounded call: the evaluations split into bound-only and guarded ones, at most the hypotheses
    beyond K per pair left unscored, at most every pair fallen back; stage A's bound-only evaluations are known."""
    assert s["K"] == K
    assert s["bound_evals"] + s["guarded_evals"] == s["evals"]
    assert 0 <= s["not_fully_scored"] <= sum(max(0, h - K) for h in batch.H)
    assert 0 <= s["fallback_pairs"] <= batch.P
    if K >= max(batch.H):                  # every hypothesis is a candidate: nothing to prune, nothing to fall back
        assert s["not_fully_scored"] == 0 and s["fallback_pairs"] == 0
    stage_a = sum(min(n, windows(n, bound_prefix, rho0)[1] * KSUB) * h for n, h in zip(batch.N, batch.H))
    prefix = sum(min(n, windows(n)[2] * KSUB) * h for n, h in zip(batch.N, batch.H))
    if not bound_prefix:
        assert s["bound_evals"] == 0
    else:
        assert stage_a <= s["bound_evals"] <= prefix
        if rho0 >= RHO:
            assert s["bound_evals"] == stage_a


def _prefix_rows(batch, F_all, p):
    """(H, N) FP64 inlier decisions (mode 0) of the pair's hypotheses."""
    p1, p2 = batch.split(p)
    return np.array([orc.distance(F, p1, p2) < THR for F in F_all[p]], dtype=bool).reshape(len(F_all[p]), -1)


def test_batch_reaches_every_window_regime(rt, ragged):
    """The ragged batch really holds pairs of all three window regimes under the default rho / rho0, H on both sides of
    the default K, H = 0 between other pairs, a pair with no inlier anywhere, and tie groups cut by K = 1, 7 and 512."""
    seen = {}
    for n, h, name in zip(ragged.N, ragged.H, ragged.names):
        G, gA0, gA = windows(n)
        seen.setdefault(regime(n), []).append(name)
        print(f"{name:>24}: G = {G:5d}, gA0 = {gA0:4d}, gA = {gA:4d}  ->  {regime(n)}")
    assert set(seen) == {"gA == G", "gA0 == gA < G", "gA0 < gA < G"}
    assert {0, 1, 255, 256, 257, 511, 512, 513, 4097} <= set(ragged.H)
    assert {8, 9, 255, 256, 257, 568, 569} <= set(ragged.N)
    assert ragged.H[2] == 0 and 0 < 2 < ragged.P - 1
    ref = oracle(rt, ragged, 0)
    assert ref[0][6][0] == -1 and ref[0][6][1] == 0                       # every count of the NaN pair is 0
    # the K-th largest exact prefix count lies inside a group of equal counts
    n = ragged.N[TIE_PAIR]
    k = min(n, windows(n, False)[2] * KSUB)
    pre = np.sort(_prefix_rows(ragged, ref["F_all"], TIE_PAIR)[:, :k].sum(axis=1))[::-1]
    for K in (1, 7, 512):
        assert pre[K - 1] == pre[K], K


def test_planted_pairs_need_stage_b(rt, ragged):
    """In the planted pairs the first maximum is hypothesis 0, which K = 1 leaves out of the candidates and the two-step
    prefix can only keep through stage B: below L after stage A plus the rest, reaching L (tie) or beyond it with its
    count over the whole prefix.  The bound-only counts equal these exact counts: no distance is near the threshold."""
    ref = oracle(rt, ragged, 0)
    for p, tie in zip(PLANTED, (True, False)):
        n = ragged.N[p]
        assert regime(n) == "gA0 < gA < G"
        _, gA0, gA = windows(n)
        k0, k = gA0 * KSUB, gA * KSUB
        p1, p2 = ragged.split(p)
        for F in ref["F_all"][p][:2]:
            d = orc.distance(F, p1, p2)
            assert np.all((d < 1.0) | (d > 2.5))
        rows = _prefix_rows(ragged, ref["F_all"], p)
        full, c0, ck = rows.sum(axis=1), rows[:, :k0].sum(axis=1), rows[:, :k].sum(axis=1)
        assert np.array_equal(full, ref["counts"][p])
        assert int(np.lexsort((np.arange(len(c0)), -c0))[0]) == 1           # the only candidate at K = 1
        L = int(full[1])
        assert c0[0] + (n - k) < L <= c0[0] + (n - k0)
        assert (ck[0] + (n - k) == L) if tie else (ck[0] + (n - k) > L)
        assert ref[0][p][0] == 0 and ref[1][p][0] == 0


@pytest.mark.parametrize("prefix", list(PREFIX))
@pytest.mark.parametrize("mode", [0, 1])
def test_ragged_batch_against_the_oracle(rt, ragged, mode, prefix):
    bound_prefix, rho0 = PREFIX[prefix]
    ref = oracle(rt, ragged, mode)
    for tie_mode in (0, 1):
        full, sf, _ = _call(rt, ragged, mode, tie_mode, {12: 0})
        assert sf["K"] == 0
        _check(ragged, full, ref, tie_mode, None, "full sweep")
        for K in (1, 7, 512, max(ragged.H)):
            for pipe in (0, 1):
                opts = {6: PASS_EVALS, 10: pipe, 14: K, 15: bound_prefix, 16: rho0}
                r, s, ls = _call(rt, ragged, mode, tie_mode, opts)
                _check(ragged, r, ref, tie_mode, full, (tie_mode, opts))
                _check_stats(ragged, s, K, bound_prefix, rho0)
                assert ls["passes"] == 5


@pytest.mark.parametrize("mode", [0, 1])
def test_many_tiny_pairs_in_one_pass(rt, tiny, mode):
    ref = oracle(rt, tiny, mode)
    full, _, _ = _call(rt, tiny, mode, 0, {2: 1, 12: 0})
    _check(tiny, full, ref, 0, None, "full sweep")
    for K in (1, 7, 512, max(tiny.H)):
        for bound_prefix in (0, 1):
            r, s, ls = _call(rt, tiny, mode, 0, {2: 1, 14: K, 15: bound_prefix})
            _check(tiny, r, ref, 0, full, (K, bound_prefix))
            _check_stats(tiny, s, K, bound_prefix, RHO0)
            assert ls["passes"] == 1


def test_device_entry_point(rt, rg, ragged):
    import torch
    ref = oracle(rt, ragged, 0)
    full, _, _ = _call(rt, ragged, 0, 0, {12: 0})
    dv = rg.device
    d_pts = torch.from_numpy(np.concatenate(ragged.pts)).cuda()
    d_idx = torch.from_numpy(np.concatenate(ragged.idx)).cuda()
    po, ho = dv.offsets(ragged.N), dv.offsets(ragged.H)
    o = dv.FOutputs(ragged.P, int(po[-1]), device=d_pts.device.index, want_mask=True)
    try:
        rt.set_option(6, PASS_EVALS)
        rt.set_option(14, 1)
        dv.f_ransac(d_pts, po, d_idx, ho, o, flags=rg.FLAG_BOUNDED)
        torch.cuda.synchronize()
        s = rt.bounded_stats()
    finally:
        rt.set_option(6, DEFAULTS[6])
        rt.set_option(14, DEFAULTS[14])
    mask = o.mask.cpu().numpy()
    r = {"best_idx": o.best_idx.cpu().numpy(), "best_count": o.best_count.cpu().numpy(),
         "F": o.F.cpu().numpy().reshape(-1, 3, 3), "mask": [mask[po[p]:po[p + 1]] for p in range(ragged.P)]}
    _check(ragged, r, ref, 0, full, "device entry point")
    _check_stats(ragged, s, 1, True, RHO0)
