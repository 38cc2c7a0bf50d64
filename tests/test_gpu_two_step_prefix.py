"""The two-step bound-only prefix of the bounded sweep (option 16 = rho0): stage A scores every hypothesis over the first
rho0 share, stage B extends only the hypotheses still alive (S) to the full prefix.  Winner index, count, F and inlier mask
must equal, bit for bit, those of the full sweep (option 12 = 0) for rho0 below, near and at rho (450), on the batches of
tests/test_gpu_bound_prefix.py.  Stage B's evaluations are checked against S recomputed on the host from stage A's counts."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
from bounded_sweep_model import prefix_points  # noqa: E402

pytestmark = pytest.mark.gpu
SEED = 20261018
RHO0 = (340, 380, 450)
DEFAULT_RHO0 = 380


@pytest.fixture(scope="module")
def rt(rg):
    return rg.runtime


def _config5(rg, P, N, first_pair=0, **kw):
    d, _ = rg.device.synth_two_view(P, N, first_pair=first_pair, seed_base=1000, **kw)
    a = d.cpu().numpy()
    return [np.ascontiguousarray(a[p]) for p in range(P)]


def _run(rt, bounded, rho0, pts, idx=None, **kw):
    rt.set_option(12, 1 if bounded else 0)
    rt.set_option(16, rho0)
    try:
        r = rt.f_ransac_batched(pts, idx, sample_seed=SEED, **kw)
        return r, rt.bounded_stats()
    finally:
        rt.set_option(12, 1)
        rt.set_option(16, DEFAULT_RHO0)


def _same(a, b):
    assert np.array_equal(a["best_idx"], b["best_idx"])
    assert np.array_equal(a["best_count"], b["best_count"])
    assert np.array_equal(a["F"].view(np.uint64), b["F"].view(np.uint64))
    for ma, mb in zip(a["mask"], b["mask"]):
        assert np.array_equal(ma, mb)


def _stage_a_evals(pts, H, rho0):
    return sum(prefix_points(len(p), min(rho0, 450) / 1000.0) * h for p, h in zip(pts, H))


def _check(rt, pts, idx=None, expect_fallback=None, n_hyp=None, **kw):
    """Every rho0 of RHO0 against the full sweep; returns the bounded statistics per rho0.  expect_fallback: the number of
    pairs that must fall back at every rho0."""
    H = [len(i) for i in idx] if idx is not None else ([n_hyp] * len(pts) if np.isscalar(n_hyp) else n_hyp)
    full, _ = _run(rt, False, DEFAULT_RHO0, pts, idx, n_hyp=n_hyp, **kw)
    out = {}
    for rho0 in RHO0:
        r, s = _run(rt, True, rho0, pts, idx, n_hyp=n_hyp, **kw)
        _same(full, r)
        assert s["K"] == 512 and s["bound_evals"] + s["guarded_evals"] == s["evals"]
        stage_b = s["bound_evals"] - _stage_a_evals(pts, H, rho0)
        assert stage_b >= 0
        if rho0 >= 450:
            assert stage_b == 0
        if expect_fallback is not None:
            assert s["fallback_pairs"] == expect_fallback
        out[rho0] = s
    return out


def test_multi_pass_config5_slice(rt, rg):
    P, N, H = 6, 50000, 8192
    pts = _config5(rg, P, N)
    rt.set_option(6, 2 * N * H)                             # three passes of two pairs: the pipelined three-set schedule
    try:
        st = _check(rt, pts, n_hyp=H)
    finally:
        rt.set_option(6, 0)
    assert rt.last_stats()["passes"] >= 3
    for rho0 in (DEFAULT_RHO0, 450):             # no fallback at the default: the candidates of stage A hold the winners
        assert st[rho0]["fallback_pairs"] == 0
        assert st[rho0]["not_fully_scored"] == P * (H - 512)
        assert st[rho0]["guarded_evals"] == P * 512 * N
    assert st[DEFAULT_RHO0]["bound_evals"] < st[450]["bound_evals"]


@pytest.mark.parametrize("order", ["inliers_first", "random"])
def test_point_orders(rt, rg, order):
    pts = _config5(rg, 4, 20000, first_pair=7)
    rng = np.random.default_rng(5)
    out = []
    for p in pts:
        perm = np.r_[np.arange(6000, 20000), np.arange(6000)] if order == "inliers_first" else rng.permutation(len(p))
        out.append(np.ascontiguousarray(p[perm]))
    _check(rt, out, n_hyp=4096)


def test_dino_pairs(rt, rg):
    pairs = [rg.synth.dino_noisy_pair(i, i + 1) for i in range(35)]
    pts = [np.ascontiguousarray(np.hstack([a, b])) for a, b in pairs]
    _check(rt, pts, n_hyp=2048)


def test_low_inlier_ratio_falls_back(rt, rg):
    """60 % outliers: no hypothesis can be pruned after stage A and every pair is certain to fall back, so stage B
    has nothing to do."""
    P, N, H = 3, 20000, 4096
    pts = _config5(rg, P, N, first_pair=20, outlier_frac=0.6)
    st = _check(rt, pts, n_hyp=H, expect_fallback=3)
    k0 = prefix_points(N, 0.34)
    assert st[340]["not_fully_scored"] == 0
    assert st[340]["bound_evals"] == P * H * k0


@pytest.mark.parametrize("tie_mode", [0, 1])
def test_exact_ties(rt, rg, tie_mode):
    pts = _config5(rg, 2, 20000, first_pair=30)
    idx = []
    for p in range(2):
        base = rg.philox.sample_indices(20000, 1024, 8, SEED, 30 + p)
        idx.append(np.ascontiguousarray(np.repeat(base, 2, axis=0).astype(np.int32)))    # every hypothesis twice
    _check(rt, pts, idx, tie_mode=tie_mode)


def test_sampson(rt, rg):
    _check(rt, _config5(rg, 3, 20000, first_pair=40), n_hyp=4096, mode=1)


@pytest.mark.parametrize("option,value", [(9, 8000), (8, 100)])
def test_wide_band_and_list_overflow(rt, rg, option, value):
    pts = _config5(rg, 2, 20000, first_pair=50)
    rt.set_option(option, value)
    try:
        _check(rt, pts, n_hyp=2048)
        if option == 8:
            assert rt.last_stats()["overflow"] > 0
    finally:
        rt.set_option(option, 1000 if option == 9 else 0)


def test_device_entry_point(rt, rg, torch):
    dv = rg.device
    P, N, H = 4, 20000, 4096
    d, _ = dv.synth_two_view(P, N, first_pair=70, seed_base=1000)
    po, ho = dv.offsets([N] * P), dv.offsets([H] * P)
    outs = []
    for flags, rho0 in [(0, DEFAULT_RHO0)] + [(rg.FLAG_BOUNDED, r) for r in RHO0]:
        rt.set_option(16, rho0)
        try:
            o = dv.FOutputs(P, P * N, device=d.device.index, want_mask=True)
            dv.f_ransac(d, po, None, ho, o, seed=SEED, first_pair=70, flags=flags)
            torch.cuda.synchronize()
        finally:
            rt.set_option(16, DEFAULT_RHO0)
        outs.append((o.best_idx.cpu().numpy(), o.best_count.cpu().numpy(), o.F.cpu().numpy(), o.mask.cpu().numpy()))
        st = rt.bounded_stats()
        assert st["K"] == (512 if flags else 0)
        if flags:
            assert st["bound_evals"] >= P * H * prefix_points(N, min(rho0, 450) / 1000.0)
    for other in outs[1:]:
        for a, b in zip(outs[0], other):
            assert np.array_equal(a, b)


def test_option_16_is_validated(rt):
    for bad in (0, 1001):
        with pytest.raises(ValueError, match="option 16"):
            rt.set_option(16, bad)


def _extremes_first(p):
    """The same correspondences with the ones on the bounding box moved to the front: every prefix that holds them has
    the pair's bounding box, hence its scoring frame."""
    ext = np.unique(np.r_[np.argmin(p, axis=0), np.argmax(p, axis=0)])
    rest = np.setdiff1d(np.arange(len(p)), ext)
    return np.ascontiguousarray(p[np.r_[ext, rest]])


def test_stage_b_matches_the_host(rt, rg):
    """Stage B's evaluation count equals sum_p |S_p| * (k - k0) over the pairs not certain to fall back, and the pairs that
    fall back are those where a member of S reaches L with its bound over the whole prefix, all recomputed on the host:
    stage A's and the prefix's bound counts (the bound-only scorer over the first k0 / k correspondences, in the pair's
    frame), the top K of stage A's, L from the exact full counts of the full sweep.  With a small K some pairs survive
    stage A uncertain and escape only once stage B's counts are added, which pins down bnd_check's add."""
    P, N, H = 3, 20000, 4096
    pts = [_extremes_first(p) for p in _config5(rg, P, N, first_pair=80)]
    full = rt.f_ransac_batched(pts, None, n_hyp=H, sample_seed=SEED, want_counts=True, want_F_all=True)
    k = prefix_points(N, 0.45)
    c_k = [rt.epi_score_count(pts[p][:k], full["F_all"][p], 1.5, score_path=2).astype(np.int64) for p in range(P)]
    escaped_after_b = 0
    for rho0, K in ((340, 512), (380, 512), (300, 8), (340, 8), (340, 64)):
        k0 = prefix_points(N, rho0 / 1000.0)
        expect_b, expect_fb = 0, 0
        for p in range(P):
            c0 = rt.epi_score_count(pts[p][:k0], full["F_all"][p], 1.5, score_path=2).astype(np.int64)
            cand = np.zeros(H, bool)
            cand[np.lexsort((np.arange(H), -c0))[:K]] = True
            L = int(full["counts"][p][cand].max())
            S = ~cand & (c0 + (N - k0) >= L)
            certain = bool(np.any(c0[S] + (N - k) >= L))        # (such a pair skips stage B)
            escapes = bool(np.any(c_k[p][S] + (N - k) >= L))
            expect_b += 0 if certain else int(S.sum()) * (k - k0)
            expect_fb += int(escapes)
            escaped_after_b += int(escapes and not certain)
        rt.set_option(14, K)
        try:
            r, s = _run(rt, True, rho0, pts, None, n_hyp=H)
        finally:
            rt.set_option(14, 512)
        _same(full, r)
        assert s["bound_evals"] - P * H * k0 == expect_b, (rho0, K)
        assert s["fallback_pairs"] == expect_fb, (rho0, K)
    assert escaped_after_b > 0


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch
