"""The bound-only prefix stage of the bounded sweep (option 15 = 1, EpiBoundPolicy) must leave every result of the sweep
unchanged: winner index, count, F and inlier mask equal, bit for bit, those of the exact prefix (option 15 = 0) and of the
full sweep (option 12 = 0) on the batches of tests/test_gpu_bounded_sweep.py.  Its counts are upper bounds of the exact
counts, checked here through the stage entry point on points at and around the threshold and in extreme frames."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
SEED = 20261018


@pytest.fixture(scope="module")
def rt(rg):
    return rg.runtime


def _config5(rg, P, N, first_pair=0, **kw):
    d, _ = rg.device.synth_two_view(P, N, first_pair=first_pair, seed_base=1000, **kw)
    a = d.cpu().numpy()
    return [np.ascontiguousarray(a[p]) for p in range(P)]


def _run(rt, bounded, bound_prefix, pts, idx=None, **kw):
    rt.set_option(12, 1 if bounded else 0)
    rt.set_option(15, 1 if bound_prefix else 0)
    try:
        r = rt.f_ransac_batched(pts, idx, sample_seed=SEED, **kw)
        return r, rt.bounded_stats()
    finally:
        rt.set_option(12, 1)
        rt.set_option(15, 1)


def _same(a, b):
    assert np.array_equal(a["best_idx"], b["best_idx"])
    assert np.array_equal(a["best_count"], b["best_count"])
    assert np.array_equal(a["F"].view(np.uint64), b["F"].view(np.uint64))
    for ma, mb in zip(a["mask"], b["mask"]):
        assert np.array_equal(ma, mb)


def _check(rt, pts, idx=None, expect_fallback=None, **kw):
    full, sf = _run(rt, False, False, pts, idx, **kw)
    exact, se = _run(rt, True, False, pts, idx, **kw)
    bound, sb = _run(rt, True, True, pts, idx, **kw)
    _same(full, exact)
    _same(full, bound)
    assert sf["K"] == 0 and se["K"] == 512 and sb["K"] == 512
    assert sf["bound_evals"] == 0 and se["bound_evals"] == 0 and sb["bound_evals"] > 0
    for s in (sf, se, sb):
        assert s["bound_evals"] + s["guarded_evals"] == s["evals"]
    if expect_fallback is not None:
        assert sb["fallback_pairs"] == expect_fallback
    return sb


def test_multi_pass_config5_slice(rt, rg):
    P, N, H = 6, 50000, 8192
    pts = _config5(rg, P, N)
    rt.set_option(6, 2 * N * H)                             # three passes of two pairs: the pipelined three-set schedule
    try:
        st = _check(rt, pts, n_hyp=H, expect_fallback=0)
    finally:
        rt.set_option(6, 0)
    assert rt.last_stats()["passes"] >= 3
    assert st["not_fully_scored"] == P * (H - 512)
    # no fallback: the guarded scorer only saw the candidates, over the whole pair
    assert st["guarded_evals"] == P * 512 * N
    assert st["bound_evals"] < 0.5 * P * N * H


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
    pts = _config5(rg, 3, 20000, first_pair=20, outlier_frac=0.6)
    st = _check(rt, pts, n_hyp=4096, expect_fallback=3)
    assert st["not_fully_scored"] == 0


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
        if option == 8:                # with the bound-only prefix the list only serves the candidate stage
            assert rt.last_stats()["overflow"] > 0
    finally:
        rt.set_option(option, 1000 if option == 9 else 0)


def test_device_entry_point(rt, rg, torch):
    dv = rg.device
    P, N, H = 4, 20000, 4096
    d, _ = dv.synth_two_view(P, N, first_pair=70, seed_base=1000)
    po, ho = dv.offsets([N] * P), dv.offsets([H] * P)
    outs = []
    for flags, bound_prefix in ((0, 1), (rg.FLAG_BOUNDED, 0), (rg.FLAG_BOUNDED, 1)):
        rt.set_option(15, bound_prefix)
        try:
            o = dv.FOutputs(P, P * N, device=d.device.index, want_mask=True)
            dv.f_ransac(d, po, None, ho, o, seed=SEED, first_pair=70, flags=flags)
            torch.cuda.synchronize()
        finally:
            rt.set_option(15, 1)
        outs.append((o.best_idx.cpu().numpy(), o.best_count.cpu().numpy(), o.F.cpu().numpy(), o.mask.cpu().numpy()))
        st = rt.bounded_stats()
        assert st["K"] == (512 if flags else 0)
        assert (st["bound_evals"] > 0) == bool(flags and bound_prefix)
    for other in outs[1:]:
        for a, b in zip(outs[0], other):
            assert np.array_equal(a, b)


def test_option_15_is_validated(rt):
    with pytest.raises(ValueError, match="option 15"):
        rt.set_option(15, 2)


# ---- the bound itself: bound count >= FP64 count for every hypothesis ----------------------------------------------
def _hypotheses(rg, pts, H, seed):
    idx = rg.sampling.fast(len(pts), H, 8, seed=seed)
    F, _ = rg.runtime.f8pt_solve(pts, idx)
    return F


def _bound_vs_exact(rt, pts, F, thr, mode):
    exact = rt.epi_score_count(pts, F, thr, mode=mode, score_path=1)
    bound = rt.epi_score_count(pts, F, thr, mode=mode, score_path=2)
    assert np.all(bound >= exact), (thr, mode, np.flatnonzero(bound < exact)[:8])
    return bound, exact


@pytest.mark.parametrize("mode", [0, 1])
def test_bound_dominates_exact_at_the_threshold(rt, rg, mode):
    """Thresholds equal to actual distances (and one ulp either side) put points exactly on and just around the
    threshold of every hypothesis."""
    pts, _ = rg.synth.two_view(3000, seed=31)
    F = _hypotheses(rg, pts, 256, seed=3)
    from oracle import f_path as orc
    d = np.stack([orc.distance(f, pts[:, :2].T, pts[:, 2:].T, mode) for f in F[:4]])
    finite = np.sort(d[np.isfinite(d)])
    for q in (0.1, 0.3, 0.6):
        t = float(finite[int(q * (len(finite) - 1))])
        for thr in (np.nextafter(t, 0.0), t, np.nextafter(t, np.inf)):
            _bound_vs_exact(rt, pts, F, float(thr), mode)


@pytest.mark.parametrize("shift,scale,thr", [(0.0, 1.0, 1.5), (1e6, 1.0, 1.5), (0.0, 1e-4, 1e-4), (0.0, 1e4, 3e3),
                                             (-3e5, 50.0, 1e-3)])
def test_bound_dominates_exact_in_extreme_frames(rt, rg, shift, scale, thr):
    pts, _ = rg.synth.two_view(2000, seed=41)
    pts = pts * scale + shift
    F = _hypotheses(rg, pts, 256, seed=4)
    for mode in (0, 1):
        _bound_vs_exact(rt, pts, F, thr, mode)


def test_unbounded_band_counts_every_finite_point(rt, rg):
    """A frame outside the FP32 analysis (B >= 1e12) has G = T = inf: every finite correspondence passes the bound (the
    pair then falls back to the full sweep), a NaN correspondence never does."""
    pts, _ = rg.synth.two_view(1000, seed=51)
    F = _hypotheses(rg, pts, 64, seed=5)
    pts = pts.copy()
    pts[7] = np.nan
    bound, exact = _bound_vs_exact(rt, pts, F, 1e-11, 0)
    assert np.all(bound == len(pts) - 1)


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch
