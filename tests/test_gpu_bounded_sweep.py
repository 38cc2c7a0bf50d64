"""The bounded sweep (option 12, csrc/bounded.cuh) must return exactly what the full sweep returns: winner index, count,
F and inlier mask, bit for bit, on every kind of batch — several passes, ragged pairs, any point order, pairs where the
bound fails and everything is scored, exact ties under both tie rules, Sampson scoring, a wide guard band and a flag list
that overflows inside a window."""
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


def _run(rt, bounded, pts, idx=None, **kw):
    rt.set_option(12, 1 if bounded else 0)
    try:
        r = rt.f_ransac_batched(pts, idx, sample_seed=SEED, **kw)
        return r, rt.bounded_stats()
    finally:
        rt.set_option(12, 1)


def _same(a, b):
    assert np.array_equal(a["best_idx"], b["best_idx"])
    assert np.array_equal(a["best_count"], b["best_count"])
    assert np.array_equal(a["F"].view(np.uint64), b["F"].view(np.uint64))
    for ma, mb in zip(a["mask"], b["mask"]):
        assert np.array_equal(ma, mb)


def _check(rt, pts, idx=None, expect_fallback=None, **kw):
    full, sf = _run(rt, False, pts, idx, **kw)
    bnd, sb = _run(rt, True, pts, idx, **kw)
    _same(full, bnd)
    assert sf["K"] == 0 and sb["K"] == 512
    if expect_fallback is not None:
        assert sb["fallback_pairs"] == expect_fallback
    return sb


def test_multi_pass_config5_slice(rt, rg):
    pts = _config5(rg, 6, 50000)
    rt.set_option(6, 2 * 50000 * 8192)                      # three passes of two pairs: the pipelined three-set schedule
    try:
        st = _check(rt, pts, n_hyp=8192, expect_fallback=0)
    finally:
        rt.set_option(6, 0)
    assert rt.last_stats()["passes"] >= 3
    assert st["not_fully_scored"] == 6 * (8192 - 512)
    assert st["evals"] < 0.6 * 6 * 50000 * 8192


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
        if option == 8:
            assert rt.last_stats()["overflow"] > 0
    finally:
        rt.set_option(option, 1000 if option == 9 else 0)


def test_counts_request_runs_the_full_sweep(rt, rg):
    pts = _config5(rg, 2, 20000, first_pair=60)
    r = rt.f_ransac_batched(pts, None, n_hyp=2048, sample_seed=SEED, want_counts=True)
    assert rt.bounded_stats()["K"] == 0
    for p in range(2):
        assert int(r["counts"][p].max()) == int(r["best_count"][p])
        assert int(np.argmax(r["counts"][p])) == int(r["best_idx"][p])


def test_device_entry_point(rt, rg, torch):
    dv = rg.device
    P, N, H = 4, 20000, 4096
    d, _ = dv.synth_two_view(P, N, first_pair=70, seed_base=1000)
    po, ho = dv.offsets([N] * P), dv.offsets([H] * P)
    outs = []
    for flags in (0, rg.FLAG_BOUNDED):
        o = dv.FOutputs(P, P * N, device=d.device.index, want_mask=True)
        dv.f_ransac(d, po, None, ho, o, seed=SEED, first_pair=70, flags=flags)
        torch.cuda.synchronize()
        outs.append((o.best_idx.cpu().numpy(), o.best_count.cpu().numpy(), o.F.cpu().numpy(), o.mask.cpu().numpy()))
        assert rt.bounded_stats()["K"] == (512 if flags else 0)
    for a, b in zip(*outs):
        assert np.array_equal(a, b)


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch
