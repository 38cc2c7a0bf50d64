"""The pipelined bounded sweep (option 10 = 1) spreads each pass over two streams and four workspace sets: the scorers
of a pass run on the caller's stream, the small kernels between them on a side stream beside the next pass's scorers, and
a pass lives from two passes before its prefix stage to two passes after it.  Six passes wrap the four-set rotation; two
pairs with 60 % outliers in a middle pass are certain to fall back, so that pass's fallback stage has work while the
passes after it are in flight.  Winners, counts, F and masks must equal, bit for bit, those of the same call run one
pass after the other (option 10 = 0) and those of the full sweep (option 12 = 0); the statistics of the pipelined and
the serial bounded sweep must be equal.  Both the device entry point (six passes through option 6) and the host entry
point (six sub-batches of one pass through option 2) are checked."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
SEED = 20261022
P, N, H = 12, 20000, 4096
FALLBACK_PAIRS = (5, 6)                 # pass 2 of the device entry point's six passes of two pairs
STATS = ("recheck_groups", "band_evals", "flips", "overflow", "bad_index_hyps", "passes", "launches")


@pytest.fixture(scope="module")
def rt(rg):
    return rg.runtime


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


@pytest.fixture(scope="module")
def d_pts(rg):
    d, _ = rg.device.synth_two_view(P, N, first_pair=300, seed_base=1000)
    p0 = FALLBACK_PAIRS[0]
    o, _ = rg.device.synth_two_view(len(FALLBACK_PAIRS), N, first_pair=300 + p0, seed_base=1000, outlier_frac=0.6)
    d[p0:p0 + len(FALLBACK_PAIRS)] = o
    return d


def _settings(rt, piped, bounded, extra):
    rt.set_option(10, piped)
    rt.set_option(12, bounded)
    for k, v in extra.items():
        rt.set_option(k, v)


def _reset(rt, extra):
    rt.set_option(10, 1)
    rt.set_option(12, 1)
    for k in extra:
        rt.set_option(k, 0)


def _same(a, b):
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert np.array_equal(a[2].view(np.uint64), b[2].view(np.uint64))
    assert len(a[3]) == len(b[3]) and all(np.array_equal(x, y) for x, y in zip(a[3], b[3]))


def _compare(rt, run):
    """run(piped, bounded) -> (best_idx, best_count, F, masks); checks the three settings against each other."""
    out = {}
    for piped, bounded in ((1, 1), (0, 1), (1, 0)):
        res = run(piped, bounded)
        out[piped, bounded] = (res, rt.last_stats(), rt.bounded_stats())
    (pip, pst, pbs), (ser, sst, sbs), (full, fst, _) = out[1, 1], out[0, 1], out[1, 0]
    _same(pip, ser)
    _same(pip, full)
    for key in STATS:
        assert pst[key] == sst[key], key
    assert pbs == sbs
    assert pst["passes"] == 6 and fst["passes"] == 6
    assert pbs["K"] == 512 and pbs["fallback_pairs"] == len(FALLBACK_PAIRS)
    assert pbs["not_fully_scored"] > 0
    return pbs


@pytest.mark.parametrize("mode", [0, 1])
def test_device_entry_point(rt, rg, torch, d_pts, mode):
    dv = rg.device
    po, ho = dv.offsets([N] * P), dv.offsets([H] * P)
    extra = {6: 2 * N * H}                                  # six passes of two pairs

    def run(piped, bounded):
        _settings(rt, piped, bounded, extra)
        try:
            o = dv.FOutputs(P, P * N, device=d_pts.device.index, want_mask=True)
            dv.f_ransac(d_pts, po, None, ho, o, mode=mode, seed=SEED, first_pair=300)
            torch.cuda.synchronize()
            mask = o.mask.cpu().numpy()
            return (o.best_idx.cpu().numpy(), o.best_count.cpu().numpy(), o.F.cpu().numpy(),
                    [mask[po[p]:po[p + 1]] for p in range(P)])
        finally:
            _reset(rt, extra)

    _compare(rt, run)


def test_host_entry_point_sub_batches(rt, d_pts):
    pts = [np.ascontiguousarray(d_pts[p].cpu().numpy()) for p in range(P)]
    extra = {2: 6}                                          # six sub-batches of the one pass

    def run(piped, bounded):
        _settings(rt, piped, bounded, extra)
        try:
            r = rt.f_ransac_batched(pts, None, n_hyp=H, sample_seed=SEED, first_pair=300, want_mask=True)
            return r["best_idx"], r["best_count"], r["F"], r["mask"]
        finally:
            _reset(rt, extra)

    _compare(rt, run)
