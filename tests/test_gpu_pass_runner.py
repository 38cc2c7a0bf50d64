"""The host entry point runs the bounded sweep in sub-batches (option 2), pipelined (option 10 = 1) or one after the other
(option 10 = 0).  Pairs are independent, so winners, counts, F, masks and every statistic of the call must be those of
one sub-batch, under both scoring modes.  A call reports one pass per sub-batch, empty ones included (eight sub-batches of
nine pairs can leave some empty, depending on the rates the context has measured)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
SEED = 20261021
SIZES = [30000, 12000, 25000, 9000, 20000, 16000, 28000, 10000, 22000]
HYPS = [4096, 2048, 3000, 1024, 4096, 2500, 1500, 3500, 2048]


@pytest.fixture(scope="module")
def rt(rg):
    return rg.runtime


@pytest.fixture(scope="module")
def pairs(rg):
    out = []
    for p, n in enumerate(SIZES):       # config-5 pairs of ragged sizes
        d, _ = rg.device.synth_two_view(1, n, first_pair=100 + p, seed_base=1000)
        out.append(np.ascontiguousarray(d[0].cpu().numpy()))
    return out


def _run(rt, pts, slices, piped, mode):
    rt.set_option(2, slices)
    rt.set_option(10, piped)
    try:
        r = rt.f_ransac_batched(pts, None, n_hyp=HYPS, sample_seed=SEED, mode=mode, want_mask=True)
        return r, rt.last_stats(), rt.bounded_stats()
    finally:
        rt.set_option(2, 0)
        rt.set_option(10, 1)


@pytest.mark.parametrize("mode", [0, 1])
def test_host_sub_batches_of_the_bounded_sweep(rt, pairs, mode):
    ref, ref_st, ref_bs = _run(rt, pairs, 1, 1, mode)
    assert ref_st["passes"] == 1 and ref_bs["K"] == 512 and ref_bs["not_fully_scored"] > 0
    for slices in (1, 2, 3, 8):
        for piped in (0, 1):
            out, st, bs = _run(rt, pairs, slices, piped, mode)
            assert st["passes"] == slices, (slices, piped)
            assert np.array_equal(out["best_idx"], ref["best_idx"]) and np.array_equal(out["best_count"], ref["best_count"])
            assert np.array_equal(out["F"].view(np.uint64), ref["F"].view(np.uint64))
            for a, b in zip(out["mask"], ref["mask"]):
                assert np.array_equal(a, b)
            for key in ("recheck_groups", "band_evals", "flips"):
                assert st[key] == ref_st[key], (key, slices, piped)
            for key in ("evals", "not_fully_scored", "fallback_pairs", "K"):
                assert bs[key] == ref_bs[key], (key, slices, piped)
