"""CPU checks of the robust-loss checker of the PnP pose refinement and of the gold-standard refinement
(tools/robust_refine_oracle.py), and of the argument validation of their Python layers.

With loss="linear" the numpy iterations are the oracle's own functions; the gradient J^T Om r of every robust loss is
the gradient of the robust cost; on small views / pairs the numpy iterations end at a robust cost not above SciPy's
least_squares(loss=, f_scale=) minimum.
"""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import robust_refine_oracle as rro  # noqa: E402
from oracle import gs_path as ogs  # noqa: E402
from oracle import pnp_refine_path as opr  # noqa: E402


@pytest.fixture(scope="module")
def view(rg):
    """Dino view 5 (C-normalised y, its K without skew), 5 % of the image points replaced, a perturbed start pose."""
    X, y, K = rg.synth.dino_view_2d3d(5)
    K = np.triu(K)
    K[0, 1] = 0.0
    yo, idx = rro.pnp_with_outliers(y)
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pnp_golden.npz"))
    R0 = opr.rodrigues(np.array([2e-3, -1e-3, 1.5e-3])) @ g["R"][5]
    t0 = g["t"][5] * (1.0 + 1e-3)
    return X, yo, K, R0, t0, idx


@pytest.fixture(scope="module")
def pair(gs_golden):
    """The first 60 correspondences of the noisy Dino pair (0, 1), 6 of them with the right point moved by 20-40 px."""
    in1, in2 = gs_golden["in1"][:, :60].copy(), gs_golden["in2"][:, :60].copy()
    rng = np.random.default_rng(3)
    in2[:, ::10] += rng.choice([-1.0, 1.0], (2, 6)) * rng.uniform(20.0, 40.0, (2, 6))
    return gs_golden["F0"], in1, in2


def test_linear_iterations_are_the_oracle_functions(view, pair):
    X, y, K, R0, t0, _ = view
    for k in (None, K):
        a = rro.pnp_refine_lm(X, y, R0, t0, K=k)
        b = opr.pnp_refine_lm(X, y, R0, t0, K=k)
        assert all(np.array_equal(a[n], b[n]) for n in ("R", "t", "cost", "iters", "status"))
    F0, in1, in2 = pair
    a = rro.gold_standard_lm(F0, in1, in2, max_iter=8)
    b = ogs.gold_standard_lm(F0, in1, in2, max_iter=8)
    assert all(np.array_equal(u, v) for u, v in zip(a, b))
    assert rro.gs_cost(*ogs.start_point(F0, in1, in2)[::2], in1, in2) == ogs.cost(*ogs.start_point(F0, in1, in2)[::2], in1, in2)


@pytest.mark.parametrize("loss", rro.ROBUST)
def test_gradients_match_central_differences_of_the_robust_cost(view, pair, loss):
    X, y, K, R0, t0, _ = view
    fs = 2.0                                                          # pixels (K given)

    def pc(p):
        return rro.pnp_cost(opr.rodrigues(p[:3]) @ R0, t0 + p[3:], X, y, K, loss, fs)

    g = rro.pnp_gradient(R0, t0, X, y, K, loss, fs)
    for k in range(6):
        h = 1e-7 if k < 3 else 1e-7 * np.abs(t0).max()
        e = np.zeros(6)
        e[k] = h
        fd = (pc(e) - pc(-e)) / (2 * h)
        assert abs(fd - g[k]) <= 1e-5 * np.abs(g).max(), (k, fd, g[k])
    F0, in1, in2 = pair
    C1, _, Xp = ogs.start_point(F0, in1, in2)
    p0 = np.hstack((C1.ravel(), Xp.T.ravel()))
    gg = rro.gs_gradient(C1, Xp, in1, in2, loss, 1.0)

    def gc(p):
        return rro.gs_cost(p[:12].reshape(3, 4), p[12:].reshape(-1, 3).T, in1, in2, loss, 1.0)

    for k in list(range(12)) + [12, 13, 14, 40, 41, 42]:
        h = 1e-5 * max(abs(p0[k]), 1e-5)                             # C1 spans 1e-7 .. 1: a step relative to the entry
        e = np.zeros_like(p0)
        e[k] = h
        fd = (gc(p0 + e) - gc(p0 - e)) / (2 * h)
        assert abs(fd - gg[k]) <= 1e-5 * max(np.abs(gg).max(), 1e-12), (k, fd, gg[k])


@pytest.mark.parametrize("loss", rro.ROBUST)
@pytest.mark.parametrize("with_K", [False, True])
def test_pnp_iteration_reaches_the_scipy_robust_minimum(view, loss, with_K):
    X, y, K, R0, t0, _ = view
    k = K if with_K else None
    fs = 1.0 if with_K else 1.0 / K[0, 0]                             # 1 px either way
    o = rro.pnp_refine_lm(X, y, R0, t0, K=k, loss=loss, f_scale=fs, max_iter=200)
    assert o["status"] == 2
    _, _, cs = rro.pnp_refine_scipy(X, y, R0, t0, K=k, loss=loss, f_scale=fs)
    assert o["cost"] <= cs * (1 + 1e-9)
    assert abs(rro.pnp_cost(o["R"], o["t"], X, y, k, loss, fs) - o["cost"]) <= 1e-12 * o["cost"]


@pytest.mark.parametrize("loss", rro.ROBUST)
def test_gold_standard_iteration_reaches_the_scipy_robust_minimum(pair, loss):
    F0, in1, in2 = pair
    Fo, co, ito, C1o, Xo = rro.gold_standard_lm(F0, in1, in2, max_iter=100, loss=loss, f_scale=1.0)
    _, sol = rro.gold_standard_scipy(F0, in1, in2, loss=loss, f_scale=1.0)
    assert co <= sol.cost * (1 + 1e-9)
    assert abs(rro.gs_cost(C1o, Xo, in1, in2, loss, 1.0) - co) <= 1e-12 * co


def test_convex_losses_on_a_pair_with_outliers_are_sensitive_to_rounding(rg):
    """The start point of the gold standard triangulates every correspondence optimally, and for the outliers of a 30 %
    outlier pair that is sensitive to rounding: a 1e-15 relative change of the points moves the soft_l1 start cost by
    ~1e-8 relative and the first trial cost by ~3e-7 (a convex loss keeps those residuals in the cost; a redescending one
    flattens them).  On such pairs the device is compared with the iteration's own sensitivity
    (tests/test_gpu_robust_refine.py), not with a fixed tolerance."""
    pts, _ = rg.synth.two_view(2000, seed=5)
    Ps = rg.synth.dino()["Ps"]
    F0 = rro.og.fmatrix_from_cameras(Ps[0], Ps[1])
    in1, in2 = pts[:, :2].T.copy(), pts[:, 2:].T.copy()
    ta, tb = [], []
    rro.gold_standard_lm(F0, in1, in2, loss="soft_l1", max_iter=1, trace=ta)
    rro.gold_standard_lm(F0, in1, in2 * (1 + 1e-15), loss="soft_l1", max_iter=1, trace=tb)
    assert abs(ta[0]["cost"] - tb[0]["cost"]) > 1e-10 * ta[0]["cost"]
    assert abs(ta[0]["cost_trial"] - tb[0]["cost_trial"]) > 1e-8 * ta[0]["cost"]


BAD = [("cauchy ", 1.0), ("Cauchy", 1.0), (len, 1.0), (None, 1.0), ("cauchy", 0.0), ("cauchy", -1.0),
       ("cauchy", float("nan")), ("cauchy", float("inf")), ("cauchy", "x"), ("linear", 0.0)]


@pytest.mark.parametrize("loss,f_scale", BAD)
def test_argument_errors_raise_without_a_gpu(rg, view, pair, loss, f_scale):
    X, y, K, R0, t0, _ = view
    F0, in1, in2 = pair
    pts = np.ascontiguousarray(np.hstack([in1.T, in2.T]))
    calls = [lambda: rg.runtime.pnp_refine(X, y, R0, t0, loss=loss, f_scale=f_scale),
             lambda: rg.runtime.pnp_refine_batched([X], [y], R0[None], t0[None], loss=loss, f_scale=f_scale),
             lambda: rg.runtime.gold_standard([pts], F0[None], loss=loss, f_scale=f_scale),
             lambda: rg.pnp.pnp_refine(X, y, R0, t0, loss=loss, f_scale=f_scale),
             lambda: rg.fun.gold_standard_device(F0, in1, in2, np.arange(60), loss=loss, f_scale=f_scale),
             lambda: rg.fun.gold_standard(F0, in1, in2, np.arange(60), loss=loss, f_scale=f_scale),
             lambda: rg.fun.getFFromLabCode(in1, in2, refine="device", loss=loss, f_scale=f_scale),
             lambda: rg.runtime.bundle_adjust(np.zeros((1, 3, 4)), np.zeros((0, 3)), np.zeros((0, 2)), [], [], loss=loss,
                                              f_scale=f_scale)]
    for call in calls:
        with pytest.raises(ValueError, match="loss must be|f_scale must be"):
            call()


def test_tables_refuses_a_robust_loss_without_the_lm_refinement(rg):
    T = rg.tables.Tables()
    y = np.zeros((8, 3))
    with pytest.raises(ValueError, match="needs refine='lm'"):
        T.addNewView(np.eye(3), 0, y, y, y, y, loss="cauchy")
    with pytest.raises(ValueError, match="loss must be"):
        T.addNewView(np.eye(3), 0, y, y, y, y, refine="lm", loss="l2")
