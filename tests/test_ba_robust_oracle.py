"""CPU checks of the robust-loss bundle adjustment's checker (tools/ba_robust_oracle.py) and of the argument validation of
``runtime.bundle_adjust(loss=, f_scale=)``.

The losses and the cost are SciPy's (least_squares.py, construct_loss_function).  On the Dino goldens with 5 % of the
observations replaced by uniform draws over the image (the outlier recipe of ``with_outliers``), the numpy IRLS iteration
that the device runs must end at a robust cost not above SciPy's at the reference's ftol, and the redescending losses
(cauchy, arctan) must recover the outlier-free optimum while the squared loss cannot.
"""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import ba_robust_oracle as bro  # noqa: E402

F_SCALE = 2.0 / bro.FOCAL_PX            # 2 px in C-normalised coordinates


@pytest.fixture(scope="module")
def ba_golden():
    from conftest import _load
    return _load("ba_golden.npz")


def _scene(g, nv):
    p = f"v{nv}_"
    return g[p + "cams0"], g[p + "pts0"], g[p + "uv"], g[p + "cam_idx"], g[p + "pt_idx"]


@pytest.mark.parametrize("f_scale", [1e-4, 1.0])
@pytest.mark.parametrize("loss", bro.LOSSES)
def test_rho_and_cost_equal_scipy(loss, f_scale):
    from scipy.optimize._lsq.least_squares import construct_loss_function
    z = np.r_[0.0, np.logspace(-6, 6, 61), 1.0, np.nextafter(1.0, 0.0), np.nextafter(1.0, 2.0), 0.5, 2.0, 1e12]
    f = f_scale * np.sqrt(z) * np.where(np.arange(z.size) % 2 == 0, 1.0, -1.0)
    zz = (f / f_scale) ** 2
    r0, r1 = bro.rho(loss, zz)
    if loss == "linear":
        assert np.array_equal(r1, np.ones_like(zz)) and np.array_equal(r0, zz)
        assert bro.robust_cost_of_residuals(f, loss, f_scale) == 0.5 * float(f @ f)
        return
    fn = construct_loss_function(f.size, loss, f_scale)
    ref = fn(f)
    np.testing.assert_allclose(f_scale ** 2 * r0, ref[0], rtol=1e-15, atol=0)
    np.testing.assert_allclose(r1, ref[1], rtol=1e-15, atol=0)
    assert abs(bro.robust_cost_of_residuals(f, loss, f_scale) - fn(f, cost_only=True)) <= 1e-14 * fn(f, cost_only=True)
    if loss == "huber":                 # the kink belongs to the quadratic branch, as in SciPy (mask = z <= 1)
        k = np.flatnonzero(zz == 1.0)
        assert k.size and np.all(r1[k] == 1.0) and np.all(r0[k] == 1.0)


def test_robust_cost_of_linear_is_the_reference_cost(ba_golden):
    cams, pts, uv, ci, pi = _scene(ba_golden, 8)
    assert bro.robust_cost(cams, pts, uv, ci, pi) == bro.oba.cost(cams, pts, uv, ci, pi)
    r = bro.bundle_adjust_lm(cams, pts, uv, ci, pi, ftol=1e-4)
    o = bro.oba.bundle_adjust_lm(cams, pts, uv, ci, pi, ftol=1e-4)
    assert r[2:] == o[2:] and np.array_equal(r[0], o[0]) and np.array_equal(r[1], o[1])


@pytest.mark.parametrize("nv", [3, 8])
@pytest.mark.parametrize("loss", bro.ROBUST)
def test_irls_cost_not_above_scipy_with_outliers(ba_golden, nv, loss):
    cams, pts, uv, ci, pi = _scene(ba_golden, nv)
    uvo, _ = bro.with_outliers(uv)
    _, _, sol = bro.bundle_adjust_scipy(cams, pts, uvo, ci, pi, loss=loss, f_scale=F_SCALE)
    C, X, c, it, st = bro.bundle_adjust_lm(cams, pts, uvo, ci, pi, ftol=1e-4, loss=loss, f_scale=F_SCALE)
    assert st in (2, 4) and 1 <= it <= 50
    assert c <= sol.cost
    assert abs(bro.robust_cost(C, X, uvo, ci, pi, loss, F_SCALE) - c) <= 1e-12 * c


def test_redescending_losses_recover_the_outlier_free_optimum(ba_golden):
    cams, pts, uv, ci, pi = _scene(ba_golden, 8)
    uvo, idx = bro.with_outliers(uv)
    C0, X0 = bro.oba.unpack(ba_golden["v8_scipy_x"], len(cams), len(pts))
    clean_opt = bro.clean_rms_px(C0, X0, uv, ci, pi, idx)           # SciPy's optimum without outliers (~0.57 px)
    assert clean_opt < 0.7
    for loss in ("cauchy", "arctan"):
        C, X, c, it, st = bro.bundle_adjust_lm(cams, pts, uvo, ci, pi, ftol=1e-4, loss=loss, f_scale=F_SCALE)
        assert bro.clean_rms_px(C, X, uv, ci, pi, idx) <= 1.2 * clean_opt, loss
    C, X, *_ = bro.bundle_adjust_lm(cams, pts, uvo, ci, pi, ftol=1e-4)
    assert bro.clean_rms_px(C, X, uv, ci, pi, idx) > 10.0


def test_convex_losses_on_8_views_are_sensitive_to_rounding(ba_golden):
    """Why the GPU tests compare huber / soft_l1 on the 8-view golden with the numpy iteration over 6 iterations only:
    run to convergence, the numpy iteration itself changes its iteration count when uv changes by 1e-15 relative,
    while cauchy and the 3-view scene reproduce themselves."""
    cams, pts, uv, ci, pi = _scene(ba_golden, 8)
    uvo, _ = bro.with_outliers(uv)
    run = lambda u, loss, **kw: bro.bundle_adjust_lm(cams, pts, u, ci, pi, loss=loss, f_scale=F_SCALE, **kw)[2:]  # noqa: E731
    assert run(uvo, "huber", ftol=1e-4)[1] != run(uvo * (1 + 1e-15), "huber", ftol=1e-4)[1]
    a, b = run(uvo, "cauchy", ftol=1e-4), run(uvo * (1 + 1e-15), "cauchy", ftol=1e-4)
    assert a[1:] == b[1:] and abs(a[0] - b[0]) < 1e-9 * a[0]
    a, b = run(uvo, "huber", ftol=1e-9, max_iter=6), run(uvo * (1 + 1e-15), "huber", ftol=1e-9, max_iter=6)
    assert a[1:] == b[1:] and abs(a[0] - b[0]) < 1e-8 * a[0]


def test_bad_loss_or_f_scale_is_rejected_before_the_library(rg, monkeypatch):
    rt = rg.runtime

    def no_call(*a, **k):
        raise AssertionError("the library was called")

    monkeypatch.setattr(rt, "_call", no_call)
    cams, pts = np.zeros((2, 3, 4)), np.zeros((1, 3))
    uv, ci, pi = np.zeros((2, 2)), np.array([0, 1]), np.array([0, 0])
    for loss in ("tukey", "Huber", "", None, 2, lambda z: z):
        with pytest.raises(ValueError):
            rt.bundle_adjust(cams, pts, uv, ci, pi, loss=loss)
    for fs in (0.0, -1.0, np.nan, np.inf, -np.inf, "x", None):
        with pytest.raises(ValueError):
            rt.bundle_adjust(cams, pts, uv, ci, pi, loss="cauchy", f_scale=fs)
    with pytest.raises(ValueError):
        rg.tables.Tables().BundleAdjustment2(loss="tukey")
    assert rg._cabi.LOSS_LINEAR == 0 and rg._cabi.LOSS_ARCTAN == 4
    assert [rt.BA_LOSSES[k] for k in bro.LOSSES] == [0, 1, 2, 3, 4]
