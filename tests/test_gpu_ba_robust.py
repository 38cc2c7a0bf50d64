"""GPU tests of the robust losses of the device bundle adjustment (``rg_bundle_adjust_host2`` / ``_dev2``,
``runtime.bundle_adjust(loss=, f_scale=)``, ``Tables.BundleAdjustment2(loss=, f_scale=)``) against
  * the squared-loss entry points (RG_LOSS_LINEAR must be bit-identical to ``rg_bundle_adjust_host``),
  * the numpy IRLS iteration of tools/ba_robust_oracle.py (same iterates up to rounding), and
  * SciPy's ``least_squares(loss=, f_scale=)`` at the reference's ftol (final cost not above SciPy's).
Outliers: 5 % (Dino goldens) or 10 % (synthetic scenes) of the observations replaced by uniform draws over the image.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import ba_robust_oracle as bro  # noqa: E402

pytestmark = pytest.mark.gpu

F_SCALE = 2.0 / bro.FOCAL_PX            # 2 px in C-normalised coordinates
LOSS_ID = {k: i for i, k in enumerate(bro.LOSSES)}


@pytest.fixture(scope="module")
def rt(rg):
    return rg.runtime


@pytest.fixture(scope="module")
def ba_golden():
    from conftest import _load
    return _load("ba_golden.npz")


def _scene(g, nv):
    p = f"v{nv}_"
    return g[p + "cams0"], g[p + "pts0"], g[p + "uv"], g[p + "cam_idx"], g[p + "pt_idx"]


def _host(rg, name, cams, pts, uv, ci, pi, ftol, *loss_args, max_iter=50):
    """rg_bundle_adjust_host (no loss_args) or rg_bundle_adjust_host2 (loss, f_scale) called through the C ABI."""
    c, p = np.array(cams, dtype=np.float64), np.array(pts, dtype=np.float64)
    cost, its = np.full(1, np.nan), np.zeros(2, dtype=np.int32)
    rg._cabi.call(name, rg._cabi.context(), 0, len(c), len(p), len(uv), c, p, np.ascontiguousarray(uv, dtype=np.float64),
                  np.ascontiguousarray(ci, dtype=np.int32), np.ascontiguousarray(pi, dtype=np.int32), 1, max_iter, ftol,
                  *loss_args, cost, its[:1], its[1:])
    return {"cams": c, "pts": p, "cost": float(cost[0]), "iters": int(its[0]), "status": int(its[1])}


def _dev2(rg, cams, pts, uv, ci, pi, ftol, loss, f_scale, max_iter=50):
    """rg_bundle_adjust_dev2 on device buffers and a side stream; returns the return code and the results."""
    import torch
    lib, ctx = rg._cabi.load_library(), rg._cabi.context()
    vp, pi32 = C.c_void_p, C.POINTER(C.c_int32)
    d_c, d_p = torch.from_numpy(np.array(cams)).cuda(), torch.from_numpy(np.array(pts)).cuda()
    d_uv = torch.from_numpy(np.ascontiguousarray(uv, dtype=np.float64)).cuda()
    d_cost = torch.zeros(1, dtype=torch.float64, device="cuda")
    d_is = torch.zeros(2, dtype=torch.int32, device="cuda")
    ci32, pi32a = np.ascontiguousarray(ci, dtype=np.int32), np.ascontiguousarray(pi, dtype=np.int32)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        rc = lib.rg_bundle_adjust_dev2(vp(ctx), vp(stream.cuda_stream), len(cams), len(pts), len(uv), vp(d_c.data_ptr()),
                                       vp(d_p.data_ptr()), vp(d_uv.data_ptr()), ci32.ctypes.data_as(pi32),
                                       pi32a.ctypes.data_as(pi32), 1, max_iter, ftol, loss, f_scale, vp(d_cost.data_ptr()),
                                       vp(d_is.data_ptr()), vp(d_is[1:].data_ptr()))
    stream.synchronize()
    return rc, {"cams": d_c.cpu().numpy(), "pts": d_p.cpu().numpy(), "cost": float(d_cost.item()),
                "iters": int(d_is[0].item()), "status": int(d_is[1].item())}


def _same(a, b):
    return (a["iters"], a["status"]) == (b["iters"], b["status"]) and np.array_equal(
        np.float64(a["cost"]), np.float64(b["cost"])) and np.array_equal(a["cams"], b["cams"]) and np.array_equal(a["pts"], b["pts"])


@pytest.mark.parametrize("nv", [3, 8, 36])
def test_linear_loss_is_bit_identical_to_the_squared_loss_entry(rg, ba_golden, nv):
    sc = _scene(ba_golden, nv)
    ref = _host(rg, "rg_bundle_adjust_host", *sc, 1e-6)
    for f_scale in (1.0, 1e-4):                     # f_scale has no effect on the linear loss
        assert _same(_host(rg, "rg_bundle_adjust_host2", *sc, 1e-6, 0, f_scale), ref)
        rc, d = _dev2(rg, *sc, 1e-6, 0, f_scale)
        assert rc == 0 and _same(d, ref)
    assert _same(rg.runtime.bundle_adjust(*sc, ftol=1e-6), ref)


# 8 views with the convex losses: once lambda reaches its floor the iteration amplifies rounding about tenfold per step
# (the numpy iteration itself moves from 18 to 33 iterations for huber when uv changes by 1e-15 relative, see
# tests/test_ba_robust_oracle.py), so the device is compared with it over the first 6 iterations only
ROUNDING_BOUND = {(8, "huber"), (8, "soft_l1")}


@pytest.mark.parametrize("nv", [3, 8])
@pytest.mark.parametrize("loss", bro.ROBUST)
def test_robust_losses_equal_the_numpy_iteration(rt, ba_golden, nv, loss):
    cams, pts, uv, ci, pi = _scene(ba_golden, nv)
    uvo, _ = bro.with_outliers(uv)
    for ftol, max_iter in ((1e-9, 6),) if (nv, loss) in ROUNDING_BOUND else ((1e-4, 50), (1e-9, 6)):
        res = rt.bundle_adjust(cams, pts, uvo, ci, pi, max_iter=max_iter, ftol=ftol, loss=loss, f_scale=F_SCALE)
        Co, Xo, co, ito, sto = bro.bundle_adjust_lm(cams, pts, uvo, ci, pi, max_iter=max_iter, ftol=ftol, loss=loss,
                                                    f_scale=F_SCALE)
        assert (res["iters"], res["status"]) == (ito, sto)
        assert abs(res["cost"] - co) < 1e-7 * co
        ra = bro.oba.residuals(bro.oba.pack(res["cams"], res["pts"]), uvo[:, 0], uvo[:, 1], ci, pi, len(cams), len(pts))
        rb = bro.oba.residuals(bro.oba.pack(Co, Xo), uvo[:, 0], uvo[:, 1], ci, pi, len(cams), len(pts))
        assert np.abs(ra - rb).max() < 1e-6 * np.abs(rb).max()


@pytest.mark.parametrize("loss", bro.ROBUST)
def test_dino_36_views_with_outliers(rt, ba_golden, loss):
    cams, pts, uv, ci, pi = _scene(ba_golden, 36)
    uvo, idx = bro.with_outliers(uv)
    res = rt.bundle_adjust(cams, pts, uvo, ci, pi, ftol=1e-4, loss=loss, f_scale=F_SCALE)
    assert res["status"] in (2, 4)
    _, _, sol = bro.bundle_adjust_scipy(cams, pts, uvo, ci, pi, loss=loss, f_scale=F_SCALE)
    assert res["cost"] <= sol.cost
    assert abs(bro.robust_cost(res["cams"], res["pts"], uvo, ci, pi, loss, F_SCALE) - res["cost"]) < 1e-10 * res["cost"]
    assert np.array_equal(res["cams"][0], cams[0])
    if loss in ("cauchy", "arctan"):
        C0, X0 = bro.oba.unpack(ba_golden["v36_scipy_x"], len(cams), len(pts))
        clean_opt = bro.clean_rms_px(C0, X0, uv, ci, pi, idx)           # outlier-free optimum, ~0.60 px
        assert bro.clean_rms_px(res["cams"], res["pts"], uv, ci, pi, idx) <= 1.2 * clean_opt


@pytest.mark.parametrize("n_views,n_points,track", [(24, 2000, 6), (60, 3000, 8)])
def test_synthetic_scenes_reproducible_over_solver_variants(rt, rg, n_views, n_points, track):
    cams, pts, uv, ci, pi, _ = rg.synth.ba_scene(n_views, n_points, track=track)
    uvo, _ = bro.with_outliers(uv, frac=0.10, seed=1)
    for loss in ("huber", "cauchy"):
        kw = dict(ftol=1e-6, max_iter=20, loss=loss, f_scale=F_SCALE)
        base = rt.bundle_adjust(cams, pts, uvo, ci, pi, **kw)
        assert base["cost"] < bro.robust_cost(cams, pts, uvo, ci, pi, loss, F_SCALE)
        assert _same(rt.bundle_adjust(cams, pts, uvo, ci, pi, **kw), base)              # repeated call
        try:
            for cl in (1, 2, 4, 8):
                rt.set_option(3, cl)
                assert _same(rt.bundle_adjust(cams, pts, uvo, ci, pi, **kw), base), (loss, cl)
            rt.set_option(3, 0)
            rt.set_option(4, 1)                                                           # L2 variant of the solver
            assert _same(rt.bundle_adjust(cams, pts, uvo, ci, pi, **kw), base), (loss, "L2")
        finally:
            rt.set_option(3, 0)
            rt.set_option(4, 0)


def test_dev2_equals_host2_and_invalid_arguments(rt, rg, ba_golden):
    cams, pts, uv, ci, pi = _scene(ba_golden, 8)
    uvo, _ = bro.with_outliers(uv)
    for loss in ("soft_l1", "cauchy"):
        h = _host(rg, "rg_bundle_adjust_host2", cams, pts, uvo, ci, pi, 1e-6, LOSS_ID[loss], F_SCALE)
        rc, d = _dev2(rg, cams, pts, uvo, ci, pi, 1e-6, LOSS_ID[loss], F_SCALE)
        assert rc == 0 and _same(d, h)
        assert _same(rt.bundle_adjust(cams, pts, uvo, ci, pi, ftol=1e-6, loss=loss, f_scale=F_SCALE), h)
    for loss, fs in ((5, 1.0), (-1, 1.0), (3, 0.0), (3, -1.0), (3, float("nan")), (3, float("inf")), (0, 0.0)):
        rc, _ = _dev2(rg, cams, pts, uvo, ci, pi, 1e-6, loss, fs)
        assert rc == -2, (loss, fs)
        with pytest.raises(ValueError):
            _host(rg, "rg_bundle_adjust_host2", cams, pts, uvo, ci, pi, 1e-6, loss, fs)


def test_tables_bundle_adjustment2_with_a_robust_loss(rt, rg, ba_golden):
    cams, pts, uv, ci, pi = _scene(ba_golden, 8)
    uvo, _ = bro.with_outliers(uv)
    T = rg.tables.Tables()
    for i, Cm in enumerate(cams):
        T.addView(i, rg.help_classes.CameraPose(Cm[:, :3].copy(), Cm[:, 3].copy()))
    for X in pts:
        T.addPoint(X.copy())
    T.K = np.eye(3)
    for y, k, j in zip(uvo, ci, pi):
        T.addObs(np.array([y[0], y[1], 1.0]), int(k), int(j))
    info = T.BundleAdjustment2(loss="cauchy", f_scale=F_SCALE)
    ref = rt.bundle_adjust(cams, pts, uvo, ci, pi, n_fixed=1, max_iter=50, ftol=1e-4, loss="cauchy", f_scale=F_SCALE)
    assert (info["cost"], info["iters"], info["status"]) == (ref["cost"], ref["iters"], ref["status"])
    C1 = np.stack([v.camera_pose.GetCameraMatrix() for v in T.T_views])
    X1 = np.stack([p.point for p in T.T_points])
    assert np.abs(C1 - ref["cams"]).max() < 1e-12 and np.array_equal(X1, ref["pts"])
