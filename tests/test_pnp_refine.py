"""CPU checks of the PnP pose refinement's contract (DESIGN.md section 4.7): the numpy restatement of the device
iteration (oracle.pnp_refine_path.pnp_refine_lm) reaches the minimum of SciPy's least_squares(method='lm') and of
OpenCV's solvePnP(SOLVEPNP_ITERATIVE, useExtrinsicGuess=True) — the final stage of the reference's cv.solvePnPRansac
(tables.py:141) — from the algebraic DLT pose; the public entry points reject bad arguments before touching a device."""
import numpy as np
import pytest

from oracle import pnp_path as opnp
from oracle import pnp_refine_path as opr

THR2 = (1.5 / 3217.0) ** 2
FTOL = 1e-16          # the minimum to ~1e-12 rad; the default 1e-12 stops up to ~1e-10 rad before it at 0.5 px


def _start(rg, n, seed, sigma):
    """synth.pnp_scene and the algebraic pose fitted on its true inliers (the last 70 %)."""
    X, y, gt = rg.synth.pnp_scene(n, seed=seed, sigma_px=sigma)
    inl = np.zeros(n, bool)
    inl[int(round(0.3 * n)):] = True
    Xh = np.hstack([X, np.ones((n, 1))])
    yh = np.hstack([y, np.ones((n, 1))])
    R0, t0 = opnp.pnp_minimize(Xh[inl], yh[inl])
    return X, y, inl, R0, t0, gt


def _dino_K(rg, skew=True):
    K = rg.synth.calibration(rg.synth.dino()["Ps"][17])
    K[1, 0] = 0.0                   # exactly upper triangular (RQ leaves ~1e-13 there)
    if not skew:
        K[0, 1] = 0.0
    return K


@pytest.mark.parametrize("sigma", [0.05, 0.5])
@pytest.mark.parametrize("with_K", [False, True])
def test_oracle_lm_reaches_scipy_minimum(rg, sigma, with_K):
    X, y, inl, R0, t0, (Rgt, _) = _start(rg, 2000, 13, sigma)
    K = _dino_K(rg) if with_K else None
    o = opr.pnp_refine_lm(X, y, R0, t0, mask=inl, K=K, ftol=FTOL)
    Rs, ts, cs = opr.pnp_refine_reference(X, y, R0, t0, mask=inl, K=K)
    assert o["status"] == 2 and o["iters"] <= 10
    assert opnp.rotation_angle(o["R"], Rs) < 1e-10
    assert np.linalg.norm(o["t"] - ts) < 1e-10 * np.linalg.norm(ts)
    assert abs(o["cost"] - cs) <= 1e-10 * cs
    assert np.abs(o["R"] @ o["R"].T - np.eye(3)).max() < 1e-12
    # the geometric minimum is closer to the truth than the algebraic start
    assert opnp.rotation_angle(o["R"], Rgt) < 0.5 * opnp.rotation_angle(R0, Rgt)


@pytest.mark.parametrize("with_K", [False, True])
def test_oracle_lm_matches_opencv_solvepnp_iterative(rg, with_K):
    cv2 = pytest.importorskip("cv2")
    X, y, inl, R0, t0, _ = _start(rg, 2000, 13, 0.5)
    # OpenCV's pinhole model has no skew term: the Dino K is compared with its skew set to zero
    K = _dino_K(rg, skew=False) if with_K else np.eye(3)
    px = np.ascontiguousarray((np.hstack([y[inl], np.ones((int(inl.sum()), 1))]) @ K.T)[:, :2])
    ok, rv, tv = cv2.solvePnP(X[inl], px, K, None, cv2.Rodrigues(R0)[0], t0.reshape(3, 1).copy(), True,
                              cv2.SOLVEPNP_ITERATIVE)
    assert ok
    Rc, tc = cv2.Rodrigues(rv)[0], tv.ravel()
    o = opr.pnp_refine_lm(X, y, R0, t0, mask=inl, K=K if with_K else None, ftol=FTOL)
    # OpenCV's own stopping rule (at most 20 LM iterations, step / cost change below DBL_EPSILON) leaves it ~1e-10 rad
    # from the minimum in pixel units
    assert opnp.rotation_angle(o["R"], Rc) < 5e-10
    assert np.linalg.norm(o["t"] - tc) < 5e-10 * np.linalg.norm(tc)
    cost_cv = 0.5 * float(np.sum(opr.reprojection_residuals(Rc, tc, X[inl], y[inl], K[:2, :2]) ** 2))
    assert abs(o["cost"] - cost_cv) <= 1e-10 * cost_cv


def test_oracle_lm_rounds_and_edge_cases(rg):
    X, y, inl, R0, t0, _ = _start(rg, 2000, 13, 0.2)
    one = opr.pnp_refine_lm(X, y, R0, t0, mask=inl, thr2=THR2, want_mask=True)
    two = opr.pnp_refine_lm(X, y, R0, t0, mask=inl, thr2=THR2, rounds=2)
    assert one["mask"].sum() <= inl.sum() and two["mask"][inl].mean() > 0.99
    few = opr.pnp_refine_lm(X[:2], y[:2], R0, t0)
    assert few["status"] == 5 and few["iters"] == 0 and np.array_equal(few["R"], R0)
    bad = opr.pnp_refine_lm(X, y, np.full((3, 3), np.nan), t0)
    assert bad["status"] == 1
    assert opr.pnp_refine_lm(X, y, R0, t0, max_iter=0)["status"] == 4


def test_rodrigues_is_a_rotation():
    for w in ([0.0, 0.0, 0.0], [1e-9, -2e-9, 3e-9], [0.3, -1.2, 0.7], [np.pi, 0.0, 0.0]):
        E = opr.rodrigues(w)
        assert np.abs(E @ E.T - np.eye(3)).max() < 1e-15 and abs(np.linalg.det(E) - 1.0) < 1e-15


def test_argument_errors_raise_value_error(rg):
    X, y, inl, R0, t0, _ = _start(rg, 200, 1, 0.1)
    rt = rg.runtime
    Kbad = np.eye(3)
    Kbad[2, 0] = 1.0
    Klow = np.eye(3)
    Klow[1, 0] = 2.0
    for kw in ({"K": Kbad}, {"K": Klow}, {"K": np.eye(4)}, {"rounds": 0}, {"rounds": 2}):
        with pytest.raises(ValueError):
            rt.pnp_refine(X, y, R0, t0, **kw)
        if "K" in kw and kw["K"].shape == (3, 3):
            with pytest.raises(ValueError):
                opr.pnp_refine_lm(X, y, R0, t0, **kw)
    with pytest.raises(ValueError):
        rt.pnp_refine(X, y[:10], R0, t0)
    with pytest.raises(ValueError):
        rt.pnp_refine_batched([X], [y], np.stack([R0, R0]), np.stack([t0, t0]))
    with pytest.raises(ValueError):
        rt.pnp_refine(X, y, R0, t0, mask=inl[:5])
    with pytest.raises(ValueError):
        rg.pnp.pnp_refine(X, y[:, :1], R0, t0)
    with pytest.raises(ValueError):
        opr.pnp_refine_lm(X, y, R0, t0, rounds=2)
    with pytest.raises(ValueError):
        rg.tables.Tables().addNewView(np.eye(3), 1, np.zeros((6, 3)), np.zeros((6, 3)), np.zeros((6, 2)),
                                      np.zeros((6, 2)), refine="nonlinear")
