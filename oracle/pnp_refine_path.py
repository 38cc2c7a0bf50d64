"""TEST INFRASTRUCTURE ONLY — CPU (numpy, float64) restatement of the device refinement of PnP poses
(csrc/pnp_refine_kernels.cuh) and the reference minimiser it is pinned against.

The reference's live PnP call is OpenCV's ``cv.solvePnPRansac`` (tables.py:141), which ends with
``solvePnP(SOLVEPNP_ITERATIVE, useExtrinsicGuess)`` on the inliers: a Levenberg-Marquardt minimisation of the
reprojection error.  The cost restated here (DESIGN.md section 4.7):

    C(R, t) = 1/2 sum_k || W (pi(R X_k + t) - y_k) ||^2,   pi(p) = (p0 / p2, p1 / p2),   W = [[fx, s], [0, fy]] (or I)

The principal point of K cancels.  pi is sign-agnostic: the points of synth.pnp_scene all have negative depth.

  * ``pnp_refine_lm``        — the device iteration step by step (same parametrisation R <- exp([dw]_x) R, t <- t + dt,
                               same Marquardt damping schedule, same accept / stop rules and status codes), dense numpy;
  * ``pnp_refine_reference`` — SciPy ``least_squares(method="lm")`` on the same cost: the reference minimum.
"""
from __future__ import annotations

import numpy as np

from .pnp_path import reprojection_error_sq

LAMBDA0 = 1e-3
XTOL = 1e-14          # a step below this (radians; relative for t) is rounding: converged


def rodrigues(w) -> np.ndarray:
    """exp([w]_x) in FP64; (1 - cos th) / th^2 is formed as 2 sin^2(th/2) / th^2 (no cancellation for small th)."""
    w = np.asarray(w, dtype=np.float64)
    th = float(np.sqrt(w @ w))
    if th == 0.0:
        a, b = 1.0, 0.5
    else:
        a = np.sin(th) / th
        h = np.sin(0.5 * th) / (0.5 * th)
        b = 0.5 * h * h
    Wx = np.array([[0.0, -w[2], w[1]], [w[2], 0.0, -w[0]], [-w[1], w[0], 0.0]])
    return np.eye(3) + a * Wx + b * (Wx @ Wx)


def weight_from_K(K) -> np.ndarray:
    """Upper-left 2x2 of K; ValueError unless K is (3, 3) with bottom row (0, 0, 1) and K[1, 0] == 0."""
    if K is None:
        return np.eye(2)
    K = np.asarray(K, dtype=np.float64)
    if K.shape != (3, 3) or K[1, 0] != 0.0 or not np.array_equal(K[2], [0.0, 0.0, 1.0]):
        raise ValueError("K must be (3, 3) with K[1, 0] == 0 and bottom row (0, 0, 1)")
    return K[:2, :2].copy()


def reprojection_residuals(R, t, X, y, W=None) -> np.ndarray:
    """(N, 2) residuals W (pi(R X + t) - y)."""
    p = np.asarray(X, dtype=np.float64) @ np.asarray(R, dtype=np.float64).T + np.asarray(t, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        d = p[:, :2] / p[:, 2:3] - np.asarray(y, dtype=np.float64)
    return d if W is None else d @ np.asarray(W, dtype=np.float64).T


def _system(R, t, X, y, W):
    """Normal equations at (R, t): A = J^T J (6x6), g = J^T r, r; J_k = W Pi_k [-[R X_k]_x | I]."""
    q = X @ R.T
    p = q + t
    with np.errstate(divide="ignore", invalid="ignore"):
        iz = 1.0 / p[:, 2]
        u, v = p[:, 0] * iz, p[:, 1] * iz
    r = np.stack([u - y[:, 0], v - y[:, 1]], axis=1) @ W.T
    n = X.shape[0]
    Pi = np.zeros((n, 2, 3))
    Pi[:, 0, 0] = iz
    Pi[:, 0, 2] = -u * iz
    Pi[:, 1, 1] = iz
    Pi[:, 1, 2] = -v * iz
    a = np.einsum("ij,njk->nik", W, Pi)                         # (n, 2, 3) rows of W Pi
    J = np.concatenate([np.cross(q[:, None, :], a), a], axis=2)  # row a times -[q]_x = q x a
    A = np.einsum("nia,nib->ab", J, J)
    g = np.einsum("nia,ni->a", J, r)
    return A, g, r


def _solve(A, g, lam):
    """(A + lam diag A) dx = -g by Cholesky; None when the damped system is not positive definite / not finite."""
    if not (np.all(np.isfinite(A)) and np.all(np.isfinite(g))):
        return None
    M = A + lam * np.diag(np.diag(A))
    try:
        L = np.linalg.cholesky(M)
    except np.linalg.LinAlgError:
        return None
    dx = -np.linalg.solve(L.T, np.linalg.solve(L, g))
    return dx if np.all(np.isfinite(dx)) else None


def _refine_once(X, y, R, t, W, max_iter, ftol):
    """One LM run on the selected points.  Returns R, t, cost, iters, status."""
    if not (np.all(np.isfinite(R)) and np.all(np.isfinite(t))):
        return R, t, float("nan"), 0, 1
    A, g, r = _system(R, t, X, y, W)
    cost = 0.5 * float(np.sum(r * r))
    if X.shape[0] < 3:
        return R, t, cost, 0, 5
    lam, iters = LAMBDA0, 0
    while True:
        if iters >= max_iter:
            return R, t, cost, iters, 4
        dx = _solve(A, g, lam)
        better = False
        if dx is not None:
            # decrease the linear model predicts: 1/2 dx^T A dx + lam dx^T diag(A) dx (a sum of positive terms).  When it
            # is below ftol * cost the step is not taken: the actual decrease would be below the rounding error of the cost
            pred = 0.5 * float(dx @ A @ dx) + lam * float(np.sum(np.diag(A) * dx * dx))
            # ... or the step would move the pose by no more than rounding (zero-residual data reach that floor)
            tiny = np.sqrt(dx[:3] @ dx[:3]) <= XTOL and np.sqrt(dx[3:] @ dx[3:]) <= XTOL * np.sqrt(t @ t)
            if pred <= ftol * cost or tiny:
                return R, t, cost, iters, 2
            Rn, tn = rodrigues(dx[:3]) @ R, t + dx[3:]
            An, gn, rn = _system(Rn, tn, X, y, W)
            cost_t = 0.5 * float(np.sum(rn * rn))
            better = cost_t < cost                                  # NaN: not better
        iters += 1
        if better:
            conv = cost - cost_t <= ftol * cost
            R, t, A, g, cost = Rn, tn, An, gn, cost_t
            lam = max(lam * 0.1, 1e-15)
            if conv:
                return R, t, cost, iters, 2
        else:
            lam *= 10.0
            if lam > 1e12:
                return R, t, cost, iters, 3


def pnp_refine_lm(X, y, R, t, mask=None, K=None, max_iter=50, ftol=1e-12, rounds=1, thr2=None, want_mask=False) -> dict:
    """The device refinement of ONE view, restated.  X (N, 3), y (N, 2) C-normalised, (R, t) the start pose; mask (N,)
    selects the points of the first round (default: all).  rounds > 1 (or want_mask) re-scores the consensus
    ``thr2 >= e`` (ransac.py:104-105, e in C-normalised units) at the refined pose after every round; the next round
    refines on it.  Returns {R, t, cost, iters, status[, mask]} of the last round."""
    X = np.asarray(X, dtype=np.float64).reshape(-1, 3)
    y = np.asarray(y, dtype=np.float64).reshape(-1, 2)
    R = np.asarray(R, dtype=np.float64).reshape(3, 3)
    t = np.asarray(t, dtype=np.float64).reshape(3)
    W = weight_from_K(K)
    sel = np.ones(X.shape[0], bool) if mask is None else np.asarray(mask).astype(bool)
    rounds = int(rounds)
    if rounds < 1:
        raise ValueError("rounds must be >= 1")
    if (rounds > 1 or want_mask) and thr2 is None:
        raise ValueError("rounds > 1 or a consensus mask needs thr2")
    out = {}
    for k in range(rounds):
        R, t, cost, iters, status = _refine_once(X[sel], y[sel], R, t, W, int(max_iter), float(ftol))
        out = {"R": R, "t": t, "cost": cost, "iters": iters, "status": status}
        if rounds > 1 or want_mask:
            with np.errstate(invalid="ignore"):
                sel = float(thr2) >= reprojection_error_sq(R, t, X, np.hstack([y, np.ones((y.shape[0], 1))]))
            out["mask"] = sel.astype(np.uint8)
    return out


def pnp_refine_reference(X, y, R, t, mask=None, K=None):
    """SciPy least_squares(method='lm') on the same cost, parametrised as R = exp([w]_x) R0, t; tolerances at their
    floor so that it stops at the minimum.  Returns R, t, cost."""
    from scipy.optimize import least_squares
    X = np.asarray(X, dtype=np.float64).reshape(-1, 3)
    y = np.asarray(y, dtype=np.float64).reshape(-1, 2)
    if mask is not None:
        sel = np.asarray(mask).astype(bool)
        X, y = X[sel], y[sel]
    R0 = np.asarray(R, dtype=np.float64).reshape(3, 3)
    W = weight_from_K(K)

    def fun(p):
        return reprojection_residuals(rodrigues(p[:3]) @ R0, p[3:], X, y, W).ravel()

    def jac(p):
        # d r / d w = (W Pi [-[R X]_x]) J_l(w): the derivative for a left increment times the left Jacobian of exp
        w = p[:3]
        th = float(np.sqrt(w @ w))
        Wx = np.array([[0.0, -w[2], w[1]], [w[2], 0.0, -w[0]], [-w[1], w[0], 0.0]])
        if th < 1e-4:
            b, c = 0.5 - th * th / 24.0, 1.0 / 6.0 - th * th / 120.0
        else:
            b, c = (1.0 - np.cos(th)) / th ** 2, (th - np.sin(th)) / th ** 3
        Jl = np.eye(3) + b * Wx + c * (Wx @ Wx)
        Rp = rodrigues(w) @ R0
        q = X @ Rp.T
        pc = q + p[3:]
        iz = 1.0 / pc[:, 2]
        Pi = np.zeros((X.shape[0], 2, 3))
        Pi[:, 0, 0] = iz
        Pi[:, 0, 2] = -pc[:, 0] * iz * iz
        Pi[:, 1, 1] = iz
        Pi[:, 1, 2] = -pc[:, 1] * iz * iz
        a = np.einsum("ij,njk->nik", W, Pi)
        Jrot = np.cross(q[:, None, :], a) @ Jl
        return np.concatenate([Jrot, a], axis=2).reshape(-1, 6)

    p0 = np.r_[np.zeros(3), np.asarray(t, dtype=np.float64).reshape(3)]
    ls = least_squares(fun, p0, jac=jac, method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=2000)
    return rodrigues(ls.x[:3]) @ R0, ls.x[3:].copy(), float(ls.cost)
