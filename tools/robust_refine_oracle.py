"""CPU (numpy / SciPy, float64) checker of the robust losses of the PnP pose refinement (``rg_pnp_refine_*2``,
``runtime.pnp_refine_batched(loss=, f_scale=)``) and of the gold-standard refinement (``rg_gold_standard_*2``,
``runtime.gold_standard(loss=, f_scale=)``).  Test and measurement infrastructure only: the product package never imports it.

It extends ``oracle/pnp_refine_path.py`` and ``oracle/gs_path.py`` without changing them; with ``loss="linear"`` the two
iterations here ARE those functions.  SciPy's losses (``rho``) come from tools/ba_robust_oracle.py: every scalar residual f
gets z = (f / C)^2, C = f_scale, and the cost is 0.5 * sum C^2 rho(z) (SciPy's ``sol.cost``).
  * ``pnp_refine_lm`` ............ the device PnP iteration with the loss linearised by IRLS (w = rho'(z) between the two
                                    factors of J^T J and J^T r), the cost and the accept / stop tests on the robust cost
  * ``pnp_refine_scipy`` ......... least_squares(method="trf", loss=, f_scale=) on the residuals and the analytic Jacobian of
                                    oracle.pnp_refine_path.pnp_refine_reference, tolerances at their floor
  * ``gold_standard_lm`` ......... the device gold-standard iteration (Schur complement of the point blocks) with IRLS
                                    weights Wl, Wr per correspondence
  * ``gold_standard_scipy`` ...... the reference's least_squares call (fun.py:358) with loss / f_scale and a jac_sparsity
                                    block pattern (small pairs only: finite differences)
  * ``pnp_with_outliers`` ........ the outlier recipe of the tests and tools/robust_refine_bench.py
"""
from __future__ import annotations

import os
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
for _p in (_ROOT, _HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)
from oracle import geom_path as og  # noqa: E402
from oracle import gs_path as ogs  # noqa: E402
from oracle import pnp_path as opnp  # noqa: E402
from oracle import pnp_refine_path as opr  # noqa: E402
from ba_robust_oracle import LOSSES, ROBUST, rho, robust_cost_of_residuals  # noqa: E402,F401


# ---------------------------------------------------------------------------------------------------------------------
# PnP pose refinement
# ---------------------------------------------------------------------------------------------------------------------
def _pnp_system(R, t, X, y, W, loss, f_scale):
    """IRLS normal equations at (R, t): A = J^T Om J, g = J^T Om r, robust cost; Om = diag(rho'(z)) per scalar residual."""
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
    a = np.einsum("ij,njk->nik", W, Pi)
    J = np.concatenate([np.cross(q[:, None, :], a), a], axis=2)
    rh, w = rho(loss, (r / f_scale) ** 2)
    A = np.einsum("nia,ni,nib->ab", J, w, J)
    g = np.einsum("nia,ni->a", J, w * r)
    return A, g, 0.5 * f_scale ** 2 * float(np.sum(rh))


def _pnp_refine_once(X, y, R, t, W, max_iter, ftol, loss, f_scale):
    """opr._refine_once with the robust cost and the IRLS system (same damping, accept and stop rules)."""
    if not (np.all(np.isfinite(R)) and np.all(np.isfinite(t))):
        return R, t, float("nan"), 0, 1
    A, g, cost = _pnp_system(R, t, X, y, W, loss, f_scale)
    if X.shape[0] < 3:
        return R, t, cost, 0, 5
    lam, iters = opr.LAMBDA0, 0
    while True:
        if iters >= max_iter:
            return R, t, cost, iters, 4
        dx = opr._solve(A, g, lam)
        better = False
        if dx is not None:
            pred = 0.5 * float(dx @ A @ dx) + lam * float(np.sum(np.diag(A) * dx * dx))
            tiny = np.sqrt(dx[:3] @ dx[:3]) <= opr.XTOL and np.sqrt(dx[3:] @ dx[3:]) <= opr.XTOL * np.sqrt(t @ t)
            if pred <= ftol * cost or tiny:
                return R, t, cost, iters, 2
            Rn, tn = opr.rodrigues(dx[:3]) @ R, t + dx[3:]
            An, gn, cost_t = _pnp_system(Rn, tn, X, y, W, loss, f_scale)
            better = cost_t < cost
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


def pnp_refine_lm(X, y, R, t, mask=None, K=None, max_iter=50, ftol=1e-12, rounds=1, thr2=None, want_mask=False,
                  loss="linear", f_scale=1.0) -> dict:
    """oracle.pnp_refine_path.pnp_refine_lm with a robust loss; "linear" is that function itself."""
    if loss == "linear":
        return opr.pnp_refine_lm(X, y, R, t, mask=mask, K=K, max_iter=max_iter, ftol=ftol, rounds=rounds, thr2=thr2,
                                 want_mask=want_mask)
    rho(loss, 0.0)                                                  # unknown loss: ValueError
    X = np.asarray(X, dtype=np.float64).reshape(-1, 3)
    y = np.asarray(y, dtype=np.float64).reshape(-1, 2)
    R = np.asarray(R, dtype=np.float64).reshape(3, 3)
    t = np.asarray(t, dtype=np.float64).reshape(3)
    W = opr.weight_from_K(K)
    sel = np.ones(X.shape[0], bool) if mask is None else np.asarray(mask).astype(bool)
    if (int(rounds) > 1 or want_mask) and thr2 is None:
        raise ValueError("rounds > 1 or a consensus mask needs thr2")
    out = {}
    for _ in range(int(rounds)):
        R, t, cost, iters, status = _pnp_refine_once(X[sel], y[sel], R, t, W, int(max_iter), float(ftol), loss,
                                                     float(f_scale))
        out = {"R": R, "t": t, "cost": cost, "iters": iters, "status": status}
        if int(rounds) > 1 or want_mask:
            with np.errstate(invalid="ignore"):
                sel = float(thr2) >= opnp.reprojection_error_sq(R, t, X, np.hstack([y, np.ones((y.shape[0], 1))]))
            out["mask"] = sel.astype(np.uint8)
    return out


def pnp_cost(R, t, X, y, K=None, loss="linear", f_scale=1.0) -> float:
    return robust_cost_of_residuals(opr.reprojection_residuals(R, t, X, y, opr.weight_from_K(K)).ravel(), loss, f_scale)


def pnp_refine_scipy(X, y, R, t, mask=None, K=None, loss="linear", f_scale=1.0):
    """least_squares(method="trf", loss=, f_scale=) on the cost of pnp_refine_reference (same residuals, same analytic
    Jacobian, R = exp([w]_x) R0), tolerances at their floor.  Returns R, t, cost (SciPy's robust sol.cost)."""
    from scipy.optimize import least_squares
    X = np.asarray(X, dtype=np.float64).reshape(-1, 3)
    y = np.asarray(y, dtype=np.float64).reshape(-1, 2)
    if mask is not None:
        sel = np.asarray(mask).astype(bool)
        X, y = X[sel], y[sel]
    R0 = np.asarray(R, dtype=np.float64).reshape(3, 3)
    W = opr.weight_from_K(K)

    def fun(p):
        return opr.reprojection_residuals(opr.rodrigues(p[:3]) @ R0, p[3:], X, y, W).ravel()

    def jac(p):
        w = p[:3]
        th = float(np.sqrt(w @ w))
        Wx = np.array([[0.0, -w[2], w[1]], [w[2], 0.0, -w[0]], [-w[1], w[0], 0.0]])
        if th < 1e-4:
            b, c = 0.5 - th * th / 24.0, 1.0 / 6.0 - th * th / 120.0
        else:
            b, c = (1.0 - np.cos(th)) / th ** 2, (th - np.sin(th)) / th ** 3
        Jl = np.eye(3) + b * Wx + c * (Wx @ Wx)
        q = X @ (opr.rodrigues(w) @ R0).T
        pc = q + p[3:]
        iz = 1.0 / pc[:, 2]
        Pi = np.zeros((X.shape[0], 2, 3))
        Pi[:, 0, 0] = iz
        Pi[:, 0, 2] = -pc[:, 0] * iz * iz
        Pi[:, 1, 1] = iz
        Pi[:, 1, 2] = -pc[:, 1] * iz * iz
        a = np.einsum("ij,njk->nik", W, Pi)
        return np.concatenate([np.cross(q[:, None, :], a) @ Jl, a], axis=2).reshape(-1, 6)

    p0 = np.r_[np.zeros(3), np.asarray(t, dtype=np.float64).reshape(3)]
    ls = least_squares(fun, p0, jac=jac, method="trf", loss=loss, f_scale=float(f_scale), xtol=1e-15, ftol=1e-15,
                       gtol=1e-15, max_nfev=2000)
    return opr.rodrigues(ls.x[:3]) @ R0, ls.x[3:].copy(), float(ls.cost)


def pnp_with_outliers(y, frac=0.05, seed=0):
    """A copy of the image points y (N, 2) with int(frac * N) rows replaced by uniform draws over their bounding box
    (numpy default_rng(seed)).  Returns (y_out, indices of the replaced rows)."""
    y = np.asarray(y, dtype=np.float64)
    rng = np.random.default_rng(seed)
    n = int(frac * len(y))
    idx = np.sort(rng.choice(len(y), n, replace=False))
    out = y.copy()
    out[idx] = rng.uniform(y.min(axis=0), y.max(axis=0), (n, 2))
    return out, idx


# ---------------------------------------------------------------------------------------------------------------------
# gold-standard refinement
# ---------------------------------------------------------------------------------------------------------------------
def gs_cost(C1, X, in1, in2, loss="linear", f_scale=1.0) -> float:
    if loss == "linear":
        return ogs.cost(C1, X, in1, in2)
    return robust_cost_of_residuals(ogs.fmatrix_residuals_gs(np.hstack((C1.ravel(), X.T.ravel())), in1, in2), loss,
                                    f_scale)


def gold_standard_lm(F, in1, in2, max_iter=50, ftol=1e-12, lam=1e-3, loss="linear", f_scale=1.0, trace=None):
    """oracle.gs_path.gold_standard_lm with a robust loss: per correspondence the IRLS weights Wl (left residuals) and Wr
    (right residuals) enter M = P2^T Wl P2, T = P2^T Wl Q, D = Q^T Wl Q + Pr^T Wr Pr, g_p = -(Q^T Wl rl + Pr^T Wr rr) and the
    right-hand side P2^T Wl rl + T D'^-1 g_p; the cost and the accept test are on 0.5 sum C^2 rho.  "linear" is that
    function itself.  Returns F_gold, cost, iterations, C1, X."""
    if loss == "linear":
        return ogs.gold_standard_lm(F, in1, in2, max_iter=max_iter, ftol=ftol, lam=lam)
    rho(loss, 0.0)
    C1, C2, X = ogs.start_point(F, in1, in2)
    N = in1.shape[1]
    c = gs_cost(C1, X, in1, in2, loss, f_scale)
    it = 0
    for it in range(1, max_iter + 1):
        Xh = np.vstack([X, np.ones(N)])
        y = C1 @ Xh
        rl = in1 - y[:2] / y[2]
        rr = in2 - X[:2] / X[2]
        wl = rho(loss, (rl / f_scale) ** 2)[1]
        wr = rho(loss, (rr / f_scale) ** 2)[1]
        S = np.zeros((12, 12)); rhs = np.zeros(12); dA = np.zeros(12)
        blocks = []
        for i in range(N):
            Wl, Wr = np.diag(wl[:, i]), np.diag(wr[:, i])
            P2 = np.array([[1, 0, -y[0, i] / y[2, i]], [0, 1, -y[1, i] / y[2, i]]]) / y[2, i]
            Q = P2 @ C1[:, :3]
            Pr = np.array([[1, 0, -X[0, i] / X[2, i]], [0, 1, -X[1, i] / X[2, i]]]) / X[2, i]
            M, T = P2.T @ Wl @ P2, P2.T @ Wl @ Q
            D = Q.T @ Wl @ Q + Pr.T @ Wr @ Pr
            gp = -(Q.T @ Wl @ rl[:, i]) - Pr.T @ Wr @ rr[:, i]
            Di = np.linalg.inv(D + lam * np.diag(np.diag(D)))
            XX = np.outer(Xh[:, i], Xh[:, i])
            S += np.kron(M - T @ Di @ T.T, XX)
            dA += np.kron(np.diag(M), np.diag(XX))
            rhs += np.kron(P2.T @ Wl @ rl[:, i] + T @ Di @ gp, Xh[:, i])
            blocks.append((T, Di, gp))
        try:
            dc = np.linalg.solve(S + lam * np.diag(dA), rhs).reshape(3, 4)
        except np.linalg.LinAlgError:
            lam *= 10.0
            continue
        Xn = X.copy()
        for i in range(N):
            T, Di, gp = blocks[i]
            Xn[:, i] = X[:, i] + Di @ (-gp - T.T @ (dc @ Xh[:, i]))
        cn = gs_cost(C1 + dc, Xn, in1, in2, loss, f_scale)
        if trace is not None:
            trace.append(dict(it=it, lam=lam, cost=c, cost_trial=cn))
        if cn < c:
            conv = c - cn <= ftol * c
            C1, X, c = C1 + dc, Xn, cn
            lam = max(lam * 0.1, 1e-15)
            if conv:
                break
        else:
            lam *= 10.0
            if lam > 1e12:
                break
    return og.fmatrix_from_cameras(C1, C2), c, it, C1, X


def gs_gradient(C1, X, in1, in2, loss, f_scale):
    """The exact gradient J^T Om r of gs_cost (in the sign convention of the residuals, r = measured - predicted: the
    gradient of the cost is -J_pred^T Om r) over params = [C1.ravel(), X.T.ravel()], from the same blocks as
    gold_standard_lm.  For the finite-difference check of the tests."""
    N = in1.shape[1]
    Xh = np.vstack([X, np.ones(N)])
    y = C1 @ Xh
    rl = in1 - y[:2] / y[2]
    rr = in2 - X[:2] / X[2]
    wl = rho(loss, (rl / f_scale) ** 2)[1]
    wr = rho(loss, (rr / f_scale) ** 2)[1]
    gC = np.zeros(12)
    gX = np.zeros((3, N))
    for i in range(N):
        P2 = np.array([[1, 0, -y[0, i] / y[2, i]], [0, 1, -y[1, i] / y[2, i]]]) / y[2, i]
        Q = P2 @ C1[:, :3]
        Pr = np.array([[1, 0, -X[0, i] / X[2, i]], [0, 1, -X[1, i] / X[2, i]]]) / X[2, i]
        gC -= np.kron(P2.T @ (wl[:, i] * rl[:, i]), Xh[:, i])
        gX[:, i] = -(Q.T @ (wl[:, i] * rl[:, i]) + Pr.T @ (wr[:, i] * rr[:, i]))
    return np.concatenate([gC, gX.T.ravel()])


def pnp_gradient(R, t, X, y, K, loss, f_scale):
    """J^T Om r of the PnP cost in the device's parametrisation (left rotation increment, t increment)."""
    return _pnp_system(np.asarray(R, float), np.asarray(t, float), np.asarray(X, float), np.asarray(y, float),
                       opr.weight_from_K(K), loss, f_scale)[1]


def gs_sparsity(N):
    """jac_sparsity of fmatrix_residuals_gs: residual rows [leftx (N), lefty (N), rightx (N), righty (N)] over
    params [C1 (12), X.T.ravel() (3N)] — the left rows see C1 and their point, the right rows only their point."""
    from scipy.sparse import lil_matrix
    S = lil_matrix((4 * N, 12 + 3 * N), dtype=int)
    for i in range(N):
        for k in range(2):
            S[k * N + i, :12] = 1
        for k in range(4):
            S[k * N + i, 12 + 3 * i:15 + 3 * i] = 1
    return S


def gold_standard_scipy(F, in1, in2, loss="linear", f_scale=1.0):
    """The reference's call (fun.py:358: xtol=2.22e-14, tr_solver='lsmr') with loss / f_scale and the block
    jac_sparsity pattern.  Returns F_gold and the OptimizeResult (sol.cost = 0.5 sum C^2 rho)."""
    from scipy.optimize import least_squares
    C1, C2, X = ogs.start_point(F, in1, in2)
    sol = least_squares(ogs.fmatrix_residuals_gs, np.hstack((C1.ravel(), X.T.ravel())), xtol=2.22e-14, tr_solver='lsmr',
                        jac_sparsity=gs_sparsity(in1.shape[1]), loss=loss, f_scale=float(f_scale), args=(in1, in2))
    return og.fmatrix_from_cameras(sol.x[:12].reshape(3, 4), C2), sol
