"""CPU (numpy / SciPy, float64) checker of the robust-loss bundle adjustment (``runtime.bundle_adjust(loss=, f_scale=)``,
``rg_bundle_adjust_host2``).  Test and measurement infrastructure only: the product package never imports it.

It extends ``oracle/ba_path.py`` without changing it; with ``loss="linear"`` every function here returns exactly what the
corresponding ``oracle.ba_path`` function returns.
  * ``rho`` / ``robust_cost`` ...... SciPy's losses (scipy/optimize/_lsq/least_squares.py, construct_loss_function): every
                                      scalar residual f of EpsilonBA gets z = (f / C)^2, C = f_scale, and the cost is
                                      0.5 * sum C^2 rho(z) (SciPy's ``sol.cost``)
  * ``bundle_adjust_scipy`` ........ the reference's least_squares call (tables.py:317) with ``loss`` / ``f_scale`` added
  * ``bundle_adjust_lm`` ........... the numpy restatement of the device iteration (oracle.ba_path.bundle_adjust_lm) with the
                                      robust loss linearised by IRLS: each residual row and its Jacobian row weighted by
                                      sqrt(rho'(z)), the cost and the accept test on the robust cost
  * ``with_outliers`` / ``clean_rms_px``  the outlier recipe of the tests and tools/ba_robust_bench.py
"""
from __future__ import annotations

import os
import sys

import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if _ROOT not in sys.path:
    sys.path.insert(0, _ROOT)
from oracle import ba_path as oba  # noqa: E402

LOSSES = ("linear", "soft_l1", "huber", "cauchy", "arctan")
ROBUST = LOSSES[1:]
FOCAL_PX = 3217.0            # K[0, 0] of the Dino data: one pixel in C-normalised coordinates is 1 / FOCAL_PX


def rho(loss, z):
    """(rho(z), rho'(z)) of SciPy's loss ``loss`` (least_squares.py: linear, soft_l1, huber, cauchy, arctan)."""
    z = np.asarray(z, dtype=np.float64)
    if loss == "linear":
        return z.copy(), np.ones_like(z)
    if loss == "soft_l1":
        t = 1.0 + z
        return 2.0 * (t ** 0.5 - 1.0), t ** -0.5
    if loss == "huber":
        mask = z <= 1.0
        r0 = np.where(mask, z, 2.0 * np.sqrt(np.where(mask, 1.0, z)) - 1.0)
        r1 = np.where(mask, 1.0, np.where(mask, 1.0, z) ** -0.5)
        return r0, r1
    if loss == "cauchy":
        return np.log1p(z), 1.0 / (1.0 + z)
    if loss == "arctan":
        return np.arctan(z), 1.0 / (1.0 + z ** 2)
    raise ValueError(f"unknown loss {loss!r}")


def robust_cost_of_residuals(r, loss="linear", f_scale=1.0) -> float:
    if loss == "linear":
        return 0.5 * float(r @ r)
    return 0.5 * f_scale ** 2 * float(np.sum(rho(loss, (r / f_scale) ** 2)[0]))


def robust_cost(cams, pts, uv, cam_idx, pt_idx, loss="linear", f_scale=1.0) -> float:
    """0.5 * sum C^2 rho((f / C)^2) over the interleaved EpsilonBA residuals (= oracle.ba_path.cost for "linear")."""
    if loss == "linear":
        return oba.cost(cams, pts, uv, cam_idx, pt_idx)
    r = oba.residuals(oba.pack(cams, pts), uv[:, 0], uv[:, 1], cam_idx, pt_idx, len(cams), len(pts))
    return robust_cost_of_residuals(r, loss, f_scale)


def bundle_adjust_scipy(cams, pts, uv, cam_idx, pt_idx, loss="linear", f_scale=1.0, ftol=1e-4):
    """The reference's least_squares call (tables.py:317) with loss / f_scale passed through."""
    if loss == "linear" and ftol == 1e-4:
        return oba.bundle_adjust_scipy(cams, pts, uv, cam_idx, pt_idx)
    from scipy.optimize import least_squares
    n_C, n_P = len(cams), len(pts)
    sol = least_squares(oba.residuals, oba.pack(cams, pts), args=(uv[:, 0], uv[:, 1], cam_idx, pt_idx, n_C, n_P),
                        jac_sparsity=oba.sparsity_mask(cam_idx, pt_idx, n_C, n_P), x_scale="jac", ftol=ftol, method="trf",
                        loss=loss, f_scale=f_scale)
    C, X = oba.unpack(sol.x, n_C, n_P)
    return C, X, sol


def bundle_adjust_lm(cams, pts, uv, cam_idx, pt_idx, n_fixed=1, max_iter=50, ftol=1e-12, lam=1e-3, loss="linear",
                     f_scale=1.0, trace=None):
    """oracle.ba_path.bundle_adjust_lm with a robust loss (IRLS weights w = rho'(z) per residual component, recomputed at
    every linearisation); "linear" is that function itself.  Returns cameras, points, cost, iterations, status."""
    if loss == "linear":
        return oba.bundle_adjust_lm(cams, pts, uv, cam_idx, pt_idx, n_fixed=n_fixed, max_iter=max_iter, ftol=ftol,
                                    lam=lam, trace=trace)
    rho(loss, 0.0)                                                  # unknown loss: ValueError
    C = np.array(cams, dtype=np.float64).reshape(-1, 3, 4)
    X = np.array(pts, dtype=np.float64).reshape(-1, 3)
    uv = np.asarray(uv, dtype=np.float64)
    cam_idx = np.asarray(cam_idx, dtype=np.int64)
    pt_idx = np.asarray(pt_idx, dtype=np.int64)
    n_C, n_P, n_O = len(C), len(X), len(uv)
    n_free = n_C - n_fixed

    def cost_of(Cc, Xc):
        return robust_cost(Cc, Xc, uv, cam_idx, pt_idx, loss, f_scale)

    c = cost_of(C, X)
    floor = 0.5 * float(np.sum(uv * uv)) * (64.0 * np.finfo(np.float64).eps) ** 2
    status, it = 4, 0
    if n_free <= 0 and n_P == 0:
        return C, X, c, 0, 2
    for it in range(1, max_iter + 1):
        Xh = np.concatenate([X, np.ones((n_P, 1))], axis=1)
        xo = Xh[pt_idx]
        y = np.einsum("oab,ob->oa", C[cam_idx], xo)
        iy = 1.0 / y[:, 2]
        pred = y[:, :2] * iy[:, None]
        r = uv - pred
        W = rho(loss, (r / f_scale) ** 2)[1]                         # (O, 2) IRLS weights
        Wr = W * r
        P2 = np.zeros((n_O, 2, 3))
        P2[:, 0, 0] = iy; P2[:, 1, 1] = iy
        P2[:, 0, 2] = -pred[:, 0] * iy; P2[:, 1, 2] = -pred[:, 1] * iy
        Q = np.einsum("oka,oac->okc", P2, C[cam_idx][:, :, :3])
        M = np.einsum("oka,ok,okb->oab", P2, W, P2)
        T = np.einsum("oka,ok,okc->oac", P2, W, Q)
        V = np.zeros((n_P, 3, 3)); gp = np.zeros((n_P, 3))
        np.add.at(V, pt_idx, np.einsum("oka,ok,okb->oab", Q, W, Q))
        np.add.at(gp, pt_idx, np.einsum("oka,ok->oa", Q, Wr))
        Vd = V + lam * np.einsum("pab,ab->pab", V, np.eye(3))
        seen = np.zeros(n_P, dtype=bool); seen[pt_idx] = True
        Vd[~seen] = np.eye(3)
        Vi = np.linalg.inv(Vd)
        Vi[~seen] = 0.0
        e = np.einsum("pab,pb->pa", Vi, gp)
        XX = np.einsum("oa,ob->oab", xo, xo)
        n = 12 * n_C
        S = np.zeros((n, n)); rhs = np.zeros(n); dU = np.zeros(n)
        U = np.einsum("oab,ocd->oacbd", M, XX).reshape(n_O, 12, 12)
        z = np.einsum("oka,ok->oa", P2, Wr) - np.einsum("oac,oc->oa", T, e[pt_idx])
        for o in range(n_O):
            k = cam_idx[o]
            S[12 * k:12 * k + 12, 12 * k:12 * k + 12] += U[o]
            dU[12 * k:12 * k + 12] += np.diag(U[o])
            rhs[12 * k:12 * k + 12] += np.kron(z[o], xo[o])
        order = np.argsort(pt_idx, kind="stable")
        starts = np.searchsorted(pt_idx[order], np.arange(n_P + 1))
        for j in range(n_P):
            oj = order[starts[j]:starts[j + 1]]
            for o in oj:
                for o2 in oj:
                    k, l = cam_idx[o], cam_idx[o2]
                    S[12 * k:12 * k + 12, 12 * l:12 * l + 12] -= np.kron(T[o] @ Vi[j] @ T[o2].T, XX[o])
        S[np.arange(n), np.arange(n)] += np.where(dU > 0.0, lam * dU, 1.0)
        f0 = 12 * n_fixed
        dc = np.zeros(n)
        ok = True
        if n_free > 0:
            try:
                L = np.linalg.cholesky(S[f0:, f0:])
                dc[f0:] = np.linalg.solve(L.T, np.linalg.solve(L, rhs[f0:]))
            except np.linalg.LinAlgError:
                ok = False
        if ok:
            dC = dc.reshape(n_C, 3, 4)
            q = np.einsum("oab,ob->oa", dC[cam_idx], xo)
            back = np.zeros((n_P, 3))
            np.add.at(back, pt_idx, np.einsum("oac,oa->oc", T, q))
            dX = np.einsum("pab,pb->pa", Vi, gp - back)
            Cn, Xn = C + dC, X + dX
            cn = cost_of(Cn, Xn)
            if not np.isfinite(cn):
                cn = np.inf
        if trace is not None:
            trace.append(dict(it=it, lam=lam, cost=c, cost_trial=cn if ok else np.nan, ok=ok))
        if ok and cn < c:
            gain = c - cn
            conv = gain <= ftol * c or cn <= floor
            C, X, c = Cn, Xn, cn
            lam = max(lam * 0.1, 1e-15)
            if conv:
                status = 2
                break
        else:
            lam *= 10.0
            if lam > 1e12:
                status = 3
                break
    return C, X, c, it, status


def with_outliers(uv, frac=0.05, seed=0):
    """A copy of uv with n = int(frac * O) observations (frac = 0.05: O // 20) replaced by uniform draws over the bounding
    box of uv (numpy default_rng(seed)).  Returns (uv_out, indices of the replaced observations)."""
    uv = np.asarray(uv, dtype=np.float64)
    rng = np.random.default_rng(seed)
    n = len(uv) // 20 if frac == 0.05 else int(frac * len(uv))
    idx = np.sort(rng.choice(len(uv), n, replace=False))
    out = uv.copy()
    out[idx] = rng.uniform(uv.min(axis=0), uv.max(axis=0), (n, 2))
    return out, idx


def clean_rms_px(cams, pts, uv_clean, cam_idx, pt_idx, outlier_idx, focal=FOCAL_PX) -> float:
    """Reprojection RMS (pixels, x focal): root mean of |uv - projection|^2 over the observations the outlier recipe
    left untouched."""
    r = oba.residuals(oba.pack(cams, pts), uv_clean[:, 0], uv_clean[:, 1], cam_idx, pt_idx, len(cams), len(pts))
    keep = np.ones(len(uv_clean), dtype=bool)
    keep[outlier_idx] = False
    rr = r.reshape(-1, 2)[keep]
    return float(np.sqrt(np.mean(np.sum(rr * rr, axis=1)))) * focal
