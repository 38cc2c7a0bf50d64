"""Mirror of the reference's ``pnp`` module.

``pnp_minimize(_3d_pts, img_pts, m)`` implements the algorithm that the reference only specifies as a docstring outline
(pnp.py:132-152; its code body pnp.py:163-196 is unfinished and returns undefined names): DLT over the rows of
[y_k]_x x_k^T, smallest right singular vector -> C0 = (A|b), tau = sign det A, R = U V^T of tau*A, t = 3 tau / tr(S) b.
The arithmetic runs on the GPU (Givens-QR reduction + register-resident one-sided Jacobi, csrc/tall.cuh).

``p3p`` is kept importable because main.py:11, tables.py:6 and ransac.py:2 import the name; the reference body is an
OpenCV call that raises on its own return unpacking (pnp.py:7-10) — out of scope (SURVEY.md section 2, row 6).
"""
from __future__ import annotations

import numpy as np

from . import runtime as _rt


def _split_inputs(_3d_pts, img_pts, m):
    X = np.asarray(_3d_pts, dtype=np.float64)
    y = np.asarray(img_pts, dtype=np.float64)
    if X.ndim != 2 or y.ndim != 2 or X.shape[0] != y.shape[0]:
        raise ValueError("_3d_pts must be (m, 4) or (m, 3) and img_pts (m, 3) or (m, 2), with the same m")
    if m is not None:
        X, y = X[:m], y[:m]
    if X.shape[1] == 4:                      # homogeneous world points -> inhomogeneous
        X = X[:, :3] / X[:, 3:4]
    elif X.shape[1] != 3:
        raise ValueError("_3d_pts must have 3 or 4 columns")
    if y.shape[1] == 3:                      # C-normalised homogeneous image points -> inhomogeneous
        y = y[:, :2] / y[:, 2:3]
    elif y.shape[1] != 2:
        raise ValueError("img_pts must have 2 or 3 columns")
    return np.ascontiguousarray(X), np.ascontiguousarray(y)


def pnp_minimize(_3d_pts, img_pts, m=None):
    """PnP by algebraic minimisation.

    _3d_pts : (m, 4) homogeneous (or (m, 3)) world points, m >= 6
    img_pts : (m, 3) C-normalised homogeneous (or (m, 2)) image points
    m       : number of correspondences to use (default: all)
    Returns R (3, 3), t (3,).  Raises ValueError for m < 6."""
    X, y = _split_inputs(_3d_pts, img_pts, m)
    if X.shape[0] < 6:
        raise ValueError("pnp_minimize needs m >= 6 correspondences")
    return _rt.pnp_minimize(X, y)


def pnp_refine(_3d_pts, img_pts, R, t, K=None, m=None, mask=None, max_iter=50, ftol=1e-12):
    """Geometric refinement of a pose (the final stage of OpenCV's solvePnP(SOLVEPNP_ITERATIVE, useExtrinsicGuess) that
    the reference's cv.solvePnPRansac runs, tables.py:141): Levenberg-Marquardt on 1/2 sum |W (pi(R X + t) - y)|^2 on
    the GPU, W = K[:2, :2] (cost in pixels) or I (C-normalised units).

    _3d_pts, img_pts, m : as pnp_minimize;  R (3, 3), t (3,) : start pose, e.g. from pnp_minimize or ransac_robust
    Returns dict(R, t, cost, iters, status) (see runtime.pnp_refine_batched)."""
    X, y = _split_inputs(_3d_pts, img_pts, m)
    if mask is not None and m is not None:
        mask = np.asarray(mask)[:m]
    return _rt.pnp_refine(X, y, R, t, mask=mask, K=K, max_iter=max_iter, ftol=ftol)


def p3p(_3d_pts, img_pts, K):
    """Name kept for import compatibility (main.py:11, tables.py:6, ransac.py:2).  The reference implementation is a
    cv2.solvePnP call whose 3-tuple result is unpacked into two names, i.e. it always raises ValueError (pnp.py:7-10);
    a minimal 3-point solver is outside the accelerated path (SURVEY.md section 2 row 6)."""
    raise ValueError("p3p is not part of the accelerated path (the reference's p3p raises as well: pnp.py:7-10); "
                     "use pnp_minimize / ransac.ransac_robust with n >= 6")
