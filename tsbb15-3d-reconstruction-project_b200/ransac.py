"""Mirror of the reference's ``ransac`` module (PnP-RANSAC).

The reference's ``ransac_robust`` (ransac.py:37-113) is a non-running skeleton: it calls ``p3p`` with the wrong arity
(:82), indexes ``len(D_high[0])`` (:77) and ``C_est[0]`` of an empty list (:108).  Its semantics are kept:

    repeat r times: draw n correspondences from D_high (gen_rnd_indices, :12-19, :77-78); solve a pose; for every
    correspondence of D_med and D_high compute y' = R x + t (:34-35, :96-97) and e = |pnorm(y) - pnorm(y')|^2
    (:31-32, :100-101); the consensus set is ``thresh >= e`` (inclusive, :104-105); keep the pose whose D_med consensus
    is the largest (``len(C[0])``, :108; strict > so the first maximum wins); return R_est, t_est, C_est.

with the pose solver the reference specifies in pnp.py:132-152 (``pnp.pnp_minimize``), which needs n >= 6 — for n == 3
and n == 4 the reference's own error behaviour is kept (:81-89).  Solving and scoring run on the GPU.

Data layout: ``D[:, 0]`` are C-normalised homogeneous image points and ``D[:, 1]`` world points (ransac.py:67-70,
96-97), i.e. a float array of shape (N, 2, 3).
"""
from __future__ import annotations

import numpy as np

from . import runtime as _rt
from .sampling import gen_rnd_indices  # noqa: F401  (same name and behaviour as ransac.py:12-19)


def calc_p(w, n, r):
    """Probability that at least one of r samples of size n is outlier-free (ransac.py:6-7)."""
    return 1 - np.power(1 - np.power(w, n), r)


def calc_r(w, n, p):
    """Number of trials needed to reach success probability p (ransac.py:9-10)."""
    return np.log(1 - p) / np.log(1 - np.power(w, n))


def norm_p(v):
    """P-normalise: divide by the last coordinate; returns a list like the reference (ransac.py:21-23)."""
    v = np.array(v)
    return np.ndarray.tolist(v / v[-1])


def cart(v):
    return norm_p(v)[0:-1]


def dpp(y1, y2):
    d = np.asarray(norm_p(y1)) - np.asarray(norm_p(y2))
    return np.sqrt(np.dot(d, d))


def dpp_squared(y1, y2):
    d = np.asarray(norm_p(y1)) - np.asarray(norm_p(y2))
    return np.dot(d, d)


def calc_y_prim(x, R, t):
    return (R @ x) + t


def _as_pairs(D, name):
    D = np.asarray(D, dtype=np.float64)
    if D.ndim != 3 or D.shape[1] != 2 or D.shape[2] != 3:
        raise ValueError(f"{name} must have shape (N, 2, 3): [:, 0] C-normalised image points, [:, 1] 3D points")
    return D


def ransac_robust(D_med, D_high, r, thresh, n, sample_idx=None, seed=None, refine=False):
    """RANSAC estimation of the camera pose.

    D_med, D_high : (N, 2, 3) correspondences, [:, 0] = C-normalised homogeneous image point, [:, 1] = 3D point
    r             : number of trials
    thresh        : consensus threshold on the squared image distance (inclusive)
    n             : sample size; n >= 6 uses the DLT pose of pnp.pnp_minimize (6, 7 or 8)
    sample_idx    : optional (r, n) host-drawn indices into D_high (otherwise gen_rnd_indices is called r times; with
                    ``seed`` the global ``random`` module is seeded first)
    refine        : False (default): the winner's algebraic DLT pose.  True: the winner is refined on its consensus set
                    (Levenberg-Marquardt on the reprojection error in C-normalised units, runtime.pnp_refine) and C_est
                    is re-scored at the refined pose
    Returns R_est, t_est, C_est as one-element lists like the reference intends (:109-111): [R], [t],
    [[D_med consensus rows, D_high consensus rows]]; three empty lists if no pose has any D_med consensus."""
    if n == 3:
        from .pnp import p3p
        return p3p(None, None, None)           # reference :81-82 -> raises
    if n == 4:
        raise ValueError("Not implemented yet")                                   # reference :84-86
    if n < 6 or n > 8:
        raise ValueError("No PnP algorithm with the given n is implemented")      # reference :88-89
    D_med = _as_pairs(D_med, "D_med")
    D_high = _as_pairs(D_high, "D_high")
    n_high = D_high.shape[0]
    if sample_idx is None:
        if seed is not None:
            import random
            random.seed(seed)
        sample_idx = np.array([gen_rnd_indices(n_high, n) for _ in range(int(r))], dtype=np.int32).reshape(-1, n)
    sample_idx = np.ascontiguousarray(sample_idx, dtype=np.int32)
    if sample_idx.ndim != 2 or sample_idx.shape[1] != n:
        raise ValueError("sample_idx must be (r, n)")
    n_med = D_med.shape[0]
    # selection votes on D_med only (reference :108); both sets are scored for the returned consensus
    both = np.concatenate([D_med, D_high], axis=0)
    y = both[:, 0, :2] / both[:, 0, 2:3]
    X = both[:, 1, :]
    res = _rt.pnp_ransac(X, y, sample_idx + n_med, float(thresh), n_sel=n_med, want_mask=True)
    if res["best_idx"] < 0:
        return [], [], []
    R, t, mask = res["R"], res["t"], res["mask"].astype(bool)
    if refine:
        ref = _rt.pnp_refine(X, y, R, t, mask=mask, thr2=float(thresh))
        R, t, mask = ref["R"], ref["t"], ref["mask"].astype(bool)
    C = [D_med[mask[:n_med]], D_high[mask[n_med:]]]
    return [R], [t], [C]
