"""Mirror of the reference's ``fun`` module for the F-matrix RANSAC entry point.

``getFFromLabCode(p1, p2)`` keeps the reference's name, argument layout ((2, N) pixel coordinates, as ``main.py:39``
passes them) and return value (the gold-standard refined F, fun.py:291-369).  The 10 000-trial loop of fun.py:303-328
— sample, 8-point solve, epipolar residuals of all N correspondences, threshold, best-hypothesis update — runs as ONE
batched call into the CUDA library; the SciPy Levenberg-Marquardt refinement (fun.py:342-369) stays on the host exactly
as in the reference (SURVEY.md section 8b).

The reference's hard-coded literals are keyword arguments with the same defaults: r=10000 trials (fun.py:302),
thr=1.5 px (fun.py:317), 8 points per sample (fun.py:306).
"""
from __future__ import annotations

import numpy as np

from . import lab3
from .correspondences import Correspondences  # noqa: F401  (fun.Correspondences, main.py:28)
from . import runtime as _rt
from . import sampling as _sampling
from ._cabi import MODE_EPI_MAX, SCORE_FP32_GUARDED, SOLVER_QR, TIE_FIRST, TIE_REFERENCE


def MakeHomogenous(K, coord):
    """C-normalise pixel coordinates: (N, 2) -> (N, 3) rows K^-1 (u, v, 1)^T (fun.py:48-55)."""
    coord = np.asarray(coord, dtype=np.float64).T
    hom = np.ones((3, coord.shape[1]))
    hom[:2] = coord[:2]
    return np.linalg.solve(np.asarray(K, dtype=np.float64), hom).T


def crossProductMat(vec3):
    """[v]_x (fun.py:23-34)."""
    return lab3.cross_matrix(np.asarray(vec3, dtype=np.float64))


def getEFromCameras(C1, C2):
    """Essential matrix of two CameraPose objects: R = R2 R1^T, t = t2 - R t1, E = R^T [t]_x (fun.py:12-21)."""
    R = C2.R @ C1.R.T
    t = C2.t - (C2.R @ C1.R.T @ C1.t)
    return R.T @ crossProductMat(t)


def camera_resectioning(C):
    """K, R, t of a (3, 4) camera C = K [R | t] (fun.py:260-283): K upper triangular with positive diagonal and
    K[2, 2] = 1; signs follow LAPACK's RQ as the reference's do.  GPU (one thread per camera)."""
    C = np.asarray(C, dtype=np.float64)
    if C.shape != (3, 4):
        raise ValueError('C must be a (3, 4) camera matrix')
    K, R, t = _rt.camera_resectioning(C)
    return K[0], R[0], t[0]


def getCameraMatrices(path='BAdino2.mat'):
    """fun.py:75-89: the (1, 36, 3, 4) camera array of BAdino2.mat (read from the working directory like the reference)."""
    import scipy.io as sio
    return np.asarray(sio.loadmat(path)['newPs'].tolist())


def reshapeToCamera3DPoints2(x0, n_C, n_P):
    """fun.py:282-289: the bundle-adjustment parameter vector back to (n_C, 3, 4) cameras and (n_P, 3) points."""
    x0 = np.asarray(x0)
    return np.reshape(x0[:n_C * 12], [n_C, 3, 4]), np.reshape(x0[n_C * 12:], [n_P, 3])


def getEAndK(C, F):
    """E = K^T F K with K taken from the LAST camera of C (1, n, 3, 4), as the reference does (fun.py:91-102)."""
    C = np.asarray(C, dtype=np.float64)
    if C.ndim != 4 or C.shape[2:] != (3, 4):
        raise ValueError('C must have shape (1, n, 3, 4)')
    K, _, _ = _rt.camera_resectioning(C[0])
    K = K[-1]
    return np.matmul(np.matmul(np.transpose(K), np.asarray(F, dtype=np.float64)), K), K


def relative_camera_pose(E, y1, y2):
    """R, t of the second camera from an essential matrix and ONE C-normalised correspondence (fun.py:209-258): the
    first of the four (V W U^T | +-v3), (V W^T U^T | +-v3) candidates whose optimally triangulated point lies in front
    of both cameras.  Returns None when no candidate passes (the reference falls off the end of the function).  GPU:
    four lanes per pair, one candidate each (``relative_camera_pose_batch`` takes P pairs at once)."""
    res = _rt.relative_pose(np.asarray(E, dtype=np.float64).reshape(1, 3, 3), np.asarray(y1, dtype=np.float64).ravel()[:2],
                            np.asarray(y2, dtype=np.float64).ravel()[:2])
    if res["which"][0] < 0:
        return None
    return res["R"][0], res["t"][0]


def relative_camera_pose_batch(M, y1, y2, K=None):
    """P pairs in one call: M (P,3,3) essential matrices (or fundamental matrices with K given), y1, y2 (P, 2).
    Returns dict(R, t, which, npass); which[p] = -1 where the reference would return None."""
    return _rt.relative_pose(M, y1, y2, K=K)


def f_ransac(p1, p2, r=10000, thr=1.5, sample_idx=None, seed=None, sampler="reference", tie="reference",
             mode=MODE_EPI_MAX, solver=SOLVER_QR, score_path=SCORE_FP32_GUARDED, device=None):
    """The RANSAC part of getFFromLabCode (fun.py:298-328) on the GPU.

    sample_idx : optional (H, 8) int array of host-drawn index sets (then ``r`` / ``seed`` / ``sampler`` are ignored).
    sampler    : "reference" replays the reference's own draw ``np.random.choice(arange(N), 8, replace=False)`` from
                 numpy's global state (after ``np.random.seed(s)`` the index sets equal the reference's);
                 "fast" draws from ``default_rng(seed)`` in O(1) per sample.
    tie        : "reference" replays the tie rule of fun.py:324-328, "first" keeps the first maximum.
    Returns dict(F, inliers (index array S_RANSAC), best (hypothesis index), count, idx).
    """
    p1 = np.asarray(p1, dtype=np.float64)
    p2 = np.asarray(p2, dtype=np.float64)
    if p1.shape != p2.shape or p1.ndim != 2 or p1.shape[0] != 2:
        raise ValueError("p1 and p2 must be (2, N) arrays of the same shape")
    n = p1.shape[1]
    if sample_idx is None:
        if sampler == "reference":
            if seed is not None:
                np.random.seed(seed)
            sample_idx = _sampling.reference_stream(n, r, 8)
        elif sampler == "fast":
            sample_idx = _sampling.fast(n, r, 8, seed)
        else:
            raise ValueError("sampler must be 'reference' or 'fast'")
    sample_idx = np.ascontiguousarray(sample_idx, dtype=np.int32)
    if sample_idx.ndim != 2 or sample_idx.shape[1] != 8:
        raise ValueError("sample_idx must be (H, 8)")
    pts = _rt.pack_pairs(p1, p2)
    res = _rt.f_ransac_batched([pts], [sample_idx], thr=thr, mode=mode,
                               tie_mode=TIE_REFERENCE if tie == "reference" else TIE_FIRST, solver=solver,
                               score_path=score_path, want_mask=True, device=device)
    best = int(res["best_idx"][0])
    F = res["F"][0] if best >= 0 else None
    return {"F": F, "inliers": np.flatnonzero(res["mask"][0]), "best": best, "count": int(res["best_count"][0]),
            "idx": sample_idx}


def gold_standard(F_guess, p1, p2, inliers, loss="linear", f_scale=1.0):
    """Gold-standard refinement of fun.py:342-369: cameras from F, optimal triangulation of the inliers, sparse-free
    LM over (C1, X) with C2 = [I|0], F from the refined cameras.  loss / f_scale (pixels) are passed to the
    least_squares call, as a SciPy user adds them there."""
    from scipy.optimize import least_squares
    _rt.loss_args(loss, f_scale)
    C1, C2 = lab3.fmatrix_cameras(F_guess)
    in1 = p1[:, inliers]
    in2 = p2[:, inliers]
    X = lab3.triangulate_optimal_batch(C1, C2, in1.T, in2.T).T          # fun.py:352 loop, one GPU call
    params = np.hstack((C1.ravel(), X.T.ravel()))
    kw = {} if loss == "linear" else {"loss": loss, "f_scale": float(f_scale)}
    sol = least_squares(lab3.fmatrix_residuals_gs, params, xtol=2.22e-14, tr_solver='lsmr', args=(in1, in2), **kw).x
    C1 = sol[:12].reshape(3, 4)
    C2 = np.hstack([np.eye(3), np.zeros((3, 1))])
    return lab3.fmatrix_from_cameras(C1, C2)


def gold_standard_device(F_guess, p1, p2, inliers, max_iter=50, ftol=1e-12, full_output=False, loss="linear", f_scale=1.0):
    """The same minimisation as ``gold_standard`` — cameras from F, optimal triangulation, cost of
    lab3.fmatrix_residuals_gs, F from the refined cameras (fun.py:342-369) — but solved on the GPU by Levenberg-Marquardt
    with a Schur complement instead of SciPy's finite-difference trust-region solver: milliseconds instead of minutes,
    and it reaches the minimum of the cost where the reference's solver stops early on ftol (DESIGN.md 4.5).
    loss / f_scale: SciPy's robust loss options (f_scale in pixels), see runtime.gold_standard."""
    p1 = np.asarray(p1, dtype=np.float64)
    p2 = np.asarray(p2, dtype=np.float64)
    pts = _rt.pack_pairs(p1[:, inliers], p2[:, inliers])
    res = _rt.gold_standard([pts], np.asarray(F_guess, dtype=np.float64).reshape(1, 3, 3), max_iter=max_iter, ftol=ftol,
                            loss=loss, f_scale=f_scale)
    if full_output:
        return res["F"][0], {"cost": float(res["cost"][0]), "iters": int(res["iters"][0]), "status": int(res["status"][0])}
    return res["F"][0]


def getFFromLabCode(p1, p2, r=10000, thr=1.5, sample_idx=None, seed=None, sampler="reference", tie="reference",
                    refine=True, device=None, loss="linear", f_scale=1.0):
    """Drop-in for fun.getFFromLabCode(p1, p2) (fun.py:291-369): RANSAC over ``r`` 8-point hypotheses followed by the
    gold-standard refinement on the consensus set.  Returns the (3, 3) F_gold (or the RANSAC F if ``refine=False``).

    refine=True      the reference's own stage: SciPy least_squares on the host (same call, same stopping behaviour);
    refine="device"  the same cost minimised on the GPU (``gold_standard_device``);
    refine=False     the RANSAC winner.
    loss, f_scale    robust loss of the refine stage that runs (SciPy's names; f_scale in pixels)."""
    _rt.loss_args(loss, f_scale)
    p1 = np.asarray(p1, dtype=np.float64)
    p2 = np.asarray(p2, dtype=np.float64)
    res = f_ransac(p1, p2, r=r, thr=thr, sample_idx=sample_idx, seed=seed, sampler=sampler, tie=tie, device=device)
    if res["F"] is None:
        # the reference would crash in the gold standard with F_RANSAC = None (fun.py:343); say why instead
        raise ValueError("RANSAC found no hypothesis with a non-empty consensus set")
    if not refine:
        return res["F"]
    if refine == "device":
        return gold_standard_device(res["F"], p1, p2, res["inliers"], loss=loss, f_scale=f_scale)
    return gold_standard(res["F"], p1, p2, res["inliers"], loss=loss, f_scale=f_scale)
