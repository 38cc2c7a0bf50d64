"""Batched entry points (one library call for many image pairs / one view): what ``main.py``-style drivers and the
benchmark use instead of calling ``fun.getFFromLabCode`` pair by pair (SURVEY.md section 7, steps 5-7)."""
from __future__ import annotations

import numpy as np

from . import runtime as _rt
from . import sampling as _sampling
from ._cabi import MODE_EPI_MAX, SCORE_FP32_GUARDED, SOLVER_QR, TIE_FIRST


def _rows(pairs) -> list:
    """pairs of (2, N_p) arrays (p1, p2) in the reference layout, or (N_p, 4) arrays -> (N_p, 4) rows (x0, x1, y0, y1)."""
    return [_rt.pack_pairs(pr[0], pr[1]) if isinstance(pr, (tuple, list)) else
            np.ascontiguousarray(pr, dtype=np.float64).reshape(-1, 4) for pr in pairs]


def f_ransac_pairs(pairs, n_hyp=10000, thr=1.5, seed=0, idx_list=None, host_sampling=False, **kw) -> dict:
    """pairs: list of (p1, p2) with (2, N_p) arrays (reference layout) or of (N_p, 4) arrays.  Unless ``idx_list`` is given,
    the sample index sets are drawn ON THE DEVICE from ``seed`` (Philox; ``philox.sample_indices(N_p, n_hyp, 8, seed, p)``
    replays pair p's samples on the host) — drawing 35 x 10 000 index sets with numpy and uploading their 11 MB cost 88 ms
    and 0.8 ms against 0.5 ms for the whole call.  host_sampling=True restores the host draw (``sampling.fast_batch``)."""
    pts = _rows(pairs)
    if idx_list is None and not host_sampling:
        return _rt.f_ransac_batched(pts, None, thr=thr, n_hyp=n_hyp, sample_seed=seed, **kw)
    if idx_list is None:
        idx_list = _sampling.fast_batch([p.shape[0] for p in pts], n_hyp, 8, seed)       # one buffer: no concatenation
    return _rt.f_ransac_batched(pts, idx_list, thr=thr, **kw)


def pnp_ransac_view(X, y, n_hyp=1024, thr2=(1.5 / 3217.0) ** 2, n=6, seed=0, idx=None, **kw) -> dict:
    """DLT-PnP RANSAC of one view: X (N, 3), y (N, 2) C-normalised."""
    X = np.asarray(X, dtype=np.float64)
    if idx is None:
        idx = _sampling.fast(X.shape[0], n_hyp, n, seed)
    return _rt.pnp_ransac(X, y, idx, thr2, **kw)


def pnp_ransac_views(views, n_hyp=1024, thr2=(1.5 / 3217.0) ** 2, n=6, seed=0, idx_list=None, **kw) -> dict:
    """DLT-PnP RANSAC of many views in one library call.  views: list of (X (N,3), y (N,2) C-normalised)."""
    Xs = [np.asarray(v[0], dtype=np.float64) for v in views]
    ys = [np.asarray(v[1], dtype=np.float64) for v in views]
    if idx_list is None:
        idx_list = [_sampling.fast(X.shape[0], n_hyp, n, seed + k) for k, X in enumerate(Xs)]
    return _rt.pnp_ransac_batched(Xs, ys, idx_list, thr2, **kw)


def two_view_init(pairs, F, K, masks=None, **kw) -> dict:
    """INIT2 + INIT3 of main.py:54-76 for many image pairs in one library call: relative pose (R, t) of the second camera
    from F and K, and the optimally triangulated 3-D point of every (inlier) correspondence in the first camera's frame.
    pairs: list of (p1, p2) with (2, N_p) arrays or of (N_p, 4) arrays; F: (P, 3, 3), e.g. ``f_ransac_pairs(...)["F"]``;
    masks: optional inlier masks (``...["mask"]``)."""
    return _rt.two_view_init(_rows(pairs), F, K, masks=masks, **kw)
