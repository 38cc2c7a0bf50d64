"""numpy-level wrappers over the C ABI (host-buffer entry points).

These are the only functions of the package that touch ctypes; ``lab3.py`` / ``fun.py`` / ``ransac.py`` / ``pnp.py``
(the mirrors of the reference's modules) and ``batched.py`` are written on top of them.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import _cabi as cabi
from ._cabi import (MODE_EPI_MAX, MODE_SAMPSON, SCORE_FP32_GUARDED, SCORE_FP64, SOLVER_JACOBI, SOLVER_QR, TIE_FIRST,
                    TIE_REFERENCE, TRI_LINEAR, TRI_OPTIMAL)


def _call(name, device, *args) -> None:
    """The one way the wrappers below reach the library: entry point ``name`` with the context of ``device`` as its first
    argument.  Every wrapper validates its arguments before it gets here."""
    cabi.call(name, cabi.context(device), *args)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def offsets(counts) -> np.ndarray:
    """int32 prefix table [0, c0, c0+c1, ...] (host) of per-pair counts."""
    counts = np.asarray(counts, dtype=np.int64).ravel()
    off = np.zeros(counts.size + 1, dtype=np.int64)
    off[1:] = counts.cumsum()
    if off[-1] >= 2 ** 31:
        raise ValueError("batch too large for int32 offsets")
    return off.astype(np.int32)


_STAGE: dict = {}


def _concat_into(key, arrays, tail, dtype) -> np.ndarray:
    """np.concatenate into a cached grow-only buffer: the batched entry points are called in loops with the same shapes,
    and a fresh 10 MB allocation per call costs more than the GPU work of a small batch.  The cache is keyed by the calling
    THREAD as well: ctypes releases the GIL during the library call, so two threads (one per device, say) would otherwise
    overwrite each other's staged inputs while an upload is in flight."""
    import threading
    key = (key, threading.get_ident())
    n = sum(a.shape[0] for a in arrays)
    buf = _STAGE.get(key)
    if buf is None or buf.shape[0] < n:
        buf = np.empty((n + n // 4 + 16,) + tuple(tail), dtype=dtype)
        _STAGE[key] = buf
    out = buf[:n]
    if arrays:
        np.concatenate(arrays, axis=0, out=out)
    return out


def _consecutive(arrays):
    """The arrays as ONE array without copying when they are C-contiguous row blocks that follow each other in memory
    (e.g. the blocks of sampling.fast_batch, or a single array), else None."""
    if not arrays:
        return None
    a0 = arrays[0]
    if len(arrays) > 1 and (a0.base is None or any(a.base is not a0.base for a in arrays)):
        return None                     # blocks of one buffer are views of it: a cheap test before the addresses
    addr = a0.ctypes.data
    rows = 0
    for a in arrays:
        if a.dtype != a0.dtype or a.shape[1:] != a0.shape[1:] or not a.flags.c_contiguous or a.ctypes.data != addr:
            return None
        addr += a.nbytes
        rows += a.shape[0]
    # a view of the first block stretched over all of them (so it keeps that block's memory alive), with the strides of
    # a C-ordered array: a block of one row can be C-contiguous with any stride along its first axis
    shape = (rows,) + a0.shape[1:]
    strides = tuple(math.prod(shape[k + 1:]) * a0.itemsize for k in range(len(shape)))
    return np.lib.stride_tricks.as_strided(a0, shape=shape, strides=strides)


def _pack(arrays, tail, dtype, stage=None):
    """A batch in CSR form: the arrays, each (N_i, *tail), as ONE (sum N_i, *tail) array, and the int32 row offset table.
    No copy when the arrays already are consecutive blocks of one buffer (a one-item list always is); otherwise
    ``np.concatenate``, or, given a ``stage`` key, the staging buffer of ``_concat_into``.  An empty list packs to a
    (0, *tail) array."""
    tail = tuple(tail)
    arrays = [np.ascontiguousarray(a, dtype=dtype) for a in arrays]
    rows = [a.shape[0] for a in arrays if a.shape[1:] == tail]
    if len(rows) != len(arrays):
        bad = next(a.shape for a in arrays if a.shape[1:] != tail)
        raise ValueError(f"expected arrays of shape (N, {', '.join(map(str, tail))}), got {bad}")
    off = offsets(rows)
    if len(arrays) == 1:
        return arrays[0], off                   # C-contiguous after ascontiguousarray: the caller's memory
    if not arrays:
        return np.zeros((0,) + tail, dtype=dtype), off
    flat = _consecutive(arrays)
    if flat is None:
        flat = _concat_into(stage, arrays, tail, dtype) if stage else np.concatenate(arrays)
    return flat, off


def _pack_masks(masks, off):
    """Per-item selection masks -> one uint8 array for the library, or None.  Any non-zero value selects (the kernels
    test ``!= 0``), whatever the mask's dtype."""
    if masks is None:
        return None
    if len(masks) != len(off) - 1 or any(len(m) != off[i + 1] - off[i] for i, m in enumerate(masks)):
        raise ValueError("masks must have one entry per point of every item")
    if not masks:
        return None
    return np.concatenate([np.asarray(m, dtype=bool).ravel() for m in masks]).view(np.uint8)


def _split(a, off) -> list:
    """The rows of a packed array, one array per item of the offset table."""
    return [a[off[i]:off[i + 1]] for i in range(len(off) - 1)]


def _poses(Rt):
    """(V, 12) rows [R row-major | t] -> R (V, 3, 3), t (V, 3)."""
    return Rt[:, :9].reshape(-1, 3, 3).copy(), Rt[:, 9:].copy()


def _alloc(want, off, tail=(), dtype=np.float64):
    """A zeroed optional output of off[-1] rows when requested, else None (NULL: the library skips it)."""
    return np.zeros((int(off[-1]),) + tail, dtype=dtype) if want else None


def _split_wanted(**outs) -> dict:
    """name=(output or None, its offset table) -> {name: per-item list} for the outputs that were requested."""
    return {k: _split(a, off) for k, (a, off) in outs.items() if a is not None}


def pack_pairs(p1, p2) -> np.ndarray:
    """(2, N) + (2, N) reference layout  ->  (N, 4) rows (x0, x1, y0, y1)."""
    p1 = np.asarray(p1, dtype=np.float64)
    p2 = np.asarray(p2, dtype=np.float64)
    if p1.shape != p2.shape or p1.ndim != 2 or p1.shape[0] != 2:
        raise ValueError("expected two (2, N) arrays of the same shape")
    return np.ascontiguousarray(np.concatenate([p1.T, p2.T], axis=1))


def set_option(option: int, value: int, device=None) -> None:
    _call("rg_set_option", device, option, value)


def profile(device=None, stream=0) -> dict:
    """Phase times (ms, summed) of the calls since profiling was enabled / last read: see rg_get_profile."""
    out = (C.c_double * 5)()
    n = C.c_int(0)
    _call("rg_get_profile", device, stream, out, C.byref(n))
    return {"calls": n.value, "prepare_ms": out[0], "solve_ms": out[1], "score_ms": out[2], "fixup_ms": out[3],
            "select_ms": out[4]}


def bounded_stats(device=None, stream=0) -> dict:
    """What the last F call executed: see rg_f_last_bounded_stats (K = 0: it ran the full sweep).  ``evals`` splits into
    ``bound_evals`` (bound-only prefix stages: stage A over the first rho0 = option 16 of every pair, and stage B, the
    survivors over the rest of the prefix) and ``guarded_evals`` (rg_f_last_bounded_evals)."""
    out = (C.c_longlong * 4)()
    _call("rg_f_last_bounded_stats", device, stream, out)
    split = (C.c_longlong * 2)()
    _call("rg_f_last_bounded_evals", device, stream, split)
    return {"evals": out[0], "not_fully_scored": out[1], "fallback_pairs": out[2], "K": out[3],
            "bound_evals": split[0], "guarded_evals": split[1]}


def last_stats(device=None, stream=0) -> dict:
    out = (C.c_longlong * 8)()
    _call("rg_get_last_stats", device, stream, out)
    return {"recheck_groups": out[0], "band_evals": out[1], "flips": out[2], "overflow": out[3], "bad_index_hyps": out[4],
            "h2d_mb_per_s": out[5], "passes": out[6], "launches": out[7]}


def f_ransac_batched(pts_list, idx_list, thr=1.5, mode=MODE_EPI_MAX, tie_mode=TIE_FIRST, solver=SOLVER_QR,
                     score_path=SCORE_FP32_GUARDED, want_counts=False, want_F_all=False, want_mask=True,
                     want_flags=False, device=None, stream=0, n_hyp=None, sample_seed=0, first_pair=0) -> dict:
    """F-matrix RANSAC over a batch of image pairs in ONE library call.

    pts_list[p] : (N_p, 4) float64 rows (x0, x1, y0, y1);  idx_list[p] : (H_p, 8) int sample indices (host-drawn).
    idx_list=None: ``n_hyp`` (int or per-pair list) index sets per pair are drawn ON THE DEVICE from ``sample_seed`` (pair p
    has global id ``first_pair + p``) and never cross PCIe; ``philox.sample_indices(N_p, H_p, 8, sample_seed, first_pair + p)``
    replays them on the host.
    Returns per-pair arrays ``best_idx`` (-1 = no hypothesis has any inlier), ``best_count``, ``F`` (P, 3, 3) and
    lists ``mask`` / ``counts`` / ``F_all`` / ``flags`` split per pair when requested.
    """
    P = len(pts_list)
    if idx_list is None:
        if n_hyp is None:
            raise ValueError("idx_list=None needs n_hyp")
        hyps = [int(n_hyp)] * P if np.isscalar(n_hyp) else [int(h) for h in n_hyp]
        if len(hyps) != P:
            raise ValueError("n_hyp must be an int or one value per pair")
        idx_all, hyp_off = None, offsets(hyps)
    elif len(idx_list) != P:
        raise ValueError("pts_list and idx_list must have the same length")
    else:
        # (sample indices are range-checked on the device where they are read: an index outside [0, N_p) makes the
        #  library call fail with ValueError — no host pass over the index arrays)
        idx_all, hyp_off = _pack(idx_list, (8,), np.int32, stage="f_idx")
    pts_all, pair_off = _pack(pts_list, (4,), np.float64, stage="f_pts")
    best_idx = np.full(P, -1, dtype=np.int32)
    best_count = np.zeros(P, dtype=np.int32)
    best_F = np.full((P, 3, 3), np.nan)
    mask = _alloc(want_mask, pair_off, (), np.uint8)
    counts = _alloc(want_counts, hyp_off, (), np.int32)
    F_all = _alloc(want_F_all, hyp_off, (3, 3))
    flags = _alloc(want_flags, hyp_off, (), np.uint8)
    _call("rg_f_ransac_host2", device, stream, P, pts_all, pair_off, idx_all, hyp_off, thr, mode, tie_mode, solver,
          score_path, sample_seed, first_pair, best_idx, best_count, best_F, mask, counts, F_all, flags)
    out = {"best_idx": best_idx, "best_count": best_count, "F": best_F, "pair_off": pair_off, "hyp_off": hyp_off}
    out.update(_split_wanted(mask=(mask, pair_off), counts=(counts, hyp_off), F_all=(F_all, hyp_off),
                             flags=(flags, hyp_off)))
    return out


def f8pt_solve(pts, idx, solver=SOLVER_QR, device=None, stream=0):
    """8-point F for every (H, 8) sample of one pair.  Returns (F_all (H,3,3), flags (H,))."""
    pts = _f64(pts).reshape(-1, 4)
    idx = np.ascontiguousarray(idx, dtype=np.int32).reshape(-1, 8)
    if idx.size and (idx.min() < 0 or idx.max() >= pts.shape[0]):
        raise ValueError("sample index out of range")
    H = idx.shape[0]
    F_all = np.zeros((H, 3, 3))
    flags = np.zeros(H, dtype=np.uint8)
    _call("rg_f8pt_solve_host", device, stream, pts.shape[0], pts, H, idx, solver, F_all, flags)
    return F_all, flags


def epi_score_count(pts, F_all, thr, mode=MODE_EPI_MAX, score_path=SCORE_FP32_GUARDED, device=None, stream=0):
    """Inlier count of each caller-supplied F (H, 3, 3) over the (N, 4) correspondences."""
    pts = _f64(pts).reshape(-1, 4)
    F_all = _f64(F_all).reshape(-1, 9)
    H = F_all.shape[0]
    counts = np.zeros(H, dtype=np.int32)
    _call("rg_epi_score_count_host", device, stream, pts.shape[0], pts, H, F_all, thr, mode, score_path, counts)
    return counts


def fmatrix_residuals(F, x, y, device=None, stream=0):
    F = _f64(F).reshape(9)
    x = _f64(x)
    y = _f64(y)
    N = x.shape[1]
    out = np.empty((2, N))
    _call("rg_fmatrix_residuals_host", device, stream, F, N, x, y, out)
    return out


def fmatrix_stls(pl, pr, device=None, stream=0):
    pl = _f64(pl)
    pr = _f64(pr)
    F = np.empty((3, 3))
    _call("rg_fmatrix_stls_host", device, stream, pl.shape[1], pl, pr, F)
    return F


# ---------------------------------------------------------------------------------------------------------------
# PnP
# ---------------------------------------------------------------------------------------------------------------
def pnp_ransac(X, y, idx, thr2, n_sel=None, score_path=SCORE_FP32_GUARDED, want_counts=False, want_poses=False,
               want_mask=True, want_flags=False, device=None, stream=0) -> dict:
    """DLT-PnP RANSAC on one view.  X (N,3), y (N,2) C-normalised, idx (H,n) with 6 <= n <= 8; only the first ``n_sel``
    correspondences vote (default: all).  pnp_ransac_batched for ONE view, with its per-view results unwrapped."""
    r = pnp_ransac_batched([X], [y], [idx], thr2, n_vote=[len(X) if n_sel is None else n_sel], score_path=score_path,
                           want_counts=want_counts, want_poses=want_poses, want_mask=want_mask, want_flags=want_flags,
                           device=device, stream=stream)
    out = {"best_idx": int(r["best_idx"][0]), "best_count": int(r["best_count"][0]), "R": r["R"][0], "t": r["t"][0]}
    out.update({k: r[k][0] for k in ("mask", "counts", "poses", "flags") if k in r})
    return out


def pnp_ransac_batched(X_list, y_list, idx_list, thr2, n_vote=None, score_path=SCORE_FP32_GUARDED, want_counts=False,
                       want_poses=False, want_mask=True, want_flags=False, device=None, stream=0) -> dict:
    """DLT-PnP RANSAC over V views in ONE library call.  X_list[v] (N_v,3), y_list[v] (N_v,2), idx_list[v] (H_v,n)."""
    V = len(X_list)
    if len(y_list) != V or len(idx_list) != V:
        raise ValueError("X_list, y_list and idx_list must have the same length")
    X, view_off = _pack(X_list, (3,), np.float64)
    y, y_off = _pack(y_list, (2,), np.float64)
    if view_off.tobytes() != y_off.tobytes():          # both int32 offset tables of the same length
        raise ValueError("X and y must have the same number of rows in every view")
    n = np.shape(idx_list[0])[1] if V and np.ndim(idx_list[0]) == 2 else 6
    # (sample indices are range-checked on the device where they are read: the library call fails with ValueError)
    idx, hyp_off = _pack(idx_list, (n,), np.int32)
    vote = None if n_vote is None else np.ascontiguousarray(n_vote, dtype=np.int32)
    best_idx = np.full(V, -1, dtype=np.int32)
    best_count = np.zeros(V, dtype=np.int32)
    Rt = np.full((V, 12), np.nan)
    mask = _alloc(want_mask, view_off, (), np.uint8)
    counts = _alloc(want_counts, hyp_off, (), np.int32)
    poses = _alloc(want_poses, hyp_off, (12,))
    flags = _alloc(want_flags, hyp_off, (), np.uint8)
    _call("rg_pnp_ransac_batched_host", device, stream, V, X, y, view_off, vote, idx, hyp_off, n, thr2, score_path,
          best_idx, best_count, Rt, mask, counts, poses, flags)
    R, t = _poses(Rt)
    out = {"best_idx": best_idx, "best_count": best_count, "R": R, "t": t, "view_off": view_off, "hyp_off": hyp_off}
    out.update(_split_wanted(mask=(mask, view_off), counts=(counts, hyp_off), poses=(poses, hyp_off),
                             flags=(flags, hyp_off)))
    return out


def pnp_minimize(X, y, device=None, stream=0):
    X = _f64(X).reshape(-1, 3)
    y = _f64(y).reshape(-1, 2)
    R = np.empty((3, 3))
    t = np.empty(3)
    _call("rg_pnp_minimize_host", device, stream, X.shape[0], X, y, R, t)
    return R, t


def pnp_k_table(K, V) -> np.ndarray | None:
    """K as the (V, 9) host table of rg_pnp_refine_*: None stays None, one (3, 3) is shared by every view."""
    if K is None:
        return None
    K = _f64(K)
    if K.shape == (3, 3):
        K = np.broadcast_to(K, (V, 3, 3))
    if K.shape != (V, 3, 3):
        raise ValueError("K must be (3, 3) or (V, 3, 3)")
    if np.any(K[:, 1, 0] != 0.0) or np.any(K[:, 2] != np.array([0.0, 0.0, 1.0])):
        raise ValueError("K must have K[1, 0] == 0 and bottom row (0, 0, 1)")
    return np.ascontiguousarray(K.reshape(V, 9))


def pnp_refine_batched(X_list, y_list, R, t, masks=None, K=None, max_iter=50, ftol=1e-12, rounds=1, thr2=None,
                       device=None, stream=0) -> dict:
    """Levenberg-Marquardt refinement of V PnP poses in ONE library call (rg_pnp_refine_host): per view, the minimum of
    1/2 sum |W (pi(R X + t) - y)|^2 over the selected correspondences, W = K[:2, :2] (cost in pixels) or I.
    X_list[v] (N_v, 3), y_list[v] (N_v, 2) C-normalised; R (V, 3, 3), t (V, 3) start poses; masks[v] optional selection;
    K (3, 3) or (V, 3, 3).  rounds > 1: re-score the consensus thr2 >= e at the refined pose and refine again on it.
    Returns dict(R, t, cost, iters, status) of the last round, plus the list ``mask`` of last consensus sets when thr2 is
    given.  status: 1 start pose not finite, 2 converged, 3 lambda > 1e12, 4 max_iter, 5 fewer than 3 points."""
    V = len(X_list)
    if len(y_list) != V:
        raise ValueError("X_list and y_list must have the same length")
    X, view_off = _pack(X_list, (3,), np.float64)
    y, y_off = _pack(y_list, (2,), np.float64)
    if view_off.tobytes() != y_off.tobytes():          # both int32 offset tables of the same length
        raise ValueError("X and y must have the same number of rows in every view")
    R = _f64(R).reshape(-1, 3, 3)
    t = _f64(t).reshape(-1, 3)
    if R.shape[0] != V or t.shape[0] != V:
        raise ValueError("R must be (V, 3, 3) and t (V, 3)")
    if int(rounds) < 1:
        raise ValueError("rounds must be >= 1")
    if int(rounds) > 1 and thr2 is None:
        raise ValueError("rounds > 1 needs thr2 (the consensus threshold)")
    mask = _pack_masks(masks, view_off)
    Kt = pnp_k_table(K, V)
    Rt = np.ascontiguousarray(np.concatenate([R.reshape(V, 9), t], axis=1))
    cost = np.full(V, np.nan)
    iters = np.zeros(V, dtype=np.int32)
    status = np.zeros(V, dtype=np.int32)
    mask_out = np.zeros(max(int(view_off[-1]), 1), dtype=np.uint8) if thr2 is not None else None
    _call("rg_pnp_refine_host", device, stream, V, X, y, view_off, Kt, mask, Rt, max_iter, ftol, rounds,
          0.0 if thr2 is None else thr2, mask_out, cost, iters, status)
    R, t = _poses(Rt)
    out = {"R": R, "t": t, "cost": cost, "iters": iters, "status": status, "view_off": view_off}
    out.update(_split_wanted(mask=(mask_out, view_off)))
    return out


def pnp_refine(X, y, R, t, mask=None, K=None, max_iter=50, ftol=1e-12, rounds=1, thr2=None, device=None, stream=0) -> dict:
    """pnp_refine_batched for ONE view: X (N, 3), y (N, 2), R (3, 3), t (3,), mask (N,) optional, K (3, 3) optional.
    Returns dict(R, t, cost, iters, status[, mask])."""
    r = pnp_refine_batched([X], [y], _f64(R).reshape(1, 3, 3), _f64(t).reshape(1, 3),
                           masks=None if mask is None else [mask], K=K, max_iter=max_iter, ftol=ftol, rounds=rounds,
                           thr2=thr2, device=device, stream=stream)
    out = {"R": r["R"][0], "t": r["t"][0], "cost": float(r["cost"][0]), "iters": int(r["iters"][0]),
           "status": int(r["status"][0])}
    if "mask" in r:
        out["mask"] = r["mask"][0]
    return out


def pnp_score_count(X, y, poses, thr2, score_path=SCORE_FP32_GUARDED, device=None, stream=0):
    X = _f64(X).reshape(-1, 3)
    y = _f64(y).reshape(-1, 2)
    poses = _f64(poses).reshape(-1, 12)
    counts = np.zeros(poses.shape[0], dtype=np.int32)
    _call("rg_pnp_score_count_host", device, stream, X.shape[0], X, y, poses.shape[0], poses, thr2, score_path, counts)
    return counts


# ---------------------------------------------------------------------------------------------------------------
# two-view geometry (SURVEY.md section 8f rows N1-N3)
# ---------------------------------------------------------------------------------------------------------------
def triangulate(C1, C2, x1_list, x2_list, method=TRI_OPTIMAL, device=None, stream=0):
    """Triangulates every correspondence of P camera pairs in ONE library call.

    C1, C2 : (P, 3, 4) (or (3, 4) for one pair);  x1_list[p], x2_list[p] : (N_p, 2) image points.
    Returns a list of (N_p, 3) arrays (lab3.triangulate_optimal / triangulate_linear per correspondence)."""
    C1 = _f64(C1).reshape(-1, 3, 4)
    C2 = _f64(C2).reshape(-1, 3, 4)
    P = C1.shape[0]
    if C2.shape[0] != P or len(x1_list) != P or len(x2_list) != P:
        raise ValueError("C1, C2, x1_list and x2_list must describe the same number of camera pairs")
    x1, off = _pack(x1_list, (2,), np.float64)
    x2, off2 = _pack(x2_list, (2,), np.float64)
    if off.tobytes() != off2.tobytes():                 # both int32 offset tables of the same length
        raise ValueError("x1 and x2 must have the same shape in every pair")
    X = np.full((int(off[-1]), 3), np.nan)
    _call("rg_triangulate_host", device, stream, P, C1, C2, off, x1, x2, method, X)
    return _split(X, off)


def fmatrix_from_cameras(C1, C2, device=None, stream=0):
    """lab3.fmatrix_from_cameras for P camera pairs: (P, 3, 4) x 2 -> (P, 3, 3)."""
    C1 = _f64(C1).reshape(-1, 3, 4)
    C2 = _f64(C2).reshape(-1, 3, 4)
    if C1.shape != C2.shape:
        raise ValueError("C1 and C2 must have the same shape")
    F = np.full((C1.shape[0], 3, 3), np.nan)
    _call("rg_fmatrix_from_cameras_host", device, stream, C1.shape[0], C1, C2, F)
    return F


def relative_pose(M, y1, y2, K=None, device=None, stream=0) -> dict:
    """fun.relative_camera_pose for P pairs in one call.  M (P,3,3) essential matrices — or fundamental matrices when
    K ((3,3) shared or (P,3,3)) is given, E = K^T M K being formed on the device; y1, y2 (P,2) C-normalised.
    Returns dict(R (P,3,3), t (P,3), which (P,) candidate index or -1, npass (P,))."""
    M = _f64(M).reshape(-1, 3, 3)
    P = M.shape[0]
    y1 = _f64(y1).reshape(-1, 2)
    y2 = _f64(y2).reshape(-1, 2)
    if y1.shape[0] != P or y2.shape[0] != P:
        raise ValueError("one correspondence per pair expected")
    per_pair = 0
    if K is not None:
        K = _f64(K)
        if K.shape == (P, 3, 3) and P != 0 and K.ndim == 3:
            per_pair = 1
        elif K.shape != (3, 3):
            raise ValueError("K must be (3, 3) or (P, 3, 3)")
    Rt = np.full((P, 12), np.nan)
    which = np.full(P, -1, dtype=np.int32)
    npass = np.zeros(P, dtype=np.int32)
    _call("rg_relative_pose_host", device, stream, P, M, K, per_pair, y1, y2, Rt, which, npass)
    R, t = _poses(Rt)
    return {"R": R, "t": t, "which": which, "npass": npass}


def two_view_init(pts_list, F, K, masks=None, device=None, stream=0) -> dict:
    """main.py:54-76 (E = K^T F K, C-normalisation, relative pose, triangulation of every correspondence) for P image
    pairs in ONE library call.  pts_list[p]: (N_p, 4) pixel rows (x0, x1, y0, y1); F: (P, 3, 3); K: (3, 3);
    masks[p] (optional): (N_p,), zero = skip.  Returns dict(R (P,3,3), t (P,3), which (P,), X list of (N_p,3))."""
    P = len(pts_list)
    F = _f64(F).reshape(-1, 3, 3)
    K = _f64(K)
    if F.shape[0] != P or K.shape != (3, 3):
        raise ValueError("F must be (P, 3, 3) and K (3, 3)")
    pts, off = _pack(pts_list, (4,), np.float64)
    mask = _pack_masks(masks, off)
    Rt = np.full((P, 12), np.nan)
    which = np.full(P, -1, dtype=np.int32)
    X = np.full((int(off[-1]), 3), np.nan)
    _call("rg_two_view_init_host", device, stream, P, pts, off, F, K, mask, Rt, which, X)
    R, t = _poses(Rt)
    return {"R": R, "t": t, "which": which, "X": _split(X, off)}


def gold_standard(pts_list, F0, masks=None, max_iter=50, ftol=1e-12, want_points=False, device=None, stream=0) -> dict:
    """Gold-standard refinement (second half of fun.getFFromLabCode, fun.py:342-369) of P pairs in ONE library call.
    pts_list[p]: (N_p, 4) pixel rows; F0: (P, 3, 3); masks[p] optional inlier masks (zero = skip).
    Returns dict(F (P,3,3), cost (P,), iters (P,), status (P,), X list when want_points)."""
    P = len(pts_list)
    F0 = _f64(F0).reshape(-1, 3, 3)
    if F0.shape[0] != P:
        raise ValueError("F0 must be (P, 3, 3)")
    pts, off = _pack(pts_list, (4,), np.float64)
    mask = _pack_masks(masks, off)
    F = np.full((P, 3, 3), np.nan)
    cost = np.full(P, np.nan)
    iters = np.zeros(P, dtype=np.int32)
    status = np.zeros(P, dtype=np.int32)
    X = np.full((int(off[-1]), 3), np.nan) if want_points else None
    _call("rg_gold_standard_host", device, stream, P, pts, off, F0, mask, max_iter, ftol, F, cost, iters, status, X)
    out = {"F": F, "cost": cost, "iters": iters, "status": status}
    out.update(_split_wanted(X=(X, off)))
    return out


def fmatrix_residuals_gs(params, pl, pr, device=None, stream=0):
    """lab3.fmatrix_residuals_gs on the GPU: params (12 + 3N,), pl / pr (2, N) -> (4N,)."""
    params = _f64(params).ravel()
    pl = _f64(pl)
    pr = _f64(pr)
    N = pl.shape[1]
    out = np.empty(4 * N)
    _call("rg_fmatrix_residuals_gs_host", device, stream, N, params, pl, pr, out)
    return out


def bundle_adjust(cams, pts, uv, cam_idx, pt_idx, n_fixed=1, max_iter=50, ftol=1e-4, device=None, stream=0) -> dict:
    """Bundle adjustment (the minimisation of tables.Tables.BundleAdjustment2, tables.py:260-333) in ONE library call.
    cams (V, 3, 4) camera matrices, pts (P, 3), uv (O, 2) observed C-normalised image points, cam_idx / pt_idx (O,) the
    view and point of every observation; the first n_fixed views are held fixed (the reference fixes view 0).
    Returns dict(cams, pts, cost = 0.5 * sum r^2, iters, status: 2 converged, 3 no further descent, 4 max_iter)."""
    cams = np.array(cams, dtype=np.float64).reshape(-1, 3, 4)
    pts = np.array(pts, dtype=np.float64).reshape(-1, 3)
    uv = _f64(uv).reshape(-1, 2)
    ci = np.ascontiguousarray(np.ravel(cam_idx), dtype=np.int32)
    pi = np.ascontiguousarray(np.ravel(pt_idx), dtype=np.int32)
    if not (ci.shape[0] == pi.shape[0] == uv.shape[0]):
        raise ValueError("uv, cam_idx and pt_idx must have one row per observation")
    cost = np.full(1, np.nan)
    it_st = np.zeros(2, dtype=np.int32)
    _call("rg_bundle_adjust_host", device, stream, cams.shape[0], pts.shape[0], uv.shape[0], cams, pts, uv, ci, pi,
          n_fixed, max_iter, ftol, cost, it_st[:1], it_st[1:])
    return {"cams": cams, "pts": pts, "cost": float(cost[0]), "iters": int(it_st[0]), "status": int(it_st[1])}


def ba_residuals(x, u, v, cam_idx, pt_idx, n_C, n_P, device=None, stream=0) -> np.ndarray:
    """EpsilonBA of tables.Tables.BundleAdjustment2 (tables.py:266-296) on the GPU: x = [cameras (n_C x 12), points (n_P x 3)]
    -> interleaved residuals (2 * n_obs,)."""
    x = _f64(x).ravel()
    if x.shape[0] != 12 * n_C + 3 * n_P:
        raise ValueError("parameter vector must hold n_C * 12 + n_P * 3 values")
    u = _f64(u).ravel()
    v = _f64(v).ravel()
    ci = np.ascontiguousarray(np.ravel(cam_idx), dtype=np.int32)
    pi = np.ascontiguousarray(np.ravel(pt_idx), dtype=np.int32)
    if not (u.shape[0] == v.shape[0] == ci.shape[0] == pi.shape[0]):
        raise ValueError("u, v, cam_idx and pt_idx must have one entry per observation")
    out = np.empty(2 * u.shape[0])
    _call("rg_ba_residuals_host", device, stream, n_C, n_P, u.shape[0], x, u, v, ci, pi, out)
    return out


def camera_resectioning(Cs, device=None, stream=0):
    """fun.camera_resectioning for V cameras: (V, 3, 4) -> K (V,3,3), R (V,3,3), t (V,3)."""
    Cs = _f64(Cs).reshape(-1, 3, 4)
    V = Cs.shape[0]
    K = np.full((V, 3, 3), np.nan)
    R = np.full((V, 3, 3), np.nan)
    t = np.full((V, 3), np.nan)
    _call("rg_camera_resectioning_host", device, stream, V, Cs, K, R, t)
    return K, R, t


def match_first_within(obs, y, tol=1e-4, device=None, stream=0) -> np.ndarray:
    """For every row of y (N, d) the index of the first row of obs (M, d) closer than tol (strict), -1 if none
    (the 2D<->3D match loop of tables.py:116-124).  d = 2 or 3."""
    obs = _f64(obs)
    y = _f64(y)
    if y.ndim != 2 or y.shape[1] not in (2, 3):
        raise ValueError("y must be (N, 2) or (N, 3)")
    d = y.shape[1]
    obs = obs.reshape(-1, d) if obs.size else np.zeros((0, d))
    idx = np.full(y.shape[0], -1, dtype=np.int32)
    _call("rg_match_first_within_host", device, stream, d, obs.shape[0], obs, y.shape[0], y, tol, idx)
    return idx


def microbench(device=None, stream=0) -> dict:
    out = (C.c_double * 6)()
    cabi.context(device)                  # rg_microbench_run takes no context handle; the library is initialised first
    cabi.call("rg_microbench_run", out, stream)
    return {"ffma_gfma_s": out[0], "ffma2_gfma_s": out[1], "mix_scalar_gevals_s": out[2],
            "mix_packed_gevals_s": out[3], "dfma_gfma_s": out[4], "sms": int(out[5])}
