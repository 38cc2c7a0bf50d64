"""numpy-level wrappers over the C ABI (host-buffer entry points).

These are the only functions of the package that touch ctypes; ``lab3.py`` / ``fun.py`` / ``ransac.py`` / ``pnp.py``
(the mirrors of the reference's modules) and ``batched.py`` are written on top of them.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _cabi as cabi
from ._cabi import (MODE_EPI_MAX, MODE_SAMPSON, SCORE_FP32_GUARDED, SCORE_FP64, SOLVER_JACOBI, SOLVER_QR, TIE_FIRST,
                    TIE_REFERENCE, TRI_LINEAR, TRI_OPTIMAL)

_vp = C.c_void_p


def _f64(a, shape_tail=None):
    arr = np.ascontiguousarray(a, dtype=np.float64)
    if shape_tail is not None and arr.shape[1:] != tuple(shape_tail):
        raise ValueError(f"expected trailing shape {shape_tail}, got {arr.shape}")
    return arr


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
    (e.g. the blocks of sampling.fast_batch), else None."""
    if not arrays:
        return None
    a0 = arrays[0]
    addr = a0.ctypes.data
    rows = 0
    for a in arrays:
        if a.dtype != a0.dtype or a.shape[1:] != a0.shape[1:] or not a.flags.c_contiguous or a.ctypes.data != addr:
            return None
        addr += a.nbytes
        rows += a.shape[0]
    if rows == 0:
        return None
    flat = np.ctypeslib.as_array((np.ctypeslib.as_ctypes_type(a0.dtype) * (rows * int(np.prod(a0.shape[1:])))).from_address(
        a0.ctypes.data))
    return flat.reshape((rows,) + a0.shape[1:])           # memory stays owned by the callers' arrays (alive during the call)


def pack_pairs(p1, p2) -> np.ndarray:
    """(2, N) + (2, N) reference layout  ->  (N, 4) rows (x0, x1, y0, y1)."""
    p1 = np.asarray(p1, dtype=np.float64)
    p2 = np.asarray(p2, dtype=np.float64)
    if p1.shape != p2.shape or p1.ndim != 2 or p1.shape[0] != 2:
        raise ValueError("expected two (2, N) arrays of the same shape")
    return np.ascontiguousarray(np.concatenate([p1.T, p2.T], axis=1))


def set_option(option: int, value: int, device=None) -> None:
    cabi.check(cabi.load_library().rg_set_option(_vp(cabi.context(device)), int(option), int(value)))


def profile(device=None, stream=0) -> dict:
    """Phase times (ms, summed) of the calls since profiling was enabled / last read: see rg_get_profile."""
    out = (C.c_double * 5)()
    n = C.c_int(0)
    cabi.check(cabi.load_library().rg_get_profile(_vp(cabi.context(device)), _vp(stream), out, C.byref(n)))
    return {"calls": n.value, "prepare_ms": out[0], "solve_ms": out[1], "score_ms": out[2], "fixup_ms": out[3],
            "select_ms": out[4]}


def last_stats(device=None, stream=0) -> dict:
    lib = cabi.load_library()
    out = (C.c_longlong * 8)()
    cabi.check(lib.rg_get_last_stats(_vp(cabi.context(device)), _vp(stream), out))
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
    lib = cabi.load_library()
    ctx = cabi.context(device)
    P = len(pts_list)
    seeded = idx_list is None
    if seeded:
        if n_hyp is None:
            raise ValueError("idx_list=None needs n_hyp")
        hyps = [int(n_hyp)] * P if np.isscalar(n_hyp) else [int(h) for h in n_hyp]
        if len(hyps) != P:
            raise ValueError("n_hyp must be an int or one value per pair")
    elif len(idx_list) != P:
        raise ValueError("pts_list and idx_list must have the same length")
    pts = [_f64(p).reshape(-1, 4) for p in pts_list]
    idx = [] if seeded else [np.ascontiguousarray(i, dtype=np.int32).reshape(-1, 8) for i in idx_list]
    pair_off = np.zeros(P + 1, dtype=np.int32)
    hyp_off = np.zeros(P + 1, dtype=np.int32)
    for p in range(P):
        pair_off[p + 1] = pair_off[p] + pts[p].shape[0]
        hyp_off[p + 1] = hyp_off[p] + (hyps[p] if seeded else idx[p].shape[0])
    # (sample indices are range-checked on the device where they are read: an index outside [0, N_p) makes the library
    #  call fail with ValueError — no host pass over the index arrays)
    Ntot, Htot = int(pair_off[-1]), int(hyp_off[-1])
    pts_all = _concat_into("f_pts", pts, (4,), np.float64)
    idx_all = None
    if not seeded:
        idx_all = _consecutive(idx)
        if idx_all is None:
            idx_all = _concat_into("f_idx", idx, (8,), np.int32)
    best_idx = np.full(P, -1, dtype=np.int32)
    best_count = np.zeros(P, dtype=np.int32)
    best_F = np.full((P, 3, 3), np.nan)
    mask = np.zeros(Ntot, dtype=np.uint8) if want_mask else None
    counts = np.zeros(Htot, dtype=np.int32) if want_counts else None
    F_all = np.zeros((Htot, 3, 3)) if want_F_all else None
    flags = np.zeros(Htot, dtype=np.uint8) if want_flags else None
    cabi.check(lib.rg_f_ransac_host2(
        _vp(ctx), _vp(stream), P, _vp(cabi.ptr(pts_all)), pair_off.ctypes.data_as(C.POINTER(C.c_int32)),
        _vp(cabi.ptr(idx_all)), hyp_off.ctypes.data_as(C.POINTER(C.c_int32)), float(thr), int(mode), int(tie_mode),
        int(solver), int(score_path), int(sample_seed), int(first_pair), _vp(cabi.ptr(best_idx)), _vp(cabi.ptr(best_count)),
        _vp(cabi.ptr(best_F)), _vp(cabi.ptr(mask)), _vp(cabi.ptr(counts)), _vp(cabi.ptr(F_all)), _vp(cabi.ptr(flags))))
    out = {"best_idx": best_idx, "best_count": best_count, "F": best_F, "pair_off": pair_off, "hyp_off": hyp_off}
    split_n = lambda a: [a[pair_off[p]:pair_off[p + 1]] for p in range(P)]
    split_h = lambda a: [a[hyp_off[p]:hyp_off[p + 1]] for p in range(P)]
    if want_mask:
        out["mask"] = split_n(mask)
    if want_counts:
        out["counts"] = split_h(counts)
    if want_F_all:
        out["F_all"] = split_h(F_all)
    if want_flags:
        out["flags"] = split_h(flags)
    return out


def f8pt_solve(pts, idx, solver=SOLVER_QR, device=None, stream=0):
    """8-point F for every (H, 8) sample of one pair.  Returns (F_all (H,3,3), flags (H,))."""
    lib = cabi.load_library()
    ctx = cabi.context(device)
    pts = _f64(pts).reshape(-1, 4)
    idx = np.ascontiguousarray(idx, dtype=np.int32).reshape(-1, 8)
    if idx.size and (idx.min() < 0 or idx.max() >= pts.shape[0]):
        raise ValueError("sample index out of range")
    H = idx.shape[0]
    F_all = np.zeros((H, 3, 3))
    flags = np.zeros(H, dtype=np.uint8)
    cabi.check(lib.rg_f8pt_solve_host(_vp(ctx), _vp(stream), pts.shape[0], _vp(cabi.ptr(pts)), H, _vp(cabi.ptr(idx)),
                                      int(solver), _vp(cabi.ptr(F_all)), _vp(cabi.ptr(flags))))
    return F_all, flags


def epi_score_count(pts, F_all, thr, mode=MODE_EPI_MAX, score_path=SCORE_FP32_GUARDED, device=None, stream=0):
    """Inlier count of each caller-supplied F (H, 3, 3) over the (N, 4) correspondences."""
    lib = cabi.load_library()
    ctx = cabi.context(device)
    pts = _f64(pts).reshape(-1, 4)
    F_all = _f64(F_all).reshape(-1, 9)
    H = F_all.shape[0]
    counts = np.zeros(H, dtype=np.int32)
    cabi.check(lib.rg_epi_score_count_host(_vp(ctx), _vp(stream), pts.shape[0], _vp(cabi.ptr(pts)), H,
                                           _vp(cabi.ptr(F_all)), float(thr), int(mode), int(score_path),
                                           _vp(cabi.ptr(counts))))
    return counts


def fmatrix_residuals(F, x, y, device=None, stream=0):
    lib = cabi.load_library()
    ctx = cabi.context(device)
    F = _f64(F).reshape(9)
    x = _f64(x)
    y = _f64(y)
    N = x.shape[1]
    out = np.empty((2, N))
    cabi.check(lib.rg_fmatrix_residuals_host(_vp(ctx), _vp(stream), _vp(cabi.ptr(F)), N, _vp(cabi.ptr(x)),
                                             _vp(cabi.ptr(y)), _vp(cabi.ptr(out))))
    return out


def fmatrix_stls(pl, pr, device=None, stream=0):
    lib = cabi.load_library()
    ctx = cabi.context(device)
    pl = _f64(pl)
    pr = _f64(pr)
    F = np.empty((3, 3))
    cabi.check(lib.rg_fmatrix_stls_host(_vp(ctx), _vp(stream), pl.shape[1], _vp(cabi.ptr(pl)), _vp(cabi.ptr(pr)),
                                        _vp(cabi.ptr(F))))
    return F


# ---------------------------------------------------------------------------------------------------------------
# PnP
# ---------------------------------------------------------------------------------------------------------------
def pnp_ransac(X, y, idx, thr2, n_sel=None, score_path=SCORE_FP32_GUARDED, want_counts=False, want_poses=False,
               want_mask=True, want_flags=False, device=None, stream=0) -> dict:
    """DLT-PnP RANSAC on one view.  X (N,3), y (N,2) C-normalised, idx (H,n) with 6 <= n <= 8."""
    lib = cabi.load_library()
    ctx = cabi.context(device)
    X = _f64(X).reshape(-1, 3)
    y = _f64(y).reshape(-1, 2)
    if X.shape[0] != y.shape[0]:
        raise ValueError("X and y must have the same number of rows")
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    if idx.ndim != 2:
        raise ValueError("idx must be (H, n)")
    H, n = idx.shape
    N = X.shape[0]
    # (sample indices are range-checked on the device where they are read: the library call fails with ValueError)
    n_sel = N if n_sel is None else int(n_sel)
    best_idx = np.full(1, -1, dtype=np.int32)
    best_count = np.zeros(1, dtype=np.int32)
    R = np.full((3, 3), np.nan)
    t = np.full(3, np.nan)
    mask = np.zeros(N, dtype=np.uint8) if want_mask else None
    counts = np.zeros(H, dtype=np.int32) if want_counts else None
    poses = np.zeros((H, 12)) if want_poses else None
    flags = np.zeros(H, dtype=np.uint8) if want_flags else None
    cabi.check(lib.rg_pnp_ransac_host(_vp(ctx), _vp(stream), N, n_sel, _vp(cabi.ptr(X)), _vp(cabi.ptr(y)), H, n,
                                      _vp(cabi.ptr(idx)), float(thr2), int(score_path), _vp(cabi.ptr(best_idx)),
                                      _vp(cabi.ptr(best_count)), _vp(cabi.ptr(R)), _vp(cabi.ptr(t)), _vp(cabi.ptr(mask)),
                                      _vp(cabi.ptr(counts)), _vp(cabi.ptr(poses)), _vp(cabi.ptr(flags))))
    out = {"best_idx": int(best_idx[0]), "best_count": int(best_count[0]), "R": R, "t": t}
    if want_mask:
        out["mask"] = mask
    if want_counts:
        out["counts"] = counts
    if want_poses:
        out["poses"] = poses
    if want_flags:
        out["flags"] = flags
    return out


def pnp_ransac_batched(X_list, y_list, idx_list, thr2, n_vote=None, score_path=SCORE_FP32_GUARDED, want_counts=False,
                       want_poses=False, want_mask=True, want_flags=False, device=None, stream=0) -> dict:
    """DLT-PnP RANSAC over V views in ONE library call.  X_list[v] (N_v,3), y_list[v] (N_v,2), idx_list[v] (H_v,n)."""
    lib = cabi.load_library()
    ctx = cabi.context(device)
    V = len(X_list)
    if len(y_list) != V or len(idx_list) != V:
        raise ValueError("X_list, y_list and idx_list must have the same length")
    Xs = [_f64(a).reshape(-1, 3) for a in X_list]
    ys = [_f64(a).reshape(-1, 2) for a in y_list]
    ids = [np.ascontiguousarray(a, dtype=np.int32) for a in idx_list]
    n = ids[0].shape[1] if V and ids[0].ndim == 2 else 6
    view_off = np.zeros(V + 1, dtype=np.int32)
    hyp_off = np.zeros(V + 1, dtype=np.int32)
    for v in range(V):
        if Xs[v].shape[0] != ys[v].shape[0]:
            raise ValueError(f"view {v}: X and y must have the same number of rows")
        if ids[v].ndim != 2 or ids[v].shape[1] != n:
            raise ValueError("every idx must be (H, n) with the same n")
        view_off[v + 1] = view_off[v] + Xs[v].shape[0]
        hyp_off[v + 1] = hyp_off[v] + ids[v].shape[0]
    N, H = int(view_off[-1]), int(hyp_off[-1])
    X = np.ascontiguousarray(np.concatenate(Xs)) if V else np.zeros((0, 3))
    y = np.ascontiguousarray(np.concatenate(ys)) if V else np.zeros((0, 2))
    idx = np.ascontiguousarray(np.concatenate(ids)) if V else np.zeros((0, n), dtype=np.int32)
    vote = None if n_vote is None else np.ascontiguousarray(n_vote, dtype=np.int32)
    best_idx = np.full(V, -1, dtype=np.int32)
    best_count = np.zeros(V, dtype=np.int32)
    Rt = np.full((V, 12), np.nan)
    mask = np.zeros(N, dtype=np.uint8) if want_mask else None
    counts = np.zeros(H, dtype=np.int32) if want_counts else None
    poses = np.zeros((H, 12)) if want_poses else None
    flags = np.zeros(H, dtype=np.uint8) if want_flags else None
    pi = C.POINTER(C.c_int32)
    cabi.check(lib.rg_pnp_ransac_batched_host(
        _vp(ctx), _vp(stream), V, _vp(cabi.ptr(X)), _vp(cabi.ptr(y)), view_off.ctypes.data_as(pi),
        vote.ctypes.data_as(pi) if vote is not None else None, _vp(cabi.ptr(idx)), hyp_off.ctypes.data_as(pi), int(n),
        float(thr2), int(score_path), _vp(cabi.ptr(best_idx)), _vp(cabi.ptr(best_count)), _vp(cabi.ptr(Rt)),
        _vp(cabi.ptr(mask)), _vp(cabi.ptr(counts)), _vp(cabi.ptr(poses)), _vp(cabi.ptr(flags))))
    out = {"best_idx": best_idx, "best_count": best_count, "R": Rt[:, :9].reshape(V, 3, 3).copy(), "t": Rt[:, 9:].copy(),
           "view_off": view_off, "hyp_off": hyp_off}
    split_n = lambda a: [a[view_off[v]:view_off[v + 1]] for v in range(V)]
    split_h = lambda a: [a[hyp_off[v]:hyp_off[v + 1]] for v in range(V)]
    if want_mask:
        out["mask"] = split_n(mask)
    if want_counts:
        out["counts"] = split_h(counts)
    if want_poses:
        out["poses"] = split_h(poses)
    if want_flags:
        out["flags"] = split_h(flags)
    return out


def pnp_minimize(X, y, device=None, stream=0):
    lib = cabi.load_library()
    ctx = cabi.context(device)
    X = _f64(X).reshape(-1, 3)
    y = _f64(y).reshape(-1, 2)
    R = np.empty((3, 3))
    t = np.empty(3)
    cabi.check(lib.rg_pnp_minimize_host(_vp(ctx), _vp(stream), X.shape[0], _vp(cabi.ptr(X)), _vp(cabi.ptr(y)),
                                        _vp(cabi.ptr(R)), _vp(cabi.ptr(t))))
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
    Xs = [_f64(a).reshape(-1, 3) for a in X_list]
    ys = [_f64(a).reshape(-1, 2) for a in y_list]
    view_off = np.zeros(V + 1, dtype=np.int32)
    for v in range(V):
        if Xs[v].shape[0] != ys[v].shape[0]:
            raise ValueError(f"view {v}: X and y must have the same number of rows")
        view_off[v + 1] = view_off[v] + Xs[v].shape[0]
    R = _f64(R).reshape(-1, 3, 3)
    t = _f64(t).reshape(-1, 3)
    if R.shape[0] != V or t.shape[0] != V:
        raise ValueError("R must be (V, 3, 3) and t (V, 3)")
    if int(rounds) < 1:
        raise ValueError("rounds must be >= 1")
    if int(rounds) > 1 and thr2 is None:
        raise ValueError("rounds > 1 needs thr2 (the consensus threshold)")
    N = int(view_off[-1])
    X = np.ascontiguousarray(np.concatenate(Xs)) if V else np.zeros((0, 3))
    y = np.ascontiguousarray(np.concatenate(ys)) if V else np.zeros((0, 2))
    mask = None
    if masks is not None:
        if len(masks) != V or any(len(m) != Xs[v].shape[0] for v, m in enumerate(masks)):
            raise ValueError("masks must match X_list")
        mask = np.ascontiguousarray(np.concatenate([np.asarray(m, dtype=bool).astype(np.uint8) for m in masks])) if V else None
    Kt = pnp_k_table(K, V)
    Rt = np.ascontiguousarray(np.concatenate([R.reshape(V, 9), t], axis=1))
    cost = np.full(V, np.nan)
    iters = np.zeros(V, dtype=np.int32)
    status = np.zeros(V, dtype=np.int32)
    mask_out = np.zeros(max(N, 1), dtype=np.uint8) if thr2 is not None else None
    lib = cabi.load_library()
    ctx = cabi.context(device)
    cabi.check(lib.rg_pnp_refine_host(
        _vp(ctx), _vp(stream), V, _vp(cabi.ptr(X)), _vp(cabi.ptr(y)), view_off.ctypes.data_as(C.POINTER(C.c_int32)),
        _vp(cabi.ptr(Kt)), _vp(cabi.ptr(mask)), _vp(cabi.ptr(Rt)), int(max_iter), float(ftol), int(rounds),
        float(thr2) if thr2 is not None else 0.0, _vp(cabi.ptr(mask_out)), _vp(cabi.ptr(cost)), _vp(cabi.ptr(iters)),
        _vp(cabi.ptr(status))))
    out = {"R": Rt[:, :9].reshape(V, 3, 3).copy(), "t": Rt[:, 9:].copy(), "cost": cost, "iters": iters, "status": status,
           "view_off": view_off}
    if mask_out is not None:
        out["mask"] = [mask_out[view_off[v]:view_off[v + 1]].copy() for v in range(V)]
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
    lib = cabi.load_library()
    ctx = cabi.context(device)
    X = _f64(X).reshape(-1, 3)
    y = _f64(y).reshape(-1, 2)
    poses = _f64(poses).reshape(-1, 12)
    counts = np.zeros(poses.shape[0], dtype=np.int32)
    cabi.check(lib.rg_pnp_score_count_host(_vp(ctx), _vp(stream), X.shape[0], _vp(cabi.ptr(X)), _vp(cabi.ptr(y)),
                                           poses.shape[0], _vp(cabi.ptr(poses)), float(thr2), int(score_path),
                                           _vp(cabi.ptr(counts))))
    return counts


# ---------------------------------------------------------------------------------------------------------------
# two-view geometry (SURVEY.md section 8f rows N1-N3)
# ---------------------------------------------------------------------------------------------------------------
def triangulate(C1, C2, x1_list, x2_list, method=TRI_OPTIMAL, device=None, stream=0):
    """Triangulates every correspondence of P camera pairs in ONE library call.

    C1, C2 : (P, 3, 4) (or (3, 4) for one pair);  x1_list[p], x2_list[p] : (N_p, 2) image points.
    Returns a list of (N_p, 3) arrays (lab3.triangulate_optimal / triangulate_linear per correspondence)."""
    lib = cabi.load_library()
    ctx = cabi.context(device)
    C1 = _f64(C1).reshape(-1, 3, 4)
    C2 = _f64(C2).reshape(-1, 3, 4)
    P = C1.shape[0]
    if C2.shape[0] != P or len(x1_list) != P or len(x2_list) != P:
        raise ValueError("C1, C2, x1_list and x2_list must describe the same number of camera pairs")
    a = [_f64(x).reshape(-1, 2) for x in x1_list]
    b = [_f64(x).reshape(-1, 2) for x in x2_list]
    off = np.zeros(P + 1, dtype=np.int32)
    for p in range(P):
        if a[p].shape != b[p].shape:
            raise ValueError(f"pair {p}: x1 and x2 must have the same shape")
        off[p + 1] = off[p] + a[p].shape[0]
    N = int(off[-1])
    x1 = np.ascontiguousarray(np.concatenate(a)) if P else np.zeros((0, 2))
    x2 = np.ascontiguousarray(np.concatenate(b)) if P else np.zeros((0, 2))
    X = np.full((N, 3), np.nan)
    cabi.check(lib.rg_triangulate_host(_vp(ctx), _vp(stream), P, _vp(cabi.ptr(C1)), _vp(cabi.ptr(C2)),
                                       off.ctypes.data_as(C.POINTER(C.c_int32)), _vp(cabi.ptr(x1)), _vp(cabi.ptr(x2)),
                                       int(method), _vp(cabi.ptr(X))))
    return [X[off[p]:off[p + 1]] for p in range(P)]


def fmatrix_from_cameras(C1, C2, device=None, stream=0):
    """lab3.fmatrix_from_cameras for P camera pairs: (P, 3, 4) x 2 -> (P, 3, 3)."""
    lib = cabi.load_library()
    ctx = cabi.context(device)
    C1 = _f64(C1).reshape(-1, 3, 4)
    C2 = _f64(C2).reshape(-1, 3, 4)
    if C1.shape != C2.shape:
        raise ValueError("C1 and C2 must have the same shape")
    F = np.full((C1.shape[0], 3, 3), np.nan)
    cabi.check(lib.rg_fmatrix_from_cameras_host(_vp(ctx), _vp(stream), C1.shape[0], _vp(cabi.ptr(C1)), _vp(cabi.ptr(C2)),
                                                _vp(cabi.ptr(F))))
    return F


def relative_pose(M, y1, y2, K=None, device=None, stream=0) -> dict:
    """fun.relative_camera_pose for P pairs in one call.  M (P,3,3) essential matrices — or fundamental matrices when
    K ((3,3) shared or (P,3,3)) is given, E = K^T M K being formed on the device; y1, y2 (P,2) C-normalised.
    Returns dict(R (P,3,3), t (P,3), which (P,) candidate index or -1, npass (P,))."""
    lib = cabi.load_library()
    ctx = cabi.context(device)
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
    cabi.check(lib.rg_relative_pose_host(_vp(ctx), _vp(stream), P, _vp(cabi.ptr(M)), _vp(cabi.ptr(K)), per_pair,
                                         _vp(cabi.ptr(y1)), _vp(cabi.ptr(y2)), _vp(cabi.ptr(Rt)), _vp(cabi.ptr(which)),
                                         _vp(cabi.ptr(npass))))
    return {"R": Rt[:, :9].reshape(P, 3, 3).copy(), "t": Rt[:, 9:].copy(), "which": which, "npass": npass}


def two_view_init(pts_list, F, K, masks=None, device=None, stream=0) -> dict:
    """main.py:54-76 (E = K^T F K, C-normalisation, relative pose, triangulation of every correspondence) for P image
    pairs in ONE library call.  pts_list[p]: (N_p, 4) pixel rows (x0, x1, y0, y1); F: (P, 3, 3); K: (3, 3);
    masks[p] (optional): (N_p,) uint8, zero = skip.  Returns dict(R (P,3,3), t (P,3), which (P,), X list of (N_p,3))."""
    lib = cabi.load_library()
    ctx = cabi.context(device)
    P = len(pts_list)
    F = _f64(F).reshape(-1, 3, 3)
    K = _f64(K)
    if F.shape[0] != P or K.shape != (3, 3):
        raise ValueError("F must be (P, 3, 3) and K (3, 3)")
    pts = [_f64(p).reshape(-1, 4) for p in pts_list]
    off = np.zeros(P + 1, dtype=np.int32)
    for p in range(P):
        off[p + 1] = off[p] + pts[p].shape[0]
    N = int(off[-1])
    allp = np.ascontiguousarray(np.concatenate(pts)) if P else np.zeros((0, 4))
    mask = None
    if masks is not None:
        if len(masks) != P or any(len(m) != pts[p].shape[0] for p, m in enumerate(masks)):
            raise ValueError("masks must match pts_list")
        mask = np.ascontiguousarray(np.concatenate([np.asarray(m, dtype=np.uint8) for m in masks])) if P else None
    Rt = np.full((P, 12), np.nan)
    which = np.full(P, -1, dtype=np.int32)
    X = np.full((N, 3), np.nan)
    cabi.check(lib.rg_two_view_init_host(_vp(ctx), _vp(stream), P, _vp(cabi.ptr(allp)), off.ctypes.data_as(C.POINTER(C.c_int32)),
                                         _vp(cabi.ptr(F)), _vp(cabi.ptr(K)), _vp(cabi.ptr(mask)), _vp(cabi.ptr(Rt)),
                                         _vp(cabi.ptr(which)), _vp(cabi.ptr(X))))
    return {"R": Rt[:, :9].reshape(P, 3, 3).copy(), "t": Rt[:, 9:].copy(), "which": which,
            "X": [X[off[p]:off[p + 1]] for p in range(P)]}


def gold_standard(pts_list, F0, masks=None, max_iter=50, ftol=1e-12, want_points=False, device=None, stream=0) -> dict:
    """Gold-standard refinement (second half of fun.getFFromLabCode, fun.py:342-369) of P pairs in ONE library call.
    pts_list[p]: (N_p, 4) pixel rows; F0: (P, 3, 3); masks[p] optional inlier masks.
    Returns dict(F (P,3,3), cost (P,), iters (P,), status (P,), X list when want_points)."""
    lib = cabi.load_library()
    ctx = cabi.context(device)
    P = len(pts_list)
    F0 = _f64(F0).reshape(-1, 3, 3)
    if F0.shape[0] != P:
        raise ValueError("F0 must be (P, 3, 3)")
    pts = [_f64(p).reshape(-1, 4) for p in pts_list]
    off = np.zeros(P + 1, dtype=np.int32)
    for p in range(P):
        off[p + 1] = off[p] + pts[p].shape[0]
    N = int(off[-1])
    allp = np.ascontiguousarray(np.concatenate(pts)) if P else np.zeros((0, 4))
    mask = None
    if masks is not None:
        if len(masks) != P or any(len(m) != pts[p].shape[0] for p, m in enumerate(masks)):
            raise ValueError("masks must match pts_list")
        mask = np.ascontiguousarray(np.concatenate([np.asarray(m, dtype=np.uint8) for m in masks])) if P else None
    F = np.full((P, 3, 3), np.nan)
    cost = np.full(P, np.nan)
    iters = np.zeros(P, dtype=np.int32)
    status = np.zeros(P, dtype=np.int32)
    X = np.full((N, 3), np.nan) if want_points else None
    cabi.check(lib.rg_gold_standard_host(_vp(ctx), _vp(stream), P, _vp(cabi.ptr(allp)), off.ctypes.data_as(C.POINTER(C.c_int32)),
                                         _vp(cabi.ptr(F0)), _vp(cabi.ptr(mask)), int(max_iter), float(ftol), _vp(cabi.ptr(F)),
                                         _vp(cabi.ptr(cost)), _vp(cabi.ptr(iters)), _vp(cabi.ptr(status)), _vp(cabi.ptr(X))))
    out = {"F": F, "cost": cost, "iters": iters, "status": status}
    if want_points:
        out["X"] = [X[off[p]:off[p + 1]] for p in range(P)]
    return out


def fmatrix_residuals_gs(params, pl, pr, device=None, stream=0):
    """lab3.fmatrix_residuals_gs on the GPU: params (12 + 3N,), pl / pr (2, N) -> (4N,)."""
    lib = cabi.load_library()
    ctx = cabi.context(device)
    params = _f64(params).ravel()
    pl = _f64(pl)
    pr = _f64(pr)
    N = pl.shape[1]
    out = np.empty(4 * N)
    cabi.check(lib.rg_fmatrix_residuals_gs_host(_vp(ctx), _vp(stream), N, _vp(cabi.ptr(params)), _vp(cabi.ptr(pl)),
                                                _vp(cabi.ptr(pr)), _vp(cabi.ptr(out))))
    return out


def bundle_adjust(cams, pts, uv, cam_idx, pt_idx, n_fixed=1, max_iter=50, ftol=1e-4, device=None, stream=0) -> dict:
    """Bundle adjustment (the minimisation of tables.Tables.BundleAdjustment2, tables.py:260-333) in ONE library call.
    cams (V, 3, 4) camera matrices, pts (P, 3), uv (O, 2) observed C-normalised image points, cam_idx / pt_idx (O,) the
    view and point of every observation; the first n_fixed views are held fixed (the reference fixes view 0).
    Returns dict(cams, pts, cost = 0.5 * sum r^2, iters, status: 2 converged, 3 no further descent, 4 max_iter)."""
    lib = cabi.load_library()
    ctx = cabi.context(device)
    cams = np.array(cams, dtype=np.float64).reshape(-1, 3, 4)
    pts = np.array(pts, dtype=np.float64).reshape(-1, 3)
    uv = _f64(uv).reshape(-1, 2)
    ci, ci_p = cabi.as_i32(np.asarray(cam_idx).ravel())
    pi, pi_p = cabi.as_i32(np.asarray(pt_idx).ravel())
    if not (ci.shape[0] == pi.shape[0] == uv.shape[0]):
        raise ValueError("uv, cam_idx and pt_idx must have one row per observation")
    cost = np.full(1, np.nan)
    it_st = np.zeros(2, dtype=np.int32)
    cabi.check(lib.rg_bundle_adjust_host(_vp(ctx), _vp(stream), cams.shape[0], pts.shape[0], uv.shape[0], _vp(cabi.ptr(cams)),
                                         _vp(cabi.ptr(pts)), _vp(cabi.ptr(uv)), ci_p, pi_p, int(n_fixed), int(max_iter), float(ftol),
                                         _vp(cabi.ptr(cost)), _vp(it_st.ctypes.data), _vp(it_st.ctypes.data + 4)))
    return {"cams": cams, "pts": pts, "cost": float(cost[0]), "iters": int(it_st[0]), "status": int(it_st[1])}


def ba_residuals(x, u, v, cam_idx, pt_idx, n_C, n_P, device=None, stream=0) -> np.ndarray:
    """EpsilonBA of tables.Tables.BundleAdjustment2 (tables.py:266-296) on the GPU: x = [cameras (n_C x 12), points (n_P x 3)]
    -> interleaved residuals (2 * n_obs,)."""
    lib = cabi.load_library()
    ctx = cabi.context(device)
    x = _f64(x).ravel()
    if x.shape[0] != 12 * n_C + 3 * n_P:
        raise ValueError("parameter vector must hold n_C * 12 + n_P * 3 values")
    u = _f64(u).ravel()
    v = _f64(v).ravel()
    ci, ci_p = cabi.as_i32(np.asarray(cam_idx).ravel())
    pi, pi_p = cabi.as_i32(np.asarray(pt_idx).ravel())
    if not (u.shape[0] == v.shape[0] == ci.shape[0] == pi.shape[0]):
        raise ValueError("u, v, cam_idx and pt_idx must have one entry per observation")
    out = np.empty(2 * u.shape[0])
    cabi.check(lib.rg_ba_residuals_host(_vp(ctx), _vp(stream), int(n_C), int(n_P), u.shape[0], _vp(cabi.ptr(x)), _vp(cabi.ptr(u)),
                                        _vp(cabi.ptr(v)), ci_p, pi_p, _vp(cabi.ptr(out))))
    return out


def camera_resectioning(Cs, device=None, stream=0):
    """fun.camera_resectioning for V cameras: (V, 3, 4) -> K (V,3,3), R (V,3,3), t (V,3)."""
    lib = cabi.load_library()
    ctx = cabi.context(device)
    Cs = _f64(Cs).reshape(-1, 3, 4)
    V = Cs.shape[0]
    K = np.full((V, 3, 3), np.nan)
    R = np.full((V, 3, 3), np.nan)
    t = np.full((V, 3), np.nan)
    cabi.check(lib.rg_camera_resectioning_host(_vp(ctx), _vp(stream), V, _vp(cabi.ptr(Cs)), _vp(cabi.ptr(K)),
                                               _vp(cabi.ptr(R)), _vp(cabi.ptr(t))))
    return K, R, t


def match_first_within(obs, y, tol=1e-4, device=None, stream=0) -> np.ndarray:
    """For every row of y (N, d) the index of the first row of obs (M, d) closer than tol (strict), -1 if none
    (the 2D<->3D match loop of tables.py:116-124).  d = 2 or 3."""
    lib = cabi.load_library()
    ctx = cabi.context(device)
    obs = _f64(obs)
    y = _f64(y)
    if y.ndim != 2 or y.shape[1] not in (2, 3):
        raise ValueError("y must be (N, 2) or (N, 3)")
    d = y.shape[1]
    obs = obs.reshape(-1, d) if obs.size else np.zeros((0, d))
    idx = np.full(y.shape[0], -1, dtype=np.int32)
    cabi.check(lib.rg_match_first_within_host(_vp(ctx), _vp(stream), d, obs.shape[0], _vp(cabi.ptr(obs)), y.shape[0],
                                              _vp(cabi.ptr(y)), float(tol), _vp(cabi.ptr(idx))))
    return idx


def microbench(device=None, stream=0) -> dict:
    lib = cabi.load_library()
    cabi.context(device)
    out = (C.c_double * 6)()
    cabi.check(lib.rg_microbench_run(out, _vp(stream)))
    return {"ffma_gfma_s": out[0], "ffma2_gfma_s": out[1], "mix_scalar_gevals_s": out[2],
            "mix_packed_gevals_s": out[3], "dfma_gfma_s": out[4], "sms": int(out[5])}
