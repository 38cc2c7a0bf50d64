"""TEST INFRASTRUCTURE ONLY — generates tests/golden/*.npz by running the UNMODIFIED reference code.

Run with RG_REFERENCE_DIR set to the original project's source tree:   python -m oracle.gen_golden
Apart from tests/test_oracle_vs_reference.py, the tests read these fixtures and never the original project.

What is recorded
  dino_data.npz      the reference's own input data (BAdino2.mat cameras / 3-D points / clean 2-D tracks, the noisy
                     imgdata/points.txt tracks as exact integers x100) and its shipped artefacts Fmatrix.npy,
                     clean_data_eval.npy
  f_path_golden.npz  outputs of lab3.fmatrix_stls, lab3.fmatrix_residuals, the fun.py:303-328 loop replayed with the
                     real lab3 functions on seeded np.random.choice draws, and fun.getFFromLabCode itself (seeded)
  pnp_golden.npz     fun.camera_resectioning(newPs[i]) = ground-truth (K, R, t) of the exact synthetic Dino cameras
  gs_golden.npz      the gold-standard stage of fun.getFFromLabCode (fun.py:342-369) replayed with the reference's functions
                     on the RANSAC winner / inliers of the noisy pair (0,1): lab3.fmatrix_cameras, triangulate_optimal,
                     scipy least_squares on lab3.fmatrix_residuals_gs (cost, nfev, status, F_gold), residual vectors
  geom_golden.npz    lab3.triangulate_optimal / triangulate_linear per correspondence (clean, noisy and gross-outlier
                     points of pair (0,1)) and fun.relative_camera_pose on all 35 consecutive clean pairs
"""
from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import _refimport as ri  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def noisy_pair(tracks: np.ndarray, i1: int, i2: int):
    """The commented 'noisy' branch of correspondences.getCorrByIndices (correspondences.py:19-22, 29-34)."""
    y1 = tracks[:, i1 * 2:i1 * 2 + 2]
    y2 = tracks[:, i2 * 2:i2 * 2 + 2]
    ok = np.logical_and(np.any(y1 != -1, axis=1), np.any(y2 != -1, axis=1))
    return np.array(y1[ok]), np.array(y2[ok])


def main() -> None:
    import scipy.io as sio
    lab3, fun = ri.import_reference("lab3", "fun")
    os.makedirs(OUT, exist_ok=True)
    ref = ri.REFERENCE_DIR

    mat = sio.loadmat(os.path.join(ref, "BAdino2.mat"))
    Ps = np.asarray(mat["newPs"].tolist())[0]                 # (36, 3, 4)
    x2d = np.asarray(mat["newPoints2D"].tolist())[0]          # (36, 2, 676), -1 = not visible
    X3d = np.asarray(mat["newPoints3D"])                      # (676, 3)
    tracks = np.loadtxt(os.path.join(ref, "imgdata", "points.txt"))
    tracks_i = np.rint(tracks * 100.0).astype(np.int32)
    assert np.array_equal(tracks_i / 100.0, tracks), "points.txt is not exactly 2-decimal"
    Fmatrix = np.load(os.path.join(ref, "Fmatrix.npy"), allow_pickle=True)
    clean_eval = np.load(os.path.join(ref, "clean_data_eval.npy"), allow_pickle=True)
    np.savez_compressed(os.path.join(ROOT, "tsbb15-3d-reconstruction-project_b200", "data", "dino_data.npz"), Ps=Ps, x2d=x2d, X3d=X3d, tracks_x100=tracks_i,
                        Fmatrix=Fmatrix, clean_data_eval=clean_eval)

    g = {}
    # ---- lab3.fmatrix_stls / fmatrix_residuals on the noisy pair (0,1) --------------------------------------------
    y1, y2 = noisy_pair(tracks, 0, 1)
    p1, p2 = y1.T.copy(), y2.T.copy()                         # (2, N) as main.py:39 passes them
    N = p1.shape[1]
    rng = np.random.RandomState(7)
    K = 64
    stls_idx = np.stack([rng.choice(N, 8, replace=False) for _ in range(K)]).astype(np.int32)
    g["stls_idx"] = stls_idx
    g["stls_F"] = np.stack([lab3.fmatrix_stls(p1[:, s], p2[:, s]) for s in stls_idx])
    g["stlsN_F_noisy01"] = lab3.fmatrix_stls(p1, p2)
    g["resid_F"] = g["stls_F"][:4]
    g["resid_out"] = np.stack([lab3.fmatrix_residuals(F, p1, p2) for F in g["resid_F"]])

    # ---- the loop fun.py:303-328, replayed with the real lab3 functions, indices = seeded reference draw -----------
    H = 3000
    np.random.seed(0)
    idx = np.empty((H, 8), dtype=np.int32)
    counts = np.empty(H, dtype=np.int32)
    F_RANSAC, S_RANSAC, d_RANSAC, best = None, [], [], -1
    first_best, first_best_count = -1, 0
    for i in range(H):
        index_points = np.arange(0, p1.shape[1], 1)
        sel = np.random.choice(index_points, 8, replace=False)
        idx[i] = sel
        F = lab3.fmatrix_stls(p1[:, sel], p2[:, sel])
        d = lab3.fmatrix_residuals(F, p1, p2)
        d = np.max(np.abs(d), axis=0)
        S = np.flatnonzero(d < 1.5)
        counts[i] = len(S)
        if len(S) > first_best_count:
            first_best, first_best_count = i, len(S)
        if len(S) > len(S_RANSAC):
            S_RANSAC, F_RANSAC, d_RANSAC, best = S, F, np.std(d), i
        elif len(S) == len(S_RANSAC):
            if np.linalg.norm(d_RANSAC) > np.linalg.norm(d):
                S_RANSAC, F_RANSAC, d_RANSAC, best = S, F, np.std(d), i
    mask = np.zeros(N, dtype=np.uint8)
    mask[S_RANSAC] = 1
    g["ransac_idx"] = idx
    g["ransac_counts"] = counts
    g["ransac_best_reference_rule"] = np.int32(best)
    g["ransac_best_first_max"] = np.int32(first_best)
    g["ransac_mask"] = mask
    g["ransac_F"] = F_RANSAC

    # ---- fun.getFFromLabCode itself (10000 trials + gold standard), seeded -----------------------------------------
    with ri.reference_cwd():
        c = fun.Correspondences()
        yc1, yc2 = c.getCorrByIndices(0, 1)                   # clean pair (0,1), N = 37
    np.random.seed(0)
    g["getF_clean01_seed0"] = fun.getFFromLabCode(yc1.T, yc2.T)
    g["clean01_y1"] = yc1
    g["clean01_y2"] = yc2
    np.random.seed(0)
    g["getF_noisy01_seed0"] = fun.getFFromLabCode(p1, p2)
    # clean consecutive pairs: F from the cameras (what every correct 8-point solve must reproduce)
    g["F_from_cameras"] = np.stack([lab3.fmatrix_from_cameras(Ps[i], Ps[i + 1]) for i in range(35)])
    np.savez_compressed(os.path.join(OUT, "f_path_golden.npz"), **g)

    # ---- PnP ground truth from the reference's own camera decomposition ---------------------------------------------
    Ks, Rs, ts = [], [], []
    for i in range(36):
        K_, R_, t_ = fun.camera_resectioning(Ps[i])
        Ks.append(K_); Rs.append(R_); ts.append(t_)
    np.savez_compressed(os.path.join(OUT, "pnp_golden.npz"), K=np.stack(Ks), R=np.stack(Rs), t=np.stack(ts))
    # ---- two-view geometry around the RANSAC path (SURVEY.md section 8f) ----------------------------------------------
    gg = {}
    rng = np.random.RandomState(11)
    a = np.concatenate([yc1, yc1 + rng.normal(0, 0.5, yc1.shape), yc1 + rng.normal(0, 4.0, yc1.shape),
                        rng.uniform(0, 600, yc1.shape)])
    b = np.concatenate([yc2, yc2 + rng.normal(0, 0.5, yc2.shape), yc2 + rng.normal(0, 4.0, yc2.shape),
                        rng.uniform(0, 600, yc2.shape)])
    gg["tri_C1"], gg["tri_C2"], gg["tri_x1"], gg["tri_x2"] = Ps[0], Ps[1], a, b
    gg["tri_X_optimal"] = np.stack([lab3.triangulate_optimal(Ps[0], Ps[1], p.copy(), q.copy()) for p, q in zip(a, b)])
    gg["tri_X_linear"] = np.stack([lab3.triangulate_linear(Ps[0], Ps[1], p.copy(), q.copy()) for p, q in zip(a, b)])
    rel = {k: [] for k in ("E", "F", "K", "y1", "y2", "R", "t")}
    with ri.reference_cwd():
        for i in range(35):
            y1, y2 = c.getCorrByIndices(i, i + 1)
            K_, _, _ = fun.camera_resectioning(Ps[i])
            F_ = lab3.fmatrix_from_cameras(Ps[i], Ps[i + 1])
            E_ = np.matmul(np.matmul(np.transpose(K_), F_), K_)                 # fun.py:100-101
            h1, h2 = fun.MakeHomogenous(K_, y1), fun.MakeHomogenous(K_, y2)
            out = fun.relative_camera_pose(E_, h1[0, :2].T, h2[0, :2].T)        # as main.py:62 calls it
            if out is None:
                continue
            for k, v in zip(("E", "F", "K", "y1", "y2", "R", "t"), (E_, F_, K_, h1[0, :2], h2[0, :2], out[0], out[1])):
                rel[k].append(np.array(v, dtype=np.float64))
    for k, v in rel.items():
        gg["rel_" + k] = np.stack(v)
    np.savez_compressed(os.path.join(OUT, "geom_golden.npz"), **gg)
    # ---- gold-standard stage (SURVEY.md section 8f N4): the reference's SciPy refinement, with its own stopping point ----
    from scipy.optimize import least_squares
    gs = {}
    sel = np.flatnonzero(mask)
    in1, in2 = p1[:, sel], p2[:, sel]
    C1g, C2g = lab3.fmatrix_cameras(F_RANSAC)
    Xg = np.vstack([lab3.triangulate_optimal(C1g, C2g, a_, b_) for a_, b_ in zip(in1.T, in2.T)]).T
    par0 = np.hstack((C1g.ravel(), Xg.T.ravel()))
    sol = least_squares(lab3.fmatrix_residuals_gs, par0, xtol=2.22e-14, tr_solver='lsmr', args=(in1, in2))
    gs["F0"], gs["in1"], gs["in2"], gs["params0"] = F_RANSAC, in1, in2, par0
    gs["resid0"] = lab3.fmatrix_residuals_gs(par0, in1, in2)
    gs["scipy_cost"], gs["scipy_nfev"], gs["scipy_status"] = sol.cost, sol.nfev, sol.status
    gs["scipy_params"] = sol.x
    gs["F_gold"] = lab3.fmatrix_from_cameras(sol.x[:12].reshape(3, 4), C2g)
    np.savez_compressed(os.path.join(OUT, "gs_golden.npz"), **gs)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
