"""TEST INFRASTRUCTURE ONLY — generates tests/golden/ba_golden.npz by running the UNMODIFIED reference bundle adjustment.

Run with RG_REFERENCE_DIR set to the original project's source tree:   python -m oracle.gen_golden_ba
(kept apart from gen_golden.py, whose gold-standard stage alone runs for several minutes).

The reference's ``Tables()`` constructor loads ``../images/*.ppm`` (fun.getImages, fun.py:59,71 — not in the repository),
so the tables are created with ``object.__new__`` and filled with the reference's own record classes
(help_classes.View / CameraPose / Point_3D / Observation) exactly as ``addView`` / ``addPoint`` / ``addObs`` would
(tables.py:21-38).  ``Tables.BundleAdjustment2`` (tables.py:260-333) itself then runs unmodified; its SciPy call is
observed through a recording wrapper around ``tables.least_squares`` (the wrapper only forwards).

What is recorded, per scene (3, 8 and all 36 Dino views; built by oracle.ba_path.dino_scene with the reference's
``fun.camera_resectioning``):
  cams0, pts0, uv, cam_idx, pt_idx      the problem, as arrays
  resid0                                the reference's EpsilonBA (tables.py:266-296) at the start
  mask_nnz / mask_rowsum / mask_colsum  signature of the reference's sparsity_mask() (tables.py:346-380)
  scipy_x, scipy_cost, scipy_nfev, scipy_status
  cams1, pts1                           what updateCameras3Dpoints2 wrote back into the tables (tables.py:384-390)
"""
from __future__ import annotations

import contextlib
import io
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import _refimport as ri  # noqa: E402
from oracle import ba_path  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def reference_tables(tables, hc, cams, pts, uv, cam_idx, pt_idx):
    T = object.__new__(tables.Tables)
    T.T_obs = np.array([], dtype="object")
    T.T_views = np.array([], dtype="object")
    T.T_points = np.array([], dtype="object")
    T.K = np.eye(3)
    for i, C in enumerate(cams):
        T.T_views = np.append(T.T_views, np.array([hc.View(i, hc.CameraPose(C[:, :3].copy(), C[:, 3].copy()))]))
    for X in pts:
        T.T_points = np.append(T.T_points, np.array([hc.Point_3D(X.copy())]))
    for y, k, j in zip(uv, cam_idx, pt_idx):
        T.T_obs = np.append(T.T_obs, np.array([hc.Observation(np.array([y[0], y[1], 1.0]), int(k), int(j), None)]))
    return T


def main() -> None:
    tables, fun, hc = ri.import_reference("tables", "fun", "help_classes")
    d = np.load(os.path.join(os.path.dirname(OUT), "..", "tsbb15-3d-reconstruction-project_b200", "data", "dino_data.npz"))
    out = {}
    real = tables.least_squares
    for nv in (3, 8, 36):
        cams, pts, uv, ci, pi = ba_path.dino_scene(d["Ps"], d["x2d"], d["X3d"], nv, camera_resectioning=fun.camera_resectioning)
        T = reference_tables(tables, hc, cams, pts, uv, ci, pi)
        rec = {}

        def spy(f, x0, **kw):
            rec["resid0"] = np.array(f(x0, *kw["args"]))
            rec["mask"] = kw["jac_sparsity"].tocsr()
            rec["kw"] = {k: v for k, v in kw.items() if k not in ("args", "jac_sparsity")}
            kw = dict(kw, verbose=0)
            rec["sol"] = real(f, x0, **kw)
            return rec["sol"]

        tables.least_squares = spy
        try:
            with contextlib.redirect_stdout(io.StringIO()):
                T.BundleAdjustment2()
        finally:
            tables.least_squares = real
        assert rec["kw"] == dict(verbose=2, x_scale="jac", ftol=1e-4, method="trf"), rec["kw"]
        sol, m = rec["sol"], rec["mask"]
        p = f"v{nv}_"
        out[p + "cams0"], out[p + "pts0"], out[p + "uv"] = cams, pts, uv
        out[p + "cam_idx"], out[p + "pt_idx"] = ci.astype(np.int32), pi.astype(np.int32)
        out[p + "resid0"] = rec["resid0"]
        out[p + "mask_nnz"] = np.int64(m.nnz)
        out[p + "mask_rowsum"] = np.asarray(m.sum(axis=1)).ravel().astype(np.int32)
        out[p + "mask_colsum"] = np.asarray(m.sum(axis=0)).ravel().astype(np.int32)
        out[p + "scipy_x"] = sol.x
        out[p + "scipy_cost"], out[p + "scipy_nfev"], out[p + "scipy_status"] = sol.cost, sol.nfev, sol.status
        out[p + "cams1"] = np.stack([v.camera_pose.GetCameraMatrix() for v in T.T_views])
        out[p + "pts1"] = np.stack([q.point for q in T.T_points])
        print(nv, "views:", len(pts), "points", len(uv), "observations; cost", 0.5 * float(rec["resid0"] @ rec["resid0"]),
              "->", sol.cost, "nfev", sol.nfev, "status", sol.status)
    np.savez_compressed(os.path.join(OUT, "ba_golden.npz"), **out)
    print("ba_golden.npz", os.path.getsize(os.path.join(OUT, "ba_golden.npz")))


if __name__ == "__main__":
    main()
