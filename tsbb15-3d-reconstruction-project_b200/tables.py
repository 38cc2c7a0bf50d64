"""Mirror of the part of the reference's ``tables`` module that calls the accelerated path (SURVEY.md section 8f row N1):
``Tables.addNewView`` (tables.py:104-159), the live consumer of PnP-RANSAC, plus the table bookkeeping it needs
(``addView`` / ``addPoint`` / ``addObs`` / ``getObsAsArrays`` / ``getCamerasForEvaluation``, tables.py:21-38, 57-73,
221-230) and the two triangulation call sites (``triangulateAndAddPoints`` tables.py:233-247, ``addNewPoints``
tables.py:161-176).

What runs on the GPU
  * the O(N x M) 2D<->3D match loop of tables.py:116-124 (first observation of the last view within 1e-4 of the query)
    -> ``runtime.match_first_within`` (one thread per query, observations tiled through shared memory; indices are
    bit-exact with the Python loop);
  * the pose of the new view: the reference calls OpenCV's ``cv.solvePnPRansac`` (tables.py:141, third-party, unpinned);
    here it is this library's DLT-PnP RANSAC (``runtime.pnp_ransac``; algorithm of ransac.py:37-113 + pnp.py:132-152)
    followed by the algebraic refit on the consensus set (``runtime.pnp_minimize``) — OpenCV's estimator is NOT matched
    (DESIGN.md, "parity unpinned at the OpenCV boundary");
  * triangulation of the new points: one batched ``lab3.triangulate_optimal_batch`` call instead of a Python loop.

  * bundle adjustment (SURVEY.md section 8f row N4): ``BundleAdjustment2`` (tables.py:260-333) gathers the tables into
    arrays as the reference does and minimises the same cost (EpsilonBA, tables.py:266-296, first view fixed as in
    sparsity_mask tables.py:376) in one ``runtime.bundle_adjust`` call — Levenberg-Marquardt with the Schur complement
    on the device instead of SciPy's finite-difference trust-region solver (same cost, not the same iterates);
    ``updateCameras3Dpoints2`` (tables.py:384-390) and ``sparsity_mask`` (tables.py:346-380) keep their behaviour.

Out of scope (SURVEY.md section 2): the dead first version ``BundleAdjustment`` (tables.py:75-102, never called, its cost
is a scalar that least_squares cannot use), plotting, colours/normals export.
The reference's constructor loads ``../images/*.ppm`` (fun.getImages, absent from the repository); here ``images`` is an
optional constructor argument and observation colours are ``None`` without it.
"""
from __future__ import annotations

import numpy as np

from . import lab3
from . import runtime as _rt
from . import sampling as _sampling
from .help_classes import CameraPose, Observation, Point_3D, View


class Tables:
    def __init__(self, images=None):
        self.T_obs = np.array([], dtype='object')
        self.T_views = np.array([], dtype='object')
        self.T_points = np.array([], dtype='object')
        self.images = images
        self.K = np.zeros([3, 3])

    # ---- bookkeeping (tables.py:21-38) ------------------------------------------------------------------------
    def addView(self, image, pose):
        self.T_views = np.append(self.T_views, np.array([View(image, pose)]))
        return self.T_views.size - 1

    def addPoint(self, coord):
        self.T_points = np.append(self.T_points, np.array([Point_3D(coord)]))
        return self.T_points.size - 1

    def addObs(self, coord, view_index, point_index):
        color = None
        if self.images is not None:
            px = self.K @ coord
            color = self.images[view_index, int(px[1]), int(px[0])]
        self.T_obs = np.append(self.T_obs, np.array([Observation(coord, view_index, point_index, color)]))
        k = self.T_obs.size - 1
        v, p = self.T_views[view_index], self.T_points[point_index]
        v.observations_index = np.concatenate((v.observations_index, [k]), axis=0)
        p.observations_index = np.concatenate((p.observations_index, [k]), axis=0)

    def getObsAsArrays(self):
        yij = np.asarray([o.image_coordinates for o in self.T_obs])
        Rktk = np.asarray([self.T_views[o.view_index].camera_pose.GetCameraMatrix() for o in self.T_obs])
        xj = np.asarray([[*self.T_points[o.point_3D_index].point[:3], 1.0] for o in self.T_obs])
        return yij, Rktk, xj

    def getCamerasForEvaluation(self):
        Rs = np.stack([v.camera_pose.R for v in self.T_views]) if self.T_views.size else np.zeros([0, 3, 3])
        ts = np.stack([v.camera_pose.t for v in self.T_views]) if self.T_views.size else np.zeros([0, 3])
        return Rs, ts

    # ---- BA (tables.py:260-390) -------------------------------------------------------------------------------
    def observationArrays(self):
        """The observation table as arrays, in table order: uv (O, 2), view index (O,), point index (O,)."""
        uv = np.array([o.image_coordinates[:2] for o in self.T_obs], dtype=np.float64).reshape(-1, 2)
        cam_idx = np.array([o.view_index for o in self.T_obs], dtype=np.int32)
        pt_idx = np.array([o.point_3D_index for o in self.T_obs], dtype=np.int32)
        return uv, cam_idx, pt_idx

    def BundleAdjustment2(self, max_iter=50, ftol=1e-4, loss="linear", f_scale=1.0):
        """tables.py:298-333: all camera matrices (first view fixed) and all points refined against every observation.
        ftol is the reference's (tables.py:317); here it bounds the relative cost decrease of an accepted LM step.
        loss / f_scale: the robust loss options of the reference's least_squares call, with SciPy's names and defaults
        (see runtime.bundle_adjust); observations are C-normalised, so a scale of s pixels is f_scale = s / K[0, 0].
        Returns the solver record (cost, iters, status) — the reference returns None."""
        Rktk = np.empty((len(self.T_views), 3, 4))
        xj = np.empty((len(self.T_points), 3))
        for i, o in enumerate(self.T_views):
            Rktk[i] = o.camera_pose.GetCameraMatrix()
        for i, o in enumerate(self.T_points):
            xj[i] = o.point
        uv, cam_idx, pt_idx = self.observationArrays()
        res = _rt.bundle_adjust(Rktk, xj, uv, cam_idx, pt_idx, n_fixed=1, max_iter=max_iter, ftol=ftol, loss=loss,
                               f_scale=f_scale)
        self.updateCameras3Dpoints2(res["cams"], res["pts"])
        return {k: res[k] for k in ("cost", "iters", "status")}

    def sparsity_mask(self):
        """tables.py:346-380: the Jacobian sparsity pattern the reference gives SciPy (first view's columns cleared)."""
        from scipy.sparse import lil_matrix
        _, camera_idx, point_idx = self.observationArrays()
        n_obs = len(self.T_obs)
        A = lil_matrix((n_obs * 2, len(self.T_views) * 12 + len(self.T_points) * 3), dtype='int')
        i = np.arange(n_obs)
        for s in range(12):
            A[2 * i, camera_idx * 12 + s] = 1
            A[2 * i + 1, camera_idx * 12 + s] = 1
        for s in range(3):
            A[2 * i, len(self.T_views) * 12 + point_idx * 3 + s] = 1
            A[2 * i + 1, len(self.T_views) * 12 + point_idx * 3 + s] = 1
        A[:, 0:12] = 0
        return A

    def updateCameras3Dpoints2(self, new_pose, new_points):
        for i, o in enumerate(self.T_views):
            o.camera_pose = CameraPose(new_pose[i, :3, :3], new_pose[i, :, 3])
        for i, o in enumerate(self.T_points):
            o.point = new_points[i]

    # ---- EXT2 + EXT3 (tables.py:104-159) ----------------------------------------------------------------------
    def matchLastView(self, y1_hom):
        """For every row of y1_hom the index into T_obs of the first observation of the last added view within 1e-4
        (tables.py:116-124), -1 where there is none.  GPU."""
        obs_idx = np.asarray(self.T_views[len(self.T_views) - 1].observations_index, dtype=np.int64)
        coords = np.array([self.T_obs[v].image_coordinates for v in obs_idx], dtype=np.float64).reshape(-1, 3)
        hit = _rt.match_first_within(coords, np.asarray(y1_hom, dtype=np.float64).reshape(-1, 3), 1e-4)
        return np.where(hit >= 0, obs_idx[np.maximum(hit, 0)], -1)

    def addNewView(self, K, img_index, y1_hom, y2_hom, y1, y2, r=1024, reproj_px=8.0, n=6, seed=0, sample_idx=None,
                   refine="algebraic", loss="linear", f_scale=1.0):
        """Adds the view seen in image ``img_index``: pose from the 2D<->3D correspondences found through the last view
        (PnP-RANSAC), consensus observations appended to the tables.  Returns (A_y1, A_y2): the putative
        correspondences without a 3-D point yet, exactly as the reference does.

        r, reproj_px, n, seed / sample_idx : PnP-RANSAC controls (the reference relies on OpenCV's defaults: 100
        iterations, 8 px reprojection error); reproj_px is converted to C-normalised units with K[0, 0].
        refine : "algebraic" (default) refits the pose algebraically on the consensus set (runtime.pnp_minimize);
        "lm" minimises the reprojection error in pixels with K on the consensus set (runtime.pnp_refine), the final
        stage of OpenCV's solvePnPRansac; the consensus appended is RANSAC's, as solvePnPRansac returns it.
        loss, f_scale : robust loss of the "lm" refinement (SciPy's names, see runtime.pnp_refine_batched); f_scale is in
        pixels.  A loss other than "linear" needs refine="lm"."""
        if refine not in ("algebraic", "lm"):
            raise ValueError("refine must be 'algebraic' or 'lm'")
        _rt.loss_args(loss, f_scale)
        if loss != "linear" and refine != "lm":
            raise ValueError(f"loss={loss!r} needs refine='lm' (the algebraic refit has no loss)")
        y1_hom = np.asarray(y1_hom, dtype=np.float64)
        y2_hom = np.asarray(y2_hom, dtype=np.float64)
        y1 = np.asarray(y1, dtype=np.float64)
        y2 = np.asarray(y2, dtype=np.float64)
        obs_of = self.matchLastView(y1_hom)
        found = obs_of >= 0
        x_i = np.array([self.T_obs[v].point_3D_index for v in obs_of[found]], dtype='int')
        D_3Dpoints = np.array([self.T_points[j].point for j in x_i], dtype=np.float64).reshape(-1, 3)
        D_imgcoords_hom = y2_hom[found]
        A_y1, A_y2 = y1[~found], y2[~found]
        m = D_3Dpoints.shape[0]
        if m < n:
            raise ValueError(f"addNewView: only {m} 2D<->3D correspondences, PnP needs at least {n}")
        if sample_idx is None:
            sample_idx = _sampling.fast(m, int(r), n, seed)
        yn = D_imgcoords_hom[:, :2] / D_imgcoords_hom[:, 2:3]
        thr2 = (float(reproj_px) / float(np.asarray(K)[0, 0])) ** 2
        res = _rt.pnp_ransac(D_3Dpoints, yn, sample_idx, thr2, want_mask=True)
        if res["best_idx"] < 0:
            raise ValueError("addNewView: PnP-RANSAC found no pose with a non-empty consensus set")
        inl = np.flatnonzero(res["mask"])
        R, t = res["R"], res["t"]
        if refine == "lm":
            # np.triu: K of an RQ factorisation can carry rounding dust below the diagonal
            ref = _rt.pnp_refine(D_3Dpoints, yn, R, t, mask=res["mask"], K=np.triu(np.asarray(K, dtype=np.float64)),
                                 loss=loss, f_scale=f_scale)
            R, t = ref["R"], ref["t"]
        elif inl.size >= 6:                                 # refit on the consensus set (OpenCV refines its winner too)
            R, t = _rt.pnp_minimize(D_3Dpoints[inl], yn[inl])
        view_index = self.addView(img_index, CameraPose(R, t))
        for yy, x in zip(D_imgcoords_hom[inl], x_i[inl]):
            self.addObs(yy, view_index, x)
        return A_y1, A_y2

    # ---- EXT5 (tables.py:161-176) and INIT3 (tables.py:233-247): triangulation call sites -----------------------
    def addNewPoints(self, A_y1_hom, A_y2_hom, view_index_1, view_index_2, E=None):
        """Triangulates the putative correspondences that satisfy the epipolar constraint |y1^T E y2| < 0.1
        (tables.py:166-168) — all of them in one GPU call — and adds points + observations.  Returns the count.
        E defaults to fun.getEFromCameras(C1, C2) of the two stored poses (tables.py:165)."""
        C1 = self.T_views[view_index_1].camera_pose
        C2 = self.T_views[view_index_2].camera_pose
        A_y1_hom = np.asarray(A_y1_hom, dtype=np.float64).reshape(-1, 3)
        A_y2_hom = np.asarray(A_y2_hom, dtype=np.float64).reshape(-1, 3)
        if E is None:
            from .fun import getEFromCameras
            E = getEFromCameras(C1, C2)
        keep = np.abs(np.einsum("ni,ij,nj->n", A_y1_hom, E, A_y2_hom)) < 0.1
        X = lab3.triangulate_optimal_batch(C1.GetCameraMatrix(), C2.GetCameraMatrix(), A_y1_hom[keep], A_y2_hom[keep])
        for x, a, b in zip(X, A_y1_hom[keep], A_y2_hom[keep]):
            k = self.addPoint(x)
            self.addObs(a, view_index_1, k)
            self.addObs(b, view_index_2, k)
        return int(keep.sum())

    def triangulateAndAddPoints(self, view_index_1, view_index_2, C1, C2, y1_hom, y2_hom):
        y1_hom = np.asarray(y1_hom, dtype=np.float64).reshape(-1, 3)
        y2_hom = np.asarray(y2_hom, dtype=np.float64).reshape(-1, 3)
        X = lab3.triangulate_optimal_batch(C1.GetCameraMatrix(), C2.GetCameraMatrix(), y1_hom[:, :2], y2_hom[:, :2])
        for x, a, b in zip(X, y1_hom, y2_hom):
            k = self.addPoint(x)
            self.addObs(a, view_index_1, k)
            self.addObs(b, view_index_2, k)
