"""The numpy oracle (oracle/) against the golden vectors produced by the UNMODIFIED reference (oracle/gen_golden.py).
CPU only.  This is what pins the oracle; the GPU tests then compare the CUDA path with the oracle."""
import numpy as np
import pytest

from oracle import f_path as orc
from oracle import pnp_path as opnp


def _nerr(Fa, Fb):
    Fb = orc.normalise_F(Fb)
    return np.linalg.norm(orc.normalise_F(Fa, Fb) - Fb)


def test_fmatrix_stls_matches_reference_8pt(f_golden, noisy01):
    p1, p2 = noisy01
    for sel, Fref in zip(f_golden["stls_idx"], f_golden["stls_F"]):
        F = orc.fmatrix_stls(p1[:, sel], p2[:, sel])
        assert np.allclose(F, Fref, rtol=0, atol=1e-12 * np.abs(Fref).max()) or _nerr(F, Fref) < 1e-11


def test_fmatrix_stls_matches_reference_all_points(f_golden, noisy01):
    p1, p2 = noisy01
    assert _nerr(orc.fmatrix_stls(p1, p2), f_golden["stlsN_F_noisy01"]) < 1e-12


def test_fmatrix_stls_shape_error():
    with pytest.raises(ValueError):
        orc.fmatrix_stls(np.zeros((2, 8)), np.zeros((2, 9)))


def test_fmatrix_residuals_matches_reference(f_golden, noisy01):
    p1, p2 = noisy01
    for F, ref in zip(f_golden["resid_F"], f_golden["resid_out"]):
        out = orc.fmatrix_residuals(F, p1, p2)
        assert out.shape == ref.shape == (2, p1.shape[1])
        assert np.allclose(out, ref, rtol=1e-12, atol=1e-12)
    with pytest.raises(ValueError):
        orc.fmatrix_residuals(np.eye(3), p1, p2[:, :-1])


def test_ransac_loop_matches_reference(f_golden, noisy01):
    """fun.py:303-328 replayed by the reference itself with seeded draws: counts, both selection rules, inlier set."""
    p1, p2 = noisy01
    idx = f_golden["ransac_idx"]
    res = orc.f_ransac(p1, p2, idx, thr=1.5, tie="reference")
    assert np.array_equal(res["counts"], f_golden["ransac_counts"])
    assert res["best"] == int(f_golden["ransac_best_reference_rule"])
    assert np.array_equal(res["mask"], f_golden["ransac_mask"])
    assert _nerr(res["F"], f_golden["ransac_F"]) < 1e-12
    assert orc.select_first_max(res["counts"]) == int(f_golden["ransac_best_first_max"])


def test_clean_pairs_reproduce_camera_F(dino, f_golden):
    """BAdino2.mat is exact synthetic data: any 8 visible correspondences give the F of the two cameras."""
    x2d = dino["x2d"]
    rng = np.random.default_rng(0)
    for i in (0, 7, 20, 34):
        y1, y2 = x2d[i].T, x2d[i + 1].T
        ok = np.logical_and(np.any(y1 != -1, axis=1), np.any(y2 != -1, axis=1))
        p1, p2 = y1[ok].T, y2[ok].T
        F = orc.fmatrix_stls(p1, p2)
        assert _nerr(F, f_golden["F_from_cameras"][i]) < 1e-7
        assert orc.inliers(F, p1, p2, 1.5).size == p1.shape[1]
        sel = rng.choice(p1.shape[1], 8, replace=False)
        F8 = orc.fmatrix_stls(p1[:, sel], p2[:, sel])
        assert orc.inliers(F8, p1, p2, 1.5).size >= 8


def test_shipped_Fmatrix_is_the_clean_pair_F(dino, f_golden):
    """The reference's own artefact Fmatrix.npy (output of getFFromLabCode on clean pair (0,1))."""
    assert _nerr(dino["Fmatrix"], f_golden["F_from_cameras"][0]) < 1e-9
    assert _nerr(f_golden["getF_clean01_seed0"], dino["Fmatrix"]) < 1e-9


def test_pnp_oracle_recovers_ground_truth_cameras(dino, pnp_golden):
    """pnp.py:132-152 restated: on the exact Dino data the DLT pose equals fun.camera_resectioning's (R, t)."""
    for i in (0, 5, 17, 35):
        vis = np.any(dino["x2d"][i] != -1, axis=0)
        X = dino["X3d"][vis]
        px = dino["x2d"][i][:, vis]
        K = pnp_golden["K"][i]
        yh = np.linalg.solve(K, np.vstack([px, np.ones(px.shape[1])])).T
        Xh = np.hstack([X, np.ones((X.shape[0], 1))])
        R, t = opnp.pnp_minimize(Xh, yh)
        assert opnp.rotation_angle(R, pnp_golden["R"][i]) < 1e-9
        assert np.linalg.norm(t - pnp_golden["t"][i]) < 1e-9 * max(1.0, np.linalg.norm(t))
        # 6-point minimal sample of exact data gives the same pose
        R6, t6 = opnp.pnp_minimize(Xh[:6], yh[:6])
        assert opnp.rotation_angle(R6, pnp_golden["R"][i]) < 1e-6
        e = opnp.reprojection_error_sq(R, t, X, yh)
        assert e.max() < 1e-20


def test_pnp_oracle_consensus_is_inclusive():
    R, t = np.eye(3), np.zeros(3)
    X = np.array([[0.0, 0.0, 1.0], [0.5, 0.0, 1.0]])
    y = np.array([[0.0, 0.0, 1.0], [0.0, 0.0, 1.0]])
    e = opnp.reprojection_error_sq(R, t, X, y)
    assert np.allclose(e, [0.0, 0.25])
    assert opnp.consensus(R, t, X, y, 0.25).tolist() == [True, True]          # thresh >= e (ransac.py:104)
    assert opnp.consensus(R, t, X, y, 0.2499).tolist() == [True, False]
    with pytest.raises(ValueError):
        opnp.pnp_minimize(np.ones((5, 4)), np.ones((5, 3)))


# ---- two-view geometry oracle (oracle/geom_path.py) against the reference's outputs -----------------------------------
def test_geom_oracle_triangulation_matches_reference_golden(geom_golden):
    from oracle import geom_path as og
    g = geom_golden
    Xo = og.triangulate_optimal_batch(g["tri_C1"], g["tri_C2"], g["tri_x1"], g["tri_x2"])
    Xl = og.triangulate_linear_batch(g["tri_C1"], g["tri_C2"], g["tri_x1"], g["tri_x2"])
    scale = np.abs(g["tri_X_optimal"]).max()
    assert np.abs(Xo - g["tri_X_optimal"]).max() < 1e-10 * scale
    assert np.abs(Xl - g["tri_X_linear"]).max() < 1e-10 * scale


def test_geom_oracle_relative_pose_and_resectioning_match_reference_golden(geom_golden, pnp_golden, dino):
    from oracle import geom_path as og
    g = geom_golden
    for k in range(len(g["rel_E"])):
        R, t = og.relative_camera_pose(g["rel_E"][k], g["rel_y1"][k], g["rel_y2"][k])
        assert np.abs(R - g["rel_R"][k]).max() < 1e-12 and np.abs(t - g["rel_t"][k]).max() < 1e-12
        assert np.allclose(og.essential_from_F(g["rel_K"][k], g["rel_F"][k]), g["rel_E"][k], rtol=1e-13, atol=0)
    assert np.abs(g["rel_R"][0] - dino["clean_data_eval"][1]).max() < 1e-6     # the reference's shipped artefact
    for k in (0, 9, 35):
        K, R, t = og.camera_resectioning(dino["Ps"][k])
        assert np.allclose(K, pnp_golden["K"][k], rtol=1e-13) and np.allclose(R, pnp_golden["R"][k], atol=1e-13)
        assert np.allclose(t, pnp_golden["t"][k], rtol=1e-12)


def test_geom_oracle_match_loop_semantics():
    from oracle import geom_path as og
    obs = np.array([[0.0, 0.0, 1.0], [1.0, 0.0, 1.0], [0.0, 0.0, 1.0]])
    y = np.array([[0.0, 5e-5, 1.0], [1.0, 1e-4, 1.0], [5.0, 5.0, 1.0]])
    assert og.match_first_within(obs, y, 1e-4).tolist() == [0, -1, -1]       # first of duplicates; strict <
    assert og.match_first_within(np.zeros((0, 3)), y).tolist() == [-1, -1, -1]


# ---- gold-standard stage (oracle/gs_path.py) against the reference's own run ------------------------------------------
def test_gs_oracle_residuals_and_start_point_match_reference_golden(gs_golden):
    from oracle import gs_path as ogs
    g = gs_golden
    assert np.allclose(ogs.fmatrix_residuals_gs(g["params0"], g["in1"], g["in2"]), g["resid0"], rtol=1e-13, atol=1e-13)
    C1, C2, X = ogs.start_point(g["F0"], g["in1"], g["in2"])
    par = np.hstack((C1.ravel(), X.T.ravel()))
    # cameras from F carry the arbitrary sign of an SVD vector: compare through the residuals, which do not
    assert np.allclose(ogs.fmatrix_residuals_gs(par, g["in1"], g["in2"]), g["resid0"], rtol=1e-8, atol=1e-8)
    r = ogs.fmatrix_residuals_gs(g["scipy_params"], g["in1"], g["in2"])
    assert abs(0.5 * r @ r - float(g["scipy_cost"])) < 1e-10 * float(g["scipy_cost"])
    with pytest.raises(ValueError):
        ogs.fmatrix_residuals_gs(g["params0"][:-3], g["in1"], g["in2"])


def test_package_host_helpers_match_reference_golden(gs_golden, rg):
    """The package's lab3 mirror at the reference's own gold-standard start point: lab3.fmatrix_cameras of the RANSAC
    winner and lab3.fmatrix_residuals_gs, as the reference computed them (oracle/gen_golden.py)."""
    g = gs_golden
    C1, _ = rg.lab3.fmatrix_cameras(g["F0"])
    assert np.allclose(C1.ravel(), g["params0"][:12], rtol=1e-12, atol=1e-15)
    assert np.allclose(rg.lab3.fmatrix_residuals_gs(g["params0"], g["in1"], g["in2"]), g["resid0"], rtol=1e-12, atol=1e-12)


def test_gs_dense_lm_beats_the_reference_stopping_point(gs_golden):
    """The reference's SciPy run stops on ftol at cost 8.288 after 5482 residual evaluations; the LM / Schur iteration
    that the CUDA path implements reaches 5.7407 in ~10 iterations.  F_gold stays within the tolerance of the LM stage."""
    from oracle import gs_path as ogs
    g = gs_golden
    F, c, it, C1, X = ogs.gold_standard_lm(g["F0"], g["in1"], g["in2"])
    assert c < float(g["scipy_cost"]) and it < 40
    assert abs(c - ogs.cost(C1, X, g["in1"], g["in2"])) < 1e-12 * c
    assert _nerr(F, g["F_gold"]) < 2e-3


# ---- bundle adjustment (SURVEY.md section 8f row N4, multi-view half) -------------------------------------------------
@pytest.fixture(scope="module")
def ba_golden():
    from conftest import _load
    return _load("ba_golden.npz")


@pytest.mark.parametrize("nv", [3, 8, 36])
def test_ba_oracle_residuals_and_mask_match_reference_golden(ba_golden, dino, nv):
    from oracle import ba_path as oba
    g, p = ba_golden, f"v{nv}_"
    cams, pts, uv, ci, pi = g[p + "cams0"], g[p + "pts0"], g[p + "uv"], g[p + "cam_idx"], g[p + "pt_idx"]
    # the scene builder is deterministic: the committed problem is what dino_scene makes from the Dino data
    c2, p2, uv2, ci2, pi2 = oba.dino_scene(dino["Ps"], dino["x2d"], dino["X3d"], nv)
    assert np.abs(c2 - cams).max() < 1e-9 and np.abs(p2 - pts).max() < 1e-12 and np.abs(uv2 - uv).max() < 1e-12
    assert np.array_equal(ci2, ci) and np.array_equal(pi2, pi)
    # EpsilonBA (tables.py:266-296) at the start and at SciPy's solution
    r0 = oba.residuals(oba.pack(cams, pts), uv[:, 0], uv[:, 1], ci, pi, len(cams), len(pts))
    assert r0.shape == g[p + "resid0"].shape and np.abs(r0 - g[p + "resid0"]).max() < 1e-13
    r1 = oba.residuals(g[p + "scipy_x"], uv[:, 0], uv[:, 1], ci, pi, len(cams), len(pts))
    assert abs(0.5 * r1 @ r1 - float(g[p + "scipy_cost"])) < 1e-12 * float(g[p + "scipy_cost"])
    # what the reference wrote back into its tables is SciPy's solution (updateCameras3Dpoints2, tables.py:384-390)
    C1, X1 = oba.unpack(g[p + "scipy_x"], len(cams), len(pts))
    assert np.array_equal(C1, g[p + "cams1"]) and np.array_equal(X1, g[p + "pts1"])
    assert np.array_equal(C1[0], cams[0])                      # first view fixed by the sparsity mask
    # sparsity_mask (tables.py:346-380)
    m = oba.sparsity_mask(ci, pi, len(cams), len(pts)).tocsr()
    assert m.nnz == int(g[p + "mask_nnz"])
    assert np.array_equal(np.asarray(m.sum(axis=1)).ravel(), g[p + "mask_rowsum"])
    assert np.array_equal(np.asarray(m.sum(axis=0)).ravel(), g[p + "mask_colsum"])


def test_ba_oracle_scipy_call_reproduces_the_reference_run(ba_golden):
    """Same SciPy call on the vectorised residual function: same stopping point as the reference's Python-loop residuals
    up to what the rounding of the residuals does to SciPy's finite-difference path (6e-5 of the cost, measured)."""
    from oracle import ba_path as oba
    g, p = ba_golden, "v3_"
    C, X, sol = oba.bundle_adjust_scipy(g[p + "cams0"], g[p + "pts0"], g[p + "uv"], g[p + "cam_idx"], g[p + "pt_idx"])
    assert sol.status == int(g[p + "scipy_status"])
    assert sol.nfev == int(g[p + "scipy_nfev"])
    assert abs(sol.cost - float(g[p + "scipy_cost"])) < 1e-3 * float(g[p + "scipy_cost"])


@pytest.mark.parametrize("nv", [3, 8])
def test_ba_lm_iteration_not_above_the_reference_stopping_point(ba_golden, nv):
    from oracle import ba_path as oba
    g, p = ba_golden, f"v{nv}_"
    cams, pts, uv, ci, pi = g[p + "cams0"], g[p + "pts0"], g[p + "uv"], g[p + "cam_idx"], g[p + "pt_idx"]
    C, X, c, it, st = oba.bundle_adjust_lm(cams, pts, uv, ci, pi, ftol=1e-4)
    assert st == 2 and c <= float(g[p + "scipy_cost"]) and np.array_equal(C[0], cams[0])
    assert abs(oba.cost(C, X, uv, ci, pi) - c) < 1e-12 * c
