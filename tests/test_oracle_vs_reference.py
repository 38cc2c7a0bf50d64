"""Pins the oracle restatements and the package's numpy host helpers against the UNMODIFIED reference code, imported
from the original project's source tree named by RG_REFERENCE_DIR.  Skipped where that tree is not available; the
golden vectors under tests/golden/ (tests/test_oracle_golden.py) pin the oracle's F, triangulation, pose and
resectioning functions without it."""
import numpy as np
import pytest

from oracle import _refimport as ri
from oracle import f_path as orc

pytestmark = pytest.mark.skipif(not ri.reference_available(),
                                reason="original project not available (set RG_REFERENCE_DIR to its source tree)")


@pytest.fixture(scope="module")
def ref_lab3():
    return ri.import_reference("lab3")


def test_stls_and_residuals_random(ref_lab3):
    rng = np.random.default_rng(3)
    for n in (8, 9, 30):
        pl = rng.uniform(0, 640, (2, n))
        pr = pl + rng.normal(0, 5, (2, n))
        Fr = ref_lab3.fmatrix_stls(pl, pr)
        Fo = orc.fmatrix_stls(pl, pr)
        Frn = orc.normalise_F(Fr)
        assert np.linalg.norm(orc.normalise_F(Fo, Frn) - Frn) < 1e-10
        assert np.allclose(orc.fmatrix_residuals(Fr, pl, pr), ref_lab3.fmatrix_residuals(Fr, pl, pr), rtol=1e-12, atol=1e-12)


def test_package_host_helpers_match_reference(ref_lab3, rg):
    """lab3 mirror: the numpy helpers used by the gold-standard refinement."""
    lab3 = rg.lab3
    rng = np.random.default_rng(5)
    C1 = rng.normal(size=(3, 4))
    C2 = rng.normal(size=(3, 4))
    F = ref_lab3.fmatrix_from_cameras(C1, C2)      # (the mirror's fmatrix_from_cameras / triangulate_* run on the GPU)
    A1, A2 = ref_lab3.fmatrix_cameras(F)
    B1, B2 = lab3.fmatrix_cameras(F)
    assert np.allclose(A1, B1) and np.allclose(A2, B2)
    e1r, e2r = ref_lab3.fmatrix_epipoles(F.copy())
    e1, e2 = lab3.fmatrix_epipoles(F)
    assert np.allclose(e1, e1r) and np.allclose(e2, e2r)
    X = rng.normal(size=3) + np.array([0, 0, 5.0])
    assert np.allclose(lab3.project(X, C1), ref_lab3.project(X, C1))
    assert np.allclose(lab3.homog(np.array([1.0, 2.0])), ref_lab3.homog(np.array([1.0, 2.0])))
    assert np.allclose(lab3.homog(np.ones((2, 3))), ref_lab3.homog(np.ones((2, 3))))
    assert np.allclose(lab3.cross_matrix(X), ref_lab3.cross_matrix(X))
    n = 5
    Xs = rng.normal(size=(3, n)) + np.array([[0], [0], [5.0]])
    params = np.hstack((C1.ravel(), Xs.T.ravel()))
    pl, pr = rng.normal(size=(2, n)), rng.normal(size=(2, n))
    assert np.allclose(lab3.fmatrix_residuals_gs(params, pl, pr), ref_lab3.fmatrix_residuals_gs(params, pl, pr))
    with pytest.raises(ValueError):
        lab3.fmatrix_residuals_gs(params, pl[:, :-1], pr[:, :-1])


def test_reference_broken_pnp_is_really_broken():
    """Documents why the PnP rows are restated from the docstring outline: the reference functions raise."""
    pnp, ransac = ri.import_reference("pnp", "ransac")
    with pytest.raises(Exception):
        pnp.pnp_minimize(np.ones((6, 4)), np.ones((6, 3)), 6)
    with pytest.raises(Exception):
        ransac.ransac_robust(np.ones((10, 2, 3)), np.ones((10, 2, 3)), 5, 1e-3, 3)
    assert ransac.calc_p(0.5, 3, 10) == pytest.approx(1 - (1 - 0.5 ** 3) ** 10)


def test_package_ransac_helpers_match_reference(rg):
    ransac_ref = ri.import_reference("ransac")
    r = rg.ransac
    assert r.calc_p(0.7, 6, 100) == ransac_ref.calc_p(0.7, 6, 100)
    assert r.calc_r(0.7, 6, 0.99) == ransac_ref.calc_r(0.7, 6, 0.99)
    assert r.norm_p([2.0, 4.0, 2.0]) == ransac_ref.norm_p([2.0, 4.0, 2.0])
    assert r.cart([2.0, 4.0, 2.0]) == ransac_ref.cart([2.0, 4.0, 2.0])
    import random
    random.seed(3); a = r.gen_rnd_indices(20, 6)
    random.seed(3); b = ransac_ref.gen_rnd_indices(20, 6)
    assert a == b
    with pytest.raises(ValueError):
        r.gen_rnd_indices(3, 6)
    with pytest.raises(ValueError):
        ransac_ref.gen_rnd_indices(3, 6)


def test_geom_oracle_matches_reference_functions(ref_lab3, dino):
    """oracle/geom_path.py against the unmodified lab3 / fun functions on fresh random inputs."""
    from oracle import geom_path as og
    fun = ri.import_reference("fun")
    rng = np.random.default_rng(21)
    Ps = dino["Ps"]
    for (i, j) in ((0, 1), (10, 14)):
        F = ref_lab3.fmatrix_from_cameras(Ps[i], Ps[j])
        assert np.allclose(og.fmatrix_from_cameras(Ps[i], Ps[j]), F, rtol=1e-12, atol=1e-12 * np.abs(F).max())
        e1, e2 = ref_lab3.fmatrix_epipoles(F.copy())
        o1, o2 = og.fmatrix_epipoles(F)
        assert np.allclose(e1, o1) and np.allclose(e2, o2)
        A1, A2 = ref_lab3.fmatrix_cameras(F)
        B1, B2 = og.fmatrix_cameras(F)
        assert np.allclose(A1, B1) and np.allclose(A2, B2)
        X = np.array([rng.uniform(-0.04, 0.04), rng.uniform(-0.07, 0.02), rng.uniform(-0.7, -0.55)])
        for noise in (0.0, 1.0, 30.0):
            x1 = ref_lab3.project(X, Ps[i]) + rng.normal(0, noise, 2)
            x2 = ref_lab3.project(X, Ps[j]) + rng.normal(0, noise, 2)
            a = ref_lab3.triangulate_optimal(Ps[i], Ps[j], x1.copy(), x2.copy())
            b = og.triangulate_optimal(Ps[i], Ps[j], x1, x2)
            assert np.abs(a - b).max() < 1e-10 * np.abs(a).max()
            a = ref_lab3.triangulate_linear(Ps[i], Ps[j], x1.copy(), x2.copy())
            b = og.triangulate_linear(Ps[i], Ps[j], x1, x2)
            assert np.abs(a - b).max() < 1e-10 * np.abs(a).max()
    M = rng.normal(size=(3, 3))
    U, S, Vt = fun.specSVD(M.copy())
    Uo, So, Vto = og.spec_svd(M)
    assert np.allclose(U, Uo) and np.allclose(S, So) and np.allclose(Vt, Vto)
    for k in (0, 17):
        K, R, t = fun.camera_resectioning(Ps[k])
        Ko, Ro, to = og.camera_resectioning(Ps[k])
        assert np.allclose(K, Ko) and np.allclose(R, Ro) and np.allclose(t, to)


def test_package_data_loaders_match_reference(rg, dino):
    """fun.getCameraMatrices / correspondences.Correspondences (main.py:24-30): same arrays as the reference's loaders."""
    import os
    from oracle import _refimport as ri
    if not ri.reference_available():
        pytest.skip("reference tree not mounted")
    path = os.path.join(ri.REFERENCE_DIR, "BAdino2.mat")
    C = rg.fun.getCameraMatrices(path)
    assert C.shape == (1, 36, 3, 4) and np.array_equal(C[0], dino["Ps"])
    c = rg.correspondences.Correspondences(path)
    ref_fun = ri.import_reference("fun")
    with ri.reference_cwd():
        rc = ref_fun.Correspondences()
        assert np.array_equal(ref_fun.getCameraMatrices(), C)
    for i1, i2 in ((0, 1), (7, 8), (34, 35), (3, 10)):
        a, b = c.getCorrByIndices(i1, i2)
        ra, rb = rc.getCorrByIndices(i1, i2)
        assert np.array_equal(a, ra) and np.array_equal(b, rb)
    assert rg.fun.Correspondences is rg.correspondences.Correspondences
