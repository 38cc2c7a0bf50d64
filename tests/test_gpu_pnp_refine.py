"""GPU tests of the refinement of PnP poses (csrc/pnp_refine_kernels.cuh, DESIGN.md section 4.7): exact Dino views return
the ground truth, noisy scenes reach the SciPy / OpenCV minimum with the iteration count of the numpy restatement, the
config-4 chain RANSAC -> refinement runs on one stream, the one-CTA and multi-CTA paths agree, and the drop-in layers
(ransac_robust(refine=True), Tables.addNewView(refine="lm")) use it."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import pnp_path as opnp
from oracle import pnp_refine_path as opr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THR2 = (1.5 / 3217.0) ** 2


@pytest.fixture(scope="module")
def rt(rg):
    return rg.runtime


def _perturb(R, t, seed, size=1e-3):
    rng = np.random.default_rng(seed)
    return opr.rodrigues(size * rng.standard_normal(3)) @ R, t + size * np.abs(t).max() * rng.standard_normal(3)


def _scene(rg, n, seed, sigma):
    X, y, gt = rg.synth.pnp_scene(n, seed=seed, sigma_px=sigma)
    inl = np.zeros(n, bool)
    inl[int(round(0.3 * n)):] = True
    # the algebraic start on the device (TSQR): the numpy oracle's full SVD of the (3m, 12) design matrix would need
    # (3m)^2 doubles for the 200 000-point scene
    R0, t0 = rg.runtime.pnp_minimize(X[inl], y[inl])
    return X, y, inl, R0, t0, gt


def _K(rg):
    K = rg.synth.calibration(rg.synth.dino()["Ps"][17])
    K[1, 0] = 0.0
    K[0, 1] = 0.0                     # OpenCV's pinhole model has no skew: keep the comparison on the same cost
    return K


def test_exact_dino_views_return_ground_truth_and_batch_equals_single(rt, rg, pnp_golden):
    views = [rg.synth.dino_view_2d3d(i) for i in range(36)]
    starts = [_perturb(pnp_golden["R"][i], pnp_golden["t"][i], i) for i in range(36)]
    R0 = np.stack([s[0] for s in starts])
    t0 = np.stack([s[1] for s in starts])
    b = rt.pnp_refine_batched([v[0] for v in views], [v[1] for v in views], R0, t0)
    assert rt.last_stats()["launches"] <= 4
    for i in range(36):
        assert opnp.rotation_angle(b["R"][i], pnp_golden["R"][i]) < 1e-10, i
        assert np.linalg.norm(b["t"][i] - pnp_golden["t"][i]) < 1e-10 * np.linalg.norm(pnp_golden["t"][i]), i
        assert b["status"][i] == 2 and b["cost"][i] < 1e-20
        one = rt.pnp_refine(views[i][0], views[i][1], R0[i], t0[i])
        assert np.array_equal(one["R"], b["R"][i]) and np.array_equal(one["t"], b["t"][i])
        assert one["cost"] == b["cost"][i] and one["iters"] == b["iters"][i] and one["status"] == b["status"][i]
    # with K: the cost in pixels has the same exact minimum
    bk = rt.pnp_refine_batched([v[0] for v in views], [v[1] for v in views], R0, t0,
                               K=np.stack([np.triu(v[2]) for v in views]))
    for i in range(36):
        assert opnp.rotation_angle(bk["R"][i], pnp_golden["R"][i]) < 1e-10, i


def test_device_entry_equals_host_entry_and_rejects_strided_tensors(rt, rg, pnp_golden):
    """device.pnp_refine on the 36 Dino views (one CTA per view) gives the host entry point's results bit for bit; the
    Dino image points are Fortran-ordered arrays, whose torch.from_numpy view is strided and must be refused."""
    import torch
    dev = rg.device
    views = [rg.synth.dino_view_2d3d(i) for i in range(36)]
    starts = [_perturb(pnp_golden["R"][i], pnp_golden["t"][i], 100 + i) for i in range(36)]
    R0 = np.stack([s[0] for s in starts])
    t0 = np.stack([s[1] for s in starts])
    h = rt.pnp_refine_batched([v[0] for v in views], [v[1] for v in views], R0, t0)
    view_off = dev.offsets([len(v[0]) for v in views])
    d_X = torch.from_numpy(np.ascontiguousarray(np.concatenate([v[0] for v in views]))).cuda()
    y = np.concatenate([v[1] for v in views])
    d_y = torch.from_numpy(np.ascontiguousarray(y)).cuda()
    out = dev.PnpOutputs(36)
    out.Rt.copy_(torch.from_numpy(np.concatenate([R0.reshape(36, 9), t0], axis=1)).cuda())
    r = dev.pnp_refine(d_X, d_y, view_off, out)
    torch.cuda.synchronize()
    Rt = out.Rt.cpu().numpy()
    assert np.array_equal(Rt[:, :9].reshape(36, 3, 3), h["R"]) and np.array_equal(Rt[:, 9:], h["t"])
    assert np.array_equal(r.iters.cpu().numpy(), h["iters"]) and np.array_equal(r.status.cpu().numpy(), h["status"])
    assert np.array_equal(r.cost.cpu().numpy(), h["cost"])
    assert not y.flags["C_CONTIGUOUS"]
    with pytest.raises(ValueError):
        dev.pnp_refine(d_X, torch.from_numpy(y).cuda(), view_off, out)
    with pytest.raises(ValueError):
        dev.pnp_refine(d_X.float(), d_y, view_off, out)
    with pytest.raises(ValueError):
        dev.pnp_refine(d_X[:10], d_y, view_off, out)


@pytest.mark.parametrize("sigma", [0.05, 0.5])
@pytest.mark.parametrize("with_K", [False, True])
def test_noisy_scene_reaches_scipy_and_opencv_minimum(rt, rg, sigma, with_K):
    cv2 = pytest.importorskip("cv2")
    X, y, inl, R0, t0, _ = _scene(rg, 2000, 13, sigma)
    K = _K(rg) if with_K else None
    d = rt.pnp_refine(X, y, R0, t0, mask=inl, K=K)
    o = opr.pnp_refine_lm(X, y, R0, t0, mask=inl, K=K)
    assert (d["iters"], d["status"]) == (o["iters"], o["status"]) and d["status"] == 2
    Rs, ts, cs = opr.pnp_refine_reference(X, y, R0, t0, mask=inl, K=K)
    Kc = K if with_K else np.eye(3)
    px = np.ascontiguousarray((np.hstack([y[inl], np.ones((int(inl.sum()), 1))]) @ Kc.T)[:, :2])
    _, rv, tv = cv2.solvePnP(X[inl], px, Kc, None, cv2.Rodrigues(R0)[0], t0.reshape(3, 1).copy(), True,
                             cv2.SOLVEPNP_ITERATIVE)
    for Rm, tm in ((Rs, ts), (cv2.Rodrigues(rv)[0], tv.ravel())):
        assert opnp.rotation_angle(d["R"], Rm) < 1e-9
        assert np.linalg.norm(d["t"] - tm) < 1e-9 * np.linalg.norm(tm)
    assert abs(d["cost"] - cs) <= 1e-10 * cs
    assert opnp.rotation_angle(d["R"], o["R"]) < 1e-9 and abs(d["cost"] - o["cost"]) <= 1e-12 * o["cost"]
    assert np.abs(d["R"] @ d["R"].T - np.eye(3)).max() < 1e-12


def test_config4_chain_ransac_then_refine_on_one_stream(rg):
    import torch
    dev = rg.device
    X, y, (Rgt, tgt) = rg.synth.pnp_scene(1000000, seed=4, sigma_px=0.05)
    idx = rg.sampling.fast(X.shape[0], 1024, 6, seed=2)
    d_X = torch.from_numpy(X).cuda()
    d_y = torch.from_numpy(y).cuda()
    d_idx = torch.from_numpy(np.ascontiguousarray(idx, dtype=np.int32)).cuda()
    view_off = dev.offsets([X.shape[0]])
    hyp_off = dev.offsets([idx.shape[0]])
    torch.cuda.synchronize()
    out = dev.PnpOutputs(1, X.shape[0], want_mask=True)
    dev.pnp_ransac(d_X, d_y, view_off, d_idx, hyp_off, out, THR2)
    Rt_ransac = out.Rt.clone()                         # device copies on the same stream: no host synchronisation
    mask_ransac = out.mask.clone()
    res = dev.pnp_refine(d_X, d_y, view_off, out, d_mask=out.mask, rounds=2, thr2=THR2, mask_out=out.mask)
    torch.cuda.synchronize()
    Rt0 = Rt_ransac.cpu().numpy()[0]
    m0 = mask_ransac.cpu().numpy()
    Rt1 = out.Rt.cpu().numpy()[0]
    m1 = out.mask.cpu().numpy()
    o = opr.pnp_refine_lm(X, y, Rt0[:9].reshape(3, 3), Rt0[9:], mask=m0, rounds=2, thr2=THR2)
    assert opnp.rotation_angle(Rt1[:9].reshape(3, 3), o["R"]) < 1e-9
    assert np.linalg.norm(Rt1[9:] - o["t"]) < 1e-9 * np.linalg.norm(o["t"])
    assert int(res.status[0]) == o["status"] and int(res.iters[0]) == o["iters"]
    assert abs(float(res.cost[0]) - o["cost"]) <= 1e-10 * o["cost"]
    # the consensus is exact except at FP64 near-ties of thr2 >= e (the two poses agree to ~1e-12, not bit for bit)
    e = opnp.reprojection_error_sq(Rt1[:9].reshape(3, 3), Rt1[9:], X, np.hstack([y, np.ones((X.shape[0], 1))]))
    near = np.abs(e - THR2) <= 1e-9 * THR2
    assert np.array_equal(m1[~near], o["mask"][~near]) and int(near.sum()) <= 10
    assert m1.sum() > 0.6 * X.shape[0]
    assert opnp.rotation_angle(Rt1[:9].reshape(3, 3), Rgt) < opnp.rotation_angle(Rt0[:9].reshape(3, 3), Rgt)


def test_one_cta_and_multi_cta_paths_agree_and_repeat_bit_for_bit(rt, rg):
    scenes = [_scene(rg, n, 20 + k, 0.3) for k, n in enumerate((300, 2500, 4000))]
    args = ([s[0] for s in scenes], [s[1] for s in scenes], np.stack([s[3] for s in scenes]), np.stack([s[4] for s in scenes]))
    kw = {"masks": [s[2] for s in scenes], "K": _K(rg)}
    a = rt.pnp_refine_batched(*args, **kw)
    a2 = rt.pnp_refine_batched(*args, **kw)
    rt.set_option(11, 1)
    try:
        b = rt.pnp_refine_batched(*args, **kw)
        b2 = rt.pnp_refine_batched(*args, **kw)
        big = _scene(rg, 200000, 7, 0.3)
        c = rt.pnp_refine(big[0], big[1], big[3], big[4], mask=big[2])
    finally:
        rt.set_option(11, 0)
    c2 = rt.pnp_refine(big[0], big[1], big[3], big[4], mask=big[2])       # > 4096 points: multi-CTA either way
    for k in ("R", "t", "cost", "iters", "status"):
        assert np.array_equal(a[k], a2[k]) and np.array_equal(b[k], b2[k])
    assert np.array_equal(c["R"], c2["R"]) and c["cost"] == c2["cost"]
    assert np.array_equal(a["iters"], b["iters"]) and np.array_equal(a["status"], b["status"])
    assert np.abs(a["R"] - b["R"]).max() < 1e-12 and np.abs(a["t"] - b["t"]).max() < 1e-12 * np.abs(a["t"]).max()
    assert np.all(np.abs(a["cost"] - b["cost"]) <= 1e-12 * a["cost"])
    o = opr.pnp_refine_lm(big[0], big[1], big[3], big[4], mask=big[2])
    assert (c["iters"], c["status"]) == (o["iters"], o["status"]) and opnp.rotation_angle(c["R"], o["R"]) < 1e-9


def test_edge_cases(rt, rg):
    X, y, inl, R0, t0, _ = _scene(rg, 500, 3, 0.2)
    empty = rt.pnp_refine_batched([], [], np.zeros((0, 3, 3)), np.zeros((0, 3)))
    assert empty["R"].shape == (0, 3, 3)
    z = rt.pnp_refine(X, y, R0, t0, mask=np.zeros(500, np.uint8))
    assert z["status"] == 5 and z["iters"] == 0 and np.array_equal(z["R"], R0) and np.array_equal(z["t"], t0)
    two = rt.pnp_refine(X[:2], y[:2], R0, t0)
    assert two["status"] == 5 and np.array_equal(two["R"], R0)
    nan = rt.pnp_refine(X, y, np.full((3, 3), np.nan), t0)
    assert nan["status"] == 1
    zero = rt.pnp_refine(X, y, R0, t0, max_iter=0)
    assert zero["status"] == 4 and np.array_equal(zero["R"], R0)
    with pytest.raises(ValueError):
        rt.pnp_refine(X, y, R0, t0, max_iter=-1)
    # consensus outputs: one round with a mask, two rounds against the oracle
    r2 = rt.pnp_refine(X, y, R0, t0, mask=inl, rounds=2, thr2=THR2 * 4)
    o2 = opr.pnp_refine_lm(X, y, R0, t0, mask=inl, rounds=2, thr2=THR2 * 4)
    assert np.array_equal(r2["mask"], o2["mask"]) and (r2["iters"], r2["status"]) == (o2["iters"], o2["status"])


def test_dropin_layers_use_the_refinement(rg, pnp_golden):
    X, y, _ = rg.synth.pnp_scene(900, seed=8, sigma_px=0.3, outlier_frac=0.2)
    D = np.stack([np.hstack([y, np.ones((900, 1))]), X], axis=1)
    idx = rg.sampling.fast(300, 400, 6, seed=5)
    R_a, t_a, C_a = rg.ransac.ransac_robust(D[:600], D[600:], 400, THR2 * 9, 6, sample_idx=idx)
    R_b, t_b, C_b = rg.ransac.ransac_robust(D[:600], D[600:], 400, THR2 * 9, 6, sample_idx=idx, refine=True)
    both = np.concatenate([D[:600], D[600:]])
    m_a = np.zeros(900, bool)
    m_a[:600] = opnp.consensus(R_a[0], t_a[0], D[:600, 1], D[:600, 0], THR2 * 9)
    m_a[600:] = opnp.consensus(R_a[0], t_a[0], D[600:, 1], D[600:, 0], THR2 * 9)
    o = opr.pnp_refine_lm(both[:, 1], both[:, 0, :2], R_a[0], t_a[0], mask=m_a, thr2=THR2 * 9, want_mask=True)
    assert opnp.rotation_angle(R_b[0], o["R"]) < 1e-9
    assert len(C_b[0][0]) + len(C_b[0][1]) == int(o["mask"].sum()) >= len(C_a[0][0]) + len(C_a[0][1])
    Xv, yv, Kv = rg.synth.dino_view_2d3d(5)
    Rp, tp = _perturb(pnp_golden["R"][5], pnp_golden["t"][5], 1)
    p = rg.pnp.pnp_refine(np.hstack([Xv, np.ones((len(Xv), 1))]), np.hstack([yv, np.ones((len(yv), 1))]), Rp, tp,
                          K=np.triu(Kv))
    assert opnp.rotation_angle(p["R"], pnp_golden["R"][5]) < 1e-10


def test_sfm_chain_with_lm_refinement_recovers_every_pose(rg, dino, pnp_golden):
    fun = rg.fun
    Tables, CameraPose = rg.tables.Tables, rg.help_classes.CameraPose
    C = dino["Ps"][None]

    def pair(i, j):
        y1, y2 = dino["x2d"][i].T, dino["x2d"][j].T
        ok = np.logical_and(np.any(y1 != -1, axis=1), np.any(y2 != -1, axis=1))
        return np.ascontiguousarray(y1[ok]), np.ascontiguousarray(y2[ok])

    y1, y2 = pair(0, 1)
    F = fun.getFFromLabCode(y1.T, y2.T, r=2000, seed=0, refine=False)
    E, K = fun.getEAndK(C, F)
    T = Tables()
    T.K = K
    y1h, y2h = fun.MakeHomogenous(K, y1), fun.MakeHomogenous(K, y2)
    R, t = fun.relative_camera_pose(E, y1h[0, :2].T, y2h[0, :2].T)
    Rg, tg = pnp_golden["R"], pnp_golden["t"]
    R01 = Rg[1] @ Rg[0].T
    s = np.linalg.norm(tg[1] - R01 @ tg[0]) * np.sign(np.median((dino["X3d"] @ Rg[0].T + tg[0])[:, 2]))
    C1, C2 = CameraPose(), CameraPose(R, t)
    v1, v2 = T.addView(0, C1), T.addView(1, C2)
    T.triangulateAndAddPoints(v1, v2, C1, C2, y1h, y2h)
    for i in range(1, 6):
        a, b = pair(i, i + 1)
        ah, bh = fun.MakeHomogenous(K, a), fun.MakeHomogenous(K, b)
        A1, A2 = T.addNewView(K, i + 1, ah, bh, a, b, r=256, reproj_px=1.5, seed=i, refine="lm")
        view = T.T_views[-1]
        Rk = Rg[i + 1] @ Rg[0].T
        tk = (tg[i + 1] - Rk @ tg[0]) / s
        assert np.abs(view.camera_pose.R - Rk).max() < 1e-5, i
        assert np.abs(view.camera_pose.t - tk).max() < 1e-5 * np.abs(tk).max(), i
        T.addNewPoints(fun.MakeHomogenous(K, A1), fun.MakeHomogenous(K, A2), i, i + 1)


DEBUG_SCRIPT = r"""
import json, sys
import numpy as np
sys.path.insert(0, %r)
from tsbb15_b200 import runtime as rt, synth
out = {}
views = [synth.pnp_scene(n, seed=k, sigma_px=0.3, outlier_frac=0.0)[:2] for k, n in enumerate((40, 900, 5000))]
R0 = np.stack([synth.pnp_scene(10, seed=k)[2][0] for k in range(3)])
t0 = np.stack([synth.pnp_scene(10, seed=k)[2][1] for k in range(3)]) * 1.001
for opt in (0, 1):
    rt.set_option(11, opt)
    r = rt.pnp_refine_batched([v[0] for v in views], [v[1] for v in views], R0, t0, rounds=2, thr2=(1.5 / 3217.0) ** 2)
    out["o%%d" %% opt] = [r["iters"].tolist(), r["status"].tolist(), [int(m.sum()) for m in r["mask"]]]
rt.set_option(11, 0)
print("RESULT " + json.dumps(out))
""" % ROOT


def test_debug_build_refinement_runs_clean():
    lib = os.path.join(ROOT, "tsbb15-3d-reconstruction-project_b200", "librg_b200_debug.so")
    if not os.path.isfile(lib):
        pytest.skip("librg_b200_debug.so not built (python __graft_entry__.py builds it)")
    outs = []
    for env_lib in (lib, None):
        env = dict(os.environ)
        if env_lib:
            env["RG_LIB"] = env_lib
        else:
            env.pop("RG_LIB", None)
        res = subprocess.run([sys.executable, "-c", DEBUG_SCRIPT], capture_output=True, text=True, env=env, timeout=600)
        assert res.returncode == 0, res.stdout[-1500:] + res.stderr[-3000:]
        outs.append(json.loads([l for l in res.stdout.splitlines() if l.startswith("RESULT ")][-1][7:]))
    assert outs[0] == outs[1]
    assert outs[0]["o0"][0] == outs[0]["o1"][0] and outs[0]["o0"][1] == outs[0]["o1"][1]
