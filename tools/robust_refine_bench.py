"""Robust losses of the PnP pose refinement and of the gold-standard refinement on the GPU: host-call time, iterations and
cost per case and loss, the accuracy figures of tests/test_gpu_robust_refine.py, and the squared-loss entry points of
this build against another build of the library (e.g. the parent commit's), alternating call by call in one process.

Cases (f_scale = 1 px throughout):
  * pnp_dino36_out5 ..... the 36 Dino views in one call, 5 % of the image points replaced by uniform draws, with K
  * pnp_view_1m ......... one synth.pnp_scene view of 1 000 000 points (config-4 size, 30 % outliers, multi-CTA path),
                          all correspondences, with K
  * gs_noisy01 .......... the 257 correspondences of the noisy Dino pair (0, 1) (tests/golden/gs_golden.npz), all of them
  * gs_two_view_16x50k .. 16 synth.two_view pairs of 50 000 correspondences with 30 % outliers, all of them, started from
                          the F of the true cameras (multi-kernel path)
  * host_ms: wall time of one rg_*_host2 call (copies in and out, ends in a stream synchronisation), median over --reps
    calls after --warmup calls; ms_per_iter divides by the largest iteration count of the call (its items run side by side)

    python tools/robust_refine_bench.py [--ref-lib other/librg_b200.so] [--out profiles/r03_robust_refine.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import robust_refine_oracle as rro  # noqa: E402

LOSS_ID = {k: i for i, k in enumerate(rro.LOSSES)}
vp = C.c_void_p


def _p(a):
    return None if a is None else vp(a.ctypes.data)


class Lib:
    """One build of librg_b200.so loaded through ctypes, with its own context on device 0."""

    def __init__(self, path):
        self.lib = C.CDLL(path)
        self.ctx = C.c_void_p()
        if self.lib.rg_init(0, C.byref(self.ctx)) != 0:
            raise RuntimeError(f"rg_init failed for {path}")

    def pnp(self, case, loss=None):
        X, y, off, K, Rt0 = case
        V = len(off) - 1
        Rt = Rt0.copy()
        cost, it, st = np.zeros(V), np.zeros(V, np.int32), np.zeros(V, np.int32)
        a = [self.ctx, vp(0), V, _p(X), _p(y), _p(off), _p(K), None, _p(Rt), 50, C.c_double(1e-12)]
        fn = self.lib.rg_pnp_refine_host
        if loss is not None:
            fn = self.lib.rg_pnp_refine_host2
            a += [LOSS_ID[loss], C.c_double(1.0)]
        a += [1, C.c_double(0.0), None, _p(cost), _p(it), _p(st)]
        t0 = time.perf_counter()
        rc = fn(*a)
        t = (time.perf_counter() - t0) * 1e3
        if rc != 0:
            raise RuntimeError(f"pnp refinement failed ({rc})")
        return t, {"out": Rt, "cost": cost, "iters": it, "status": st}

    def gs(self, case, loss=None):
        pts, off, F0 = case
        P = len(off) - 1
        F, cost, it, st = np.zeros((P, 3, 3)), np.zeros(P), np.zeros(P, np.int32), np.zeros(P, np.int32)
        a = [self.ctx, vp(0), P, _p(pts), _p(off), _p(F0), None, 50, C.c_double(1e-12)]
        fn = self.lib.rg_gold_standard_host
        if loss is not None:
            fn = self.lib.rg_gold_standard_host2
            a += [LOSS_ID[loss], C.c_double(1.0)]
        a += [_p(F), _p(cost), _p(it), _p(st), None]
        t0 = time.perf_counter()
        rc = fn(*a)
        t = (time.perf_counter() - t0) * 1e3
        if rc != 0:
            raise RuntimeError(f"gold standard failed ({rc})")
        return t, {"out": F, "cost": cost, "iters": it, "status": st}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:                              # noqa: BLE001
        return f"unknown ({e})"


def _K(K):
    K = np.triu(np.asarray(K, dtype=np.float64))
    K[0, 1] = 0.0
    return K


def cases():
    import tsbb15_b200 as rg
    g = np.load(os.path.join(ROOT, "tests", "golden", "pnp_golden.npz"))
    X, Y, Ks, Rt = [], [], [], []
    for i in range(36):
        x, y, k = rg.synth.dino_view_2d3d(i)
        X.append(x)
        Y.append(rro.pnp_with_outliers(y, seed=i)[0])
        Ks.append(_K(k).ravel())
        R0 = rro.opr.rodrigues(2e-3 * np.array([1.0, -0.5, 0.7])) @ g["R"][i]
        Rt.append(np.r_[R0.ravel(), g["t"][i] * 1.001])
    off = np.r_[0, np.cumsum([len(x) for x in X])].astype(np.int32)
    yield "pnp_dino36_out5", "pnp", (np.ascontiguousarray(np.concatenate(X)), np.ascontiguousarray(np.concatenate(Y)), off,
                                     np.ascontiguousarray(np.stack(Ks)), np.ascontiguousarray(np.stack(Rt)))
    Xb, yb, _ = rg.synth.pnp_scene(1000000, seed=4)
    R0, t0 = rg.runtime.pnp_minimize(Xb[300000:], yb[300000:])
    K = _K(rg.synth.calibration(rg.synth.dino()["Ps"][17]))
    yield "pnp_view_1m", "pnp", (Xb, yb, np.array([0, len(Xb)], np.int32), np.ascontiguousarray(K.ravel()[None]),
                                 np.r_[R0.ravel(), t0][None].copy())
    gg = np.load(os.path.join(ROOT, "tests", "golden", "gs_golden.npz"))
    pts = np.ascontiguousarray(np.hstack([gg["in1"].T, gg["in2"].T]))
    yield "gs_noisy01", "gs", (pts, np.array([0, len(pts)], np.int32), np.ascontiguousarray(gg["F0"][None]))
    Ps = rg.synth.dino()["Ps"]
    pairs = [rg.synth.two_view(50000, seed=100 + p)[0] for p in range(16)]
    Ft = rro.og.fmatrix_from_cameras(Ps[0], Ps[1])
    off = np.r_[0, np.cumsum([len(p) for p in pairs])].astype(np.int32)
    yield "gs_two_view_16x50k", "gs", (np.ascontiguousarray(np.concatenate(pairs)), off, np.ascontiguousarray(np.stack([Ft] * 16)))


def accuracy():
    """The quantities of test_cauchy_on_all_correspondences_is_as_good_as_the_squared_loss_on_the_true_inliers."""
    import tsbb15_b200 as rg
    from oracle import f_path as orc
    rt = rg.runtime
    n = 20000
    X, y, (Rg, _) = rg.synth.pnp_scene(n, seed=4)
    inl = np.arange(n) >= int(round(0.3 * n))
    K = _K(rg.synth.calibration(rg.synth.dino()["Ps"][17]))
    r = rt.pnp_ransac(X, y, rg.sampling.fast(n, 1024, 6, seed=2), (8.0 / K[0, 0]) ** 2, want_mask=True)
    out = {"pnp_scene_20000_rot_err_rad": {
        "ransac": rro.opnp.rotation_angle(r["R"], Rg),
        "linear_true_inliers": rro.opnp.rotation_angle(rt.pnp_refine(X, y, r["R"], r["t"], mask=inl, K=K)["R"], Rg),
        "linear_ransac_consensus": rro.opnp.rotation_angle(rt.pnp_refine(X, y, r["R"], r["t"], mask=r["mask"], K=K)["R"], Rg),
        "linear_all": rro.opnp.rotation_angle(rt.pnp_refine(X, y, r["R"], r["t"], K=K)["R"], Rg)}}
    for loss in rro.ROBUST:
        out["pnp_scene_20000_rot_err_rad"][loss + "_all"] = rro.opnp.rotation_angle(
            rt.pnp_refine(X, y, r["R"], r["t"], K=K, loss=loss, f_scale=1.0)["R"], Rg)
    pts, lab = rg.synth.two_view(2000, seed=3)
    Ps = rg.synth.dino()["Ps"]
    Ft = orc.normalise_F(rro.og.fmatrix_from_cameras(Ps[0], Ps[1]))
    fr = rg.batched.f_ransac_pairs([pts], n_hyp=3000, thr=1.5, seed=2, host_sampling=True)

    def err(F):
        return float(np.linalg.norm(orc.normalise_F(F, Ft) - Ft))

    acc = {"ransac": err(fr["F"][0]),
           "linear_true_inliers": err(rt.gold_standard([pts], fr["F"], masks=[lab.astype(np.uint8)])["F"][0]),
           "linear_ransac_consensus": err(rt.gold_standard([pts], fr["F"], masks=[fr["mask"][0]])["F"][0]),
           "linear_all": err(rt.gold_standard([pts], fr["F"])["F"][0])}
    for loss in rro.ROBUST:
        acc[loss + "_all"] = err(rt.gold_standard([pts], fr["F"], loss=loss, f_scale=1.0)["F"][0])
    out["two_view_2000_F_err_normalised"] = acc
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref-lib", default=os.environ.get("RG_REF_LIB"), help="another librg_b200.so for the linear A/B")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_robust_refine.json"))
    ap.add_argument("--reps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU")
    lib = Lib(os.path.join(ROOT, "tsbb15-3d-reconstruction-project_b200", "librg_b200.so"))
    ref = Lib(os.path.abspath(args.ref_lib)) if args.ref_lib else None
    out = {"gpu": gpu_info(), "f_scale_px": 1.0, "ftol": 1e-12, "reps": args.reps, "warmup": args.warmup, "cases": {},
           "linear_ab": {}}
    for name, kind, case in cases():
        rows = {"losses": {}}
        for loss in rro.LOSSES:
            call = (lambda: getattr(lib, kind)(case, loss))  # noqa: E731
            for _ in range(args.warmup):
                call()
            ts, res = [], None
            for _ in range(args.reps):
                t, res = call()
                ts.append(t)
            it = max(int(res["iters"].max()), 1)
            rows["losses"][loss] = {"iters_max": it, "iters_sum": int(res["iters"].sum()), "status": res["status"].tolist()[:36],
                                    "cost_sum": float(res["cost"].sum()), "host_ms": float(np.median(ts)),
                                    "host_ms_min": float(np.min(ts)), "host_ms_max": float(np.max(ts)),
                                    "host_ms_per_iter": float(np.median(ts)) / it}
            print(name, loss, {k: v for k, v in rows["losses"][loss].items() if k != "status"}, flush=True)
        out["cases"][name] = rows
        if ref is not None:
            for _ in range(args.warmup):
                getattr(lib, kind)(case)
                getattr(ref, kind)(case)
            tn, to, r_new, r_old = [], [], None, None
            for rep in range(args.reps):
                for which in ((lib, ref) if rep % 2 == 0 else (ref, lib)):      # A B, then B A: no order bias
                    t, r = getattr(which, kind)(case)
                    if which is lib:
                        tn.append(t)
                        r_new = r
                    else:
                        to.append(t)
                        r_old = r
            same = all(np.array_equal(r_new[k], r_old[k]) for k in ("out", "cost", "iters", "status"))
            # the multi-kernel gold standard (pairs > 4096 correspondences) sums with floating-point atomics: two calls of
            # the SAME build differ in the last bits there, so the A/B difference is stated next to a repeat of this build
            repeat = getattr(lib, kind)(case)[1]
            it = max(int(r_new["iters"].max()), 1)
            out["linear_ab"][name] = {"iters_max": it, "bit_identical": bool(same),
                                      "max_rel_cost_diff_ab": float(np.max(np.abs(r_new["cost"] - r_old["cost"]) /
                                                                           np.abs(r_old["cost"]))),
                                      "repeat_of_this_build_bit_identical": bool(
                                          all(np.array_equal(r_new[k], repeat[k]) for k in ("out", "cost", "iters", "status"))),
                                      "max_rel_cost_diff_repeat": float(np.max(np.abs(r_new["cost"] - repeat["cost"]) /
                                                                               np.abs(r_new["cost"]))),
                                      "host_ms_per_iter_new": [t / it for t in tn], "host_ms_per_iter_ref": [t / it for t in to],
                                      "host_ms_per_iter_new_median": float(np.median(tn)) / it,
                                      "host_ms_per_iter_ref_median": float(np.median(to)) / it}
            print(name, "linear A/B", {k: v for k, v in out["linear_ab"][name].items() if not isinstance(v, list)}, flush=True)
    out["accuracy"] = accuracy()
    print("accuracy", out["accuracy"], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
