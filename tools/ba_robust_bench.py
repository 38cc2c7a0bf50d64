"""Robust-loss bundle adjustment on the GPU: time per LM iteration, iterations, final cost and clean reprojection RMS per
scene and loss, and the squared-loss path against another build of the library (e.g. the parent commit's), alternating
the two in the same process.

Scenes: the 36-view Dino golden with 5 % outliers, ring-of-cameras scenes (synth.ba_scene) of 24 / 60 / 120 views with
10 % outliers (uniform draws over the image, tools/ba_robust_oracle.with_outliers); f_scale = 2 px.
  * host_ms: wall time of one rg_bundle_adjust_host2 call (copies in and out, ends in a stream synchronisation)
  * dev_ms: CUDA events around one rg_bundle_adjust_dev2 call on a stream (device buffers); this entry point enqueues all
    max_iter = 50 iterations, those after convergence return at once, so dev_ms includes their launches
  * per-iteration figures divide by the iterations the call ran; medians over --reps calls after --warmup calls
  * clean_rms_px: root mean |uv - projection|^2 over the observations the outlier recipe left untouched, x 3217

    python tools/ba_robust_bench.py [--ref-lib other/librg_b200.so] [--out profiles/r03_ba_robust.json]
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
import ba_robust_oracle as bro  # noqa: E402

F_SCALE = 2.0 / bro.FOCAL_PX
LOSS_ID = {k: i for i, k in enumerate(bro.LOSSES)}


def scenes():
    import tsbb15_b200 as rg
    with np.load(os.path.join(ROOT, "tests", "golden", "ba_golden.npz")) as g:
        sc = tuple(g["v36_" + k] for k in ("cams0", "pts0", "uv", "cam_idx", "pt_idx"))
    uvo, idx = bro.with_outliers(sc[2])
    yield "dino36_out5", sc[0], sc[1], sc[2], uvo, sc[3], sc[4], idx
    for nv, npt, tr in ((24, 2000, 6), (60, 3000, 8), (120, 1500, 10)):
        cams, pts, uv, ci, pi, _ = rg.synth.ba_scene(nv, npt, track=tr)
        uvo, idx = bro.with_outliers(uv, frac=0.10, seed=1)
        yield f"synth{nv}_out10", cams, pts, uv, uvo, ci, pi, idx


class Lib:
    """One build of librg_b200.so loaded through ctypes, with its own context on device 0."""

    def __init__(self, path):
        self.lib = C.CDLL(path)
        self.ctx = C.c_void_p()
        rc = self.lib.rg_init(0, C.byref(self.ctx))
        if rc != 0:
            raise RuntimeError(f"rg_init failed ({rc}) for {path}")

    def host(self, cams, pts, uv, ci, pi, ftol, loss=None, f_scale=1.0, max_iter=50):
        c, p = np.array(cams, dtype=np.float64), np.array(pts, dtype=np.float64)
        cost, its = np.zeros(1), np.zeros(2, dtype=np.int32)
        vp = C.c_void_p
        a = [self.ctx, vp(0), len(c), len(p), len(uv), vp(c.ctypes.data), vp(p.ctypes.data), vp(uv.ctypes.data),
             vp(ci.ctypes.data), vp(pi.ctypes.data), 1, max_iter, C.c_double(ftol)]
        if loss is None:
            fn = self.lib.rg_bundle_adjust_host
        else:
            fn = self.lib.rg_bundle_adjust_host2
            a += [int(loss), C.c_double(f_scale)]
        a += [vp(cost.ctypes.data), vp(its.ctypes.data), vp(its[1:].ctypes.data)]
        t0 = time.perf_counter()
        rc = fn(*a)
        t = time.perf_counter() - t0
        if rc != 0:
            raise RuntimeError(f"bundle adjustment failed ({rc})")
        return t * 1e3, {"cams": c, "pts": p, "cost": float(cost[0]), "iters": int(its[0]), "status": int(its[1])}

    def dev(self, cams, pts, uv, ci, pi, ftol, loss=None, f_scale=1.0, max_iter=50):
        import torch
        vp = C.c_void_p
        d_c, d_p = torch.from_numpy(np.array(cams)).cuda(), torch.from_numpy(np.array(pts)).cuda()
        d_uv = torch.from_numpy(uv).cuda()
        d_out = torch.zeros(2, dtype=torch.float64, device="cuda")
        d_is = torch.zeros(2, dtype=torch.int32, device="cuda")
        s = torch.cuda.Stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a = [self.ctx, vp(s.cuda_stream), len(cams), len(pts), len(uv), vp(d_c.data_ptr()), vp(d_p.data_ptr()),
             vp(d_uv.data_ptr()), vp(ci.ctypes.data), vp(pi.ctypes.data), 1, max_iter, C.c_double(ftol)]
        if loss is None:
            fn = self.lib.rg_bundle_adjust_dev
        else:
            fn = self.lib.rg_bundle_adjust_dev2
            a += [int(loss), C.c_double(f_scale)]
        a += [vp(d_out.data_ptr()), vp(d_is.data_ptr()), vp(d_is[1:].data_ptr())]
        torch.cuda.synchronize()
        e0.record(s)
        rc = fn(*a)
        e1.record(s)
        s.synchronize()
        if rc != 0:
            raise RuntimeError(f"bundle adjustment failed ({rc})")
        return e0.elapsed_time(e1), int(d_is[0].item())


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:                              # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref-lib", default=os.environ.get("RG_REF_LIB"), help="another librg_b200.so for the linear A/B")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_ba_robust.json"))
    ap.add_argument("--reps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--ftol", type=float, default=1e-4)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU")
    lib = Lib(os.path.join(ROOT, "tsbb15-3d-reconstruction-project_b200", "librg_b200.so"))
    ref = Lib(os.path.abspath(args.ref_lib)) if args.ref_lib else None
    out = {"gpu": gpu_info(), "f_scale_px": 2.0, "ftol": args.ftol, "reps": args.reps, "warmup": args.warmup,
           "scenes": {}, "linear_ab": {}}
    for name, cams, pts, uv, uvo, ci, pi, idx in scenes():
        ci32, pi32 = np.ascontiguousarray(ci, dtype=np.int32), np.ascontiguousarray(pi, dtype=np.int32)
        uvo = np.ascontiguousarray(uvo, dtype=np.float64)
        rows = {"n_views": len(cams), "n_points": len(pts), "n_obs": len(uv), "n_outliers": int(len(idx)), "losses": {}}
        for loss in bro.LOSSES:
            lid = LOSS_ID[loss]
            for _ in range(args.warmup):
                lib.host(cams, pts, uvo, ci32, pi32, args.ftol, lid, F_SCALE)
                lib.dev(cams, pts, uvo, ci32, pi32, args.ftol, lid, F_SCALE)
            th, td, res = [], [], None
            for _ in range(args.reps):
                t, res = lib.host(cams, pts, uvo, ci32, pi32, args.ftol, lid, F_SCALE)
                th.append(t)
                t, it = lib.dev(cams, pts, uvo, ci32, pi32, args.ftol, lid, F_SCALE)
                td.append(t)
            it = max(res["iters"], 1)
            rows["losses"][loss] = {
                "iters": res["iters"], "status": res["status"], "cost": res["cost"],
                "clean_rms_px": bro.clean_rms_px(res["cams"], res["pts"], uv, ci, pi, idx),
                "host_ms": float(np.median(th)), "dev_ms": float(np.median(td)),
                "host_ms_per_iter": float(np.median(th)) / it, "dev_ms_per_iter": float(np.median(td)) / it,
                "dev_ms_min": float(np.min(td)), "dev_ms_max": float(np.max(td))}
            print(name, loss, rows["losses"][loss], flush=True)
        out["scenes"][name] = rows
        if ref is not None:
            # the squared-loss entry points of both builds, alternating call by call
            r_new = r_old = None
            for _ in range(args.warmup):
                lib.dev(cams, pts, uvo, ci32, pi32, args.ftol)
                ref.dev(cams, pts, uvo, ci32, pi32, args.ftol)
            dn, do, hn, ho = [], [], [], []
            for rep in range(args.reps):
                for which in ((lib, ref) if rep % 2 == 0 else (ref, lib)):      # A B, then B A: no order bias
                    t, _ = which.dev(cams, pts, uvo, ci32, pi32, args.ftol)
                    (dn if which is lib else do).append(t)
                    t, r = which.host(cams, pts, uvo, ci32, pi32, args.ftol)
                    (hn if which is lib else ho).append(t)
                    if which is lib:
                        r_new = r
                    else:
                        r_old = r
            same = (r_new["cost"] == r_old["cost"] and r_new["iters"] == r_old["iters"]
                    and np.array_equal(r_new["cams"], r_old["cams"]) and np.array_equal(r_new["pts"], r_old["pts"]))
            it = max(r_new["iters"], 1)
            out["linear_ab"][name] = {
                "iters": r_new["iters"], "bit_identical": bool(same),
                "dev_ms_per_iter_new": [t / it for t in dn], "dev_ms_per_iter_ref": [t / it for t in do],
                "host_ms_per_iter_new": [t / it for t in hn], "host_ms_per_iter_ref": [t / it for t in ho],
                "dev_ms_per_iter_new_median": float(np.median(dn)) / it, "dev_ms_per_iter_ref_median": float(np.median(do)) / it}
            print(name, "linear A/B", {k: v for k, v in out["linear_ab"][name].items() if not isinstance(v, list)}, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
