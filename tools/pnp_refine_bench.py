"""Timing of the refinement of PnP poses (rg_pnp_refine_dev) on the GPU, next to the host minimisers it replaces.

Two workloads:
  * dino36  — the 36 exact Dino views (37-204 correspondences each) in ONE batched call (the one-CTA-per-view path),
              start poses off the truth by ~1e-3;
  * config4 — the consensus of BASELINE config 4 (1 000 000 correspondences, sigma 0.05 px, 1 024 DLT-6 hypotheses):
              device.pnp_ransac, then device.pnp_refine on the RANSAC mask (the multi-CTA path); the RANSAC call is timed
              in the same run for comparison.
Device times: CUDA events around `reps` calls after `warmup` calls (the start pose is restored by a device copy inside
the window: 96 bytes per view).  Host times: SciPy least_squares(method='lm') and OpenCV solvePnP(ITERATIVE,
useExtrinsicGuess=True) on the same inputs, one view after the other.  The GPU name and power limit are read in the same
run.  Writes one JSON file (default profiles/r03_pnp_refine.json).

    python tools/pnp_refine_bench.py [--out FILE] [--reps N] [--warmup N] [--no-host]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

THR2 = (1.5 / 3217.0) ** 2
# FP64 operations per selected correspondence and pass, counted from pr_point (csrc/pnp_refine_kernels.cuh), FMA = 2:
# R X 15, depth / quotient 1 add + 1 division, u v 2, residual 2 + 4, rows of W Pi 2 + 4 + 3, J rows 9 + 5,
# J^T J 21 x 2 FMA = 84, J^T r 6 x 2 FMA = 24, |r|^2 2 FMA = 4, count 1
FLOPS_PER_POINT = 15 + 1 + 2 + 6 + 9 + 14 + 84 + 24 + 4 + 1
DIVS_PER_POINT = 1
# bytes per pass: the mask byte of every correspondence, X (24 B) and y (16 B) of the selected ones
MASK_BYTES, POINT_BYTES = 1, 40


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else q.stderr.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def time_device(fn, reset, reps, warmup):
    import torch
    for _ in range(warmup):
        reset()
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        reset()
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def host_minimisers(X_list, y_list, R0, t0, masks):
    """Seconds of SciPy and OpenCV over the views, one after the other."""
    from oracle import pnp_refine_path as opr
    out = {}
    t = time.perf_counter()
    for X, y, R, tt, m in zip(X_list, y_list, R0, t0, masks):
        opr.pnp_refine_reference(X, y, R, tt, mask=m)
    out["scipy_lm_s"] = time.perf_counter() - t
    try:
        import cv2
        t = time.perf_counter()
        for X, y, R, tt, m in zip(X_list, y_list, R0, t0, masks):
            sel = np.ones(len(X), bool) if m is None else m.astype(bool)
            cv2.solvePnP(np.ascontiguousarray(X[sel]), np.ascontiguousarray(y[sel]), np.eye(3), None, cv2.Rodrigues(R)[0],
                         tt.reshape(3, 1).copy(), True, cv2.SOLVEPNP_ITERATIVE)
        out["opencv_solvepnp_iterative_s"] = time.perf_counter() - t
    except ImportError:
        out["opencv_solvepnp_iterative_s"] = None
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_pnp_refine.json"))
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--no-host", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU and has no CPU fallback")
    import tsbb15_b200 as rg
    from oracle import pnp_refine_path as opr
    dev = rg.device
    res = {"info": gpu_info(), "reps": a.reps, "warmup": a.warmup, "flops_per_point": FLOPS_PER_POINT,
           "divisions_per_point": DIVS_PER_POINT}

    # ---- dino36 ---------------------------------------------------------------------------------------------------
    g = np.load(os.path.join(ROOT, "tests", "golden", "pnp_golden.npz"))
    views = [rg.synth.dino_view_2d3d(i) for i in range(36)]
    rng = np.random.default_rng(0)
    R0 = np.stack([opr.rodrigues(1e-3 * rng.standard_normal(3)) @ g["R"][i] for i in range(36)])
    t0 = np.stack([g["t"][i] * (1 + 1e-3 * rng.standard_normal(3)) for i in range(36)])
    view_off = dev.offsets([len(v[0]) for v in views])
    d_X = torch.from_numpy(np.ascontiguousarray(np.concatenate([v[0] for v in views]))).cuda()
    d_y = torch.from_numpy(np.ascontiguousarray(np.concatenate([v[1] for v in views]))).cuda()
    out = dev.PnpOutputs(36)
    start = torch.from_numpy(np.concatenate([R0.reshape(36, 9), t0], axis=1)).cuda()
    r = dev.PnpRefineOutputs(36)
    ms = time_device(lambda: dev.pnp_refine(d_X, d_y, view_off, out, res=r), lambda: out.Rt.copy_(start), a.reps, a.warmup)
    it = r.iters.cpu().numpy()
    n = int(view_off[-1])
    res["dino36"] = {"views": 36, "points": n, "ms_per_call": ms, "iters_max": int(it.max()), "iters_mean": float(it.mean()),
                     "ms_per_iteration": ms / max(int(it.max()), 1), "status": sorted(set(r.status.cpu().numpy().tolist())),
                     "bytes_per_iteration": n * (MASK_BYTES + POINT_BYTES)}
    if not a.no_host:
        res["dino36"]["host"] = host_minimisers([v[0] for v in views], [v[1] for v in views], R0, t0, [None] * 36)

    # ---- config4 --------------------------------------------------------------------------------------------------
    X, y, (Rgt, _) = rg.synth.pnp_scene(1000000, seed=4, sigma_px=0.05)
    idx = rg.sampling.fast(X.shape[0], 1024, 6, seed=2)
    d_X, d_y = torch.from_numpy(X).cuda(), torch.from_numpy(y).cuda()
    d_idx = torch.from_numpy(np.ascontiguousarray(idx, dtype=np.int32)).cuda()
    voff, hoff = dev.offsets([X.shape[0]]), dev.offsets([idx.shape[0]])
    out = dev.PnpOutputs(1, X.shape[0], want_mask=True)
    ms_ransac = time_device(lambda: dev.pnp_ransac(d_X, d_y, voff, d_idx, hoff, out, THR2), lambda: None,
                            max(a.reps // 10, 5), 3)
    dev.pnp_ransac(d_X, d_y, voff, d_idx, hoff, out, THR2)
    start = out.Rt.clone()
    r = dev.PnpRefineOutputs(1)
    ms = time_device(lambda: dev.pnp_refine(d_X, d_y, voff, out, d_mask=out.mask, res=r), lambda: out.Rt.copy_(start),
                     a.reps, a.warmup)
    it = int(r.iters.cpu().numpy()[0])
    n_sel = int(out.mask.sum().item())
    ms2 = time_device(lambda: dev.pnp_refine(d_X, d_y, voff, out, d_mask=out.mask, rounds=2, thr2=THR2, res=r),
                      lambda: out.Rt.copy_(start), max(a.reps // 4, 10), 5)
    Rs = start.cpu().numpy()[0]
    Rr = out.Rt.cpu().numpy()[0]
    from oracle import pnp_path as opnp
    res["config4"] = {"points": X.shape[0], "selected": n_sel, "ransac_ms_per_call": ms_ransac, "refine_ms_per_call": ms,
                      "iters": it, "passes": it + 1, "ms_per_pass": ms / (it + 1),
                      "refine_share_of_ransac": ms / ms_ransac, "refine_rounds2_ms_per_call": ms2,
                      "bytes_per_pass": X.shape[0] * MASK_BYTES + n_sel * POINT_BYTES,
                      "fp64_flops_per_pass": n_sel * FLOPS_PER_POINT,
                      "rotation_error_ransac_rad": opnp.rotation_angle(Rs[:9].reshape(3, 3), Rgt),
                      "rotation_error_refined_rad": opnp.rotation_angle(Rr[:9].reshape(3, 3), Rgt),
                      "note": "X, y and the mask (41 MB) fit in the 126 MB L2: passes after the first read L2"}
    if not a.no_host:
        m = out.mask.cpu().numpy()
        res["config4"]["host"] = host_minimisers([X], [y], [Rs[:9].reshape(3, 3)], [Rs[9:]], [m])
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
