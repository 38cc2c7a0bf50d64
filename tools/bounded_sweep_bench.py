"""Bounded sweep (option 12) against the full sweep on the same device-resident config-5 inputs, for each prefix share rho
(option 13), candidate count K (option 14) and share rho0 of the first prefix stage (option 16): step time, evaluations
executed (split into the bound-only and the guarded scorer's), hypotheses not fully scored, pairs that fell back, and
whether the answer equals the full sweep's.  Writes one JSON document (default profiles/r03_bounded_sweep.json).

    python tools/bounded_sweep_bench.py --pairs 512 --steps 3 --out profiles/r03_bounded_sweep.json
    python tools/bounded_sweep_bench.py --pairs 4096 --steps 2 --rho 450 --K 512 --rho0 340 360 380 400 450 \
        --out profiles/r03_two_step_prefix.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 20261018


def main():
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    import tsbb15_b200 as rg
    from tsbb15_b200 import parallel, runtime as rt
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=512)
    ap.add_argument("--n", type=int, default=50000)
    ap.add_argument("--hyp", type=int, default=8192)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rho", type=int, nargs="+", default=[400, 450, 500], help="thousandths")
    ap.add_argument("--K", type=int, nargs="+", default=[256, 512])
    ap.add_argument("--rho0", type=int, nargs="+", default=[380], help="thousandths (>= rho: one prefix stage)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_bounded_sweep.json"))
    args = ap.parse_args()
    sh = parallel.PairShardedRansac(args.pairs, args.n, args.hyp, want_mask=True)
    sh.generate(seed_base=1000)

    def run(option12, rho=450, K=512, rho0=380):
        rt.set_option(12, option12); rt.set_option(13, rho); rt.set_option(14, K); rt.set_option(16, rho0)
        sh.run(thr=1.5, sample_seed=SEED)                # warm-up (workspaces, plan)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            sh.run(thr=1.5, sample_seed=SEED)
        e1.record(); e1.synchronize()
        st = rt.bounded_stats()
        res = sh.unpack(sh.gather(masks=True))
        return e0.elapsed_time(e1) / args.steps, st, res

    full_ms, full_st, full = run(0)
    rows = []
    for rho in args.rho:
        for K in args.K:
            for rho0 in args.rho0:
                ms, st, res = run(1, rho, K, rho0)
                same = (np.array_equal(res["best_idx"], full["best_idx"])
                        and np.array_equal(res["best_count"], full["best_count"])
                        and np.array_equal(res["F"].view(np.uint64), full["F"].view(np.uint64))
                        and all(np.array_equal(a, b) for a, b in zip(res["mask"], full["mask"])))
                rows.append({"rho": rho / 1000.0, "K": K, "rho0": min(rho0, rho) / 1000.0, "ms_per_sweep": ms,
                             "speedup_vs_full": full_ms / ms,
                             "evals_executed": st["evals"], "evals_vs_full": st["evals"] / full_st["evals"],
                             "bound_evals": st["bound_evals"], "guarded_evals": st["guarded_evals"],
                             "not_fully_scored_per_pair": st["not_fully_scored"] / args.pairs,
                             "fallback_pairs": st["fallback_pairs"], "identical_to_full_sweep": bool(same)})
                print(json.dumps(rows[-1]), flush=True)
    rt.set_option(12, 1); rt.set_option(13, 450); rt.set_option(14, 512); rt.set_option(16, 380)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    doc = {"workload": f"config-5 pairs 0..{args.pairs - 1}: {args.pairs} x {args.n} x {args.hyp}, device-resident, "
                       f"PairShardedRansac.run, {args.steps} timed sweeps per setting",
           "gpu": smi, "full_sweep": {"ms_per_sweep": full_ms, "evals_executed": full_st["evals"]}, "bounded": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
