"""CPU model of the bounded sweep (csrc/bounded.cuh) on oracle counts.

For config-5 pairs (the device's synthetic data and sample draws, replayed on the host) it computes every hypothesis's exact
count over the prefix and over all correspondences with the numpy oracle, then applies the sweep's rule for each prefix
share rho and candidate count K: how many hypotheses escape the bound, whether the pair falls back, and which share of the
full sweep's evaluations is left.  With --rho0 it also applies the two-step prefix (option 16): the evaluations of stage A
(every hypothesis over the first k0 correspondences), |S| (the hypotheses still alive after it) and the evaluations of
stage B (S over the correspondences k0 .. k).  One pair of 50 000 x 8 192 takes about half a minute.

    python tools/bounded_sweep_model.py --pairs 0 1 2 --rho 0.40 0.45 0.50 --K 256 512
    python tools/bounded_sweep_model.py --pairs 0 1 --rho 0.45 --K 512 --rho0 0.34 0.38 0.40
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KSUB = 8


def prefix_points(n: int, rho: float) -> int:
    """Real correspondences of the prefix window: ceil(rho * G) groups of KSUB, rounded up to whole 32-group flag words."""
    G = (n + KSUB - 1) // KSUB
    g = -(-int(round(rho * 1000)) * G // 1000)
    gA = min(G, -(-g // 32) * 32)
    return min(n, gA * KSUB)


def bounded_rule(pre: np.ndarray, full: np.ndarray, rest: int, K: int) -> dict:
    """The rule bnd_select / bnd_check apply to one pair.  pre: prefix counts — exact, or upper bounds of the exact ones
    (the bound-only prefix stage, option 15) — full: exact full counts, rest: points outside the prefix.  Returns the
    candidate mask, the escapees, whether the pair falls back, and the counts the tail sees (full counts where they were
    computed, prefix counts elsewhere)."""
    H = len(pre)
    order = np.lexsort((np.arange(H), -pre))           # (prefix count desc, index asc)
    cand = np.zeros(H, bool)
    cand[order[:min(K, H)]] = True
    L = int(full[cand].max()) if cand.any() else 0
    esc = ~cand & (pre.astype(np.int64) + rest >= L)
    fallback = bool(esc.any())
    seen = full.copy() if fallback else np.where(cand, full, pre)
    return {"cand": cand, "escapees": int(esc.sum()), "fallback": fallback, "counts": seen, "L": L}


def two_step_rule(pre0: np.ndarray, pre: np.ndarray, full: np.ndarray, n: int, k0: int, k: int, K: int) -> dict:
    """The two-step prefix (bnd_select, bnd_extend, bnd_check) for one pair.  pre0 / pre: prefix counts (or upper bounds)
    over the first k0 <= k correspondences, with pre - pre0 <= k - k0.  The candidates are chosen by pre0; S = the
    non-candidates with pre0 + (n - k0) >= L, whose counts are extended to pre; the pair falls back when a member of S has
    pre + (n - k) >= L.  A pair where a member already has pre0 + (n - k) >= L is certain to fall back and skips the
    extension.  Returns bounded_rule's entries plus |S|, `certain` and the evaluations of both stages."""
    r = bounded_rule(pre0, full, n - k0, K)
    live = ~r["cand"] & (pre0.astype(np.int64) + (n - k0) >= r["L"])
    c = np.where(live, pre, pre0)
    esc = live & (c.astype(np.int64) + (n - k) >= r["L"])
    certain = bool((live & (pre0.astype(np.int64) + (n - k) >= r["L"])).any())
    fallback = bool(esc.any())
    seen = full.copy() if fallback else np.where(r["cand"], full, c)
    return {"cand": r["cand"], "live": live, "S": int(live.sum()), "escapees": int(esc.sum()), "fallback": fallback,
            "certain": certain, "counts": seen, "L": r["L"], "evals_a": k0 * len(pre0),
            "evals_b": 0 if certain else int(live.sum()) * (k - k0)}


def main():
    sys.path.insert(0, ROOT)
    from oracle import f_path as orc
    from tsbb15_b200 import philox, synth
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, nargs="+", default=[0])
    ap.add_argument("--n", type=int, default=50000)
    ap.add_argument("--hyp", type=int, default=8192)
    ap.add_argument("--seed", type=int, default=20261018)
    ap.add_argument("--rho", type=float, nargs="+", default=[0.40, 0.45, 0.50])
    ap.add_argument("--K", type=int, nargs="+", default=[256, 512])
    ap.add_argument("--rho0", type=float, nargs="*", default=[], help="stage-A shares of the two-step prefix")
    args = ap.parse_args()
    for pair in args.pairs:
        pts = philox.synth_two_view(args.n, pair, synth.dino()["Ps"], synth.DINO_BBOX)[0]
        idx = philox.sample_indices(args.n, args.hyp, 8, args.seed, pair)
        p1, p2 = pts[:, :2].T.copy(), pts[:, 2:].T.copy()
        F = orc.solve_hypotheses(p1, p2, idx)
        ks = [prefix_points(args.n, r) for r in args.rho + args.rho0]
        pre = np.zeros((args.hyp, len(ks)), np.int64)
        full = np.zeros(args.hyp, np.int64)
        for h in range(args.hyp):
            with np.errstate(all="ignore"):
                cs = np.cumsum(orc.distance(F[h], p1, p2) < 1.5)
            full[h] = cs[-1]
            pre[h] = cs[np.array(ks) - 1]
        for j, (rho, k) in enumerate(zip(args.rho, ks)):
            for K in args.K:
                r = bounded_rule(pre[:, j], full, args.n - k, K)
                Kp = min(K, args.hyp)
                evals = k * args.hyp + (args.n - k) * Kp + ((args.n - k) * args.hyp if r["fallback"] else 0)
                print(json.dumps({"pair": pair, "rho": rho, "K": K, "best": int(full.max()), "L": r["L"],
                                  "escapees": r["escapees"], "fallback": r["fallback"],
                                  "survivors": int((pre[:, j] + args.n - k >= full.max()).sum()),
                                  "evals_vs_full": evals / (args.n * args.hyp)}))
                for j0, (rho0, k0) in enumerate(zip(args.rho0, ks[len(args.rho):])):
                    if k0 >= k:
                        continue
                    t = two_step_rule(pre[:, len(args.rho) + j0], pre[:, j], full, args.n, k0, k, K)
                    Kp = min(K, args.hyp)
                    evals = t["evals_a"] + t["evals_b"] + (args.n * Kp) + (args.n * args.hyp if t["fallback"] else 0)
                    print(json.dumps({"pair": pair, "rho": rho, "rho0": rho0, "K": K, "L": t["L"], "S": t["S"],
                                      "stage_a_evals": t["evals_a"], "stage_b_evals": t["evals_b"],
                                      "fallback": t["fallback"], "evals_vs_full": evals / (args.n * args.hyp)}))


if __name__ == "__main__":
    main()
