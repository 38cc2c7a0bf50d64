"""Timeline of the pipelined bounded sweep: one device-resident sweep over config-5 pairs (default 512 pairs = 8 passes of
64) under torch.profiler with CUDA activities, in a run of its own.  A pipelined pass has four scorer launches on the
caller's stream (prefix stage A, the candidate stage, prefix stage B, the fallback); the period of a pass is the time
from the start of one prefix stage A to the next.  Per period the tool writes every kernel that starts in it (name,
stream, start, duration), the summed scorer time on the caller's stream, and the rest of the period: the time in which
the caller's stream runs something other than a scorer or waits (non-scorer time, with the gaps between consecutive
scorer launches listed one by one).  Stage B's duration and launch grid are listed per period too.

    python tools/bounded_pass_timeline.py --out profiles/r03_bounded_pass_timeline.json
    python tools/bounded_pass_timeline.py --root <other checkout> --out <file>      # the same run with another build

--root imports the package of another checkout (its library must be built); the tool itself is the same.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 20261018
LONG_BOUND_MS = 1.0          # a bound-only scorer launch this long is a prefix stage A at config 5 (stage B: well below)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=HERE, help="checkout whose package is imported")
    ap.add_argument("--pairs", type=int, default=512)
    ap.add_argument("--n", type=int, default=50000)
    ap.add_argument("--hyp", type=int, default=8192)
    ap.add_argument("--out", default=os.path.join(HERE, "profiles", "r03_bounded_pass_timeline.json"))
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    import torch
    from torch.profiler import ProfilerActivity, profile
    import tsbb15_b200  # noqa: F401
    from tsbb15_b200 import parallel, runtime as rt

    sh = parallel.PairShardedRansac(args.pairs, args.n, args.hyp, want_mask=True)
    sh.generate(seed_base=1000)
    for _ in range(2):                                    # workspaces, plan, modules
        sh.run(thr=1.5, sample_seed=SEED)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sh.run(thr=1.5, sample_seed=SEED)
        torch.cuda.synchronize()
    passes = rt.last_stats()["passes"]
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    kernels = sorted(({"name": e["name"], "stream": e["args"].get("stream"), "ts": float(e["ts"]), "dur": float(e["dur"]),
                       "grid": e["args"].get("grid")}
                      for e in trace["traceEvents"] if e.get("ph") == "X" and e.get("cat") == "kernel"),
                     key=lambda k: k["ts"])

    def is_scorer(k):
        return "score_packed" in k["name"]

    def is_bound(k):
        return "EpiBoundPolicy" in k["name"]

    scorer_time = {}
    for k in kernels:
        if is_scorer(k):
            scorer_time[k["stream"]] = scorer_time.get(k["stream"], 0.0) + k["dur"]
    caller = max(scorer_time, key=scorer_time.get)
    on_caller = [k for k in kernels if k["stream"] == caller]
    starts = [k["ts"] for k in on_caller if is_scorer(k) and is_bound(k) and k["dur"] >= LONG_BOUND_MS * 1e3]
    end = max(k["ts"] + k["dur"] for k in kernels)
    periods = []
    for i, t0 in enumerate(starts):
        t1 = starts[i + 1] if i + 1 < len(starts) else end
        mine = [k for k in kernels if t0 <= k["ts"] < t1]
        scorers = [k for k in mine if k["stream"] == caller and is_scorer(k)]
        busy = sum(k["dur"] for k in scorers)
        gaps = [round((b["ts"] - (a["ts"] + a["dur"])) * 1e-3, 4) for a, b in zip(scorers, scorers[1:])]
        stage_b = [k for k in scorers if is_bound(k) and k["dur"] < LONG_BOUND_MS * 1e3]
        periods.append({
            "period_ms": round((t1 - t0) * 1e-3, 4),
            "scorer_ms": round(busy * 1e-3, 4),
            "non_scorer_ms": round((t1 - t0 - busy) * 1e-3, 4),
            "caller_gaps_between_scorers_ms": gaps,
            "caller_non_scorer_kernels": [k["name"].split("(")[0] for k in mine if k["stream"] == caller and not is_scorer(k)],
            "stage_b": [{"ms": round(k["dur"] * 1e-3, 4), "grid": k["grid"]} for k in stage_b],
            "kernels": [{"name": k["name"].split("(")[0], "stream": k["stream"], "start_ms": round((k["ts"] - t0) * 1e-3, 4),
                         "ms": round(k["dur"] * 1e-3, 4)} for k in mine],
        })
    inner = periods[1:-1] if len(periods) > 2 else periods          # the first and the last hold the fill and the drain

    def mean(key):
        return round(sum(p[key] for p in inner) / max(len(inner), 1), 4)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    doc = {"workload": f"config-5 pairs 0..{args.pairs - 1}: {args.pairs} x {args.n} x {args.hyp}, device-resident, one "
                       f"PairShardedRansac.run under torch.profiler (CUDA activities)",
           "root": os.path.abspath(args.root), "gpu": smi, "passes": passes, "caller_stream": caller,
           "steady_periods": len(inner),
           "mean_steady": {"period_ms": mean("period_ms"), "scorer_ms": mean("scorer_ms"),
                           "non_scorer_ms": mean("non_scorer_ms")},
           "sweep_ms": round((end - kernels[0]["ts"]) * 1e-3, 3),
           "periods": periods}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps({k: doc[k] for k in ("root", "gpu", "passes", "steady_periods", "mean_steady", "sweep_ms")}))


if __name__ == "__main__":
    main()
