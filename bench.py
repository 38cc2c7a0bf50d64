#!/usr/bin/env python
"""Benchmark of the B200-native RANSAC hot path (contract: see the task brief / DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W            # our arm (torchrun launches N ranks for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm (numpy oracle port) on host cores
    python bench.py ... --dump-outputs DIR                   # also writes the last timed step's results as DIR/*.npy

Workload ("step") = BASELINE config 5 IN FULL: F-matrix RANSAC over 4096 synthetic image pairs x 50 000 correspondences x
8 192 hypotheses (30 % outliers, thr 1.5 px): hypotheses sampled and solved (8-point), every hypothesis scored against
every correspondence, best hypothesis + inlier mask selected — 1.68e12 hypothesis x correspondence evaluations per step.
The 4096 pairs are a FIXED total split over the N ranks in contiguous blocks (strong scaling, no data-path collective);
every step ends with the all-gather of the per-pair results (index, count, F, and on the device-resident leg the inlier
masks) so that every rank holds the whole answer.  The step is driven through the repo's own multi-GPU entry point
``parallel.PairShardedRansac``.  Inputs are generated on the device from seed 1000 + pair (counter-based Philox, replayable
on the host: the first 8 pairs are checked against the oracle in the run).  metric = evaluations per second, whole job.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLOP_PER_F_EVAL = 30.0       # SURVEY.md section 8d: 12 FMA + 6 other flops per evaluation (algorithmic)
FLOP_PER_PNP_EVAL = 29.0
THR2_PNP = (1.5 / 3217.0) ** 2
SAMPLE_SEED = 20261018       # one seed feeds the device sampler and (through philox.py) the oracle


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference algorithm on host cores
# ---------------------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    p1, p2, idx, thr, threads = args
    ctx = None
    if threads:
        try:
            from threadpoolctl import threadpool_limits
            ctx = threadpool_limits(threads)
        except Exception:
            ctx = None
    from oracle import f_path as orc
    F = orc.solve_hypotheses(p1, p2, idx)
    counts = orc.score_hypotheses(F, p1, p2, thr)
    del ctx
    return counts


def _pnp_cpu_worker(args):
    X, yh, idx, thr2 = args
    try:
        from threadpoolctl import threadpool_limits
        ctx = threadpool_limits(1)
    except Exception:
        ctx = None
    from oracle import pnp_path as opnp
    r = opnp.pnp_ransac(X, yh, idx, thr2)
    del ctx
    return r["counts"]


_POOL = None


def _cpu_pool(cores: int):
    global _POOL
    if _POOL is None and cores > 1:
        import multiprocessing as mp
        _POOL = mp.get_context("fork").Pool(cores)
        _POOL.map(abs, range(cores))                      # spin the workers up outside any timed region
    return _POOL


_PAIR0 = {}


def config5_pair_on_host(n_points: int, pair_id: int = 0):
    """Pair ``pair_id`` of the config-5 sweep replayed on the host (identical to what the device generates)."""
    key = (n_points, pair_id)
    if key not in _PAIR0:
        from tsbb15_b200 import philox, synth
        _PAIR0[key] = philox.synth_two_view(n_points, pair_id, synth.dino()["Ps"], synth.DINO_BBOX)[0]
    return _PAIR0[key]


def cpu_reference_sample(n_points: int, n_hyp: int, cores: int, hyp_first: int = 0):
    """Times fun.py:303-317 semantics (solve + score + threshold + count, oracle port) for ``n_hyp`` hypotheses of config-5
    pair 0 (``n_points`` correspondences, the samples the device draws for SAMPLE_SEED), hypotheses spread over ``cores``
    processes (cores == 0: this process alone with the default BLAS threading).  Returns evals/s, seconds, best count."""
    from tsbb15_b200 import philox
    pts = config5_pair_on_host(n_points)
    idx = philox.sample_indices(n_points, n_hyp, 8, SAMPLE_SEED, 0, hyp_first)
    p1, p2 = pts[:, :2].T.copy(), pts[:, 2:].T.copy()
    if cores == 0:
        t0 = time.perf_counter()
        out = [_cpu_worker((p1, p2, idx, 1.5, 0))]
        dt = time.perf_counter() - t0
    else:
        chunks = [c for c in np.array_split(idx, cores) if len(c)]
        pool = _cpu_pool(cores)
        t0 = time.perf_counter()
        if pool is not None:
            out = pool.map(_cpu_worker, [(p1, p2, c, 1.5, 1) for c in chunks])
        else:
            out = [_cpu_worker((p1, p2, chunks[0], 1.5, 1))]
        dt = time.perf_counter() - t0
    best = int(np.max(np.concatenate(out)))
    return n_points * n_hyp / dt, dt, best


def blas_info() -> dict:
    info = {"numpy": np.__version__}
    try:
        from threadpoolctl import threadpool_info
        info["threadpools"] = [{k: d.get(k) for k in ("user_api", "internal_api", "num_threads", "version")}
                               for d in threadpool_info()]
    except Exception as e:
        info["threadpools"] = repr(e)
    return info


WORKLOAD = ("BASELINE config 5 in full: synthetic multi-pair F-RANSAC, %d pairs x %d correspondences x %d hypotheses, 30%% "
            "outliers, thr 1.5 px, pairs generated from seed 1000+p")


def run_reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_hyp = max(cores * 8, 256)                       # bounded sample: ~6 ms of numpy per hypothesis at N = 50 000
    config5_pair_on_host(args.n)
    for _ in range(min(args.warmup, 1)):
        cpu_reference_sample(args.n, max(cores, 32), cores)
    times, evals = [], 0
    for s in range(args.steps):
        v, dt, _ = cpu_reference_sample(args.n, n_hyp, cores, hyp_first=(s * n_hyp) % max(args.hyp - n_hyp, 1))
        times.append(dt)
        evals += args.n * n_hyp
    total = sum(times)
    value = evals / total
    line = {
        "impl": "reference", "metric": "f_ransac_evals_per_sec", "value": value, "unit": "evals/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / max(args.steps, 1),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD % (args.pairs, args.n, args.hyp) + "; CPU step = a bounded sample of it: %d "
                               "hypotheses of pair 0 (constant cost per hypothesis x correspondence)" % n_hyp,
                   "pairs": args.pairs, "n_corr": args.n, "n_hyp": args.hyp, "hyp_per_cpu_step": n_hyp},
        "cpu_baseline": {"value": value, "unit": "evals/s", "cores": cores, "kind": "port",
                         "sample": "%d steps x %d hypotheses x %d correspondences of config-5 pair 0, numpy oracle port of "
                                   "fun.py:303-317 (lab3.fmatrix_stls + fmatrix_residuals), one process per core, BLAS "
                                   "threads=1" % (args.steps, n_hyp, args.n), "blas": blas_info()},
        "e2e": {"value": value, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# clocks sampler
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.samples = []
        self.proc = None
        self.thread = None
        self.dev = device_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.dev), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, windows):
        rows = []
        for ts, line in self.samples:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                rows.append((ts, float(parts[0]), float(parts[1]), float(parts[2]), parts[3:7]))
            except ValueError:
                continue
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        inside = [r for r in rows if any(a <= r[0] <= b for a, b in windows)] or rows
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in inside for k in range(4) if r[4][k].lower().startswith("active")})
        return {"sm_mhz": float(np.median([r[1] for r in inside])), "sm_max_mhz": inside[0][2],
                "power_w_max": max(r[3] for r in inside), "reasons": reasons, "samples": len(inside)}


# ---------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------
def run_ours(args) -> None:
    import torch
    import tsbb15_b200 as rg
    from tsbb15_b200 import _cabi as cabi, parallel, philox, runtime as rt, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    lib = cabi.load_library()
    ctx = cabi.context(local)
    stream = torch.cuda.current_stream().cuda_stream

    peaks = rt.microbench(device=local)               # measured FFMA / FFMA2 / DFMA pipe rates of THIS gpu
    fp32_peak_tflops = 2.0 * max(peaks["ffma_gfma_s"], peaks["ffma2_gfma_s"]) * 1e-3

    Pt, N, H = args.pairs, args.n, args.hyp
    sh = parallel.PairShardedRansac(Pt, N, H, device=local, want_mask=True)
    sh.generate(seed_base=1000)                        # device-side Philox: the local shard never exists on the host ...
    sh.alloc_host(want_mask=True)                      # ... except as the page-locked copy the end-to-end leg uploads
    sh.h_pts[: sh.P].copy_(sh.d_pts)
    torch.cuda.synchronize()

    def step_dev(s):
        sh.run(thr=1.5, sample_seed=SAMPLE_SEED, solver=args.solver)
        sh.gather(masks=True)

    def step_host(s):
        sh.run_host(thr=1.5, sample_seed=SAMPLE_SEED, solver=args.solver)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.time()
        e0.record()
        for s in range(steps):
            fn(s)
        e1.record()
        e1.synchronize()
        w1 = time.time()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms, (w0, w1)

    if args.host_slices:
        rt.set_option(2, args.host_slices, device=local)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for s in range(args.warmup):
        step_dev(s)
        step_host(s)
    torch.cuda.synchronize()
    host_stats = rt.last_stats(device=local, stream=stream)                 # last warm-up call was step_host
    step_dev(0)
    dev_stats = rt.last_stats(device=local, stream=stream)

    rt.set_option(1, 1, device=local)                                       # phase events on the launching stream
    ms_dev, win_dev = timed(step_dev, args.steps)
    prof = rt.profile(device=local, stream=stream)
    rt.set_option(1, 0, device=local)
    stats = rt.last_stats(device=local, stream=stream)
    res_dev = sh.unpack(sh.gather(masks=bool(args.dump_outputs)))           # the last device-resident step's answer
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, res_dev)
    ms_e2e, win_e2e = timed(step_host, args.steps)
    # the same step with the passes strictly one after the other on one stream (option 10 = 0): the scorer ALONE on the GPU.
    # In the timed region above the solver of the next pass and the fix-up / selection / masks of the previous one run beside
    # it on a second stream, which hides them but slows each scorer launch by ~2 %.
    rt.set_option(10, 0, device=local)
    step_dev(0)
    rt.set_option(1, 1, device=local)
    ms_serial, _ = timed(step_dev, 1)
    prof_serial = rt.profile(device=local, stream=stream)
    rt.set_option(1, 0, device=local)
    rt.set_option(10, 1, device=local)
    h2d_rate = rt.last_stats(device=local, stream=stream)["h2d_mb_per_s"] * 1e-3          # GB/s this rank's uploads achieved
    if dist is not None:
        t = torch.tensor([h2d_rate], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        h2d_rate = float(t.item())
    blk = (sh.h_all_block if world > 1 else sh.h_block).numpy()
    # the end-to-end leg must give the same answer as the device-resident one (same inputs, same seed)
    h_cnt = np.concatenate([blk[q * sh.per * 80:(q + 1) * sh.per * 80][sh.per * 76:].view(np.int32)[: b - a]
                            for q, (a, b) in enumerate([parallel.shard_range(Pt, q2, world) for q2 in range(world)])])
    assert np.array_equal(h_cnt, res_dev["best_count"]), "end-to-end and device-resident legs disagree"
    assert int(res_dev["best_count"].min()) > 0.5 * 0.7 * N, "benchmark produced implausible consensus sets"

    evals_per_step = float(Pt) * N * H
    value = evals_per_step * args.steps / (ms_dev * 1e-3)
    e2e = evals_per_step * args.steps / (ms_e2e * 1e-3)
    passes = max(prof["calls"], 1)
    score_ms = prof["score_ms"] / passes                                    # one scorer launch = one pass
    # passes differ in size (the first and the last pass of a call are cut into 1/8 .. 1/2 pieces: pipeline fill / drain), so the
    # scorer's rate is total evaluations over total scorer time of the profiled passes = whole steps of this rank
    steps_covered = passes / max(dev_stats["passes"], 1)
    whole_steps = abs(steps_covered - round(steps_covered)) < 1e-9 and steps_covered >= 1    # false only beyond 2048 passes
    pairs_per_pass = sh.P / max(dev_stats["passes"], 1)
    evals_per_pass = pairs_per_pass * N * H                                 # average over the passes of a step
    achieved_tflops = FLOP_PER_F_EVAL * evals_per_pass / (score_ms * 1e-3) * 1e-12 if score_ms > 0 else None
    alg_bytes = pairs_per_pass * (16.0 * N + 64.0 * H + 4.0 * H)      # FP32 points + 64-byte hypothesis records + counts
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        hbm_peak = 6650.0
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "score_kernel_traffic.json")))
    except Exception:
        pass

    oracle_check = None
    if rank == 0 and not args.no_oracle_check:
        oracle_check = check_first_pairs(args, rg, rt, philox, synth, sh, res_dev, torch)

    extras = {}
    cpu_baseline = None
    split = None
    if not args.no_split:                               # every rank: the hypothesis-split mode with its one exchange
        split = run_split(args, rg, parallel, torch, dist, dev, rank, world)
    if rank == 0 and world == 1 and not args.no_extras:
        extras = run_extras(args, rg, rt, cabi, lib, ctx, stream, dev, torch, fp32_peak_tflops)
    if rank == 0 and world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        n_hyp = max(cores * 48, 1024)
        v, dt, _ = cpu_reference_sample(N, n_hyp, cores)
        v1, dt1, _ = cpu_reference_sample(N, 192, 0)
        cpu_baseline = {"value": v, "unit": "evals/s", "cores": cores, "kind": "port",
                        "sample": "config-5 pair 0 x %d hypotheses x %d correspondences (%.1f s wall), numpy oracle port of "
                                  "fun.py:303-317, one process per core, BLAS threads=1" % (n_hyp, N, dt),
                        "single_process_default_blas": {"value": v1, "unit": "evals/s", "sample": "192 hypotheses x %d "
                                                        "correspondences (%.1f s), one process, default BLAS threading"
                                                        % (N, dt1), "blas": blas_info()}}
    if rank == 0:
        sampler.stop()
        clocks = sampler.summary([win_dev, win_e2e])
        line = {
            "metric": "f_ransac_evals_per_sec", "value": value, "unit": "evals/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32 scoring with f64 guard-band recheck; f64 solve",
            "data": "synthetic",
            "config": {"workload": WORKLOAD % (Pt, N, H), "pairs": Pt, "n_corr": N, "n_hyp": H,
                       "parallelism": "pair-sharded x%d (%d pairs per rank, %d passes of %d pairs per step and rank), results "
                                      "all-gathered every step" % (world, sh.P, dev_stats["passes"], int(round(pairs_per_pass))),
                       "l2": "inputs of one step are %.2f GB per rank, far larger than the 126 MB L2" % (sh.P * N * 32 / 1e9),
                       "sampling": "index sets drawn on the device from one seed (Philox4x32-10), replayable on the host",
                       "solver": "qr" if args.solver == 0 else "jacobi",
                       "warmup_note": "bench.py raises --warmup to at least 3" if args.warmup_raised else None},
            "e2e": {"value": e2e, "unit": "evals/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": int(sh.P) * N * 32 * world + (world > 1) * sh.per * 80 * world,
                    "d2h_bytes_per_step": (int(sh.P) * (80 + N)) * world + (world > 1) * world * world * sh.per * 80,
                    "h2d_gbs_per_rank_measured_min": h2d_rate,
                    "h2d_gbs_needed_per_rank_to_hide_uploads": int(sh.P) * N * 32 / (ms_dev / args.steps * 1e-3) * 1e-9,
                    "note": "rg_f_ransac_host2 on every rank's page-locked shard (uploads pass by pass on a second stream, "
                            "masks and per-pair results downloaded), then the all-gather of the per-pair results; bytes are "
                            "whole-job sums over the ranks"},
            "gpu_launches": int(dev_stats["launches"]) * args.steps,
            "gpu_launches_e2e_region": int(host_stats["launches"]) * args.steps,
            "roofline": {"bound": "fp32_ffma", "kernel": "score_packed<EpiPolicy>", "achieved": achieved_tflops,
                         "peak": fp32_peak_tflops, "unit": "TFLOP/s",
                         "frac": (achieved_tflops / fp32_peak_tflops) if achieved_tflops else None,
                         "traffic": (traffic or {}).get("dram_bytes_per_launch"),
                         "traffic_note": (traffic or {}).get("note"),
                         "kernel_ms_per_launch": score_ms, "launches_timed": passes,
                         "launches_cover_whole_steps": bool(whole_steps),
                         "timed_with": "pass pipelining (option 10): head of pass k+1 and tail of pass k-1 run beside the scorer "
                                       "of pass k on a second stream",
                         "kernel_alone": {
                             "kernel_ms_per_launch": prof_serial["score_ms"] / max(prof_serial["calls"], 1),
                             "frac": (FLOP_PER_F_EVAL * float(sh.P) * N * H / (prof_serial["score_ms"] * 1e-3)
                                      * 1e-12 / fp32_peak_tflops) if prof_serial["score_ms"] > 0 else None,
                             "ms_per_step_serial_passes": ms_serial,
                             "note": "one more step with option 10 = 0 (passes strictly in order on one stream), outside the "
                                     "timed region: the scorer with the GPU to itself"},
                         "units_per_launch": evals_per_pass,
                         "peak_source": "FFMA/FFMA2 chain micro-benchmark run on this GPU at start of bench.py "
                                        "(MEASURED_PEAKS.json has no FP32 figure)",
                         "algorithmic_flop_per_eval": FLOP_PER_F_EVAL,
                         "executed_fp32_lane_ops_per_eval": 16,
                         "hbm": {"algorithmic_bytes_per_launch": alg_bytes,
                                 "achieved_gbs": alg_bytes / (score_ms * 1e-3) * 1e-9 if score_ms > 0 else None,
                                 "peak_gbs": hbm_peak}},
            "phases_ms_per_pass": {k: prof[k] / passes for k in
                                   ("prepare_ms", "solve_ms", "score_ms", "fixup_ms", "select_ms")},
            "guard_band": {"band_eval_fraction": stats["band_evals"] / (sh.P * float(N) * H),
                           "flagged_groups_per_step": stats["recheck_groups"], "flips_per_step": stats["flips"],
                           "hypotheses_recounted_after_list_overflow": stats["overflow"]},
            "oracle_check": oracle_check,
            "pipes": peaks, "clocks": clocks, "cpu_baseline": cpu_baseline,
        }
        line.update(extras)
        if split is not None:
            line.update(split)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(out_dir: str, res: dict) -> None:
    """Writes what the last timed step returned to its caller as DIR/<name>.npy (float64, the inlier masks float32), so that
    two builds can be compared output for output on the same seeded inputs.  Under 60 MB in all: the per-pair results of
    every pair (a sample of 100 000 pairs beyond that) and the masks of 128 pairs (at most 4M entries).  The samples are
    drawn from a fixed seed, so the same arguments select the same pairs and points."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)
    P, N = len(res["best_idx"]), len(res["mask"][0])
    pairs = np.arange(P) if P <= 100_000 else np.sort(rng.choice(P, 100_000, replace=False))
    rows = np.sort(rng.choice(P, min(P, 128), replace=False))
    cols = np.arange(N) if len(rows) * N <= 1 << 22 else np.sort(rng.choice(N, (1 << 22) // len(rows), replace=False))
    out = {"pair_ids": pairs, "best_idx": res["best_idx"][pairs], "best_count": res["best_count"][pairs],
           "F": res["F"][pairs], "mask_pair_ids": rows, "mask_point_ids": cols}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))
    np.save(os.path.join(out_dir, "mask.npy"), np.stack([res["mask"][r][cols] for r in rows]).astype(np.float32))


def check_first_pairs(args, rg, rt, philox, synth, sh, res_dev, torch) -> dict:
    """SURVEY 8d config 5: 'check the first 8 pairs against the oracle'.  (1) the device-generated inputs of pairs 0..7 equal
    their host replay bit for bit; (2) a separate library call on the replayed inputs reproduces the sweep's winners;
    (3) the oracle (numpy port of fun.py:303-317) gives the same inlier counts for the first 40 hypotheses of every pair and
    for the winner, on the samples replayed from the seed."""
    from oracle import f_path as orc
    n_chk = min(8, sh.P)
    N, H = args.n, args.hyp
    pairs = [philox.synth_two_view(N, p, synth.dino()["Ps"], synth.DINO_BBOX)[0] for p in range(n_chk)]
    same_inputs = all(np.array_equal(sh.d_pts[p].cpu().numpy(), pairs[p]) for p in range(n_chk))
    r = rt.f_ransac_batched(pairs, None, n_hyp=H, sample_seed=SAMPLE_SEED, first_pair=0, want_counts=True, want_flags=True,
                            solver=args.solver)
    same_winner = bool(np.array_equal(r["best_idx"], res_dev["best_idx"][:n_chk]) and
                       np.array_equal(r["best_count"], res_dev["best_count"][:n_chk]) and
                       np.array_equal(r["F"], res_dev["F"][:n_chk]))
    cores = os.cpu_count() or 1
    pool = _cpu_pool(cores)
    jobs, meta = [], []
    for p in range(n_chk):
        idx = philox.sample_indices(N, H, 8, SAMPLE_SEED, p)
        sel = np.unique(np.concatenate([np.arange(40), [max(int(r["best_idx"][p]), 0)]]))
        p1, p2 = pairs[p][:, :2].T.copy(), pairs[p][:, 2:].T.copy()
        for chunk in np.array_split(sel, 4):
            jobs.append((p1, p2, idx[chunk], 1.5, 1))
            meta.append((p, chunk))
    outs = pool.map(_cpu_worker, jobs) if pool is not None else [_cpu_worker(j) for j in jobs]
    mism = checked = skipped = 0
    for (p, chunk), c in zip(meta, outs):
        ok = r["flags"][p][chunk] == 0                      # rank-deficient samples: the null vector itself is arbitrary
        mism += int((c[ok] != r["counts"][p][chunk][ok]).sum())
        checked += int(ok.sum())
        skipped += int((~ok).sum())
    assert same_inputs and same_winner and mism == 0, "config-5 oracle check failed"
    return {"pairs": n_chk, "device_inputs_equal_host_replay": bool(same_inputs), "sweep_winners_reproduced": same_winner,
            "hypotheses_checked_vs_oracle": checked, "count_mismatches": mism, "rank_deficient_skipped": skipped}


def run_split(args, rg, parallel, torch, dist, dev, rank, world) -> dict:
    """The one collective of the design (SURVEY 8e item 2), timed in the default path at every N: BASELINE config 3 (ONE pair,
    100 000 correspondences x 16 384 hypotheses) and config 4 (ONE view, PnP 1M x 8192) with the hypotheses split over the
    ranks.  Every rank holds all correspondences (prepared once), scores its block, and ONE peer-memory exchange kernel
    (NCCL all-reduce + F broadcast as the fallback / comparison) picks the winner and ships its model; every rank then computes
    the winner's inlier mask.  Device resident, CUDA events on the launching stream, max over ranks."""
    from tsbb15_b200 import device as dv, philox, sampling, synth
    out = {}

    def ev(fn, reps):
        for _ in range(3):
            fn()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); e1.synchronize()
        ms = e0.elapsed_time(e1) / reps
        if dist is not None:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---- config 3 -------------------------------------------------------------------------------------------------
    N3, H3 = 100000, 16384
    try:
        d3, _ = dv.synth_two_view(1, N3, first_pair=0, seed_base=3000, device=dev.index)
        d3 = d3[0]
        modes = ["p2p", "nccl"] if world > 1 else ["none"]
        res = {}
        for mode in modes:
            try:
                sp = parallel.SplitHypothesesF(d3, H3, exchange=mode, sample_seed=SAMPLE_SEED)
            except Exception as e:                      # P2PExchange raises on EVERY rank when any rank cannot map its peers
                res[mode] = {"error": repr(e)[:200]}
                continue
            ms = ev(lambda: sp.run(thr=1.5, want_mask=True), 20)
            r = sp.result()
            res[mode] = {"ms": ms, "evals_per_s": float(N3) * H3 / (ms * 1e-3), "winner": r["best_idx"],
                         "count": r["best_count"], "owner_rank": r["owner"], "mask_inliers": int(r["mask"].sum())}
            if mode in ("p2p", "none"):                 # the same chain replayed as ONE CUDA graph launch
                try:
                    sp.capture(thr=1.5, want_mask=True)
                    msg = ev(sp.replay, 20)
                    rg_ = sp.result()
                    res[mode + "_cuda_graph"] = {"ms": msg, "evals_per_s": float(N3) * H3 / (msg * 1e-3),
                                                 "winner": rg_["best_idx"], "count": rg_["best_count"],
                                                 "owner_rank": rg_["owner"], "mask_inliers": int(rg_["mask"].sum())}
                except Exception as e:
                    res[mode + "_cuda_graph"] = {"error": repr(e)[:200]}
            if sp.p2p is not None:
                sp.p2p.close()
        best = min((v for v in res.values() if "ms" in v), key=lambda v: v["ms"], default=None)
        entry = {"workload": "config 3: one pair, 100000 correspondences x 16384 hypotheses split over %d rank(s), samples "
                             "drawn on the device, points prepared once, inlier mask of the winner on every rank" % world,
                 "exchange": res, "ms": best["ms"] if best else None, "winner": best["winner"] if best else None,
                 "count": best["count"] if best else None}
        if rank == 0 and best is not None and world > 1:      # the same problem on one GPU: identical winner
            one = parallel.SplitHypothesesF.__new__(parallel.SplitHypothesesF)
            o1 = dv.FOutputs(1, N3, device=dev.index, want_mask=False, want_key=False)
            dv.f_ransac(d3, np.array([0, N3], np.int32), None, np.array([0, H3], np.int32), o1, seed=SAMPLE_SEED)
            entry["same_winner_as_one_gpu"] = bool(int(o1.best_idx.item()) == best["winner"] and
                                                   int(o1.best_count.item()) == best["count"])
            del one
        out["config3_split_hypotheses"] = entry
    except Exception as e:
        out["config3_split_hypotheses"] = {"error": repr(e)[:300]}

    # ---- config 4 (PnP) ---------------------------------------------------------------------------------------------
    N4, H4 = 1000000, 8192
    try:
        X, y, _ = synth.pnp_scene(N4, seed=4)
        pidx = sampling.fast(N4, H4, 6, seed=2)
        dX, dy = torch.from_numpy(X).to(dev), torch.from_numpy(y).to(dev)
        modes = ["p2p", "nccl"] if world > 1 else ["none"]
        res = {}
        for mode in modes:
            try:
                sp = parallel.SplitHypothesesPnp(dX, dy, pidx, n=6, exchange=mode)
            except Exception as e:
                res[mode] = {"error": repr(e)[:200]}
                continue
            ms = ev(lambda: sp.run(THR2_PNP), 10)
            r = sp.result()
            res[mode] = {"ms": ms, "poses_per_s": H4 / (ms * 1e-3), "winner": r["best_idx"], "count": r["best_count"]}
            if sp.p2p is not None:
                sp.p2p.close()
        best = min((v for v in res.values() if "ms" in v), key=lambda v: v["ms"], default=None)
        out["config4_split_hypotheses"] = {"workload": "config 4: one view, PnP 1000000 correspondences x 8192 six-point "
                                                       "hypotheses split over %d rank(s)" % world, "exchange": res,
                                           "ms": best["ms"] if best else None, "winner": best["winner"] if best else None,
                                           "count": best["count"] if best else None}
    except Exception as e:
        out["config4_split_hypotheses"] = {"error": repr(e)[:300]}
    return out


def run_extras(args, rg, rt, cabi, lib, ctx, stream, dev, torch, fp32_peak) -> dict:
    """Short, separately timed runs of the other BASELINE configs (reported, not the headline)."""
    from tsbb15_b200 import device as dv, philox, sampling, synth
    out = {}

    def time_dev(fn, reps):
        fn(); torch.cuda.synchronize()
        rt.set_option(1, 1)                      # phase events from here on (the warm-up call is not profiled)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); e1.synchronize()
        return e0.elapsed_time(e1) / reps

    # ---- config 3: single pair 100k x 16k, threshold sweep, both criteria -------------------------------------
    N3, H3 = 100000, 16384
    d3, _ = dv.synth_two_view(1, N3, first_pair=0, seed_base=3000, device=dev.index)
    po3, ho3 = dv.offsets([N3]), dv.offsets([H3])
    o3 = dv.FOutputs(1, N3, device=dev.index, want_mask=True)
    sweep = {}
    for mode, name in ((rg.MODE_EPI_MAX, "epi_max"), (rg.MODE_SAMPSON, "sampson")):
        for thr in ((0.25, 0.5, 1.0, 1.5, 2.0, 3.0, 4.0) if mode == rg.MODE_EPI_MAX else (1.5,)):
            ms = time_dev(lambda: dv.f_ransac(d3, po3, None, ho3, o3, thr=thr, mode=mode, seed=SAMPLE_SEED, solver=args.solver), 5)
            pr = rt.profile(stream=stream); rt.set_option(1, 0)
            st = rt.last_stats(stream=stream)
            sc = pr["score_ms"] / max(pr["calls"], 1)
            sweep["%s_thr%g" % (name, thr)] = {
                "ms": ms, "evals_per_s": N3 * H3 / (ms * 1e-3), "score_kernel_ms": sc,
                "score_kernel_frac_of_fp32_peak": FLOP_PER_F_EVAL * N3 * H3 / (sc * 1e-3) * 1e-12 / fp32_peak,
                "fixup_ms": pr["fixup_ms"] / max(pr["calls"], 1),
                "best_count": int(o3.best_count.item()), "band_eval_fraction": st["band_evals"] / (N3 * H3)}
    out["config3_single_pair_100k_x_16k"] = sweep

    # ---- config 4: PnP 1M x 8192 — the second half of the metric (poses/s) --------------------------------------------
    out["pnp"] = run_pnp_block(args, rg, rt, dv, sampling, synth, stream, dev, torch, fp32_peak)

    # ---- config 2: Dino sequence through the host API (real data shapes, launch/latency bound) ---------------------
    try:
        pairs = [np.ascontiguousarray(np.hstack(synth.dino_noisy_pair(i, i + 1))) for i in range(35)]
        ev = sum(p.shape[0] for p in pairs) * 10000.0

        def host_time(fn, reps=10):
            fn()
            t0 = time.perf_counter()
            for _ in range(reps):
                r = fn()
            return (time.perf_counter() - t0) / reps, r
        # (a) samples drawn on the device from one seed: nothing but the points (0.3 MB) crosses PCIe
        dt_seed, r = host_time(lambda: rt.f_ransac_batched(pairs, None, n_hyp=10000, sample_seed=SAMPLE_SEED, thr=1.5))
        rt.set_option(1, 1)
        rt.f_ransac_batched(pairs, None, n_hyp=10000, sample_seed=SAMPLE_SEED, thr=1.5)
        pr = rt.profile(); rt.set_option(1, 0)
        # (b) host-drawn samples (11 MB of indices uploaded), one pageable buffer
        idl = sampling.fast_batch([p.shape[0] for p in pairs], 10000, 8, seed=0)
        dt_host, _ = host_time(lambda: rt.f_ransac_batched(pairs, idl, thr=1.5))
        # (c) what a user of batched.f_ransac_pairs pays, index drawing included
        from tsbb15_b200 import batched
        dt_api, _ = host_time(lambda: batched.f_ransac_pairs(pairs, n_hyp=10000, thr=1.5, seed=0), 3)
        # CPU: the oracle port on pair 0 of the sequence, bounded sample
        cores = os.cpu_count() or 1
        p0 = pairs[0]
        nh = max(cores * 64, 1024)
        idx0 = philox.sample_indices(p0.shape[0], nh, 8, SAMPLE_SEED, 0)
        pool = _cpu_pool(cores)
        p1, p2 = p0[:, :2].T.copy(), p0[:, 2:].T.copy()
        t0 = time.perf_counter()
        if pool is not None:
            pool.map(_cpu_worker, [(p1, p2, c, 1.5, 1) for c in np.array_split(idx0, cores)])
        else:
            _cpu_worker((p1, p2, idx0, 1.5, 1))
        dtc = time.perf_counter() - t0
        views = [synth.dino_view_2d3d(i) for i in range(36)]
        vidx = [sampling.fast(v[0].shape[0], 1024, 6, seed=i) for i, v in enumerate(views)]
        Xl, yl = [v[0] for v in views], [v[1] for v in views]
        dtp, rp = host_time(lambda: rt.pnp_ransac_batched(Xl, yl, vidx, THR2_PNP), 5)
        sc = pr["score_ms"] / max(pr["calls"], 1)
        out["config2_dino_sequence"] = {
            "f_35_pairs_x_10000_hyp_host_call_ms": dt_seed * 1e3, "f_evals_per_s_e2e": ev / dt_seed,
            "f_host_call_ms_host_drawn_samples": dt_host * 1e3,
            "f_pairs_api_ms_including_host_sampling": dt_api * 1e3,
            "f_inlier_counts": [int(c) for c in r["best_count"][:5]],
            "phases_ms": {k: pr[k] / max(pr["calls"], 1) for k in ("prepare_ms", "solve_ms", "score_ms", "fixup_ms", "select_ms")},
            "roofline": {"bound": "launch latency / solver (350 000 8-point solves against 1.1e8 evaluations)",
                         "kernel": "score_packed<EpiPolicy>", "kernel_ms": sc,
                         "achieved": FLOP_PER_F_EVAL * ev / (sc * 1e-3) * 1e-12 if sc > 0 else None, "peak": fp32_peak,
                         "unit": "TFLOP/s", "frac": FLOP_PER_F_EVAL * ev / (sc * 1e-3) * 1e-12 / fp32_peak if sc > 0 else None},
            "cpu_baseline": {"value": p0.shape[0] * nh / dtc, "unit": "evals/s", "cores": cores, "kind": "port",
                             "sample": "noisy Dino pair (0,1), %d correspondences x %d hypotheses, numpy oracle port of "
                                       "fun.py:303-317, one process per core" % (p0.shape[0], nh)},
            "pnp_36_views_x_1024_hyp_one_host_call_ms": dtp * 1e3, "pnp_poses_per_s_e2e": 36 * 1024 / dtp,
            "pnp_consensus": [int(c) for c in rp["best_count"][:5]], "pnp_view_sizes": [int(v[0].shape[0]) for v in views[:5]]}
    except Exception as e:                                            # fixture missing: report, do not fail the bench
        out["config2_dino_sequence"] = {"error": repr(e)}

    # ---- rows next to the hot path (SURVEY.md section 8f N1-N3): triangulation, relative pose, 2D<->3D matching -----
    try:
        out["next_rows"] = run_next_rows(args, rg, rt, cabi, lib, ctx, stream, dev, torch)
    except Exception as e:
        out["next_rows"] = {"error": repr(e)}
    return out


def run_pnp_block(args, rg, rt, dv, sampling, synth, stream, dev, torch, fp32_peak) -> dict:
    """BASELINE config 4 (1M 2D-3D correspondences x 8192 six-point DLT hypotheses): poses/s device resident and end to end,
    roofline of the scorer (FP32) and of the solver (FP64 pipe), the oracle port on the host cores, and OpenCV's
    cv.solvePnPRansac as tables.py:141 calls it (third party, a different algorithm: reported, not matched)."""
    N4, H4 = 1000000, 8192
    X, y, _ = synth.pnp_scene(N4, seed=4)
    pidx = sampling.fast(N4, H4, 6, seed=2)
    dX, dy, dI = torch.from_numpy(X).to(dev), torch.from_numpy(y).to(dev), torch.from_numpy(pidx).to(dev)
    o = dv.PnpOutputs(1, N4, device=dev.index, want_mask=True)
    vo, ho = np.array([0, N4], np.int32), np.array([0, H4], np.int32)
    res = {"workload": "config 4: PnP-RANSAC, 1000000 correspondences x 8192 six-point DLT hypotheses, 30% outliers, "
                       "thr^2 = (1.5/3217)^2", "parity": "restated (ransac.ransac_robust / pnp.pnp_minimize raise in the "
                                                   "reference: pinned by exact Dino data, see DESIGN.md section 2)"}
    for solver, name in ((0, "givens_qr_row_jacobi"), (1, "group_jacobi_16_lanes")):
        rt.set_option(7, solver)
        dv.pnp_ransac(dX, dy, vo, dI, ho, o, THR2_PNP); torch.cuda.synchronize()
        rt.set_option(1, 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            dv.pnp_ransac(dX, dy, vo, dI, ho, o, THR2_PNP)
        e1.record(); e1.synchronize()
        ms = e0.elapsed_time(e1) / 5
        pr = rt.profile(stream=stream); rt.set_option(1, 0)
        c = max(pr["calls"], 1)
        res[name] = {"ms": ms, "poses_per_s": H4 / (ms * 1e-3), "evals_per_s": float(N4) * H4 / (ms * 1e-3),
                     "solve_ms": pr["solve_ms"] / c, "score_kernel_ms": pr["score_ms"] / c, "fixup_ms": pr["fixup_ms"] / c,
                     "best_count": int(o.best_count.item())}
    rt.set_option(7, 0)
    d = res["givens_qr_row_jacobi"]
    st = rt.last_stats(stream=stream)
    res["poses_per_s"] = d["poses_per_s"]
    res["ms"] = d["ms"]
    sc = d["score_kernel_ms"]
    peaks = rt.microbench()
    # solver: ~4.5e4 FP64 FMA-class operations per hypothesis (Givens insertion 18 x 78 x 4, ~7 sweeps x 66 rotations x 84)
    dfma_per_hyp = 18 * 78 * 4 + 7 * 66 * 84
    res["roofline"] = {
        "scorer": {"bound": "fp32_ffma", "kernel": "score_packed<PnpPolicy>", "kernel_ms_per_launch": sc,
                   "achieved": FLOP_PER_PNP_EVAL * N4 * H4 / (sc * 1e-3) * 1e-12, "peak": fp32_peak, "unit": "TFLOP/s",
                   "frac": FLOP_PER_PNP_EVAL * N4 * H4 / (sc * 1e-3) * 1e-12 / fp32_peak,
                   "algorithmic_flop_per_eval": FLOP_PER_PNP_EVAL, "band_eval_fraction": st["band_evals"] / (float(N4) * H4)},
        "solver": {"bound": "fp64 latency (one warp per SM sub-partition: 8192 hypotheses are 256 warps)",
                   "kernel": "pnp_solve_rows<6>", "kernel_ms_per_launch": d["solve_ms"],
                   "achieved": dfma_per_hyp * H4 / (d["solve_ms"] * 1e-3) * 1e-9, "peak": peaks["dfma_gfma_s"],
                   "unit": "GFMA/s (FP64)", "frac": dfma_per_hyp * H4 / (d["solve_ms"] * 1e-3) * 1e-9 / peaks["dfma_gfma_s"],
                   "fp64_fma_per_hypothesis_estimate": dfma_per_hyp,
                   "group_jacobi_ms": res["group_jacobi_16_lanes"]["solve_ms"]}}
    # end to end through rg_pnp_ransac_host (pageable numpy inputs: 40 MB up, 1 MB of mask down)
    rt.pnp_ransac(X, y, pidx, THR2_PNP)
    t0 = time.perf_counter()
    for _ in range(3):
        rh = rt.pnp_ransac(X, y, pidx, THR2_PNP)
    dth = (time.perf_counter() - t0) / 3
    res["e2e"] = {"value": H4 / dth, "unit": "poses/s", "ms": dth * 1e3, "h2d_bytes": int(X.nbytes + y.nbytes + pidx.nbytes),
                  "d2h_bytes": N4 + 112, "best_count": rh["best_count"]}
    # CPU: oracle port (pnp.py:132-152 solve + ransac.py:96-105 scoring) on all cores, bounded sample of the hypotheses
    cores = os.cpu_count() or 1
    nh = max(2 * cores, 32)
    yh = np.hstack([y, np.ones((N4, 1))])
    pool = _cpu_pool(cores)
    chunks = [c for c in np.array_split(pidx[:nh], cores) if len(c)]
    t0 = time.perf_counter()
    cnts = pool.map(_pnp_cpu_worker, [(X, yh, c, THR2_PNP) for c in chunks]) if pool is not None else \
        [_pnp_cpu_worker((X, yh, chunks[0], THR2_PNP))]
    dtc = time.perf_counter() - t0
    cnts = np.concatenate(cnts)
    g = rt.pnp_ransac(X, y, pidx[:nh], THR2_PNP, want_counts=True, want_flags=True)
    ok = g["flags"] == 0
    res["cpu_baseline"] = {"value": nh / dtc, "unit": "poses/s", "cores": cores, "kind": "port",
                           "sample": "%d hypotheses x 1000000 correspondences (%.1f s), numpy oracle port of pnp.py:132-152 + "
                                     "ransac.py:96-105, one process per core" % (nh, dtc),
                           "counts_equal_gpu": bool(np.array_equal(cnts[ok], g["counts"][ok]))}
    # OpenCV, as tables.py:141 calls it: cv.solvePnPRansac(X, y, K=I, None) with OpenCV's defaults (100 iterations,
    # reprojection error 8.0 in ITS units) — and with our threshold / iteration budget for a like-for-like wall time
    try:
        import cv2 as cv
        Xc, yc = np.ascontiguousarray(X), np.ascontiguousarray(y)
        t0 = time.perf_counter()
        okc, rvec, tvec, inl = cv.solvePnPRansac(Xc, yc, np.eye(3), None)
        dt_def = time.perf_counter() - t0
        t0 = time.perf_counter()
        ok2, rvec2, tvec2, inl2 = cv.solvePnPRansac(Xc, yc, np.eye(3), None, iterationsCount=256,
                                                    reprojectionError=float(np.sqrt(THR2_PNP)), confidence=0.999999999)
        dt_256 = time.perf_counter() - t0
        res["opencv_solvePnPRansac"] = {
            "version": cv.__version__, "note": "third party, minimal-sample P3P/EPnP + early termination: not the reference's "
                                               "DLT spec; reported as the call main.py actually makes (tables.py:141)",
            "defaults_as_in_tables_py": {"seconds": dt_def, "ok": bool(okc), "inliers": int(len(inl)) if inl is not None else 0},
            "thr_1p5px_256_iterations_max": {"seconds": dt_256, "ok": bool(ok2), "inliers": int(len(inl2)) if inl2 is not None else 0,
                                             "poses_per_s_upper_bound": 256 / dt_256}}
    except Exception as e:
        res["opencv_solvePnPRansac"] = {"unavailable": repr(e)[:200]}
    return res


def _tri_cpu_worker(a):
    from oracle import geom_path as og
    C1, C2, x1, x2 = a
    return og.triangulate_optimal_batch(C1, C2, x1, x2)


def run_next_rows(args, rg, rt, cabi, lib, ctx, stream, dev, torch) -> dict:
    """Device-resident and end-to-end rates of the kernels either side of the RANSAC path, with the numpy oracle port of
    the reference loop timed beside them (bounded sample)."""
    vp = C.c_void_p
    pi32 = C.POINTER(C.c_int32)
    from tsbb15_b200 import synth as _syn
    g = np.load(_syn.DINO_FIXTURE)
    Ps = g["Ps"]
    rng = np.random.default_rng(0)
    out = {}

    def ev_time(fn, reps):
        fn(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); e1.synchronize()
        return e0.elapsed_time(e1) / reps

    # triangulation: 1M correspondences of one camera pair, 0.5 px noise (config-4 sized point set)
    N = 1_000_000
    Xw = np.column_stack([rng.uniform(-0.045, 0.045, N), rng.uniform(-0.08, 0.03, N), rng.uniform(-0.72, -0.54, N),
                          np.ones(N)])
    proj = lambda Pm: (Xw @ Pm.T)[:, :2] / (Xw @ Pm.T)[:, 2:]
    x1 = proj(Ps[0]) + rng.normal(0, 0.5, (N, 2))
    x2 = proj(Ps[1]) + rng.normal(0, 0.5, (N, 2))
    d1, d2 = torch.from_numpy(x1).to(dev), torch.from_numpy(x2).to(dev)
    dC1, dC2 = torch.from_numpy(Ps[0:1].copy()).to(dev), torch.from_numpy(Ps[1:2].copy()).to(dev)
    dX = torch.empty((N, 3), dtype=torch.float64, device=dev)
    off = np.array([0, N], dtype=np.int32)
    tri = {}
    for method, name in ((0, "optimal"), (1, "linear")):
        def call():
            cabi.check(lib.rg_triangulate_dev(vp(ctx), vp(stream), 1, vp(dC1.data_ptr()), vp(dC2.data_ptr()),
                                              off.ctypes.data_as(pi32), vp(d1.data_ptr()), vp(d2.data_ptr()), method,
                                              vp(dX.data_ptr())))
        ms = ev_time(call, 5)
        t0 = time.perf_counter()
        rt.triangulate(Ps[0], Ps[1], [x1], [x2], method=method)
        dt = time.perf_counter() - t0
        tri[name] = {"ms": ms, "points_per_s": N / (ms * 1e-3), "e2e_points_per_s_host_call": N / dt,
                     "algorithmic_bytes_per_point": 56, "hbm_gbs": 56.0 * N / (ms * 1e-3) * 1e-9}
    cores = os.cpu_count() or 1
    per = 48
    pool = _cpu_pool(cores)
    jobs = [(Ps[0], Ps[1], x1[k * per:(k + 1) * per], x2[k * per:(k + 1) * per]) for k in range(cores)]
    t0 = time.perf_counter()
    ref = pool.map(_tri_cpu_worker, jobs) if pool is not None else [_tri_cpu_worker(jobs[0])]
    dt = time.perf_counter() - t0
    tri["cpu_baseline"] = {"value": per * len(jobs) / dt, "unit": "points/s", "cores": cores, "kind": "port",
                           "sample": "%d points, numpy oracle port of lab3.triangulate_optimal, one process per core"
                                     % (per * len(jobs))}
    got = rt.triangulate(Ps[0], Ps[1], [x1[:per]], [x2[:per]])[0]
    tri["max_rel_err_vs_oracle_sample"] = float(np.abs(got - ref[0]).max() / np.abs(ref[0]).max())
    out["triangulate_1M_points"] = tri

    # relative pose for 4096 pairs (config-5 pair count): E of random camera pairs + one correspondence each
    from oracle import geom_path as og
    Pn = 4096
    Ks = og.camera_resectioning(Ps[0])[0]
    ii = rng.integers(0, 35, Pn)
    Es, y1s, y2s = np.empty((Pn, 3, 3)), np.empty((Pn, 2)), np.empty((Pn, 2))
    Kinv = np.linalg.inv(Ks)
    Fs = [og.fmatrix_from_cameras(Ps[i], Ps[i + 1]) for i in range(35)]
    for k, i in enumerate(ii):
        Es[k] = Ks.T @ Fs[i] @ Ks
        Xp = np.array([rng.uniform(-0.04, 0.04), rng.uniform(-0.07, 0.02), rng.uniform(-0.7, -0.56), 1.0])
        a, b = Ps[i] @ Xp, Ps[i + 1] @ Xp
        y1s[k] = (Kinv @ (a / a[2]))[:2]
        y2s[k] = (Kinv @ (b / b[2]))[:2]
    dE, dy1, dy2 = (torch.from_numpy(a).to(dev) for a in (Es, y1s, y2s))
    dRt = torch.empty((Pn, 12), dtype=torch.float64, device=dev)
    dw = torch.empty(2 * Pn, dtype=torch.int32, device=dev)

    def rcall():
        cabi.check(lib.rg_relative_pose_dev(vp(ctx), vp(stream), Pn, vp(dE.data_ptr()), None, 0, vp(dy1.data_ptr()),
                                            vp(dy2.data_ptr()), vp(dRt.data_ptr()), vp(dw.data_ptr()),
                                            vp(dw[Pn:].data_ptr())))
    ms = ev_time(rcall, 5)
    t0 = time.perf_counter()
    for k in range(32):
        og.relative_camera_pose(Es[k], y1s[k], y2s[k])
    dt = time.perf_counter() - t0
    out["relative_pose_4096_pairs"] = {"ms": ms, "pairs_per_s": Pn / (ms * 1e-3), "resolved": int((dw[:Pn] >= 0).sum().item()),
                                       "cpu_baseline": {"value": 32 / dt, "unit": "pairs/s", "cores": 1, "kind": "port",
                                                        "sample": "32 pairs, numpy oracle port of fun.relative_camera_pose"}}

    # main.py:54-76 for 512 pairs x 2000 correspondences in one call (E = K^T F K, relative pose, triangulation)
    Pt, Nt = 512, 2000
    it = rng.integers(0, 35, Pt)
    tv_pts = np.empty((Pt * Nt, 4))
    tv_F = np.empty((Pt, 3, 3))
    for k, i in enumerate(it):
        Xs = np.column_stack([rng.uniform(-0.04, 0.04, Nt), rng.uniform(-0.07, 0.02, Nt), rng.uniform(-0.7, -0.56, Nt),
                              np.ones(Nt)])
        a, b = Xs @ Ps[i].T, Xs @ Ps[i + 1].T
        tv_pts[k * Nt:(k + 1) * Nt, :2] = a[:, :2] / a[:, 2:]
        tv_pts[k * Nt:(k + 1) * Nt, 2:] = b[:, :2] / b[:, 2:]
        tv_F[k] = Fs[i]
    tv_pts += rng.normal(0, 0.3, tv_pts.shape)
    d_tp, d_tF = torch.from_numpy(tv_pts).to(dev), torch.from_numpy(tv_F).to(dev)
    d_tRt = torch.empty((Pt, 12), dtype=torch.float64, device=dev)
    d_tw = torch.empty(Pt, dtype=torch.int32, device=dev)
    d_tX = torch.empty((Pt * Nt, 3), dtype=torch.float64, device=dev)
    toff = (np.arange(Pt + 1, dtype=np.int32) * Nt)
    Kc = np.ascontiguousarray(Ks)

    def tcall():
        cabi.check(lib.rg_two_view_init_dev(vp(ctx), vp(stream), Pt, vp(d_tp.data_ptr()), toff.ctypes.data_as(pi32),
                                            vp(d_tF.data_ptr()), vp(Kc.ctypes.data), None, vp(d_tRt.data_ptr()),
                                            vp(d_tw.data_ptr()), vp(d_tX.data_ptr())))
    ms = ev_time(tcall, 5)
    out["two_view_init_512_pairs_x_2000"] = {"ms": ms, "pairs_per_s": Pt / (ms * 1e-3), "points_per_s": Pt * Nt / (ms * 1e-3),
                                             "resolved": int((d_tw >= 0).sum().item()),
                                             "finite_points": int(torch.isfinite(d_tX).all(dim=1).sum().item())}

    # gold-standard refinement (second half of fun.getFFromLabCode): the reference's own case (257 inliers of the noisy
    # Dino pair (0,1); SciPy: 5482 residual evaluations, 267 s on this project's build box) and a config-5 sized batch
    try:
        gsg = np.load(os.path.join(ROOT, "tests", "golden", "gs_golden.npz"))
        gpts = np.ascontiguousarray(np.hstack([gsg["in1"].T, gsg["in2"].T]))
        rt.gold_standard([gpts], gsg["F0"][None])
        t0 = time.perf_counter()
        for _ in range(5):
            gres = rt.gold_standard([gpts], gsg["F0"][None])
        dt = (time.perf_counter() - t0) / 5
        Pg, Ng = 16, 50000
        big = []
        for k in range(Pg):
            Xs = np.column_stack([rng.uniform(-0.04, 0.04, Ng), rng.uniform(-0.07, 0.02, Ng), rng.uniform(-0.7, -0.56, Ng),
                                  np.ones(Ng)])
            a, b = Xs @ Ps[k].T, Xs @ Ps[k + 1].T
            big.append(np.hstack([a[:, :2] / a[:, 2:], b[:, :2] / b[:, 2:]]) + rng.normal(0, 0.5, (Ng, 4)))
        d_gp = torch.from_numpy(np.concatenate(big)).to(dev)
        d_gF = torch.from_numpy(np.stack([Fs[k] for k in range(Pg)])).to(dev)
        d_gout = torch.empty((Pg, 9), dtype=torch.float64, device=dev)
        d_gcost = torch.empty(Pg, dtype=torch.float64, device=dev)
        d_git = torch.empty(2 * Pg, dtype=torch.int32, device=dev)
        goff = (np.arange(Pg + 1, dtype=np.int32) * Ng)

        def gcall():
            cabi.check(lib.rg_gold_standard_dev(vp(ctx), vp(stream), Pg, vp(d_gp.data_ptr()), goff.ctypes.data_as(pi32),
                                                vp(d_gF.data_ptr()), None, 50, 1e-12, vp(d_gout.data_ptr()),
                                                vp(d_gcost.data_ptr()), vp(d_git.data_ptr()), vp(d_git[Pg:].data_ptr()), None))
        msg = ev_time(gcall, 3)
        out["gold_standard"] = {
            "dino_noisy_pair_257_inliers": {"host_call_ms": dt * 1e3, "cost": float(gres["cost"][0]),
                                            "iters": int(gres["iters"][0]), "status": int(gres["status"][0]),
                                            "reference_scipy": {"cost": float(gsg["scipy_cost"]), "nfev": int(gsg["scipy_nfev"]),
                                                                "seconds_on_build_box": 267}},
            "batch_16_pairs_x_50000": {"ms": msg, "points_per_s": Pg * Ng / (msg * 1e-3),
                                       "iters": [int(v) for v in d_git[:Pg].cpu().numpy()[:4]],
                                       "status": [int(v) for v in d_git[Pg:].cpu().numpy()[:4]],
                                       "cost_per_point": float(d_gcost.mean().item()) / Ng}}
    except Exception as e:
        out["gold_standard"] = {"error": repr(e)}

    # bundle adjustment (Tables.BundleAdjustment2): the 36-view Dino scene the golden file holds (reference: SciPy trf with
    # a finite-difference Jacobian, 14 residual sweeps, ~8 s) and the oracle's SciPy call timed here on the 8-view scene
    try:
        from oracle import ba_path as oba
        bag = np.load(os.path.join(ROOT, "tests", "golden", "ba_golden.npz"))
        bsc = lambda nv: tuple(bag[f"v{nv}_" + k] for k in ("cams0", "pts0", "uv", "cam_idx", "pt_idx"))
        b36 = bsc(36)
        rt.bundle_adjust(*b36, ftol=1e-4)
        t0 = time.perf_counter()
        for _ in range(5):
            bres = rt.bundle_adjust(*b36, ftol=1e-4)
        dt = (time.perf_counter() - t0) / 5
        d_bc = torch.from_numpy(b36[0].copy()).to(dev)
        d_bp = torch.from_numpy(b36[1].copy()).to(dev)
        d_buv = torch.from_numpy(b36[2].copy()).to(dev)
        d_bout = torch.empty(1, dtype=torch.float64, device=dev)
        d_bit = torch.empty(2, dtype=torch.int32, device=dev)
        bci = np.ascontiguousarray(b36[3], dtype=np.int32)
        bpi = np.ascontiguousarray(b36[4], dtype=np.int32)
        n_it = 8                                     # fixed number of LM iterations from the same start: per-iteration device time

        def bcall():
            d_bc.copy_(torch.from_numpy(b36[0]), non_blocking=False)
            d_bp.copy_(torch.from_numpy(b36[1]), non_blocking=False)
            cabi.check(lib.rg_bundle_adjust_dev(vp(ctx), vp(stream), 36, b36[1].shape[0], b36[2].shape[0], vp(d_bc.data_ptr()),
                                                vp(d_bp.data_ptr()), vp(d_buv.data_ptr()), bci.ctypes.data_as(pi32),
                                                bpi.ctypes.data_as(pi32), 1, n_it, 0.0, vp(d_bout.data_ptr()),
                                                vp(d_bit.data_ptr()), vp(d_bit[1:].data_ptr())))
        msb = ev_time(bcall, 3)
        b8 = bsc(8)
        t0 = time.perf_counter()
        _, _, sol8 = oba.bundle_adjust_scipy(*b8)
        dt8 = time.perf_counter() - t0
        r8 = rt.bundle_adjust(*b8, ftol=1e-4)
        t0 = time.perf_counter()
        for _ in range(5):
            r8 = rt.bundle_adjust(*b8, ftol=1e-4)
        dt8g = (time.perf_counter() - t0) / 5
        from tsbb15_b200 import synth as _synth
        big = _synth.ba_scene(36, 20000, track=8)
        rbig = rt.bundle_adjust(*big[:5], ftol=1e-6)
        t0 = time.perf_counter()
        rbig = rt.bundle_adjust(*big[:5], ftol=1e-6)
        dtbig = time.perf_counter() - t0
        out["bundle_adjust"] = {
            "synthetic_36_views_20000_points_160000_obs": {"host_call_ms": dtbig * 1e3, "cost": rbig["cost"],
                                                           "iters": rbig["iters"], "status": rbig["status"],
                                                           "observations_per_s_per_iteration":
                                                               160000 * rbig["iters"] / dtbig},
            "dino_36_views_676_points_4165_obs": {
                "host_call_ms": dt * 1e3, "cost": bres["cost"], "iters": bres["iters"], "status": bres["status"],
                "device_ms_per_lm_iteration": msb / n_it,
                "reference_scipy": {"cost": float(bag["v36_scipy_cost"]), "nfev": int(bag["v36_scipy_nfev"]),
                                    "seconds_on_build_box": 8.1}},
            "dino_8_views_113_points_560_obs": {
                "host_call_ms": dt8g * 1e3, "cost": r8["cost"], "iters": r8["iters"],
                "cpu_baseline": {"value": dt8 * 1e3, "unit": "ms per bundle adjustment", "cores": 1, "kind": "port",
                                 "cost": float(sol8.cost), "nfev": int(sol8.nfev),
                                 "sample": "the reference's SciPy call (tables.py:317) on the oracle's vectorised EpsilonBA, "
                                           "whole problem"}}}
    except Exception as e:
        out["bundle_adjust"] = {"error": repr(e)}

    # 2D<->3D match loop of Tables.addNewView: 20 000 queries against 20 000 observations, 2/3 of them present
    M = Nq = 20000
    obs = np.column_stack([rng.uniform(-0.1, 0.1, (M, 2)), np.ones(M)])
    q = np.column_stack([rng.uniform(-0.1, 0.1, (Nq, 2)), np.ones(Nq)])
    take = rng.uniform(size=Nq) < 0.67
    q[take] = obs[rng.integers(0, M, int(take.sum()))]
    dobs, dq = torch.from_numpy(obs).to(dev), torch.from_numpy(q).to(dev)
    dm = torch.empty(Nq, dtype=torch.int32, device=dev)

    def mcall():
        cabi.check(lib.rg_match_first_within_dev(vp(ctx), vp(stream), 3, M, vp(dobs.data_ptr()), Nq, vp(dq.data_ptr()),
                                                 1e-4, vp(dm.data_ptr())))
    ms = ev_time(mcall, 5)
    t0 = time.perf_counter()
    refm = og.match_first_within(obs, q[:24], 1e-4)
    dt = time.perf_counter() - t0
    out["match_20000_x_20000"] = {"ms": ms, "queries_per_s": Nq / (ms * 1e-3),
                                  "matched": int((dm >= 0).sum().item()),
                                  "bit_exact_vs_oracle_sample": bool(np.array_equal(dm[:24].cpu().numpy(), refm)),
                                  "cpu_baseline": {"value": 24 / dt, "unit": "queries/s", "cores": 1, "kind": "port",
                                                   "sample": "24 queries x 20000 observations, the literal loop of "
                                                             "tables.py:116-124"}}
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=4096, help="image pairs of the sweep (fixed total, split over the ranks)")
    ap.add_argument("--n", type=int, default=50000)
    ap.add_argument("--hyp", type=int, default=8192)
    ap.add_argument("--solver", type=int, default=0)
    ap.add_argument("--host-slices", type=int, default=0, help="sub-batches of the host entry point (0 = automatic)")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-split", action="store_true", help="skip the hypothesis-split legs (configs 3 and 4)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-oracle-check", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup_raised = args.impl == "ours" and args.warmup < 3
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup      # timing rules: W >= 3 (noted in config)
    try:
        if args.impl == "reference":
            run_reference_arm(args)
        else:
            run_ours(args)
    finally:
        if _POOL is not None:                       # CPU-baseline workers: shut down before interpreter teardown
            _POOL.close()
            _POOL.join()


if __name__ == "__main__":
    main()
