// Host orchestration + C ABI of the F-matrix RANSAC path.  See include/rg_b200.h for the contract of each entry point.
//
// One call = one or more PASSES.  A pass is the launch chain
//   memset(state) -> [f_bbox -> f_normalise] -> f8_solve (draws its own samples when idx is NULL) -> score_packed -> fixup_list -> argmax_counts
//   -> [f_tie_stats -> f_tie_resolve] -> f_mask
// over a contiguous block of pairs whose workspaces (hypotheses, FP32 points, flag list) stay bounded; BASELINE config 5
// (4096 pairs x 50 000 x 8 192) runs as 64 passes of 64 pairs.  A call that wants no per-hypothesis counts runs the bounded
// sweep instead of score_packed -> fixup_list (bounded.cuh): bound-only prefix stage A, candidates, candidate stage,
// extension of the prefix for the hypotheses still alive (stage B), check, fallback.  The per-pass PairInfo table is
// planned on the host into double-buffered pinned staging, so the host plans pass k+1 while pass k runs.
#include "f_kernels.cuh"
#include "bounded.cuh"
#include "jacobi.cuh"
#include "philox.cuh"
#include "plan.cuh"
#include <algorithm>
#include <vector>

namespace rg {

enum : int { FLAG_REUSE_POINTS = 1, FLAG_BOUNDED = 2 };

constexpr double kDefaultPassEvals = 2.7e10;        // 64 pairs of the config-5 shape
constexpr long long kMaxPassHyp = 1ll << 22;        // hypotheses per pass (F64 workspace 288 MB)

struct ScoreState {
    unsigned* bbox; int* counts; int* work; unsigned* list_n; unsigned char* ovf;
    size_t off_counts, bytes;
    // bounded sweep (Ctot >= 0): work counters / list sizes of the candidate (c) and fallback (f) stages, the fallback's
    // item count, suffix counts, marks of the pairs that fell back, overflow marks; stage B's work counter, item count,
    // counts (compact, as its records) and |S| per pair
    int *c_work, *f_work, *f_items, *sfx_c, *sfx_f, *mark;
    int *b_work, *b_items, *cnt_b, *n_s;
    unsigned *c_list_n, *f_list_n;
    unsigned char *ovf_c, *ovf_f;
};

// [bbox keys: P x words][counts: H][work counter][list size][pad][ovf: H bytes]
//   + bounded sweep: [8 counters][sfx_c: C][sfx_f: H][mark: P][cnt_b: B][n_s: P][ovf_c: C bytes][ovf_f: H bytes]
// — one cudaMemsetAsync clears a pass's state
int score_state_layout(Ctx* c, int P, long long Htot, int bbox_words, ScoreState& s, long long Ctot = -1,
                       long long Btot = 0) {
    const size_t H = (size_t)std::max<long long>(Htot, 1);
    const size_t bbox_bytes = (((size_t)std::max(P, 1) * bbox_words * 4) + 15) / 16 * 16;
    const size_t cnt_bytes = ((H + 2) * 4 + 15) / 16 * 16;
    const size_t ovf_bytes = (H + 15) / 16 * 16;
    const size_t C = (size_t)std::max<long long>(Ctot, 1);
    const size_t B = (size_t)std::max<long long>(Btot, 1), P1 = (size_t)std::max(P, 1);
    const size_t bnd_ints = Ctot >= 0 ? ((8 + C + H + P1 + B + P1) * 4 + 15) / 16 * 16 : 0;
    const size_t bnd_ovf = Ctot >= 0 ? (C + H + 15) / 16 * 16 : 0;
    s.off_counts = bbox_bytes;
    s.bytes = bbox_bytes + cnt_bytes + ovf_bytes + bnd_ints + bnd_ovf;
    int rc = ensure(c->state, s.bytes);
    if (rc) return rc;
    char* base = (char*)c->state.ptr;
    s.bbox = (unsigned*)base;
    s.counts = (int*)(base + bbox_bytes);
    s.work = s.counts + H;
    s.list_n = (unsigned*)(s.counts + H + 1);
    s.ovf = (unsigned char*)(base + bbox_bytes + cnt_bytes);
    if (Ctot >= 0) {
        int* b = (int*)(base + bbox_bytes + cnt_bytes + ovf_bytes);
        s.c_work = b; s.c_list_n = (unsigned*)(b + 1); s.f_work = b + 2; s.f_list_n = (unsigned*)(b + 3); s.f_items = b + 4;
        s.b_work = b + 5; s.b_items = b + 6;
        s.sfx_c = b + 8; s.sfx_f = s.sfx_c + C; s.mark = s.sfx_f + H; s.cnt_b = s.mark + P1; s.n_s = s.cnt_b + B;
        s.ovf_c = (unsigned char*)(base + bbox_bytes + cnt_bytes + ovf_bytes + bnd_ints);
        s.ovf_f = s.ovf_c + C;
    }
    c->counts_ptr = s.counts;
    c->ovf_ptr = s.ovf;
    return RG_OK;
}

// per-set workspace of the bounded sweep: [compact Hyp32 records: C][map: C][sel: P int4][live fallback table: P]
//   [stage B's compact Hyp32 records: B][its map: B][live stage-B table: P]
struct BndWs { Hyp32* hypc; int* map; int4* sel; PairInfo* fb; Hyp32* hypb; int* mapb; PairInfo* bt; };
static int bnd_workspace(Ctx* c, const FPlan& plan, BndWs& w) {
    const size_t C = (size_t)std::max<long long>(plan.Ctot, 1), P = (size_t)std::max(plan.P, 1);
    const size_t B = (size_t)std::max<long long>(plan.Btot, 1);
    const size_t o_map = C * sizeof(Hyp32), o_sel = o_map + (C * 4 + 63) / 64 * 64, o_fb = o_sel + P * sizeof(int4);
    const size_t o_hypb = o_fb + P * sizeof(PairInfo), o_mapb = o_hypb + B * sizeof(Hyp32);
    const size_t o_bt = o_mapb + (B * 4 + 63) / 64 * 64;
    int rc = ensure(c->bnd, o_bt + P * sizeof(PairInfo));
    if (rc) return rc;
    char* b = (char*)c->bnd.ptr;
    w.hypc = (Hyp32*)b; w.map = (int*)(b + o_map); w.sel = (int4*)(b + o_sel); w.fb = (PairInfo*)(b + o_fb);
    w.hypb = (Hyp32*)(b + o_hypb); w.mapb = (int*)(b + o_mapb); w.bt = (PairInfo*)(b + o_bt);
    return RG_OK;
}

// blocks of the fix-up kernel: one full wave for big passes, a few blocks for small ones (a pass of 2048 hypotheses x
// 100 000 correspondences flags ~90 000 groups: 4736 mostly idle warps cost more to launch and to retire than the work)
int fixup_grid(const Ctx* c, double evals) {
    const double expected_records = evals * 6.0e-4;              // measured 4.5e-4 flagged groups per evaluation
    const long long want = (long long)(expected_records / 256.0) + 1;     // ~one record per thread
    return (int)std::max<long long>(8, std::min<long long>(want, (long long)c->sm_count * 4));
}

FlagList flag_list_for(Ctx* c, const ScoreState& s, double evals, int* rc_out) {
    FlagList L{nullptr, s.list_n, 0u, s.ovf};
    double want = evals / 512.0 + 65536.0;            // ~4.3x the measured 4.5e-4 records per evaluation
    if (c->opt_list_cap > 0) want = (double)c->opt_list_cap;
    const unsigned cap = (unsigned)std::min(want, 1.0e9);
    *rc_out = ensure(c->flag_list, sizeof(int2) * (size_t)cap);
    L.rec = (int2*)c->flag_list.ptr;
    L.cap = cap;
    return L;
}

struct FCall {
    int P = 0;
    const double* pts64 = nullptr; const int* pair_off = nullptr;
    const int* idx = nullptr;      const int* hyp_off = nullptr;
    double thr = 1.5;
    int mode = MODE_EPI_MAX, tie_mode = TIE_FIRST, solver = SOLVER_QR, score_path = SCORE_FP32_GUARDED, flags = 0;
    unsigned long long sample_seed = 0; int first_pair = 0; int hyp_first = 0;
    bool bounded = false;          // bounded sweep (bounded.cuh): the per-hypothesis counts are not all full counts
    int* best_idx = nullptr; int* best_count = nullptr; double* best_F = nullptr; unsigned char* mask = nullptr;
    unsigned long long* keys = nullptr;
};

// ---- pass pipelining (Ctx::spare, common.cuh; the schedules are in f_run_piped below) ----
// Single-pass calls never switch: their launch chain stays on the caller's stream in the current set (capturable in a CUDA
// graph, RG_FLAG_REUSE_POINTS finds its prepared points).
static void ws_exchange(Ctx* c, Ctx::PassSet& o) {
    std::swap(c->pair_info, o.pair_info);   std::swap(c->pair_frame, o.pair_frame);
    std::swap(c->state, o.state);           std::swap(c->pts32, o.pts32);
    std::swap(c->F64, o.F64);               std::swap(c->hyp32, o.hyp32);
    std::swap(c->flags, o.flags);           std::swap(c->flag_list, o.flag_list);
    std::swap(c->best, o.best);             std::swap(c->tie_stats, o.tie_stats);
    std::swap(c->bnd, o.bnd);
}

static void ws_use(Ctx* c, int slot) {
    if (c->ws_slot == slot) return;
    ws_exchange(c, c->spare[c->ws_slot]);        // park the current set (its spare entry was empty) ...
    ws_exchange(c, c->spare[slot]);              // ... and take the wanted one out of its entry
    c->ws_slot = slot;
    c->plan_valid = false;                       // the cached PairInfo table lives in the set that just left
    c->prep_pts = nullptr;                       // ... and so do the prepared points
}

// An SM cannot change its L1 / shared-memory split while blocks are resident.  The tail kernels of pass k are still resident
// when the scorer of pass k+1 arrives; left to the default carve-out they had switched the SM to a smaller shared-memory
// partition and only three of the scorer's four 49 KB blocks fitted until they drained (measured: scorer 15.41 -> 16.10 ms
// with the tail beside it, 15.55 ms once the tail kernels ask for the maximum carve-out too; profiles/r02_pipe_sweep.txt).
// The preference is a per-function attribute: it is switched on for pipelined passes only, so that single-pass calls (and
// the last pass of a call, whose tail runs alone) keep the large L1 the fix-up's gathers like.
static int tail_carveout(Ctx* c, bool want_max) {
    static const int off = [] { const char* e = getenv("RG_TAIL_NO_CARVEOUT"); return e ? atoi(e) : 0; }();     // experiment hook
    if (off || c->tail_carve_max == (int)want_max) return RG_OK;
    const int v = want_max ? (int)cudaSharedmemCarveoutMaxShared : (int)cudaSharedmemCarveoutDefault;
    RG_CUDA(cudaFuncSetAttribute(fixup_list<EpiFix<MODE_EPI_MAX>>, cudaFuncAttributePreferredSharedMemoryCarveout, v));
    RG_CUDA(cudaFuncSetAttribute(fixup_list<EpiFix<MODE_SAMPSON>>, cudaFuncAttributePreferredSharedMemoryCarveout, v));
    RG_CUDA(cudaFuncSetAttribute(f_mask, cudaFuncAttributePreferredSharedMemoryCarveout, v));
    RG_CUDA(cudaFuncSetAttribute(argmax_counts, cudaFuncAttributePreferredSharedMemoryCarveout, v));
    RG_CUDA(cudaFuncSetAttribute(f_tie_stats, cudaFuncAttributePreferredSharedMemoryCarveout, v));
    RG_CUDA(cudaFuncSetAttribute(f_tie_resolve, cudaFuncAttributePreferredSharedMemoryCarveout, v));
    RG_CUDA(cudaFuncSetAttribute(f8_solve_qr<MODE_EPI_MAX>, cudaFuncAttributePreferredSharedMemoryCarveout, v));
    RG_CUDA(cudaFuncSetAttribute(f8_solve_qr<MODE_SAMPSON>, cudaFuncAttributePreferredSharedMemoryCarveout, v));
    for (const void* f : {(const void*)bnd_select, (const void*)bnd_extend, (const void*)bnd_check, (const void*)bnd_live_plan,
                          (const void*)bnd_merge})
        RG_CUDA(cudaFuncSetAttribute(f, cudaFuncAttributePreferredSharedMemoryCarveout, v));
    c->tail_carve_max = (int)want_max;
    return RG_OK;
}

static int pipe_setup(Ctx* c) {
    if (!c->tail_stream) {
        static const int low = [] { const char* e = getenv("RG_TAIL_PRIO"); return e ? atoi(e) : 0; }();     // experiment hook
        int lo_p = 0, hi_p = 0;
        RG_CUDA(cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p));
        RG_CUDA(cudaStreamCreateWithPriority(&c->tail_stream, cudaStreamNonBlocking, low ? lo_p : 0));
    }
    for (int i = 0; i < 3; ++i) {
        if (!c->head_done[i]) RG_CUDA(cudaEventCreateWithFlags(&c->head_done[i], cudaEventDisableTiming));
        if (!c->score_done[i]) RG_CUDA(cudaEventCreateWithFlags(&c->score_done[i], cudaEventDisableTiming));
        if (!c->cand_done[i]) RG_CUDA(cudaEventCreateWithFlags(&c->cand_done[i], cudaEventDisableTiming));
        if (!c->sweep_done[i]) RG_CUDA(cudaEventCreateWithFlags(&c->sweep_done[i], cudaEventDisableTiming));
    }
    if (!c->tail_done) RG_CUDA(cudaEventCreateWithFlags(&c->tail_done, cudaEventDisableTiming));
    if (!c->pipe_gate) RG_CUDA(cudaEventCreateWithFlags(&c->pipe_gate, cudaEventDisableTiming));
    return RG_OK;
}

static unsigned long long hash_offsets(const int* off, int n) {
    unsigned long long h = 1469598103934665603ull;
    for (int i = 0; i <= n; ++i) { h ^= (unsigned)off[i]; h *= 1099511628211ull; }
    return h;
}

static int f_workspace(Ctx* c, const FPlan& plan) {
    int rc;
    const size_t H = (size_t)std::max<long long>(plan.Htot, 1);
    if ((rc = ensure(c->F64, sizeof(double) * 9 * H))) return rc;
    if ((rc = ensure(c->hyp32, sizeof(Hyp32) * H))) return rc;
    if ((rc = ensure(c->flags, H))) return rc;
    if ((rc = ensure(c->stats, sizeof(unsigned long long) * 8))) return rc;
    if ((rc = ensure(c->best, sizeof(int2) * (size_t)std::max(plan.P, 1)))) return rc;
    if ((rc = ensure(c->tie_stats, sizeof(double2) * H))) return rc;
    if ((rc = ensure(c->pair_frame, sizeof(PairFrame) * (size_t)std::max(plan.P, 1)))) return rc;
    if ((rc = ensure_pinned(c->h_stats, sizeof(unsigned long long) * 8))) return rc;
    return RG_OK;
}

static int f_prepare(Ctx* c, cudaStream_t st, const FPlan& plan, const ScoreState& s, const double* pts64, double thr) {
    int rc;
    if ((rc = ensure(c->pts32, sizeof(float4) * (size_t)std::max<long long>(plan.N32tot, 1)))) return rc;
    const PairInfo* pi = (const PairInfo*)c->pair_info.ptr;
    const int P = plan.P;
    const int nbx = std::max(1, std::min(64, ceil_div(plan.maxN, 256 * 4)));
    f_bbox<<<dim3(nbx, P), 256, 0, st>>>((const double4*)pts64, pi, s.bbox);
    const int nbn = std::max(1, std::min(128, ceil_div(plan.maxN / 2 + kSub, 256)));
    f_normalise<<<dim3(nbn, P), 256, 0, st>>>((const double4*)pts64, pi, s.bbox, thr, c->opt_band_scale, (PairFrame*)c->pair_frame.ptr,
                                              (float4*)c->pts32.ptr);
    c->last_stats[7] += 2;
    RG_CUDA(cudaGetLastError());
    return RG_OK;
}

template <int MODE>
static int f_solve_launch(Ctx* c, cudaStream_t st, const FPlan& plan, const double* pts64, const int* idx, int solver,
                          unsigned long long seed = 0, unsigned first_pair = 0) {
    const PairInfo* pi = (const PairInfo*)c->pair_info.ptr;
    const PairFrame* fr = (const PairFrame*)c->pair_frame.ptr;
    if (plan.Htot == 0) return RG_OK;
    if (solver == SOLVER_QR) {
        f8_solve_qr<MODE><<<ceil_div(plan.Htot, 128), 128, 0, st>>>((const double4*)pts64, idx, seed, first_pair, pi, fr, plan.P,
                                                                  (int)plan.Htot, (double*)c->F64.ptr, (Hyp32*)c->hyp32.ptr,
                                                                  (unsigned char*)c->flags.ptr);
    } else {
        const int groups_per_block = kJacobiThreads / 16;
        f8_solve_jacobi<MODE><<<ceil_div(plan.Htot, groups_per_block), kJacobiThreads, 0, st>>>(
            (const double4*)pts64, idx, seed, first_pair, pi, fr, plan.P, (int)plan.Htot, (double*)c->F64.ptr,
            (Hyp32*)c->hyp32.ptr, (unsigned char*)c->flags.ptr);
    }
    c->last_stats[7] += 1;
    RG_CUDA(cudaGetLastError());
    return RG_OK;
}

// ---- one pass = three phases that may run on different streams (pass pipelining, see f_run_piped) ----
//   head : PairInfo plan + memset(state) + [f_bbox, f_normalise] + f8_solve      (needs only the pass's inputs)
//   score: score_packed                                                          (the FP32-bound 94 % of a pass)
//   tail : fixup_list + argmax_counts [+ f_tie_stats + f_tie_resolve] + f_mask   (latency bound, needs the scorer's counts)
struct PassCtl {
    FCall a;
    std::vector<int> po, ho;              // storage behind a.pair_off / a.hyp_off when the pass is a sub-range of a call
    FPlan plan;
    ScoreState s;
    FlagList fl{nullptr, nullptr, 0u, nullptr};
    FlagList flc{nullptr, nullptr, 0u, nullptr}, flf{nullptr, nullptr, 0u, nullptr};   // bounded sweep: candidate / fallback stage
    BndWs bw{};
    bool scored = false;                  // the packed scorer ran: its flag list wants the fix-up
    int slot = 0;                         // workspace set of the pass (Ctx::spare; pipelined runs only)
    int prof_call = -1;                   // ring index of the pass's phase events (option 1)
    cudaEvent_t ready = nullptr;          // optional: the pass's inputs have arrived; the stream that runs its head waits for it
    cudaEvent_t done = nullptr;           // optional: recorded behind the pass's last tail kernel
    // optional: a copy queued on out_stream behind `done` as soon as the pass's tail is queued (host entry point: the pass's
    // inlier masks travel back while later passes are scored; queued after all passes instead, a 64-pass call had its host
    // thread stuck in the driver's launch queue and every mask download ended up behind the last scorer)
    cudaStream_t out_stream = nullptr; void* out_dst = nullptr; const void* out_src = nullptr; size_t out_bytes = 0;
    // optional: host destinations of the pass's per-hypothesis counts / F / flags, copied behind its tail (they live in the
    // pass's workspace set, which the next pass reuses: a call that wants them runs its passes one after the other)
    int* out_counts = nullptr; double* out_F_all = nullptr; unsigned char* out_flags = nullptr;
    bool wants_hypotheses() const { return out_counts || out_F_all || out_flags; }
};

// counts / work counter / flag list are already cleared by the pass's memset
template <int MODE>
static int f_score_only(Ctx* c, cudaStream_t st, PassCtl& k) {
    const FPlan& plan = k.plan;
    const PairInfo* pi = (const PairInfo*)c->pair_info.ptr;
    k.scored = false;
    if (plan.Htot == 0 || plan.Ntot == 0 || (k.a.score_path != SCORE_FP64 && plan.n_items == 0)) return RG_OK;
    if (k.a.score_path != SCORE_FP64) {
        int bps = 1, rc = score_blocks_per_sm<EpiPolicy<MODE>>(&bps);
        if (rc) return rc;
        // (the later stages of a bounded pass reuse the records once the previous stage's fix-up has read them)
        k.fl = flag_list_for(c, k.s, std::max(plan.evals, plan.evals_f), &rc);
        if (rc) return rc;
        if (plan.bounded) {
            k.flc = FlagList{k.fl.rec, k.s.c_list_n, k.fl.cap, k.s.ovf_c};
            k.flf = FlagList{k.fl.rec, k.s.f_list_n, k.fl.cap, k.s.ovf_f};
        }
        if (plan.bound_prefix || k.a.score_path == SCORE_FP32_BOUND) {      // upper-bound counts: no flags, no fix-up
            static_assert(score_smem_bytes<EpiBoundPolicy>() == score_smem_bytes<EpiPolicy<MODE>>(), "same stage ring");
            if ((rc = score_blocks_per_sm<EpiBoundPolicy>(&bps))) return rc;
            score_packed<EpiBoundPolicy><<<std::min(plan.n_items, c->sm_count * bps), kScoreThreads,
                                           score_smem_bytes<EpiBoundPolicy>(), st>>>(
                (const float4*)c->pts32.ptr, (const Hyp32*)c->hyp32.ptr, pi, plan.P, plan.n_items, k.s.counts, k.fl, k.s.work);
        } else {
            constexpr size_t smem = score_smem_bytes<EpiPolicy<MODE>>();
            const int grid = std::min(plan.n_items, c->sm_count * bps);
            score_packed<EpiPolicy<MODE>><<<grid, kScoreThreads, smem, st>>>((const float4*)c->pts32.ptr, (const Hyp32*)c->hyp32.ptr,
                                                                            pi, plan.P, plan.n_items, k.s.counts, k.fl, k.s.work);
        }
        k.scored = true;
    } else {
        const int zs = std::max(1, std::min(64, ceil_div(plan.maxN, 2048)));
        f_score_fp64<<<dim3(ceil_div(plan.maxH, 128), plan.P, zs), 128, 0, st>>>((const double4*)k.a.pts64, (const double*)c->F64.ptr,
                                                                                 pi, k.a.thr, MODE, k.s.counts);
    }
    c->last_stats[7] += 1;
    RG_CUDA(cudaGetLastError());
    return RG_OK;
}

// beside_scorer: the kernel will run NEXT TO the following pass's scorer (4 blocks x 128 threads x 96 registers per SM leave
// room for exactly one 256-thread, 64-register block): a grid of one block per SM runs beside the scorer instead of ahead of it
// stage: what the fix-up corrects — STAGE_MAIN the pass's scorer (full sweep, or the bounded sweep's exact prefix stage),
// STAGE_CAND the candidate stage (compact records, counts in sfx_c), STAGE_FALLBACK the fallback stage (counts in sfx_f)
enum : int { STAGE_MAIN = 0, STAGE_CAND = 1, STAGE_FALLBACK = 2 };
template <int MODE>
static int f_fixup_launch(Ctx* c, cudaStream_t ts, PassCtl& k, bool beside_scorer, int stage = STAGE_MAIN) {
    if (!k.scored) return RG_OK;
    const FPlan& plan = k.plan;
    const PairInfo* pi = (const PairInfo*)c->pair_info.ptr;
    const Hyp32* hyp = (const Hyp32*)c->hyp32.ptr;
    const int* map = nullptr;
    FlagList fl = k.fl;
    long long H = plan.Htot;
    int* counts = k.s.counts;
    double evals = plan.evals;
    if (stage == STAGE_CAND) {
        pi += plan.P; hyp = k.bw.hypc; map = k.bw.map; fl = k.flc; H = plan.Ctot; counts = k.s.sfx_c; evals = plan.evals_c;
    } else if (stage == STAGE_FALLBACK) {
        pi = k.bw.fb; fl = k.flf; counts = k.s.sfx_f; evals = plan.evals_f;
    }
    typename EpiFix<MODE>::Params fp{(const float4*)c->pts32.ptr, (const double4*)k.a.pts64, hyp, (const double*)c->F64.ptr,
                                     pi, (const PairFrame*)c->pair_frame.ptr, plan.P, map};
    int fgrid = fixup_grid(c, evals);
    if (beside_scorer) {
        static const int forced = [] { const char* e = getenv("RG_TAIL_GRID"); return e ? atoi(e) : 0; }();   // experiment hook
        fgrid = std::min(fgrid, forced > 0 ? forced : c->sm_count);
    }
    fixup_list<EpiFix<MODE>><<<fgrid, 256, 0, ts>>>(fp, fl, (int)H, counts, (unsigned long long*)c->stats.ptr);
    c->last_stats[7] += 1;
    RG_CUDA(cudaGetLastError());
    return RG_OK;
}

// bounded sweep, after the prefix stage: its fix-up (exact prefix only: counts c_A) and the choice of the candidates
template <int MODE>
static int f_bnd_cands(Ctx* c, cudaStream_t ts, PassCtl& k, bool beside_scorer) {
    if (k.scored) {
        int rc = k.plan.bound_prefix ? RG_OK : f_fixup_launch<MODE>(c, ts, k, beside_scorer);
        if (rc) return rc;
        const PairInfo* pi = (const PairInfo*)c->pair_info.ptr;
        bnd_select<<<k.plan.P, kSelectThreads, 0, ts>>>(k.s.counts, pi, pi + k.plan.P, (const Hyp32*)c->hyp32.ptr, k.bw.hypc,
                                                        k.bw.map, k.bw.sel);
        c->last_stats[7] += 1;
        RG_CUDA(cudaGetLastError());
    }
    prof_mark_at(c, ts, k.prof_call, 4);
    return RG_OK;
}

// bounded sweep, after the candidates: candidate stage + its fix-up, extension (bnd_extend, stage B), check, fallback
// stage.  Stage B and the fallback are queued at full grid with their item counts read from the device (bnd_live_plan;
// the fallback normally has none).  The fallback's fix-up and merge belong to the tail.
template <int MODE>
static int f_bnd_sweep(Ctx* c, cudaStream_t st, PassCtl& k) {
    if (!k.scored) return RG_OK;
    const FPlan& plan = k.plan;
    const PairInfo* pi = (const PairInfo*)c->pair_info.ptr;
    const PairInfo *pc = pi + plan.P, *pf = pi + 2 * (size_t)plan.P, *pb = pi + 3 * (size_t)plan.P;
    unsigned long long* bstats = (unsigned long long*)c->bnd_stats.ptr;
    int bps = 1, bps_b = 1, rc = score_blocks_per_sm<EpiPolicy<MODE>>(&bps);
    if (rc || (rc = score_blocks_per_sm<EpiBoundPolicy>(&bps_b))) return rc;
    constexpr size_t smem = score_smem_bytes<EpiPolicy<MODE>>();
    prof_mark_at(c, st, k.prof_call, Ctx::kProfSweep);
    if (plan.n_items_c > 0) {
        score_packed<EpiPolicy<MODE>><<<std::min(plan.n_items_c, c->sm_count * bps), kScoreThreads, smem, st>>>(
            (const float4*)c->pts32.ptr, k.bw.hypc, pc, plan.P, plan.n_items_c, k.s.sfx_c, k.flc, k.s.c_work);
        c->last_stats[7] += 1;
    }
    prof_mark_at(c, st, k.prof_call, Ctx::kProfSweep + 1);
    if (plan.n_items_c > 0 && (rc = f_fixup_launch<MODE>(c, st, k, false, STAGE_CAND))) return rc;
    bnd_extend<<<plan.P, 256, 0, st>>>(k.s.counts, k.s.sfx_c, k.bw.map, pi, pc, pb, (const Hyp32*)c->hyp32.ptr, k.bw.sel,
                                       k.bw.hypb, k.bw.mapb, k.s.n_s, k.s.mark, bstats,
                                       !plan.bound_prefix);
    c->last_stats[7] += 1;
    if (plan.n_items_b > 0) {
        bnd_live_plan<<<1, kSelectThreads, 0, st>>>(pb, k.s.n_s, plan.P, k.bw.bt, k.s.b_items);
        prof_mark_at(c, st, k.prof_call, Ctx::kProfSweep + 2);
        score_packed<EpiBoundPolicy><<<std::min(plan.n_items_b, c->sm_count * bps_b), kScoreThreads,
                                       score_smem_bytes<EpiBoundPolicy>(), st>>>(
            (const float4*)c->pts32.ptr, k.bw.hypb, k.bw.bt, plan.P, plan.n_items_b, k.s.cnt_b, k.fl, k.s.b_work, k.s.b_items);
        prof_mark_at(c, st, k.prof_call, Ctx::kProfSweep + 3);
        c->last_stats[7] += 2;
    }
    bnd_check<<<plan.P, 256, 0, st>>>(k.s.counts, k.s.sfx_c, k.bw.map, k.s.cnt_b, k.bw.mapb, k.s.n_s, pi, pc, pb, k.bw.sel,
                                      k.s.mark, bstats, !plan.bound_prefix);
    bnd_live_plan<<<1, kSelectThreads, 0, st>>>(pf, k.s.mark, plan.P, k.bw.fb, k.s.f_items);
    c->last_stats[7] += 2;
    prof_mark_at(c, st, k.prof_call, Ctx::kProfSweep + 4);
    if (plan.n_items_f > 0) {
        score_packed<EpiPolicy<MODE>><<<std::min(plan.n_items_f, c->sm_count * bps), kScoreThreads, smem, st>>>(
            (const float4*)c->pts32.ptr, (const Hyp32*)c->hyp32.ptr, k.bw.fb, plan.P, plan.n_items_f, k.s.sfx_f, k.flf,
            k.s.f_work, k.s.f_items);
        c->last_stats[7] += 1;
    }
    prof_mark_at(c, st, k.prof_call, Ctx::kProfSweep + 5);
    RG_CUDA(cudaGetLastError());
    return RG_OK;
}

// scorer + fix-up on one stream (stage entry point rg_epi_score_count_host; SCORE_FP32_BOUND: the bound-only scorer alone)
template <int MODE>
static int f_score_launch(Ctx* c, cudaStream_t st, const FPlan& plan, const ScoreState& s, const double* pts64, double thr,
                          int score_path) {
    PassCtl k;
    k.a.pts64 = pts64; k.a.thr = thr; k.a.score_path = score_path;
    k.plan = plan; k.s = s;
    int rc = f_score_only<MODE>(c, st, k);
    if (rc) return rc;
    prof_mark(c, st, 3);
    return score_path == SCORE_FP32_BOUND ? RG_OK : f_fixup_launch<MODE>(c, st, k, false);
}

static int f_select_launch(Ctx* c, cudaStream_t st, const FPlan& plan, const ScoreState& s, const double* pts64, double thr,
                           int mode, int tie_mode, unsigned char* mask, double* best_F, int* best_idx, int* best_count,
                           unsigned long long* keys) {
    if (plan.P == 0) return RG_OK;
    const PairInfo* pi = (const PairInfo*)c->pair_info.ptr;
    int2* best = (int2*)c->best.ptr;
    const bool tie = tie_mode == TIE_REFERENCE && plan.Htot > 0;
    if (!tie && mask == nullptr) {                    // nothing follows the argmax: it publishes the winners itself
        argmax_counts<<<plan.P, 256, 0, st>>>(s.counts, pi, best, (const unsigned char*)c->flags.ptr,
                                              (unsigned long long*)c->stats.ptr, keys, (const double*)c->F64.ptr, 9, best_F,
                                              best_idx, best_count);
        c->last_stats[7] += 1;
        RG_CUDA(cudaGetLastError());
        return RG_OK;
    }
    argmax_counts<<<plan.P, 256, 0, st>>>(s.counts, pi, best, (const unsigned char*)c->flags.ptr,
                                          (unsigned long long*)c->stats.ptr, tie ? nullptr : keys);
    c->last_stats[7] += 1;
    if (tie) {
        const int nb = (int)std::min<long long>(plan.Htot, (long long)c->sm_count * 8);
        f_tie_stats<<<nb, 256, 0, st>>>((const double4*)pts64, (const double*)c->F64.ptr, s.counts, pi, plan.P,
                                        (int)plan.Htot, best, mode, (double2*)c->tie_stats.ptr);
        f_tie_resolve<<<plan.P, 32, 0, st>>>(s.counts, pi, (const double2*)c->tie_stats.ptr, best, keys);
        c->last_stats[7] += 2;
    }
    const int nbx = mask ? std::max(1, std::min(64, ceil_div(plan.maxN, 256 * 4))) : 1;
    f_mask<<<dim3(nbx, plan.P), 256, 0, st>>>((const double4*)pts64, (const double*)c->F64.ptr, pi, best, thr, mode, mask, best_F,
                                              best_idx, best_count);
    c->last_stats[7] += 1;
    RG_CUDA(cudaGetLastError());
    return RG_OK;
}

// head of a pass on stream hs, in the CURRENT workspace set
static int f_pass_head(Ctx* c, cudaStream_t hs, PassCtl& k) {
    const FCall& a = k.a;
    FPlan& plan = k.plan;
    int bps = 1, rc = score_blocks_per_sm<EpiPolicy<MODE_EPI_MAX>>(&bps);
    if (rc) return rc;
    if ((rc = f_plan(c, hs, a.P, a.pair_off, a.hyp_off, plan, bps, nullptr, a.hyp_first, a.bounded ? c->opt_bounded_k : 0,
                     c->opt_rho_milli, a.bounded && c->opt_bound_prefix != 0, c->opt_rho0_milli)))
        return rc;
    for (int p = 0; p < a.P; ++p) {
        const int n = a.pair_off[p + 1] - a.pair_off[p], H = a.hyp_off[p + 1] - a.hyp_off[p];
        RG_CHECK_ARG(H == 0 || n >= 8, "a pair with hypotheses needs at least 8 correspondences");
    }
    if ((rc = f_workspace(c, plan))) return rc;
    if ((rc = score_state_layout(c, a.P, plan.Htot, 8, k.s, a.bounded ? plan.Ctot : -1, plan.Btot))) return rc;
    if (a.bounded && (rc = bnd_workspace(c, plan, k.bw))) return rc;
    if (plan.bound_prefix) {
        c->bnd_bound_evals += (long long)plan.evals;
        c->bnd_host_evals += (long long)plan.evals_c;
    } else {
        c->bnd_host_evals += (long long)(plan.evals + plan.evals_c);
    }
    const ScoreState& s = k.s;

    bool reuse = (a.flags & FLAG_REUSE_POINTS) != 0;
    const unsigned long long hsh = hash_offsets(a.pair_off, a.P);
    if (reuse) {
        RG_CHECK_ARG(c->prep_pts == (const void*)a.pts64 && c->prep_P == a.P && c->prep_N == plan.Ntot &&
                         c->prep_thr == a.thr && c->prep_hash == hsh,
                     "RG_FLAG_REUSE_POINTS: the previous pass on this context prepared different points / threshold");
    }
    k.prof_call = prof_begin(c);
    prof_mark_at(c, hs, k.prof_call, 0);
    // one memset clears the pass's state (the bounding boxes only when the points are prepared in this pass)
    const size_t from = reuse ? s.off_counts : 0;
    RG_CUDA(cudaMemsetAsync((char*)c->state.ptr + from, 0, s.bytes - from, hs));
    const int* idx = a.idx;                           // NULL: the solver draws its own sample (philox.cuh), no index array exists
    if (!reuse) {
        c->prep_pts = nullptr;
        if ((rc = f_prepare(c, hs, plan, s, a.pts64, a.thr))) return rc;
        c->prep_pts = a.pts64; c->prep_P = a.P; c->prep_N = plan.Ntot; c->prep_thr = a.thr; c->prep_hash = hsh;
    }
    prof_mark_at(c, hs, k.prof_call, 1);
    rc = (a.mode == MODE_SAMPSON)
             ? f_solve_launch<MODE_SAMPSON>(c, hs, plan, a.pts64, idx, a.solver, a.sample_seed, (unsigned)a.first_pair)
             : f_solve_launch<MODE_EPI_MAX>(c, hs, plan, a.pts64, idx, a.solver, a.sample_seed, (unsigned)a.first_pair);
    if (rc) return rc;
    prof_mark_at(c, hs, k.prof_call, 2);
    return RG_OK;
}

static int f_pass_score(Ctx* c, cudaStream_t st, PassCtl& k) {
    prof_mark_at(c, st, k.prof_call, Ctx::kProfScoreStart);
    const int rc = (k.a.mode == MODE_SAMPSON) ? f_score_only<MODE_SAMPSON>(c, st, k) : f_score_only<MODE_EPI_MAX>(c, st, k);
    prof_mark_at(c, st, k.prof_call, 3);
    return rc;
}

static int f_pass_cands(Ctx* c, cudaStream_t ts, PassCtl& k, bool beside_scorer) {
    return (k.a.mode == MODE_SAMPSON) ? f_bnd_cands<MODE_SAMPSON>(c, ts, k, beside_scorer)
                                      : f_bnd_cands<MODE_EPI_MAX>(c, ts, k, beside_scorer);
}

static int f_pass_sweep(Ctx* c, cudaStream_t st, PassCtl& k) {
    return (k.a.mode == MODE_SAMPSON) ? f_bnd_sweep<MODE_SAMPSON>(c, st, k) : f_bnd_sweep<MODE_EPI_MAX>(c, st, k);
}

static int f_pass_tail(Ctx* c, cudaStream_t ts, PassCtl& k, bool beside_scorer) {
    const FCall& a = k.a;
    const int stage = a.bounded ? STAGE_FALLBACK : STAGE_MAIN;
    int rc = (a.mode == MODE_SAMPSON) ? f_fixup_launch<MODE_SAMPSON>(c, ts, k, beside_scorer, stage)
                                      : f_fixup_launch<MODE_EPI_MAX>(c, ts, k, beside_scorer, stage);
    if (rc) return rc;
    if (a.bounded && k.scored) {
        bnd_merge<<<k.plan.P, 256, 0, ts>>>(k.s.counts, k.s.sfx_f, (const PairInfo*)c->pair_info.ptr, k.s.mark,
                                            !k.plan.bound_prefix);
        c->last_stats[7] += 1;
        RG_CUDA(cudaGetLastError());
    }
    if (!a.bounded) prof_mark_at(c, ts, k.prof_call, 4);
    if ((rc = f_select_launch(c, ts, k.plan, k.s, a.pts64, a.thr, a.mode, a.tie_mode, a.mask, a.best_F, a.best_idx, a.best_count,
                              a.keys)))
        return rc;
    prof_mark_at(c, ts, k.prof_call, 5);
    return RG_OK;
}

// the pass's downloads, queued on stream ts behind its tail: per-hypothesis results, then `done` and the copy behind it
static int f_pass_downloads(Ctx* c, cudaStream_t ts, const PassCtl& k) {
    const size_t H = (size_t)k.plan.Htot;
    if (k.out_counts && H) RG_CUDA(cudaMemcpyAsync(k.out_counts, c->counts_ptr, sizeof(int) * H, cudaMemcpyDeviceToHost, ts));
    if (k.out_F_all && H) RG_CUDA(cudaMemcpyAsync(k.out_F_all, c->F64.ptr, sizeof(double) * 9 * H, cudaMemcpyDeviceToHost, ts));
    if (k.out_flags && H) RG_CUDA(cudaMemcpyAsync(k.out_flags, c->flags.ptr, H, cudaMemcpyDeviceToHost, ts));
    if (!k.done) return RG_OK;
    RG_CUDA(cudaEventRecord(k.done, ts));
    if (k.out_stream && k.out_bytes) {
        RG_CUDA(cudaStreamWaitEvent(k.out_stream, k.done, 0));
        RG_CUDA(cudaMemcpyAsync(k.out_dst, k.out_src, k.out_bytes, cudaMemcpyDeviceToHost, k.out_stream));
    }
    return RG_OK;
}

// passes one after the other, everything on the caller's stream in the current workspace set
static int f_run_serial(Ctx* c, cudaStream_t st, std::vector<PassCtl>& jobs) {
    int rc;
    if (c->tail_carve_max > 0 && (rc = tail_carveout(c, false))) return rc;
    for (PassCtl& k : jobs) {
        if (k.ready) RG_CUDA(cudaStreamWaitEvent(st, k.ready, 0));
        if ((rc = f_pass_head(c, st, k)) || (rc = f_pass_score(c, st, k))) return rc;
        if (k.a.bounded && ((rc = f_pass_cands(c, st, k, false)) || (rc = f_pass_sweep(c, st, k)))) return rc;
        if ((rc = f_pass_tail(c, st, k, false)) || (rc = f_pass_downloads(c, st, k))) return rc;
    }
    return RG_OK;
}

// Several passes, software-pipelined over the caller's stream and a side stream.  The full sweep uses two workspace sets:
//
//   caller's stream :            score(0)            score(1)            score(2)         ...      join
//   side stream     :  head(0)   head(1)   tail(0)   head(2)   tail(1)   head(3)   tail(2) ...
//
// The caller's stream runs the scorers back to back; the side stream's kernels run BESIDE them: the tail of pass k and the head
// of pass k+2 need the same workspace set, which the side stream's own order serialises.  head(k+1) is queued before tail(k)
// (tail(k) has to wait for score(k), head(k+1) has not).
//
// The bounded sweep uses THREE workspace sets (pass k lives until its tail, which follows the prefix stage of pass k+1 and its
// own candidate stage):
//
//   caller's stream :  S1(0)          S1(1)  S3+FB(0)          S1(2)  S3+FB(1)          S1(3) ...  S3+FB(n-1)        join
//   side stream     :  head(0) head(1)  cands(0) head(2)  cands(1) tail(0) head(3)  cands(2) tail(1) head(4) ...  tail(n-1)
//
// S1 = prefix stage A, cands = its fix-up + bnd_select, S3+FB = candidate stage, its fix-up, bnd_extend, bnd_live_plan,
// prefix stage B, bnd_check, bnd_live_plan and the fallback stage, tail = fallback fix-up, bnd_merge, selection, masks.
// The caller's stream only waits between S3 and FB for the candidate stage's fix-up, bnd_extend, the two table kernels
// and bnd_check (small one-CTA-per-pair launches; stage B itself is a short full-grid scorer of a few hundred hypotheses
// per pair); everything else on the side stream runs beside a scorer.
// head(k+3) reuses pass k's set and is queued behind tail(k) on the side stream.
//
// Either way the caller's stream ends behind the last tail (join), and the current set is the last pass's (counts_ptr / F64 /
// flags of rg_f_last_hypotheses_dev and the prepared points).
static int f_run_piped(Ctx* c, cudaStream_t st, std::vector<PassCtl>& jobs) {
    const int n = (int)jobs.size();
    const bool bounded = jobs[0].a.bounded;
    int rc;
    if ((rc = pipe_setup(c)) || (rc = tail_carveout(c, true))) return rc;
    cudaStream_t side = c->tail_stream;
    RG_CUDA(cudaEventRecord(c->pipe_gate, st));       // the side stream may not overtake what the caller queued before the call
    RG_CUDA(cudaStreamWaitEvent(side, c->pipe_gate, 0));
    for (int k = 0; k < n; ++k) jobs[k].slot = (c->ws_slot + 1 + k) % (bounded ? 3 : 2);
    auto head = [&](int k) -> int {                   // side stream
        PassCtl& j = jobs[k];
        ws_use(c, j.slot);
        if (j.ready) RG_CUDA(cudaStreamWaitEvent(side, j.ready, 0));
        int r = f_pass_head(c, side, j);
        if (r) return r;
        RG_CUDA(cudaEventRecord(c->head_done[j.slot], side));
        return RG_OK;
    };
    auto score = [&](int k) -> int {                  // caller's stream
        PassCtl& j = jobs[k];
        RG_CUDA(cudaStreamWaitEvent(st, c->head_done[j.slot], 0));
        ws_use(c, j.slot);
        int r = f_pass_score(c, st, j);
        if (r) return r;
        RG_CUDA(cudaEventRecord(c->score_done[j.slot], st));
        return RG_OK;
    };
    auto tail = [&](int k, cudaEvent_t gate, bool beside) -> int {      // side stream, behind `gate` of the caller's stream
        PassCtl& j = jobs[k];
        RG_CUDA(cudaStreamWaitEvent(side, gate, 0));
        ws_use(c, j.slot);
        int r = f_pass_tail(c, side, j, beside);
        return r ? r : f_pass_downloads(c, side, j);
    };
    if ((rc = head(0))) return rc;
    if (!bounded) {
        for (int k = 0; k < n; ++k) {
            if ((rc = score(k))) return rc;
            if (k + 1 < n && (rc = head(k + 1))) return rc;
            if ((rc = tail(k, c->score_done[jobs[k].slot], k + 1 < n))) return rc;
        }
    } else {
        auto sweep = [&](int k) -> int {              // caller's stream
            PassCtl& j = jobs[k];
            RG_CUDA(cudaStreamWaitEvent(st, c->cand_done[j.slot], 0));
            ws_use(c, j.slot);
            int r = f_pass_sweep(c, st, j);
            if (r) return r;
            RG_CUDA(cudaEventRecord(c->sweep_done[j.slot], st));
            return RG_OK;
        };
        if (n > 1 && (rc = head(1))) return rc;
        for (int k = 0; k < n; ++k) {
            PassCtl& j = jobs[k];
            if ((rc = score(k))) return rc;
            if (k > 0 && (rc = sweep(k - 1))) return rc;
            RG_CUDA(cudaStreamWaitEvent(side, c->score_done[j.slot], 0));
            ws_use(c, j.slot);
            if ((rc = f_pass_cands(c, side, j, k + 1 < n))) return rc;
            RG_CUDA(cudaEventRecord(c->cand_done[j.slot], side));
            if (k > 0 && (rc = tail(k - 1, c->sweep_done[jobs[k - 1].slot], true))) return rc;
            if (k + 2 < n && (rc = head(k + 2))) return rc;
        }
        if ((rc = sweep(n - 1)) || (rc = tail(n - 1, c->sweep_done[jobs[n - 1].slot], false))) return rc;
    }
    RG_CUDA(cudaEventRecord(c->tail_done, side));
    RG_CUDA(cudaStreamWaitEvent(st, c->tail_done, 0));
    return RG_OK;
}

static int f_check_call(const FCall& a) {
    RG_CHECK_ARG(a.P >= 0 && a.pair_off && a.hyp_off, "bad pair table");
    RG_CHECK_ARG(a.thr > 0.0 && std::isfinite(a.thr), "thr must be positive and finite");
    RG_CHECK_ARG(a.mode == MODE_EPI_MAX || a.mode == MODE_SAMPSON, "unknown scoring mode");
    RG_CHECK_ARG(a.tie_mode == TIE_FIRST || a.tie_mode == TIE_REFERENCE, "unknown tie mode");
    RG_CHECK_ARG(a.solver == SOLVER_QR || a.solver == SOLVER_JACOBI, "unknown solver");
    RG_CHECK_ARG(a.score_path == SCORE_FP32_GUARDED || a.score_path == SCORE_FP64, "unknown scoring path");
    RG_CHECK_ARG((a.flags & ~(FLAG_REUSE_POINTS | FLAG_BOUNDED)) == 0, "unknown flag bits");
    RG_CHECK_ARG(a.hyp_first >= 0 && a.first_pair >= 0, "negative index base");
    if (a.P > 0) {
        RG_CHECK_ARG(a.pair_off[0] == 0 && a.hyp_off[0] == 0, "offset arrays must start at 0");
        for (int p = 0; p < a.P; ++p)
            RG_CHECK_ARG(a.pair_off[p + 1] >= a.pair_off[p] && a.hyp_off[p + 1] >= a.hyp_off[p],
                         "offset arrays must be non-decreasing");
    }
    return RG_OK;
}

static double pair_evals(const FCall& a, int p) {
    return (double)(a.pair_off[p + 1] - a.pair_off[p]) * (double)(a.hyp_off[p + 1] - a.hyp_off[p]);
}

// pass boundaries: contiguous blocks of pairs with bounded evaluations / hypotheses (every pass holds at least one pair)
static void f_pass_bounds(const Ctx* c, const FCall& a, std::vector<int>& bounds) {
    const double budget = c->opt_pass_evals > 0 ? (double)c->opt_pass_evals : kDefaultPassEvals;
    bounds.clear();
    bounds.push_back(0);
    double ev = 0.0;
    long long hy = 0;
    for (int p = 0; p < a.P; ++p) {
        const double e = pair_evals(a, p);
        const long long h = a.hyp_off[p + 1] - a.hyp_off[p];
        if (p > bounds.back() && (ev + e > budget || hy + h > kMaxPassHyp || p - bounds.back() >= 32768)) {
            bounds.push_back(p);
            ev = 0.0; hy = 0;
        }
        ev += e; hy += h;
    }
    bounds.push_back(a.P);
}

// Sub-batches of the host entry point: the passes of f_pass_bounds, the first of them cut further when that hides a
// worthwhile part of the upload.  The scoring and upload times are estimated with the rates MEASURED on this context by
// earlier calls.  Every sub-batch is a sub-range of a pass of f_pass_bounds, and therefore one pass itself (its limits are
// monotone).  A plan may hold empty sub-batches.
static void f_host_batches(const Ctx* c, const FCall& a, double evals, double bytes_per_hyp, std::vector<int>& bounds) {
    const int P = a.P;
    f_pass_bounds(c, a, bounds);
    const double r_ev = c->rate_evals_per_s > 0.0 ? c->rate_evals_per_s : 1.5e12;       // until measured: round-1 figures
    const double r_up = c->rate_h2d_bytes_per_s > 0.0 ? c->rate_h2d_bytes_per_s : 5.0e10;
    // how many extra passes are affordable: each costs ~0.1 ms of small kernels; spend at most 1 % of the call on them
    const int levels = (int)std::min(5.0, std::floor(0.01 * (evals / r_ev) / 1.0e-4));
    if (levels >= 2 && c->opt_host_slices == 0 && !c->opt_profile) {
        // Large batch: nothing hides the upload of the FIRST pass (102 MB for 64 config-5 pairs: 2 ms at 55 GB/s, 17 ms
        // when eight ranks share the host link), so the first pass is cut into sub-passes of doubling size — 1/2^levels of
        // it first — each of which covers the upload of the next one.
        const int p_end = bounds[1];
        double first_evals = 0.0;
        for (int p = 0; p < p_end; ++p) first_evals += pair_evals(a, p);
        std::vector<int> nb;
        nb.push_back(0);
        double target = first_evals / (double)(1 << levels), acc = 0.0;
        for (int p = 0; p < p_end; ++p) {
            acc += pair_evals(a, p);
            if (acc >= target && p + 1 < p_end) {
                nb.push_back(p + 1);
                acc = 0.0;
                target *= 2.0;
            }
        }
        for (size_t k = 1; k < bounds.size(); ++k) nb.push_back(bounds[k]);
        bounds.swap(nb);
    } else if (bounds.size() == 2 && P >= 2 && !c->opt_profile && c->opt_host_slices != 1) {
        // a batch that fits one pass: the first sub-batch is the smallest whose scoring time covers the upload of the rest
        int first = 1;
        double score_s = 0.0;
        auto rest_bytes = [&](int f) {
            return 32.0 * (double)(a.pair_off[P] - a.pair_off[f]) + bytes_per_hyp * (double)(a.hyp_off[P] - a.hyp_off[f]);
        };
        for (first = 1; first < P; ++first) {
            score_s += pair_evals(a, first - 1) / r_ev;
            if (score_s >= rest_bytes(first) / r_up) break;
        }
        first = std::max(1, std::min(first, std::max(1, P / 2)));
        double sc = 0.0;
        for (int q = 0; q < first; ++q) sc += pair_evals(a, q) / r_ev;
        const double hidden_s = std::min(sc, rest_bytes(first) / r_up);
        int S = c->opt_host_slices > 0 ? c->opt_host_slices : (hidden_s > 1.5e-4 ? 2 : 1);     // a pass costs ~0.1 ms of small kernels
        S = std::max(1, std::min(S, P));
        if (S > 1) {
            bounds.clear();
            bounds.push_back(0);
            for (int k = 1; k <= S; ++k) bounds.push_back(first + (int)((long long)(P - first) * (k - 1) / (S - 1)));
        }
    }
}

// sub-call of pairs [p0, p1) with offsets rebased to the pass
static FCall f_sub_call(const FCall& a, int p0, int p1, std::vector<int>& po, std::vector<int>& ho) {
    FCall s = a;
    const int Pk = p1 - p0;
    const size_t n0 = (size_t)a.pair_off[p0], h0 = (size_t)a.hyp_off[p0];
    po.resize(Pk + 1); ho.resize(Pk + 1);
    for (int q = 0; q <= Pk; ++q) { po[q] = a.pair_off[p0 + q] - (int)n0; ho[q] = a.hyp_off[p0 + q] - (int)h0; }
    s.P = Pk;
    s.pair_off = po.data(); s.hyp_off = ho.data();
    s.pts64 = a.pts64 ? a.pts64 + 4 * n0 : nullptr;
    s.idx = a.idx ? a.idx + 8 * h0 : nullptr;
    s.first_pair = a.first_pair + p0;
    s.best_idx = a.best_idx + p0; s.best_count = a.best_count + p0; s.best_F = a.best_F + 9 * (size_t)p0;
    s.mask = a.mask ? a.mask + n0 : nullptr;
    s.keys = a.keys ? a.keys + p0 : nullptr;
    return s;
}

// Runs the passes of one F call (one job per pass, from f_sub_call) and owns the call's statistics (rg_get_last_stats,
// rg_f_last_bounded_stats).  Several passes are pipelined (f_run_piped, option 10) unless a pass wants its per-hypothesis
// results; otherwise they run one after the other on the caller's stream, so a single-pass call never swaps sets or
// streams: it stays capturable in a CUDA graph and RG_FLAG_REUSE_POINTS finds its prepared points.  Asynchronous with
// respect to the host except for the PairInfo staging; the caller's stream ends behind every pass, i.e. the call keeps the
// stream semantics of a plain sequence of launches.
// (Cutting the first / last pass into 1/8 .. 1/2 pieces to shorten the exposed head and tail was tried: the smaller passes
// cost the scorer as much as they save — 512-pair sweep 126.96 -> 127.32 ms resident, full sweep end to end 987.1 -> 988.6
// ms; profiles/r02_taper.txt.)
static int f_run_passes(Ctx* c, cudaStream_t st, bool bounded, std::vector<PassCtl>& jobs) {
    c->last_passes = (int)jobs.size();                // (the empty sub-batches of a host call count, and run nothing)
    jobs.erase(std::remove_if(jobs.begin(), jobs.end(), [](const PassCtl& j) { return j.a.P == 0; }), jobs.end());
    const bool piped = jobs.size() > 1 && c->opt_pipeline &&
                       std::none_of(jobs.begin(), jobs.end(), [](const PassCtl& j) { return j.wants_hypotheses(); });
    const size_t stats_bytes = sizeof(unsigned long long) * 8, bnd_bytes = sizeof(unsigned long long) * 4;
    const int rc = [&]() -> int {
        int r;
        if ((r = ensure(c->stats, stats_bytes)) || (r = ensure_pinned(c->h_stats, stats_bytes)) ||
            (r = ensure(c->bnd_stats, bnd_bytes)))
            return r;
        RG_CUDA(cudaMemsetAsync(c->stats.ptr, 0, stats_bytes, st));
        RG_CUDA(cudaMemsetAsync(c->bnd_stats.ptr, 0, bnd_bytes, st));
        c->bnd_host_evals = 0;
        c->bnd_bound_evals = 0;
        c->last_bounded = bounded;
        c->last_stats[7] = 0;
        if ((r = piped ? f_run_piped(c, st, jobs) : f_run_serial(c, st, jobs))) return r;
        RG_CUDA(cudaMemcpyAsync(c->h_stats.ptr, c->stats.ptr, stats_bytes, cudaMemcpyDeviceToHost, st));
        return RG_OK;
    }();
    if (rc) {                                         // leave nothing in flight behind an error return
        cudaStreamSynchronize(st);
        if (piped && c->tail_stream) cudaStreamSynchronize(c->tail_stream);
        for (const PassCtl& j : jobs) {
            if (j.ready) cudaEventSynchronize(j.ready);       // (the host entry point's uploads)
            if (j.out_stream) cudaStreamSynchronize(j.out_stream);
        }
    }
    return rc;
}

static int f_ransac_dev(Ctx* c, cudaStream_t st, const FCall& a_in) {
    int rc = f_check_call(a_in);
    if (rc) return rc;
    FCall a = a_in;
    a.bounded = a.bounded && a.score_path == SCORE_FP32_GUARDED;      // (the FP64 path always scores everything)
    RG_CUDA(cudaSetDevice(c->device));
    std::vector<int> bounds;
    f_pass_bounds(c, a, bounds);
    const int n_pass = a.P > 0 ? (int)bounds.size() - 1 : 0;
    RG_CHECK_ARG(n_pass <= 1 || !(a.flags & FLAG_REUSE_POINTS), "RG_FLAG_REUSE_POINTS needs a call that fits one pass");
    std::vector<PassCtl> jobs(n_pass);
    for (int k = 0; k < n_pass; ++k) jobs[k].a = f_sub_call(a, bounds[k], bounds[k + 1], jobs[k].po, jobs[k].ho);
    return f_run_passes(c, st, a.bounded, jobs);
}

}  // namespace rg

using namespace rg;

extern "C" {

int rg_f_ransac_dev2(void* ctx, void* stream, int P, const double* pts64_dev, const int* pair_off_host, const int* idx_dev,
                     const int* hyp_off_host, double thr, int mode, int tie_mode, int solver, int score_path, int flags,
                     unsigned long long sample_seed, int first_pair_id, int hyp_index_base, int* best_idx_dev,
                     int* best_count_dev, double* best_F_dev, unsigned char* mask_dev, unsigned long long* key_dev) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(best_idx_dev && best_count_dev && best_F_dev, "output pointers are null");
    FCall a;
    a.P = P; a.pts64 = pts64_dev; a.pair_off = pair_off_host; a.idx = idx_dev; a.hyp_off = hyp_off_host;
    a.thr = thr; a.mode = mode; a.tie_mode = tie_mode; a.solver = solver; a.score_path = score_path; a.flags = flags;
    a.sample_seed = sample_seed; a.first_pair = first_pair_id; a.hyp_first = hyp_index_base;
    a.bounded = (flags & FLAG_BOUNDED) != 0 && ((Ctx*)ctx)->opt_bounded != 0;
    a.best_idx = best_idx_dev; a.best_count = best_count_dev; a.best_F = best_F_dev; a.mask = mask_dev; a.keys = key_dev;
    return f_ransac_dev((Ctx*)ctx, (cudaStream_t)stream, a);
}

int rg_f_ransac_dev(void* ctx, void* stream, int P, const double* pts64_dev, const int* pair_off_host, const int* idx_dev,
                    const int* hyp_off_host, double thr, int mode, int tie_mode, int solver, int score_path,
                    int* best_idx_dev, int* best_count_dev, double* best_F_dev, unsigned char* mask_dev) {
    RG_CHECK_ARG(P == 0 || hyp_off_host == nullptr || hyp_off_host[P] == 0 || idx_dev != nullptr,
                 "idx_dev is null (use rg_f_ransac_dev2 for device-drawn samples)");
    return rg_f_ransac_dev2(ctx, stream, P, pts64_dev, pair_off_host, idx_dev, hyp_off_host, thr, mode, tie_mode, solver,
                            score_path, 0, 0ull, 0, 0, best_idx_dev, best_count_dev, best_F_dev, mask_dev, nullptr);
}

// the k = 8 sample index sets rg_f_ransac_*2 draws for (seed, first_pair_id, hyp_index_base) when idx is NULL: lets a caller
// (or the oracle) see exactly the samples a seeded call used.  n_points_host[p] points, hypotheses CSR hyp_off_host.
int rg_sample_indices_dev(void* ctx, void* stream, int P, const int* n_points_host, const int* hyp_off_host, int k,
                          unsigned long long seed, int first_pair_id, int hyp_index_base, int* idx_out_dev) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(P >= 0 && n_points_host && hyp_off_host, "bad pair table");
    RG_CHECK_ARG(k == 6 || k == 7 || k == 8, "sample size k must be 6, 7 or 8");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    if (P == 0 || hyp_off_host[P] == 0) return RG_OK;
    RG_CHECK_ARG(idx_out_dev != nullptr, "idx_out_dev is null");
    std::vector<int> po(P + 1, 0);
    for (int p = 0; p < P; ++p) {
        RG_CHECK_ARG(n_points_host[p] >= k || hyp_off_host[p + 1] == hyp_off_host[p], "a pair with hypotheses needs at least k points");
        po[p + 1] = po[p] + n_points_host[p];
    }
    FPlan plan;
    int rc = f_plan(c, st, P, po.data(), hyp_off_host, plan, 1, nullptr, hyp_index_base);
    if (rc) return rc;
    const PairInfo* pi = (const PairInfo*)c->pair_info.ptr;
    const int H = (int)plan.Htot, grid = ceil_div(H, 256);
    if (k == 8) sample_indices_kernel<8><<<grid, 256, 0, st>>>(pi, P, H, seed, (unsigned)first_pair_id, idx_out_dev);
    else if (k == 7) sample_indices_kernel<7><<<grid, 256, 0, st>>>(pi, P, H, seed, (unsigned)first_pair_id, idx_out_dev);
    else sample_indices_kernel<6><<<grid, 256, 0, st>>>(pi, P, H, seed, (unsigned)first_pair_id, idx_out_dev);
    c->prep_pts = nullptr;              // the PairInfo table of a prepared pass was overwritten
    RG_CUDA(cudaGetLastError());
    return RG_OK;
}

// synthetic two-view correspondences of BASELINE configs 3-5, generated on the device (philox.cuh).
// cams_host: n_cams x 12 camera matrices; bbox6_host: lo/hi of the world box per axis.
int rg_synth_two_view_dev(void* ctx, void* stream, int P, int first_pair_id, int N, const double* cams_host, int n_cams,
                          const double* bbox6_host, unsigned long long seed_base, double outlier_frac, double sigma_px,
                          double width, double height, double* pts_out_dev, int* cam_pair_out_dev) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(P >= 0 && P <= 65535 && N >= 0 && n_cams >= 2 && cams_host && bbox6_host, "bad arguments");
    RG_CHECK_ARG(outlier_frac >= 0.0 && outlier_frac <= 1.0, "outlier_frac must be in [0, 1]");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    if (P == 0 || N == 0) return RG_OK;
    RG_CHECK_ARG(pts_out_dev != nullptr, "pts_out_dev is null");
    int rc;
    if ((rc = ensure(c->geom, sizeof(double) * 12 * (size_t)n_cams))) return rc;
    RG_CUDA(cudaMemcpyAsync(c->geom.ptr, cams_host, sizeof(double) * 12 * (size_t)n_cams, cudaMemcpyHostToDevice, st));
    SynthParams prm;
    for (int k = 0; k < 6; ++k) prm.bbox[k] = bbox6_host[k];
    prm.sigma_px = sigma_px; prm.width = width; prm.height = height;
    prm.n_out = (int)std::floor(outlier_frac * (double)N + 0.5);
    prm.n_cams = n_cams;
    const int nbx = std::max(1, std::min(64, ceil_div(N, 256)));
    synth_two_view_kernel<<<dim3(nbx, P), 256, 0, st>>>((const double*)c->geom.ptr, prm, N, seed_base, (unsigned)first_pair_id,
                                                        (double4*)pts_out_dev, cam_pair_out_dev);
    RG_CUDA(cudaGetLastError());
    RG_CUDA(cudaStreamSynchronize(st));               // cams_host may be pageable: do not return before it was read
    return RG_OK;
}

// inlier mask (FP64 reference criterion, fun.py:315-317) of one caller-supplied F per pair; everything on the device
int rg_f_inlier_mask_dev(void* ctx, void* stream, int P, const double* pts64_dev, const int* pair_off_host, const double* F_dev,
                         double thr, int mode, unsigned char* mask_dev) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(P >= 0 && pair_off_host, "bad pair table");
    RG_CHECK_ARG(thr > 0.0 && std::isfinite(thr), "thr must be positive and finite");
    RG_CHECK_ARG(mode == MODE_EPI_MAX || mode == MODE_SAMPSON, "unknown scoring mode");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    if (P == 0 || pair_off_host[P] == 0) return RG_OK;
    RG_CHECK_ARG(pts64_dev && F_dev && mask_dev, "null buffers");
    for (int p0 = 0; p0 < P; p0 += 64) {
        const int Pk = std::min(64, P - p0);
        MaskPairs mp;
        int maxn = 1;
        for (int q = 0; q <= Pk; ++q) mp.off[q] = pair_off_host[p0 + q];
        for (int q = 0; q < Pk; ++q) maxn = std::max(maxn, mp.off[q + 1] - mp.off[q]);
        const int nbx = std::max(1, std::min(c->sm_count * 2, ceil_div(maxn, 256 * 4)));
        f_mask_given<<<dim3(nbx, Pk), 256, 0, st>>>((const double4*)pts64_dev, mp, F_dev + 9 * (size_t)p0, thr, mode, mask_dev);
    }
    RG_CUDA(cudaGetLastError());
    return RG_OK;
}

// device pointers to the per-hypothesis results of the LAST call on this context (valid until the next call; a call that
// ran in several passes only keeps its last pass, and is refused here).  After a bounded sweep *counts_dev is NULL: the
// hypotheses it proved unable to win hold prefix counts only.
int rg_f_last_hypotheses_dev(void* ctx, const int** counts_dev, const double** F_all_dev, const unsigned char** flags_dev) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    Ctx* c = (Ctx*)ctx;
    RG_CHECK_ARG(c->last_passes <= 1, "the last call ran in several passes: per-hypothesis results are not retained");
    if (counts_dev) *counts_dev = c->last_bounded ? nullptr : (const int*)c->counts_ptr;
    if (F_all_dev) *F_all_dev = (const double*)c->F64.ptr;
    if (flags_dev) *flags_dev = (const unsigned char*)c->flags.ptr;
    return RG_OK;
}

// out[0] guard-band groups flagged, [1] band evaluations re-done in FP64, [2] decisions changed by the recheck,
// [3] hypotheses recounted in FP64 after a flag-list overflow, [4] hypotheses with a sample index out of range,
// [5] upload rate measured by the host entry point (MB/s, running average), [6] passes of the last call, [7] kernel launches of the last call.  Synchronises the stream.
int rg_get_last_stats(void* ctx, void* stream, long long* out8) {
    RG_CHECK_ARG(ctx != nullptr && out8 != nullptr, "null argument");
    Ctx* c = (Ctx*)ctx;
    RG_CUDA(cudaSetDevice(c->device));
    RG_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    for (int i = 0; i < 8; ++i) out8[i] = 0;
    if (c->h_stats.ptr) {
        const unsigned long long* s = (const unsigned long long*)c->h_stats.ptr;
        for (int i = 0; i < 6; ++i) out8[i] = (long long)s[i];
    }
    out8[5] = (long long)(c->rate_h2d_bytes_per_s * 1e-6);        // measured upload rate of the host entry point, MB/s
    out8[6] = c->last_passes;
    out8[7] = c->last_stats[7];
    return RG_OK;
}

// out[0] hypothesis x correspondence evaluations the last F call executed, [1] hypotheses it did not score in full (proved
// unable to reach their pair's maximum), [2] pairs whose bound failed and that were scored in full, [3] candidates per pair
// (0: the call ran the full sweep).  Synchronises the stream.
static int bnd_stats_read(Ctx* c, void* stream, unsigned long long (&d)[4]) {
    RG_CUDA(cudaSetDevice(c->device));
    RG_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    if (c->bnd_stats.ptr) RG_CUDA(cudaMemcpy(d, c->bnd_stats.ptr, sizeof(d), cudaMemcpyDeviceToHost));
    return RG_OK;
}

int rg_f_last_bounded_stats(void* ctx, void* stream, long long* out4) {
    RG_CHECK_ARG(ctx != nullptr && out4 != nullptr, "null argument");
    Ctx* c = (Ctx*)ctx;
    unsigned long long d[4] = {0, 0, 0, 0};
    int rc = bnd_stats_read(c, stream, d);
    if (rc) return rc;
    out4[0] = c->bnd_bound_evals + (long long)d[3] + c->bnd_host_evals + (long long)d[0];
    out4[1] = (long long)d[1];
    out4[2] = (long long)d[2];
    out4[3] = c->last_bounded ? c->opt_bounded_k : 0;
    return RG_OK;
}

// out[0] evaluations of the last F call's bound-only prefix stages A and B (upper-bound counts; stage B's depend on the
// data and are counted on the device), [1] evaluations of its guarded scorer (exact prefix, candidate and fallback stages,
// or the full sweep); their sum is out4[0] of rg_f_last_bounded_stats.  Synchronises the stream.
int rg_f_last_bounded_evals(void* ctx, void* stream, long long* out2) {
    RG_CHECK_ARG(ctx != nullptr && out2 != nullptr, "null argument");
    Ctx* c = (Ctx*)ctx;
    unsigned long long d[4] = {0, 0, 0, 0};
    int rc = bnd_stats_read(c, stream, d);
    if (rc) return rc;
    out2[0] = c->bnd_bound_evals + (long long)d[3];
    out2[1] = c->bnd_host_evals + (long long)d[0];
    return RG_OK;
}

// Host-buffer entry point.  The pairs are processed in sub-batches of one pass each (f_host_batches).  All uploads are
// queued on a second stream (one event per sub-batch), the kernels of sub-batch k wait only for their own inputs, so the
// upload of sub-batch k+1 overlaps the scoring of sub-batch k (needs pinned host buffers to actually overlap; pageable ones
// are still correct).  Results are identical to a single batch: pairs are independent.  idx == NULL: samples drawn on the
// device from sample_seed.
int rg_f_ransac_host2(void* ctx, void* stream, int P, const double* pts64, const int* pair_off, const int* idx,
                      const int* hyp_off, double thr, int mode, int tie_mode, int solver, int score_path,
                      unsigned long long sample_seed, int first_pair_id, int* best_idx, int* best_count, double* best_F,
                      unsigned char* mask, int* counts, double* F_all, unsigned char* flags) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(best_idx && best_count && best_F, "output pointers are null");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    FCall a;
    a.P = P; a.pair_off = pair_off; a.hyp_off = hyp_off; a.thr = thr; a.mode = mode; a.tie_mode = tie_mode;
    a.solver = solver; a.score_path = score_path; a.sample_seed = sample_seed; a.first_pair = first_pair_id;
    a.bounded = counts == nullptr && c->opt_bounded != 0 && score_path == SCORE_FP32_GUARDED;
    int rc = f_check_call(a);
    if (rc) return rc;
    RG_CUDA(cudaSetDevice(c->device));
    if (P == 0) return RG_OK;
    const size_t Ntot = (size_t)pair_off[P], Htot = (size_t)hyp_off[P];
    RG_CHECK_ARG(Ntot == 0 || pts64, "pts64 is null");
    const bool seeded = idx == nullptr;
    if ((rc = ensure(c->d_in_a, sizeof(double) * 4 * std::max<size_t>(Ntot, 1)))) return rc;
    if (!seeded && (rc = ensure(c->d_in_b, sizeof(int) * 8 * std::max<size_t>(Htot, 1)))) return rc;
    if ((rc = ensure(c->d_out_a, sizeof(int) * 2 * (size_t)P))) return rc;
    if ((rc = ensure(c->d_out_b, sizeof(double) * 9 * (size_t)P))) return rc;
    if (mask && (rc = ensure(c->d_out_c, std::max<size_t>(Ntot, 1)))) return rc;

    const double bytes_per_hyp = seeded ? 0.0 : 32.0;
    double evals = 0.0;
    for (int p = 0; p < P; ++p) evals += pair_evals(a, p);
    std::vector<int> bounds;
    f_host_batches(c, a, evals, bytes_per_hyp, bounds);
    const int S = (int)bounds.size() - 1;
    if (!c->copy_stream) RG_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    if (!c->copy_gate) RG_CUDA(cudaEventCreateWithFlags(&c->copy_gate, cudaEventDisableTiming));
    while ((int)c->pass_ready.size() < S) {
        cudaEvent_t e;
        RG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        c->pass_ready.push_back(e);
    }
    for (int k = 0; k < 4; ++k)
        if (!c->rate_ev[k]) RG_CUDA(cudaEventCreate(&c->rate_ev[k]));
    // the inlier masks of pass k travel back on a third stream while pass k+1 is scored (205 MB for the config-5 sweep:
    // 3.7 ms at the end of the call otherwise)
    const bool stream_masks = mask != nullptr && S > 1;
    if (stream_masks) {
        if (!c->d2h_stream) RG_CUDA(cudaStreamCreateWithFlags(&c->d2h_stream, cudaStreamNonBlocking));
        if (!c->d2h_done) RG_CUDA(cudaEventCreateWithFlags(&c->d2h_done, cudaEventDisableTiming));
        while ((int)c->pass_done.size() < S) {
            cudaEvent_t e;
            RG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            c->pass_done.push_back(e);
        }
    }

    double* d_pts = (double*)c->d_in_a.ptr;
    int* d_ix = seeded ? nullptr : (int*)c->d_in_b.ptr;
    cudaStream_t cs = S > 1 ? c->copy_stream : st;
    if (S > 1) {                                      // uploads may not overtake earlier work queued on the caller's stream
        RG_CUDA(cudaEventRecord(c->copy_gate, st));
        RG_CUDA(cudaStreamWaitEvent(cs, c->copy_gate, 0));
    }
    RG_CUDA(cudaEventRecord(c->rate_ev[0], cs));
    for (int k = 0; k < S; ++k) {
        const int p0 = bounds[k], p1 = bounds[k + 1];
        const size_t n0 = (size_t)pair_off[p0], n1 = (size_t)pair_off[p1], h0 = (size_t)hyp_off[p0], h1 = (size_t)hyp_off[p1];
        if (n1 > n0) RG_CUDA(cudaMemcpyAsync(d_pts + 4 * n0, pts64 + 4 * n0, sizeof(double) * 4 * (n1 - n0), cudaMemcpyHostToDevice, cs));
        if (!seeded && h1 > h0) RG_CUDA(cudaMemcpyAsync(d_ix + 8 * h0, idx + 8 * h0, sizeof(int) * 8 * (h1 - h0), cudaMemcpyHostToDevice, cs));
        if (S > 1) RG_CUDA(cudaEventRecord(c->pass_ready[k], cs));
    }
    RG_CUDA(cudaEventRecord(c->rate_ev[1], cs));
    RG_CUDA(cudaEventRecord(c->rate_ev[2], st));
    int* d_idx = (int*)c->d_out_a.ptr;
    int* d_cnt = d_idx + P;
    a.pts64 = d_pts; a.idx = d_ix;
    a.best_idx = d_idx; a.best_count = d_cnt; a.best_F = (double*)c->d_out_b.ptr;
    a.mask = mask ? (unsigned char*)c->d_out_c.ptr : nullptr;
    // one job per sub-batch: its head waits for its own upload, its mask download hangs on its tail
    std::vector<PassCtl> jobs(S);
    for (int k = 0; k < S; ++k) {
        PassCtl& j = jobs[k];
        const int p0 = bounds[k], p1 = bounds[k + 1];
        const size_t n0 = (size_t)pair_off[p0], h0 = (size_t)hyp_off[p0];
        j.a = f_sub_call(a, p0, p1, j.po, j.ho);
        if (S > 1) j.ready = c->pass_ready[k];
        if (stream_masks) {
            j.done = c->pass_done[k];
            j.out_stream = c->d2h_stream;
            j.out_dst = mask + n0; j.out_src = a.mask + n0; j.out_bytes = (size_t)pair_off[p1] - n0;
        }
        if (counts) j.out_counts = counts + h0;
        if (F_all) j.out_F_all = F_all + 9 * h0;
        if (flags) j.out_flags = flags + h0;
    }
    if ((rc = f_run_passes(c, st, a.bounded, jobs))) return rc;
    if (stream_masks) {                               // the caller's stream also waits for the mask downloads
        RG_CUDA(cudaEventRecord(c->d2h_done, c->d2h_stream));
        RG_CUDA(cudaStreamWaitEvent(st, c->d2h_done, 0));
    }
    RG_CUDA(cudaEventRecord(c->rate_ev[3], st));
    RG_CUDA(cudaMemcpyAsync(best_idx, d_idx, sizeof(int) * (size_t)P, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaMemcpyAsync(best_count, d_cnt, sizeof(int) * (size_t)P, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaMemcpyAsync(best_F, c->d_out_b.ptr, sizeof(double) * 9 * (size_t)P, cudaMemcpyDeviceToHost, st));
    if (mask && Ntot && !stream_masks) RG_CUDA(cudaMemcpyAsync(mask, c->d_out_c.ptr, Ntot, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaStreamSynchronize(st));
    {   // measured rates for the next call's sub-batch model (exponential average; uploads of < 1 MB say nothing)
        float ms_up = 0.f, ms_run = 0.f;
        const double up_bytes = 32.0 * (double)Ntot + bytes_per_hyp * (double)Htot;
        if (cudaEventElapsedTime(&ms_up, c->rate_ev[0], c->rate_ev[1]) == cudaSuccess && ms_up > 0.f && up_bytes > 1e6) {
            const double r = up_bytes / (ms_up * 1e-3);
            c->rate_h2d_bytes_per_s = c->rate_h2d_bytes_per_s > 0.0 ? 0.75 * c->rate_h2d_bytes_per_s + 0.25 * r : r;
        }
        if (cudaEventElapsedTime(&ms_run, c->rate_ev[2], c->rate_ev[3]) == cudaSuccess && ms_run > 0.f && evals > 1e9) {
            const double r = evals / (ms_run * 1e-3);
            c->rate_evals_per_s = c->rate_evals_per_s > 0.0 ? 0.75 * c->rate_evals_per_s + 0.25 * r : r;
        }
    }
    // sample indices are validated where they are read (the solver clamps them and sets flag bit 2): no host pass over idx
    if (c->h_stats.ptr && ((const unsigned long long*)c->h_stats.ptr)[4] != 0) {
        set_error("invalid argument: %llu hypotheses have a sample index outside [0, N) of their pair",
                  ((const unsigned long long*)c->h_stats.ptr)[4]);
        return RG_ERR_ARG;
    }
    return RG_OK;
}

int rg_f_ransac_host(void* ctx, void* stream, int P, const double* pts64, const int* pair_off, const int* idx,
                     const int* hyp_off, double thr, int mode, int tie_mode, int solver, int score_path, int* best_idx,
                     int* best_count, double* best_F, unsigned char* mask, int* counts, double* F_all, unsigned char* flags) {
    RG_CHECK_ARG(P <= 0 || hyp_off == nullptr || hyp_off[P] == 0 || idx != nullptr,
                 "idx is null (use rg_f_ransac_host2 for device-drawn samples)");
    return rg_f_ransac_host2(ctx, stream, P, pts64, pair_off, idx, hyp_off, thr, mode, tie_mode, solver, score_path, 0ull, 0,
                             best_idx, best_count, best_F, mask, counts, F_all, flags);
}

// Stage entry point: score caller-supplied fundamental matrices (H x 9, row-major, pixel frame) on one pair.
int rg_epi_score_count_host(void* ctx, void* stream, int N, const double* pts64, int H, const double* F_all, double thr,
                            int mode, int score_path, int* counts) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(N >= 0 && H >= 0 && counts, "bad sizes / null output");
    RG_CHECK_ARG(thr > 0.0 && std::isfinite(thr), "thr must be positive and finite");
    RG_CHECK_ARG(mode == MODE_EPI_MAX || mode == MODE_SAMPSON, "unknown scoring mode");
    RG_CHECK_ARG(score_path == SCORE_FP32_GUARDED || score_path == SCORE_FP64 || score_path == SCORE_FP32_BOUND,
                 "unknown scoring path");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    if (H == 0) return RG_OK;
    const int pair_off[2] = {0, N}, hyp_off[2] = {0, H};
    FPlan plan;
    int bps = 1, rc = score_blocks_per_sm<EpiPolicy<MODE_EPI_MAX>>(&bps);
    if (rc) return rc;
    if ((rc = f_plan(c, st, 1, pair_off, hyp_off, plan, bps))) return rc;
    if ((rc = f_workspace(c, plan))) return rc;
    ScoreState s;
    if ((rc = score_state_layout(c, 1, H, 8, s))) return rc;
    if ((rc = ensure(c->d_in_a, sizeof(double) * 4 * std::max<size_t>((size_t)N, 1)))) return rc;
    if (N) RG_CUDA(cudaMemcpyAsync(c->d_in_a.ptr, pts64, sizeof(double) * 4 * (size_t)N, cudaMemcpyHostToDevice, st));
    RG_CUDA(cudaMemcpyAsync(c->F64.ptr, F_all, sizeof(double) * 9 * (size_t)H, cudaMemcpyHostToDevice, st));
    c->last_stats[7] = 0;
    c->last_passes = 1;
    c->prep_pts = nullptr;
    RG_CUDA(cudaMemsetAsync(c->state.ptr, 0, s.bytes, st));
    RG_CUDA(cudaMemsetAsync(c->stats.ptr, 0, sizeof(unsigned long long) * 8, st));
    if ((rc = f_prepare(c, st, plan, s, (const double*)c->d_in_a.ptr, thr))) return rc;
    const PairInfo* pi = (const PairInfo*)c->pair_info.ptr;
    const PairFrame* fr = (const PairFrame*)c->pair_frame.ptr;
    if (mode == MODE_SAMPSON)
        f_make_hyp32<MODE_SAMPSON><<<ceil_div(H, 256), 256, 0, st>>>((const double*)c->F64.ptr, pi, fr, 1, H, (Hyp32*)c->hyp32.ptr);
    else
        f_make_hyp32<MODE_EPI_MAX><<<ceil_div(H, 256), 256, 0, st>>>((const double*)c->F64.ptr, pi, fr, 1, H, (Hyp32*)c->hyp32.ptr);
    c->last_stats[7] += 1;
    rc = (mode == MODE_SAMPSON) ? f_score_launch<MODE_SAMPSON>(c, st, plan, s, (const double*)c->d_in_a.ptr, thr, score_path)
                                : f_score_launch<MODE_EPI_MAX>(c, st, plan, s, (const double*)c->d_in_a.ptr, thr, score_path);
    if (rc) return rc;
    RG_CUDA(cudaMemcpyAsync(c->h_stats.ptr, c->stats.ptr, sizeof(unsigned long long) * 8, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaMemcpyAsync(counts, s.counts, sizeof(int) * (size_t)H, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaStreamSynchronize(st));
    return RG_OK;
}

// Stage entry point: 8-point solve only.  idx is (H, 8) indices into the N points.
int rg_f8pt_solve_host(void* ctx, void* stream, int N, const double* pts64, int H, const int* idx, int solver, double* F_all,
                       unsigned char* flags) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(N >= 8 && H >= 0 && pts64 && F_all, "need N >= 8 and non-null buffers");
    RG_CHECK_ARG(solver == SOLVER_QR || solver == SOLVER_JACOBI, "unknown solver");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    if (H == 0) return RG_OK;
    RG_CHECK_ARG(idx != nullptr, "idx is null");
    const int pair_off[2] = {0, N}, hyp_off[2] = {0, H};
    FPlan plan;
    int bps = 1, rc = score_blocks_per_sm<EpiPolicy<MODE_EPI_MAX>>(&bps);
    if (rc) return rc;
    if ((rc = f_plan(c, st, 1, pair_off, hyp_off, plan, bps))) return rc;
    if ((rc = f_workspace(c, plan))) return rc;
    ScoreState s;
    if ((rc = score_state_layout(c, 1, H, 8, s))) return rc;
    if ((rc = ensure(c->d_in_a, sizeof(double) * 4 * (size_t)N))) return rc;
    if ((rc = ensure(c->d_in_b, sizeof(int) * 8 * (size_t)H))) return rc;
    RG_CUDA(cudaMemcpyAsync(c->d_in_a.ptr, pts64, sizeof(double) * 4 * (size_t)N, cudaMemcpyHostToDevice, st));
    RG_CUDA(cudaMemcpyAsync(c->d_in_b.ptr, idx, sizeof(int) * 8 * (size_t)H, cudaMemcpyHostToDevice, st));
    c->last_stats[7] = 0;
    c->last_passes = 1;
    c->prep_pts = nullptr;
    RG_CUDA(cudaMemsetAsync(c->state.ptr, 0, s.bytes, st));
    if ((rc = f_prepare(c, st, plan, s, (const double*)c->d_in_a.ptr, 1.0))) return rc;
    if ((rc = f_solve_launch<MODE_EPI_MAX>(c, st, plan, (const double*)c->d_in_a.ptr, (const int*)c->d_in_b.ptr, solver)))
        return rc;
    RG_CUDA(cudaMemcpyAsync(F_all, c->F64.ptr, sizeof(double) * 9 * (size_t)H, cudaMemcpyDeviceToHost, st));
    if (flags) RG_CUDA(cudaMemcpyAsync(flags, c->flags.ptr, (size_t)H, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaStreamSynchronize(st));
    return RG_OK;
}

// lab3.fmatrix_residuals drop-in arithmetic: x, y are (2, N) row-major; out is (2, N) row-major.
int rg_fmatrix_residuals_host(void* ctx, void* stream, const double* F9, int N, const double* x, const double* y, double* out) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(F9 && N >= 0, "bad arguments");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    if (N == 0) return RG_OK;
    RG_CHECK_ARG(x && y && out, "null buffers");
    int rc;
    if ((rc = ensure(c->d_in_a, sizeof(double) * (4 * (size_t)N + 16)))) return rc;
    if ((rc = ensure(c->d_out_b, sizeof(double) * 2 * (size_t)N))) return rc;
    double* d = (double*)c->d_in_a.ptr;
    RG_CUDA(cudaMemcpyAsync(d, F9, sizeof(double) * 9, cudaMemcpyHostToDevice, st));
    RG_CUDA(cudaMemcpyAsync(d + 16, x, sizeof(double) * 2 * (size_t)N, cudaMemcpyHostToDevice, st));
    RG_CUDA(cudaMemcpyAsync(d + 16 + 2 * (size_t)N, y, sizeof(double) * 2 * (size_t)N, cudaMemcpyHostToDevice, st));
    f_residuals<<<std::max(1, std::min(c->sm_count * 4, ceil_div(N, 256))), 256, 0, st>>>(d, d + 16, d + 16 + 2 * (size_t)N, N,
                                                                                         (double*)c->d_out_b.ptr);
    RG_CUDA(cudaGetLastError());
    RG_CUDA(cudaMemcpyAsync(out, c->d_out_b.ptr, sizeof(double) * 2 * (size_t)N, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaStreamSynchronize(st));
    return RG_OK;
}

}  // extern "C"
