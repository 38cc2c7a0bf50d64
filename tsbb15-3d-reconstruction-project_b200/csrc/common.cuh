// Shared declarations for librg_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <cmath>
#include <vector>
#ifdef RG_DEBUG
#include <cassert>
// bounds / invariant checks of the debug build (librg_b200_debug.so, tests/test_gpu_debug_build.py): compute-sanitizer is closed
// on this pool, so the kernels carry their own assertions; a failed one traps and the next CUDA call reports it
#define RG_ASSERT(cond) assert(cond)
#else
#define RG_ASSERT(cond) ((void)0)
#endif

namespace rg {

// ---------------------------------------------------------------------------------------------
// status codes returned through the C ABI (0 = ok, negative = failure; text via rg_last_error())
// ---------------------------------------------------------------------------------------------
enum : int {
    RG_OK = 0,
    RG_ERR_CUDA = -1,        // a CUDA runtime call failed
    RG_ERR_ARG = -2,         // invalid argument (null pointer, negative size, sample size unsupported ...)
    RG_ERR_NO_DEVICE = -3,   // no sm_100 device / wrong architecture
};

void set_error(const char* fmt, ...);

#define RG_CUDA(call)                                                                       \
    do {                                                                                    \
        cudaError_t _e = (call);                                                            \
        if (_e != cudaSuccess) {                                                            \
            ::rg::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
            return ::rg::RG_ERR_CUDA;                                                       \
        }                                                                                   \
    } while (0)

#define RG_CHECK_ARG(cond, msg)                                   \
    do {                                                          \
        if (!(cond)) {                                            \
            ::rg::set_error("invalid argument: %s", msg);         \
            return ::rg::RG_ERR_ARG;                              \
        }                                                         \
    } while (0)

// ---------------------------------------------------------------------------------------------
// scoring criteria / selection modes (values are part of the ABI, see include/rg_b200.h)
// ---------------------------------------------------------------------------------------------
enum : int { MODE_EPI_MAX = 0, MODE_SAMPSON = 1 };
enum : int { TIE_FIRST = 0, TIE_REFERENCE = 1 };
enum : int { SOLVER_QR = 0, SOLVER_JACOBI = 1 };
enum : int { SCORE_FP32_GUARDED = 0, SCORE_FP64 = 1, SCORE_FP32_BOUND = 2 };

// ---------------------------------------------------------------------------------------------
// device-side records
// ---------------------------------------------------------------------------------------------
// Per hypothesis, FP32 scorer input: F~ = M1^T F M2 scaled to unit weighted abs-sum (f), the image-2 line normal
// l2 = (F~^T x~)[:2] ROTATED by the per-hypothesis angle that removes the x0 term of its second component
// (g = c, d, e, a, b:  l2x' = c x0 + d x1 + e,  l2y' = a x1 + b;  |l2'|^2 = |l2|^2, one FMA fewer per evaluation), and the
// rigorous rounding-error band G (see DESIGN.md "guard band") and the constant T of the bound-only prefix scorer
// (r^2 < T holds for every reference inlier, DESIGN.md section 4.2).  64 bytes, 16-byte aligned.
struct __align__(16) Hyp32 {
    float f[9];
    float g[5];
    float G;
    float T;
};
static_assert(sizeof(Hyp32) == 64, "Hyp32 layout");

// PnP hypothesis for the FP32 scorer: rows P0,P1,P2 (3x4 each, in the normalised frame), band G.
struct __align__(16) Pose32 {
    float p[12];
    float G;
    float pad0, pad1, pad2;
};
static_assert(sizeof(Pose32) == 64, "Pose32 layout");

constexpr int kSub = 8;             // points per guard-band flag (FP32 scorer); a thread collects 32 flags (256 points) per list append

// ---------------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------------
// largest p with off[p] <= i  (off is non-decreasing, off[0] = 0, off[P] = total)
__device__ __forceinline__ int find_segment(const int* __restrict__ off, int P, int i) {
    int lo = 0, hi = P;           // invariant: off[lo] <= i < off[hi]
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (off[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}

// ---- mbarrier + 1-D bulk TMA (cp.async.bulk -> SASS UBLKCP) ----------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// global -> shared bulk copy, completion signalled on the mbarrier (bytes % 16 == 0, 16-B aligned)
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ---------------------------------------------------------------------------------------------
// context: one per device, owns grow-only workspaces so steady-state calls never cudaMalloc
// ---------------------------------------------------------------------------------------------
struct Buffer {
    void*  ptr = nullptr;
    size_t cap = 0;
};

// Per image pair: integer geometry of the batch (filled on the host, uploaded once per pass).
struct PairInfo {
    int pt_off, n;             // offset / count in the caller's pts64 array (points)
    int pt_off32, n_pad;       // offset / count in the normalised FP32 copy (points, multiples of kSub)
    int hyp_off, H;            // offset / count in the hypothesis arrays
    int item_off, nsplit;      // scorer work items of this pair: [item_off, item_off + ceil(H/kHypPerBlock)*nsplit)
    int groups_per_split;      // kSub-point groups handled by one item
    int n_all;                 // PnP: all correspondences of the view (n = those that vote, n <= n_all); F path: n_all == n
    int hyp_first;             // index of the pair's first hypothesis inside the pair's full hypothesis set (hypothesis-split
                               // mode: this rank holds hypotheses [hyp_first, hyp_first + H) of the pair); 0 otherwise
    int g_base, g_end;         // window of kSub-point groups the scorer's items cover (absolute groups of the pair; a full
                               // sweep has [0, n_pad / kSub), the bounded sweep scores a prefix and a suffix, bounded.cuh)
    int pad0, pad1, pad2;
};
static_assert(sizeof(PairInfo) == 64, "PairInfo layout");

// Frame of the FP32 scorer, computed on the device from the pair's bounding box (f_normalise):
// x~ = (x - c1)/thr, y~ = (y - c2)/thr  => threshold is exactly 1, |x~|,|y~| <= B.  Kept apart from PairInfo so that a
// caller who scores several hypothesis sets against the same points (hypothesis-split mode) prepares the points once.
struct PairFrame {
    double c1x, c1y, c2x, c2y;
    double thr, B;
    double band_scale;         // multiplies the guard band (1 = the proven bound; option 9 widens it for experiments)
    double pad;
};

struct FPlan {
    int P = 0;
    long long Ntot = 0, Htot = 0, N32tot = 0;
    int n_items = 0;
    int maxN = 0, maxH = 0;
    double evals = 0.0;                  // sum_p n_p * H_p (bounded sweep: of prefix stage A)
    // bounded sweep (bounded.cuh): four tables per pass, [prefix stage A | candidate stage | fallback template |
    // stage-B template]
    bool bounded = false;
    bool bound_prefix = false;           // the prefix stage counts an upper bound (EpiBoundPolicy); later stages cover [0, G)
    int K = 0;                           // candidates per pair
    long long Ctot = 0;                  // candidates of the pass (sum_p min(K, H_p))
    long long Btot = 0;                  // room for stage B's records (sum_p H_p - min(K, H_p))
    int n_items_c = 0, n_items_f = 0;    // scorer items of the candidate stage / of the fallback with every pair marked
    int n_items_b = 0;                   // scorer items of stage B with every non-candidate live (0: one-step prefix)
    double evals_c = 0.0, evals_f = 0.0; // their evaluations (real correspondences)
};

struct Ctx {
    int device = 0;
    int sm_count = 0;
    // device workspaces (grow-only)
    Buffer pair_info, pair_frame, state, pts32, F64, hyp32, flags, flag_list, stats, best, tie_stats, bbox;
    Buffer bnd;                                    // bounded sweep: candidate records, compact -> global map, selection, fallback table
    // `state` = everything one cudaMemsetAsync clears per pass: [bbox keys][counts][work counter, list size][ovf bytes]
    int* counts_ptr = nullptr;                     // inside `state` (valid after f_state_layout of the current pass)
    unsigned char* ovf_ptr = nullptr;
    // Pass pipelining (F calls of several passes): the caller's stream runs the scorers back to back; the solver ("head") of
    // pass k+1 and the fix-up / selection / mask kernels ("tail") of pass k-1 run on a second stream BESIDE the scorer of pass k
    // — they are latency bound (23 % issue active) and one of their blocks fits next to the scorer's four on every SM.  The
    // per-pass workspaces exist two or three times (the bounded sweep keeps a pass alive across the next pass's prefix
    // stage); ws_use() moves the named buffers into spare[ws_slot] and those of the wanted set out of spare[slot], so all the
    // code keeps using c->F64, c->state, ... for "the set of the pass being queued".  spare[ws_slot] is always empty.
    struct PassSet { Buffer pair_info, pair_frame, state, pts32, F64, hyp32, flags, flag_list, best, tie_stats, bnd; } spare[3];
    cudaStream_t tail_stream = nullptr;
    cudaEvent_t head_done[3] = {nullptr, nullptr, nullptr};   // recorded on the side stream after the solver of the pass in set i
    cudaEvent_t score_done[3] = {nullptr, nullptr, nullptr};  // recorded on the caller's stream after the scorer of the pass in set i
    cudaEvent_t cand_done[3] = {nullptr, nullptr, nullptr};   // bounded sweep: side stream, candidates of the pass in set i chosen
    cudaEvent_t sweep_done[3] = {nullptr, nullptr, nullptr};  // bounded sweep: caller's stream, last scorer of the pass in set i
    cudaEvent_t tail_done = nullptr;                    // recorded on the side stream behind the last tail kernel of a run
    cudaEvent_t pipe_gate = nullptr;                    // recorded on the caller's stream before the side stream starts a run
    int tail_carve_max = -1;                            // shared-memory carve-out preference of the tail kernels: -1 never set, 0 default, 1 max
    int ws_slot = 0;                                    // which set is the current one
    int opt_pipeline = 1;                               // option 10: 0 = passes strictly one after the other on one stream
    // points prepared by the last F pass (RG_FLAG_REUSE_POINTS: score another hypothesis set against the same points)
    const void* prep_pts = nullptr; int prep_P = 0; long long prep_N = 0; double prep_thr = 0.0; unsigned long long prep_hash = 0;
    int last_passes = 0;                           // passes of the last RANSAC call (per-hypothesis results cover the last pass)
    // measured rates (exponential averages over the host-buffer calls) that size the first upload sub-batch
    double rate_evals_per_s = 0.0, rate_h2d_bytes_per_s = 0.0;
    cudaEvent_t rate_ev[4] = {nullptr, nullptr, nullptr, nullptr};
    bool pnp_rows_attr_set = false;                // dynamic shared memory limit of pnp_solve_rows raised on this device
    int opt_pnp_solver = 0;                        // option 7: 0 = Givens-QR + row Jacobi (default), 1 = 16-lane group Jacobi
    long long opt_list_cap = 0;                    // option 8 (test hook): capacity of the guard-band flag list in records (0 = automatic)
    double opt_band_scale = 1.0;                   // option 9: guard-band safety factor (>= 1)
    long long opt_pass_evals = 0;                  // option 6: evaluations per pass of a large batch (0 = default)
    int opt_bounded = 1;                           // option 12: F calls without per-hypothesis counts run the bounded sweep
    int opt_rho_milli = 450;                       // option 13: prefix share rho of the bounded sweep, in thousandths
    int opt_bounded_k = 512;                       // option 14: candidates per pair of the bounded sweep
    int opt_bound_prefix = 1;                      // option 15: 1 = bound-only prefix stage, 0 = exact (guarded + fix-up) prefix
    int opt_rho0_milli = 380;                      // option 16: share rho0 of the bound-only prefix stage A, in thousandths
    bool last_bounded = false;                     // the last F call ran the bounded sweep (its counts are not full counts)
    long long bnd_host_evals = 0;                  // guarded-scorer evaluations of its prefix and candidate stages (known on the host)
    long long bnd_bound_evals = 0;                 // evaluations of its bound-only prefix stages A (option 15 = 1)
    Buffer bnd_stats;                              // device: [0] fallback evaluations, [1] hypotheses not fully scored, [2] fallback pairs,
                                                   // [3] evaluations of the bound-only prefix stages B
    // peer-to-peer argmax exchange (hypothesis-split mode over NVLink), see p2p_api.cu
    void* p2p_local = nullptr; size_t p2p_bytes = 0; int p2p_rank = 0, p2p_world = 0; unsigned p2p_seq = 0;
    void* p2p_peer[16] = {nullptr};

    Buffer d_in_a, d_in_b, d_in_c;                 // device copies of host inputs (host-buffer entry points)
    Buffer d_out_a, d_out_b, d_out_c, d_out_d;     // device outputs of host-buffer entry points
    Buffer pose64, pose32, X32;                    // PnP path
    Buffer geom;                                   // two-view geometry: PairGeom table + CSR offsets
    Buffer geom_ws;                                // two-view initialisation: normalised points, cameras, picks
    Buffer gs_ws;                                  // gold-standard refinement: per-pair state, sums, cameras, points
    Buffer ba_ws;                                  // bundle adjustment: state, step, trial points, point blocks, camera system
    int opt_ba_cluster = 0;                        // option 3: CTAs in the cluster of the camera-system factorisation (0 = 8)
    int opt_gs_multi = 0;                          // option 5: 1 = gold standard always on the multi-kernel path (no gs_fused)
    int opt_ba_l2 = 0;                             // option 4: 1 = keep the camera system in L2 (ba_solve) even when it fits in DSMEM
    Buffer pr_ws;                                  // refinement of PnP poses: per-view state, per-block partials, offsets, weights
    int opt_pr_multi = 0;                          // option 11: 1 = PnP pose refinement always on the multi-CTA path
    Buffer h_pr_flags;                             // pinned: views still running after every iteration (host entry point)
    cudaEvent_t pr_iter_ev[2] = {nullptr, nullptr};
    Buffer h_ba_items;                             // pinned: work items of ba_blocks (blocks with a common point x segments)
    Buffer h_ba_flags;                             // pinned: the solver's `done` flag after every iteration (host entry point)
    cudaEvent_t ba_iter_ev[2] = {nullptr, nullptr};
    bool ba_attr_set = false;                      // dynamic shared memory limit of ba_solve raised on this device
    // pinned host staging for the small per-call tables and the statistics read-back
    Buffer h_stage[2], h_stats;                    // PairInfo staging, double buffered: the host plans pass k+1 while pass k runs
    cudaEvent_t staging_free[2] = {nullptr, nullptr};   // recorded after the H2D that reads h_stage[i]
    int stage_turn = 0;
    // the table of the last planned pass is still on the device: a repeated call skips staging and upload (plan.cuh)
    FPlan plan_cached; unsigned long long plan_hash = 0; const void* plan_table = nullptr; bool plan_valid = false;
    // host-buffer entry points: inputs are uploaded on a second stream in sub-batches so that the copy of sub-batch
    // k+1 overlaps the kernels of sub-batch k
    static constexpr int kMaxSlices = 8;
    cudaStream_t copy_stream = nullptr;
    std::vector<cudaEvent_t> pass_ready;           // one per pass of the host entry point: its inputs have arrived
    std::vector<cudaEvent_t> pass_done;            // ... its kernels have finished (the mask download of pass k overlaps pass k+1)
    cudaStream_t d2h_stream = nullptr;
    cudaEvent_t d2h_done = nullptr;
    cudaEvent_t copy_gate = nullptr;               // recorded on the caller's stream before the first upload
    int opt_host_slices = 0;                       // option 2: 0 = automatic, n >= 1 = force n sub-batches
    long long last_stats[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    // optional phase profiling (option 1): CUDA events on the launching stream around the phases of every call
    int opt_profile = 0;
    static constexpr int kProfPhases = 5;          // prepare, solve, score kernel, fixup+repair, select
    static constexpr int kProfScoreStart = 6;      // extra boundary: the scorer's own start (pipelined passes: the solver ended long before)
    static constexpr int kProfSweep = 7;           // bounded sweep: boundaries 7/8 around the candidate stage's scorer, 9/10 stage B's,
                                                   // 11/12 the fallback's
    static constexpr int kProfEvents = 13;         // boundaries 0..5 + the scorer start + the three later scorer launches
    static constexpr int kProfRing = 2048;         // passes remembered between two reads (20 steps of a tapered 64-pass sweep)
    cudaEvent_t* prof_ev = nullptr;                // kProfRing * kProfEvents events
    int prof_cur = -1;                             // pass opened by the last prof_mark(.., 0) (sequential callers)
    int prof_calls = 0;                            // calls recorded in the ring since profiling was switched on / last read
    bool prof_open = false;                        // boundary 0 of the current call was recorded (ring not full)
    unsigned prof_masks[kProfRing] = {0};          // boundaries recorded per pass
};

int ensure_pinned(Buffer& b, size_t bytes);
void prof_mark(Ctx* c, cudaStream_t st, int boundary);   // boundary 0 opens a call, 1..kProfPhases close the phases
int prof_begin(Ctx* c);                                  // opens a pass explicitly: its ring index, or -1 (off / ring full)
void prof_mark_at(Ctx* c, cudaStream_t st, int call, int boundary);   // boundary of THAT pass (phases of passes may interleave)
void release_pinned(Buffer& b);
int ensure(Buffer& b, size_t bytes);      // grow-only cudaMalloc
void release(Buffer& b);
void p2p_release(Ctx* c);                 // p2p_api.cu

}  // namespace rg
