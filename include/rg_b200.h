/* librg_b200.so — C ABI of the B200-native robust two-view / pose estimation hot path.
 *
 * This header is the drop-in boundary: every entry point is plain C (pointers + sizes, no C++/torch types) and is
 * what a reference-side FFI (Python ctypes, see INTEGRATION.md) binds.  The reference project has no FFI of its own:
 * its boundary is a set of Python functions in flat modules.  Each entry point below names the reference function
 * (file:line in bioengstrom/tsbb15-3d-reconstruction-project) whose arithmetic it replaces.
 *
 * Conventions
 *   - every function returns 0 on success and a negative code on failure; rg_last_error() gives the text
 *     (-1 CUDA error, -2 invalid argument, -3 no sm_100 device);
 *   - there is NO CPU fallback: without a Blackwell (sm_100) device rg_init fails with -3;
 *   - "_host" entry points take HOST buffers, do the H2D / D2H copies on `stream` and synchronise it before returning;
 *     "_dev" entry points take DEVICE buffers (offset tables stay on the host) and are asynchronous on `stream`;
 *   - all matrices are row-major doubles; correspondences of a pair are an (N, 4) array (x0, x1, y0, y1) where
 *     x = image-1 point and y = image-2 point of the reference's convention x^T F y = 0 (lab3.py:196);
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); a context is bound to one device and may be
 *     used from one host thread at a time.
 */
#ifndef RG_B200_H
#define RG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- enumerations (ABI values) -------------------------------------------------------------------------------- */
#define RG_MODE_EPI_MAX 0   /* max(|d1|,|d2|) < thr : the reference criterion, fun.py:316-317 */
#define RG_MODE_SAMPSON 1   /* Sampson distance < thr : extension named by the north star, not in the reference */
#define RG_TIE_FIRST 0      /* ties on the inlier count: first hypothesis wins (strict >, fun.py:320) */
#define RG_TIE_REFERENCE 1  /* replay of the reference's tie rule norm(std(d_best)) > norm(d_new), fun.py:324-328 */
#define RG_SOLVER_QR 0      /* Householder null vector, one hypothesis per thread (default) */
#define RG_SOLVER_JACOBI 1  /* register-resident one-sided Jacobi SVD, one hypothesis per 16-lane group */
#define RG_SCORE_FP32_GUARDED 0 /* FP32 fma.rn.f32x2 scorer + rigorous guard band re-evaluated in FP64 (exact counts) */
#define RG_SCORE_FP64 1         /* every evaluation in FP64 with the reference formula */
#define RG_SCORE_FP32_BOUND 2   /* rg_epi_score_count_host only: the bounded sweep's bound-only prefix scorer, whose counts
                                   are upper bounds of the exact counts (option 15) */

/* ---- context -------------------------------------------------------------------------------------------------- */
int rg_abi_version(void);
const char* rg_last_error(void);
int rg_init(int device, void** out_ctx);
int rg_shutdown(void* ctx);
int rg_device_sm_count(void* ctx);
/* page-locked host memory for input batches built in place (the host-buffer entry points accept any host memory; uploads
 * from pageable memory are staged by the driver at a fraction of the link rate) */
int rg_host_alloc(size_t bytes, void** out);
int rg_host_free(void* p);
/* option 1 = phase profiling on/off: CUDA events on the launching stream around the phases of every RANSAC call
 * option 2 = number of sub-batches of rg_f_ransac_host (0 = automatic, 1 = monolithic, up to 8): the upload of sub-batch
 *            k+1 runs on a second stream while sub-batch k is scored; results do not depend on it
 * option 3 = CTAs in the thread-block cluster that factorises the bundle-adjustment camera system (0 = default 8; 1, 2, 4,
 *            8); results do not depend on it
 * option 4 = 1: factorise that system in global memory / L2 even when it fits in the cluster's distributed shared memory
 *            (the default picks shared memory when it fits); results do not depend on it
 * option 5 = 1: gold-standard refinement always on the multi-kernel path (default: pairs of <= 4096 correspondences run
 *            the whole Levenberg-Marquardt loop in one CTA and one launch); same iteration, sums in a different order
 * option 6 = hypothesis x correspondence evaluations per PASS of a large RANSAC batch (0 = default 2.7e10 = 64 pairs of
 *            50 000 x 8 192): a batch is processed in passes so that its workspaces stay bounded; results do not depend on it
 * option 7 = PnP minimal-sample solver: 0 = Givens QR + Jacobi on the rows of R, one thread per hypothesis (default);
 *            1 = register-resident one-sided Jacobi in a 16-lane group (the solver BASELINE.json names)
 * option 8 = test hook: capacity of the guard-band flag list in records (0 = automatic); a small value forces the
 *            FP64 recount of the hypotheses whose flags did not fit; results do not depend on it
 * option 9 = guard-band safety factor x 1000 (default 1000 = the proven FP32 rounding bound): a wider band sends more
 *            evaluations to the FP64 recheck (results do not depend on it); measures the fix-up cost of a less accurate scorer
 * option 10 = pass pipelining of F calls that run in several passes (default 1): the fix-up / selection / mask kernels of
 *            pass k run on a second stream while pass k+1 is solved and scored; 0 = one stream, strictly in order
 *            (results do not depend on it; the caller's stream sees the whole call complete either way)
 * option 11 = test hook: 1 = refinement of PnP poses (rg_pnp_refine_*) always on the multi-CTA path (default: views of
 *            <= 4096 correspondences run the whole loop in one CTA); same iteration, sums in a different order
 * option 12 = bounded sweep of F calls (default 1): rg_f_ransac_host / _host2 with counts == NULL and rg_f_ransac_dev2
 *            with RG_FLAG_BOUNDED score every hypothesis on a prefix of each pair, finish the K best prefix counts, and
 *            score in full only the pairs where another hypothesis could still reach the maximum (DESIGN.md section 4);
 *            winners, counts, F and masks are those of the full sweep; 0 = every hypothesis against every correspondence
 * option 13 = prefix share rho of the bounded sweep in thousandths, [1, 1000] (default 450); results do not depend on it
 * option 14 = candidates K per pair of the bounded sweep, [1, 65536] (default 512); results do not depend on it
 * option 15 = prefix stage of the bounded sweep: 1 (default) = bound-only FP32 scorer (counts r^2 < T, an upper bound on
 *            every hypothesis's prefix count, with no guard-band fix-up; the K candidates are then scored over the whole
 *            pair), 0 = guarded scorer + FP64 fix-up (exact prefix counts; the candidates are scored on the rest of the
 *            pair); results do not depend on it (DESIGN.md section 4)
 * option 16 = share rho0 of the bound-only prefix's first stage in thousandths, [1, 1000] (default 380): every hypothesis
 *            is scored on the first rho0 of its pair, the candidates are chosen there, and only the hypotheses that
 *            share cannot yet rule out are extended to rho; rho0 >= rho (or option 15 = 0) is a one-stage prefix;
 *            results do not depend on it */
int rg_set_option(void* ctx, int option, long long value);
/* summed milliseconds of {prepare, solve, score kernel, fixup + repair, select} over the PASSES since the last read
 * (at most 2048 passes are remembered; *out_calls = passes covered); synchronises `stream` */
int rg_get_profile(void* ctx, void* stream, double* out_ms5, int* out_calls);

/* Pipe micro-benchmarks on the context's device (roofline denominators for bench.py):
 * out6 = {FFMA GFMA/s, FFMA2 GFMA/s, scalar-mix Gevals/s, packed-mix Gevals/s, DFMA GFMA/s, SM count}. */
int rg_microbench_run(double* out6, void* stream);

/* out8 = {guard-band groups flagged by the FP32 scorer, band evaluations redone in FP64, decisions changed by that,
 *         hypotheses recounted in FP64 because the flag list was full, hypotheses with an out-of-range sample index,
 *         upload rate measured by rg_f_ransac_host* (MB/s, running average), passes of the last call, kernel launches of the last call}.  Synchronises `stream`. */
int rg_get_last_stats(void* ctx, void* stream, long long* out8);

/* ---- F-matrix RANSAC: replaces the loop of fun.getFFromLabCode (fun.py:303-328), which calls
 *      lab3.fmatrix_stls (lab3.py:269-329) and lab3.fmatrix_residuals (lab3.py:188-227) once per trial ------------- */
/* Batched over P image pairs (CSR layout).  pair_off[P+1] / hyp_off[P+1] are HOST int32 prefix tables.
 *   pts64   : (pair_off[P], 4) doubles        idx : (hyp_off[P], 8) int32 sample indices local to the pair (host-drawn)
 * Outputs per pair: best_idx (index of the selected hypothesis inside the pair, -1 if no hypothesis has an inlier),
 * best_count, best_F (3x3); mask (pair_off[P] bytes, optional) = inlier set of the selected hypothesis. */
int rg_f_ransac_dev(void* ctx, void* stream, int P, const double* pts64_dev, const int32_t* pair_off_host,
                    const int32_t* idx_dev, const int32_t* hyp_off_host, double thr, int mode, int tie_mode, int solver,
                    int score_path, int32_t* best_idx_dev, int32_t* best_count_dev, double* best_F_dev,
                    unsigned char* mask_dev /* may be NULL */);
/* Extended form (round 2).  Everything rg_f_ransac_dev does, plus
 *   idx_dev == NULL : the (H, 8) sample index sets are drawn on the DEVICE (Philox4x32-10, csrc/philox.cuh) as a pure
 *                     function of (sample_seed, first_pair_id + pair, hyp_index_base + hypothesis); they never cross
 *                     PCIe and the host replays them bit for bit (tsbb15_b200/philox.py, rg_sample_indices_dev) — the
 *                     reference draws np.random.choice(N, 8, replace=False) per trial, fun.py:305-308;
 *   flags & RG_FLAG_REUSE_POINTS : the points, pair table and threshold are those of the previous call on this context:
 *                     skip the bounding-box / FP32-copy kernels (hypothesis-split mode scores many hypothesis sets
 *                     against one pair);
 *   hyp_index_base  : hypothesis-split mode (SURVEY 8e item 2): this rank holds hypotheses [base, base + H_p) of every pair;
 *   flags & RG_FLAG_BOUNDED : run the bounded sweep when option 12 is on (the results are the same; afterwards
 *                     rg_f_last_hypotheses_dev returns no counts, since hypotheses that cannot win keep a prefix count);
 *   key_dev (P, optional) : the cross-GPU argmax key of every pair, (count << 32) | (0xFFFFFFFF - global hypothesis
 *                     index), 0 if no hypothesis of this rank has an inlier (fun.py:320-323: first maximum wins). */
#define RG_FLAG_REUSE_POINTS 1
#define RG_FLAG_BOUNDED 2
int rg_f_ransac_dev2(void* ctx, void* stream, int P, const double* pts64_dev, const int32_t* pair_off_host,
                     const int32_t* idx_dev /* may be NULL */, const int32_t* hyp_off_host, double thr, int mode,
                     int tie_mode, int solver, int score_path, int flags, unsigned long long sample_seed, int first_pair_id,
                     int hyp_index_base, int32_t* best_idx_dev, int32_t* best_count_dev, double* best_F_dev,
                     unsigned char* mask_dev /* may be NULL */, unsigned long long* key_dev /* may be NULL */);
/* the index sets a seeded call draws (k = 6, 7, 8), for callers / oracles that want to see them: idx_out (hyp_off[P], k) */
int rg_sample_indices_dev(void* ctx, void* stream, int P, const int32_t* n_points_host, const int32_t* hyp_off_host, int k,
                          unsigned long long seed, int first_pair_id, int hyp_index_base, int32_t* idx_out_dev);
/* synthetic correspondences of BASELINE configs 3-5 generated on the device (SURVEY 8d: X ~ U(box) seen by two of the
 * n_cams cameras drawn from seed_base + pair id, Gaussian pixel noise (Irwin-Hall 12), the first outlier_frac of the image-2
 * points uniform in the image); host-replayable (tsbb15_b200/philox.py).  pts_out (P x N x 4), cam_pair_out (P x 2, opt.) */
int rg_synth_two_view_dev(void* ctx, void* stream, int P, int first_pair_id, int N, const double* cams_host, int n_cams,
                          const double* bbox6_host, unsigned long long seed_base, double outlier_frac, double sigma_px,
                          double width, double height, double* pts_out_dev, int32_t* cam_pair_out_dev);
/* inlier mask (reference criterion, fun.py:315-317) of ONE caller-supplied F per pair, device buffers */
int rg_f_inlier_mask_dev(void* ctx, void* stream, int P, const double* pts64_dev, const int32_t* pair_off_host,
                         const double* F_dev, double thr, int mode, unsigned char* mask_dev);
/* per-hypothesis results of the last rg_f_ransac_dev call on this context (device pointers, valid until the next call;
 * after rg_f_ransac_host they cover only its last sub-batch — use that function's counts / F_all / flags outputs):
 * counts (hyp_off[P] int32), F_all (hyp_off[P] x 9 doubles), flags (bit0: rank-deficient sample, bit1: non-finite F,
 * bit2: a sample index outside [0, N) of the pair — the solver clamps it; rg_f_ransac_host then returns -2 and
 * rg_get_last_stats reports the number of such hypotheses in out8[4]).  *counts_dev is NULL after a bounded sweep. */
int rg_f_last_hypotheses_dev(void* ctx, const int32_t** counts_dev, const double** F_all_dev,
                             const unsigned char** flags_dev);
/* what the last F call executed: out4 = {hypothesis x correspondence evaluations, hypotheses not scored in full (proved
 * unable to reach their pair's maximum), pairs that fell back to scoring every hypothesis in full, K (0: full sweep)}.
 * Synchronises `stream`. */
int rg_f_last_bounded_stats(void* ctx, void* stream, long long* out4);
/* the evaluations of the last F call split by scorer: out2 = {bound-only prefix stages (option 15 = 1; both stages of
 * option 16, the second counted on the device), guarded scorer
 * (exact prefix, candidate and fallback stages, or the full sweep)}; out2[0] + out2[1] = out4[0] above.
 * Synchronises `stream`. */
int rg_f_last_bounded_evals(void* ctx, void* stream, long long* out2);
/* Same with host buffers; counts / F_all / flags / mask are optional (NULL = not copied back; counts == NULL runs the
 * bounded sweep when option 12 is on).  The batch is uploaded pass
 * by pass on a second stream, so the copy of pass k+1 overlaps the scoring of pass k (page-locked buffers needed for the
 * overlap; pageable ones are still correct). */
int rg_f_ransac_host(void* ctx, void* stream, int P, const double* pts64, const int32_t* pair_off, const int32_t* idx,
                     const int32_t* hyp_off, double thr, int mode, int tie_mode, int solver, int score_path,
                     int32_t* best_idx, int32_t* best_count, double* best_F, unsigned char* mask, int32_t* counts,
                     double* F_all, unsigned char* flags);

/* idx == NULL: samples drawn on the device from (sample_seed, first_pair_id), see rg_f_ransac_dev2 */
int rg_f_ransac_host2(void* ctx, void* stream, int P, const double* pts64, const int32_t* pair_off,
                      const int32_t* idx /* may be NULL */, const int32_t* hyp_off, double thr, int mode, int tie_mode,
                      int solver, int score_path, unsigned long long sample_seed, int first_pair_id, int32_t* best_idx,
                      int32_t* best_count, double* best_F, unsigned char* mask, int32_t* counts, double* F_all,
                      unsigned char* flags);

/* Stage entry points (same kernels, one pair):
 * 8-point solve of H samples — lab3.fmatrix_stls on 8 points (lab3.py:269-329) */
int rg_f8pt_solve_host(void* ctx, void* stream, int N, const double* pts64, int H, const int32_t* idx, int solver,
                       double* F_all, unsigned char* flags /* may be NULL */);
/* inlier counts of H caller-supplied F over N correspondences — fmatrix_residuals + threshold (fun.py:315-317);
 * score_path RG_SCORE_FP32_BOUND returns the bound-only scorer's upper bounds of those counts instead */
int rg_epi_score_count_host(void* ctx, void* stream, int N, const double* pts64, int H, const double* F_all, double thr,
                            int mode, int score_path, int32_t* counts);
/* lab3.fmatrix_residuals (lab3.py:188-227): x, y are (2, N) row-major, out is (2, N) signed distances */
int rg_fmatrix_residuals_host(void* ctx, void* stream, const double* F9, int N, const double* x, const double* y,
                              double* out);
/* lab3.fmatrix_stls for any N >= 8 (lab3.py:269-329): pl, pr are (2, N) row-major */
int rg_fmatrix_stls_host(void* ctx, void* stream, int N, const double* pl, const double* pr, double* F9);

/* ---- PnP-RANSAC: restates ransac.ransac_robust (ransac.py:37-113, does not run in the reference) with the DLT pose
 *      solver specified in pnp.py:132-152 (pnp.pnp_minimize, body unfinished in the reference) --------------------- */
/* One view.  X : (N, 3) world points, y : (N, 2) C-normalised image points, idx : (H, n) sample indices, n in [6, 8].
 * Inlier: squared reprojection distance e <= thr2 (inclusive, ransac.py:104).  N_sel <= N: only the first N_sel
 * correspondences vote in the selection (the reference selects on D_med, ransac.py:108); mask covers all N.
 * Outputs: best_idx, best_count, R (3x3), t (3), mask (N bytes, optional), counts (H, optional), poses (H x 12, opt). */
int rg_pnp_ransac_host(void* ctx, void* stream, int N, int N_sel, const double* X, const double* y, int H, int n,
                       const int32_t* idx, double thr2, int score_path, int32_t* best_idx, int32_t* best_count, double* R,
                       double* t, unsigned char* mask, int32_t* counts, double* poses, unsigned char* flags);
int rg_pnp_ransac_dev(void* ctx, void* stream, int N, int N_sel, const double* X_dev, const double* y_dev, int H, int n,
                      const int32_t* idx_dev, double thr2, int score_path, int32_t* best_idx_dev, int32_t* best_count_dev,
                      double* Rt_dev /* 12 doubles: R row-major then t */, unsigned char* mask_dev);
/* The same over V views in ONE call (CSR: view_off[V+1], hyp_off[V+1] host int32; idx local to the view).  n_vote
 * (host, V ints, may be NULL = all) = number of leading correspondences of each view that vote.  Outputs per view:
 * best_idx, best_count, Rt (V x 12: R row-major then t); mask covers all correspondences. */
int rg_pnp_ransac_batched_host(void* ctx, void* stream, int V, const double* X, const double* y, const int32_t* view_off,
                               const int32_t* n_vote, const int32_t* idx, const int32_t* hyp_off, int n, double thr2,
                               int score_path, int32_t* best_idx, int32_t* best_count, double* Rt, unsigned char* mask,
                               int32_t* counts, double* poses, unsigned char* flags);
int rg_pnp_ransac_batched_dev(void* ctx, void* stream, int V, const double* X_dev, const double* y_dev,
                              const int32_t* view_off_host, const int32_t* n_vote_host, const int32_t* idx_dev,
                              const int32_t* hyp_off_host, int n, double thr2, int score_path, int32_t* best_idx_dev,
                              int32_t* best_count_dev, double* Rt_dev, unsigned char* mask_dev);
/* hypothesis-split mode (see rg_f_ransac_dev2): this rank holds hypotheses [hyp_index_base, hyp_index_base + H_v) of every
 * view; key_dev (V, optional) receives the cross-GPU argmax keys (ransac.py:108: first maximum wins) */
int rg_pnp_ransac_batched_dev2(void* ctx, void* stream, int V, const double* X_dev, const double* y_dev,
                               const int32_t* view_off_host, const int32_t* n_vote_host, const int32_t* idx_dev,
                               const int32_t* hyp_off_host, int n, double thr2, int score_path, int hyp_index_base,
                               int32_t* best_idx_dev, int32_t* best_count_dev, double* Rt_dev, unsigned char* mask_dev,
                               unsigned long long* key_dev);
/* pnp.pnp_minimize(_3d_pts, img_pts, m) (pnp.py:132-152) for any m >= 6: X (m, 3), y (m, 2) -> R (3x3), t (3) */
int rg_pnp_minimize_host(void* ctx, void* stream, int m, const double* X, const double* y, double* R, double* t);
/* reprojection scoring of H caller-supplied poses (H x 12: R row-major then t) — ransac.py:96-105 */
int rg_pnp_score_count_host(void* ctx, void* stream, int N, const double* X, const double* y, int H, const double* poses,
                            double thr2, int score_path, int32_t* counts);

/* ---- refinement of PnP poses (DESIGN.md section 4.7) ------------------------------------------------------------ */
/* The reference's live PnP call is OpenCV's cv.solvePnPRansac (tables.py:141), which ends with solvePnP(ITERATIVE,
 * useExtrinsicGuess) on the inliers: a Levenberg-Marquardt minimisation of the reprojection error.  The RANSAC above
 * returns the algebraic DLT pose of pnp.py:132-152; this minimises, per view v over its selected correspondences,
 *   C_v(R, t) = 1/2 sum_k |W_v (pi(R X_k + t) - y_k)|^2,  pi(p) = (p0/p2, p1/p2),  W_v = K_v[:2, :2] (fx, s; 0, fy) or I
 * (the principal point cancels; with K the cost is in pixels) over R <- exp([dw]_x) R and t <- t + dt, batched over V
 * views, no host synchronisation.  Views of <= 4096 correspondences run the whole loop in one CTA (option 11 = 1 forces
 * the multi-CTA path of larger views); sums in a fixed order, bit-reproducible.
 *   X (view_off[V], 3), y (view_off[V], 2) C-normalised, view_off HOST int32 CSR table (layout of rg_pnp_ransac_batched_*)
 *   K : V x 9 row-major on the HOST (NULL = W = I); -2 unless K[1][0] == 0 and the bottom row is (0, 0, 1)
 *   mask (optional) selects the correspondences of the first round, e.g. the mask of rg_pnp_ransac_batched_dev
 *   Rt (V x 12, R row-major then t, as rg_pnp_ransac_* write it) is refined IN PLACE
 *   rounds >= 1: after every round the consensus thr2 >= e at the refined pose (ransac.py:104-105, FP64, C-normalised
 *   units) is recomputed over all correspondences and the next round refines on it; mask_out (optional) receives the
 *   last consensus; thr2 is required when rounds > 1 or mask_out is given
 * Outputs of the last round (optional): cost = C_v at the returned pose; iters; status: 1 = start pose not finite,
 * 2 = converged (relative decrease <= ftol, actual or predicted), 3 = lambda > 1e12, 4 = max_iter reached, 5 = fewer than
 * 3 selected correspondences (pose unchanged). */
int rg_pnp_refine_dev(void* ctx, void* stream, int V, const double* X_dev, const double* y_dev, const int32_t* view_off_host,
                      const double* K_host, const unsigned char* mask_dev, double* Rt_dev, int max_iter, double ftol,
                      int rounds, double thr2, unsigned char* mask_out_dev, double* cost_dev, int32_t* iters_dev,
                      int32_t* status_dev);
/* the same with host buffers: uploads, calls the above, downloads, synchronises `stream` */
int rg_pnp_refine_host(void* ctx, void* stream, int V, const double* X, const double* y, const int32_t* view_off,
                       const double* K, const unsigned char* mask, double* Rt, int max_iter, double ftol, int rounds,
                       double thr2, unsigned char* mask_out, double* cost, int32_t* iters, int32_t* status);
/* The same with a robust loss (SciPy's least_squares `loss` / `f_scale`; the RG_LOSS_* values and rho of
 * rg_bundle_adjust_host2 below).  Every scalar residual f of W_v (pi(R X_k + t) - y_k) gets z = (f / C)^2, C = f_scale > 0,
 * and cost = 0.5 * sum C^2 rho(z) (SciPy's sol.cost).  f_scale is in the units of the residuals: pixels when K is given,
 * C-normalised otherwise.  Linearisation by iteratively reweighted least squares (weights rho'(z)); the stopping rules
 * read the robust cost.  The consensus of rounds > 1 / mask_out is the same hard test thr2 >= e.  An unknown loss, or an
 * f_scale that is not finite and > 0 (or whose square is 0 or not finite), is an invalid argument (-2) and nothing is
 * enqueued.  RG_LOSS_LINEAR gives results bit-identical to rg_pnp_refine_dev / _host. */
int rg_pnp_refine_dev2(void* ctx, void* stream, int V, const double* X_dev, const double* y_dev, const int32_t* view_off_host,
                       const double* K_host, const unsigned char* mask_dev, double* Rt_dev, int max_iter, double ftol, int loss,
                       double f_scale, int rounds, double thr2, unsigned char* mask_out_dev, double* cost_dev,
                       int32_t* iters_dev, int32_t* status_dev);
int rg_pnp_refine_host2(void* ctx, void* stream, int V, const double* X, const double* y, const int32_t* view_off,
                        const double* K, const unsigned char* mask, double* Rt, int max_iter, double ftol, int loss,
                        double f_scale, int rounds, double thr2, unsigned char* mask_out, double* cost, int32_t* iters,
                        int32_t* status);

/* ---- two-view geometry either side of the RANSAC path (SURVEY.md section 8f, rows N1-N3), all FP64 -------------- */
#define RG_TRI_OPTIMAL 0    /* lab3.triangulate_optimal (lab3.py:382-475): Hartley-Sturm, degree-6 root solve per point */
#define RG_TRI_LINEAR 1     /* lab3.triangulate_linear (lab3.py:477-503) */
/* Triangulation of every correspondence of P camera pairs in ONE call: replaces the per-correspondence Python loops
 * around lab3.triangulate_optimal / triangulate_linear (fun.py:352, tables.py:170, tables.py:243, fun.py:240-255).
 * C1, C2: (P, 3, 4) cameras; pair_off[P+1] HOST int32 CSR table; x1, x2: (pair_off[P], 2) image points (x1 seen by C1,
 * x2 by C2); X: (pair_off[P], 3) world points.  Device x1 / x2 (and y1 / y2 below) must be 16-byte aligned. */
int rg_triangulate_host(void* ctx, void* stream, int P, const double* C1, const double* C2, const int32_t* pair_off,
                        const double* x1, const double* x2, int method, double* X);
int rg_triangulate_dev(void* ctx, void* stream, int P, const double* C1_dev, const double* C2_dev,
                       const int32_t* pair_off_host, const double* x1_dev, const double* x2_dev, int method,
                       double* X_dev);
/* lab3.fmatrix_from_cameras (lab3.py:331-351) for P camera pairs: F (P, 3, 3) with x1^T F x2 = 0, the reference's
 * scale ([C1 n]_x C1 pinv(C2), |n| = 1) up to the arbitrary sign of its SVD null vector */
int rg_fmatrix_from_cameras_host(void* ctx, void* stream, int P, const double* C1, const double* C2, double* F);
/* fun.relative_camera_pose (fun.py:209-258, with fun.specSVD fun.py:186-207) for P pairs in one call.
 * M: (P, 3, 3) essential matrices; if K != NULL, M holds fundamental matrices and E = K^T M K is formed on the device
 * (fun.getEAndK, fun.py:100-101; K is (3,3) shared, or (P,3,3) when k_per_pair != 0).  y1, y2: (P, 2) one C-normalised
 * correspondence per pair.  Rt: (P, 12) R row-major then t of the first of the four candidates whose optimally
 * triangulated point is in front of both cameras (NaN if none: the reference returns None); which: candidate index
 * 0..3 in the reference's order for THIS library's SVD sign convention, -1 if none; npass (optional): number of
 * candidates that pass (1 for a well-posed pair). */
int rg_relative_pose_host(void* ctx, void* stream, int P, const double* M, const double* K, int k_per_pair,
                          const double* y1, const double* y2, double* Rt, int32_t* which, int32_t* npass);
int rg_relative_pose_dev(void* ctx, void* stream, int P, const double* M_dev, const double* K_dev, int k_per_pair,
                         const double* y1_dev, const double* y2_dev, double* Rt_dev, int32_t* which_dev,
                         int32_t* npass_dev /* may be NULL */);
/* The two-view initialisation of main.py:54-76 (INIT2 + INIT3) for P image pairs in one call, entirely on the device:
 * E = K^T F K (fun.getEAndK), C-normalised points K^-1 (u, v, 1)^T (fun.MakeHomogenous, fun.py:48-55, first two
 * components as main.py passes them), fun.relative_camera_pose on the pair's FIRST correspondence (main.py:62; with a
 * mask: the first correspondence whose mask byte is non-zero), then lab3.triangulate_optimal of every correspondence
 * with C1 = [I | 0], C2 = [R | t] (tables.py:233-247).  pts64: (pair_off[P], 4) pixels; F: (P, 3, 3), e.g. best_F of
 * rg_f_ransac_dev; K9: HOST (3, 3); mask (optional): correspondences with 0 are not triangulated (X = NaN).
 * Outputs: Rt (P, 12), which (P, -1 = no candidate passes), X (pair_off[P], 3) in the frame of the first camera. */
int rg_two_view_init_host(void* ctx, void* stream, int P, const double* pts64, const int32_t* pair_off, const double* F,
                          const double* K9, const unsigned char* mask, double* Rt, int32_t* which, double* X);
int rg_two_view_init_dev(void* ctx, void* stream, int P, const double* pts64_dev, const int32_t* pair_off_host,
                         const double* F_dev, const double* K9_host, const unsigned char* mask_dev, double* Rt_dev,
                         int32_t* which_dev, double* X_dev);
/* ---- gold-standard refinement (SURVEY.md section 8f row N4) ------------------------------------------------------ */
/* The second half of fun.getFFromLabCode (fun.py:342-369) for P image pairs in one call, entirely on the device:
 * cameras from F (lab3.fmatrix_cameras, lab3.py:353-380), optimal triangulation of the inliers (fun.py:352), then the
 * minimisation of the cost of lab3.fmatrix_residuals_gs (lab3.py:230-266) over C1 (3x4) and the 3-D points, and
 * F_gold = lab3.fmatrix_from_cameras(C1, [I|0]) (fun.py:368).  The reference hands that cost to
 * scipy.optimize.least_squares (trust-region reflective, finite-difference Jacobian: minutes, and it stops on ftol before
 * the minimum); here it is Levenberg-Marquardt with the Schur complement of the point blocks and converges to the
 * minimum of the SAME cost — F_gold therefore differs from the reference's by what its early stop leaves (DESIGN.md).
 * pts64: (pair_off[P], 4) pixels; F0: (P, 3, 3) e.g. best_F of rg_f_ransac; mask (optional): 0 = not an inlier.
 * Outputs: F_gold (P, 3, 3); cost (P, optional) = 0.5 * sum of squared residuals at the solution (SciPy's `cost`);
 * iters (P, optional); status (P, optional): 1 = F0 not finite, 2 = converged (relative decrease <= ftol), 3 = no
 * further descent, 4 = max_iter reached; X (pair_off[P], 3, optional) = refined points (NaN for masked-out ones). */
int rg_gold_standard_host(void* ctx, void* stream, int P, const double* pts64, const int32_t* pair_off, const double* F0,
                          const unsigned char* mask, int max_iter, double ftol, double* F_gold, double* cost, int32_t* iters,
                          int32_t* status, double* X);
int rg_gold_standard_dev(void* ctx, void* stream, int P, const double* pts64_dev, const int32_t* pair_off_host,
                         const double* F0_dev, const unsigned char* mask_dev, int max_iter, double ftol, double* F_gold_dev,
                         double* cost_dev, int32_t* iters_dev, int32_t* status_dev, double* X_dev);
/* The same with a robust loss (SciPy's least_squares `loss` / `f_scale`, as a SciPy user adds them to the reference's
 * call fun.py:358; the RG_LOSS_* values and rho of rg_bundle_adjust_host2 below).  Each of the four residuals of a
 * correspondence gets z = (f / C)^2, C = f_scale > 0 in PIXELS (pts64 is in pixels), and cost = 0.5 * sum C^2 rho(z)
 * (SciPy's sol.cost).  Linearisation by iteratively reweighted least squares (weights rho'(z) between the factors of
 * every Jacobian product; the Schur structure is unchanged).  With mask == NULL every correspondence takes part, which
 * makes this a refinement without a hard inlier set.  An unknown loss, or an f_scale that is not finite and > 0 (or
 * whose square is 0 or not finite), is an invalid argument (-2) and nothing is enqueued.  RG_LOSS_LINEAR gives results
 * bit-identical to rg_gold_standard_dev / _host. */
int rg_gold_standard_dev2(void* ctx, void* stream, int P, const double* pts64_dev, const int32_t* pair_off_host,
                          const double* F0_dev, const unsigned char* mask_dev, int max_iter, double ftol, int loss, double f_scale,
                          double* F_gold_dev, double* cost_dev, int32_t* iters_dev, int32_t* status_dev, double* X_dev);
int rg_gold_standard_host2(void* ctx, void* stream, int P, const double* pts64, const int32_t* pair_off, const double* F0,
                           const unsigned char* mask, int max_iter, double ftol, int loss, double f_scale, double* F_gold,
                           double* cost, int32_t* iters, int32_t* status, double* X);
/* lab3.fmatrix_residuals_gs(params, pl, pr) (lab3.py:230-266): params = [C1.ravel() (12), X.T.ravel() (3N)], pl / pr (2, N)
 * row-major; out (4N) = leftx, lefty, rightx, righty */
int rg_fmatrix_residuals_gs_host(void* ctx, void* stream, int N, const double* params, const double* pl, const double* pr,
                                 double* out);
/* ---- bundle adjustment (SURVEY.md section 8f row N4, multi-view half) -------------------------------------------------- */
/* The minimisation of tables.Tables.BundleAdjustment2 (tables.py:260-333): cost = 0.5 * sum over the observation table of
 * (u - c1.x/c3.x)^2 + (v - c2.x/c3.x)^2 (EpsilonBA, tables.py:266-296) over all 12 entries of every view's 3x4 matrix except
 * the first n_fixed views (the reference clears the first view's Jacobian columns, tables.py:376: n_fixed = 1) and all 3-D
 * points.  The reference calls scipy.optimize.least_squares (trf, x_scale='jac', ftol=1e-4, finite differences); here it is
 * Levenberg-Marquardt with the Schur complement of the point blocks and a dense Cholesky of the reduced camera system on
 * one thread-block cluster, converging on the relative cost decrease ftol — same cost function, not the same iterates
 * (DESIGN.md section 4.6).  cams (n_views, 3, 4) and pts (n_points, 3) are refined IN PLACE; uv (n_obs, 2) observed
 * C-normalised image points; cam_idx / pt_idx (n_obs) HOST arrays in both variants.  n_views - n_fixed <= 170.
 * Outputs (optional scalars): cost at the solution, iterations, status: 2 = converged, 3 = no further descent,
 * 4 = max_iter reached. */
int rg_bundle_adjust_host(void* ctx, void* stream, int n_views, int n_points, int n_obs, double* cams, double* pts,
                          const double* uv, const int32_t* cam_idx, const int32_t* pt_idx, int n_fixed, int max_iter, double ftol,
                          double* cost, int32_t* iters, int32_t* status);
int rg_bundle_adjust_dev(void* ctx, void* stream, int n_views, int n_points, int n_obs, double* cams_dev, double* pts_dev,
                         const double* uv_dev, const int32_t* cam_idx_host, const int32_t* pt_idx_host, int n_fixed, int max_iter,
                         double ftol, double* cost_dev, int32_t* iters_dev, int32_t* status_dev);
/* The same with a robust loss: the `loss` and `f_scale` of the reference's least_squares call (tables.py:317), with
 * SciPy's definitions (scipy/optimize/_lsq/least_squares.py).  Every scalar residual f of EpsilonBA gets z = (f / C)^2,
 * C = f_scale > 0, and the cost is 0.5 * sum C^2 rho(z) (SciPy's sol.cost) with
 *   RG_LOSS_LINEAR   rho = z                                  (the entry points above; f_scale has no effect)
 *   RG_LOSS_SOFT_L1  rho = 2 (sqrt(1 + z) - 1)
 *   RG_LOSS_HUBER    rho = z for z <= 1, 2 sqrt(z) - 1 above
 *   RG_LOSS_CAUCHY   rho = log(1 + z)
 *   RG_LOSS_ARCTAN   rho = arctan(z)
 * uv is C-normalised, so a scale of s pixels is f_scale = s / K[0][0].  The linearisation is iteratively reweighted least
 * squares (each residual row and its Jacobian row weighted by sqrt(rho'(z))), not SciPy's second-order-corrected scaling
 * (DESIGN.md section 4.6).  An unknown loss, or an f_scale that is not finite and > 0, is an invalid argument (-2).
 * RG_LOSS_LINEAR gives results bit-identical to rg_bundle_adjust_host / _dev. */
#define RG_LOSS_LINEAR 0
#define RG_LOSS_SOFT_L1 1
#define RG_LOSS_HUBER 2
#define RG_LOSS_CAUCHY 3
#define RG_LOSS_ARCTAN 4
int rg_bundle_adjust_host2(void* ctx, void* stream, int n_views, int n_points, int n_obs, double* cams, double* pts,
                           const double* uv, const int32_t* cam_idx, const int32_t* pt_idx, int n_fixed, int max_iter, double ftol,
                           int loss, double f_scale, double* cost, int32_t* iters, int32_t* status);
int rg_bundle_adjust_dev2(void* ctx, void* stream, int n_views, int n_points, int n_obs, double* cams_dev, double* pts_dev,
                          const double* uv_dev, const int32_t* cam_idx_host, const int32_t* pt_idx_host, int n_fixed, int max_iter,
                          double ftol, int loss, double f_scale, double* cost_dev, int32_t* iters_dev, int32_t* status_dev);
/* EpsilonBA(x0, u, v, table) (tables.py:266-296): x = [all camera matrices raveled (n_views x 12), all points (n_points x 3)]
 * (tables.py:315, fun.reshapeToCamera3DPoints2 fun.py:282-289); out (2 * n_obs) = interleaved u / v residuals */
int rg_ba_residuals_host(void* ctx, void* stream, int n_views, int n_points, int n_obs, const double* x, const double* u,
                         const double* v, const int32_t* cam_idx, const int32_t* pt_idx, double* out);
/* fun.camera_resectioning (fun.py:260-283, fun.specRQ fun.py:174-184) for V cameras: C (V,3,4) -> K (V,3,3) upper
 * triangular with positive diagonal and K[2][2] = 1, R (V,3,3), t (V,3); signs follow LAPACK's RQ as the reference's do */
int rg_camera_resectioning_host(void* ctx, void* stream, int V, const double* C, double* K, double* R, double* t);
/* The 2D<->3D match loop of tables.Tables.addNewView (tables.py:116-124): for every row y[i] (N, dim) the index of the
 * FIRST row of obs (M, dim) with ||obs[v] - y[i]||_2 < tol (strict), -1 if none.  dim = 2 or 3. */
int rg_match_first_within_host(void* ctx, void* stream, int dim, int M, const double* obs, int N, const double* y,
                               double tol, int32_t* idx);
int rg_match_first_within_dev(void* ctx, void* stream, int dim, int M, const double* obs_dev, int N, const double* y_dev,
                              double tol, int32_t* idx_dev);

/* ---- cross-GPU argmax when ONE pair's / view's hypotheses are split over several GPUs (SURVEY.md section 8b, 8e) ------- */
/* Every rank runs rg_f_ransac_dev / rg_pnp_ransac_dev on its hypothesis block [index_offset, ...).  rg_argmax_pack_dev
 * turns the per-pair (best_idx, best_count) into the monotone key (count << 32) | (0xFFFFFFFF - (best_idx + index_offset)),
 * 0 if the block has no hypothesis with an inlier; rg_argmax_allreduce is ONE in-place ncclAllReduce(ncclMax, ncclUint64)
 * over `count` keys on `stream` (nccl_comm: the caller's ncclComm_t; libnccl.so.2 is dlopen'ed at the first call, or
 * the library named by RG_NCCL_LIB); rg_argmax_unpack_dev gives the winner's GLOBAL hypothesis index and count: larger
 * count first, then the lower index = the first maximum of the single-GPU selection (fun.py:320-323, ransac.py:108).
 * The rank that owns the winning index then publishes its F / pose and mask. */
int rg_argmax_pack_dev(void* stream, int P, const int32_t* best_idx_dev, const int32_t* best_count_dev, int index_offset,
                       unsigned long long* key_dev);
int rg_argmax_allreduce(void* nccl_comm, void* stream, unsigned long long* key_dev, int count);
int rg_argmax_unpack_dev(void* stream, int P, const unsigned long long* key_dev, int32_t* best_idx_dev, int32_t* best_count_dev);

/* The same reduction WITHOUT NCCL, fused into one kernel over NVLink peer memory (csrc/p2p_api.cu): every rank owns a small
 * buffer that its peers map through CUDA IPC; one launch stores {key, payload} into every peer's buffer, raises a flag,
 * waits (bounded) for the peers' flags and picks the maximum key with its payload (the winner's F, or R|t) — the key and
 * the winner's model arrive in the same exchange, so no second collective is needed.
 *   rg_p2p_create   every rank: allocate the buffer, return its 64-byte IPC handle
 *   rg_p2p_connect  every rank, after the host all-gathered the handles (world x 64 bytes, rank order)
 *   rg_p2p_argmax_exchange  collective on `stream`: P <= 64 keys as written by rg_f_ransac_dev2 / rg_pnp_ransac_batched_dev2
 *                   (key_dev), payload_dev (P x npay doubles, npay <= 12); outputs the winner's GLOBAL index, count and
 *                   payload on every rank; *status_dev (device int, zero it once) becomes 1 + r if rank r did not arrive
 *                   within ~3 s instead of hanging the GPU
 * One rank per GPU. */
int rg_p2p_create(void* ctx, int rank, int world, void* handle_out64);
int rg_p2p_connect(void* ctx, const void* handles_all);
int rg_p2p_destroy(void* ctx);
int rg_p2p_argmax_exchange(void* ctx, void* stream, int P, const unsigned long long* key_dev, const double* payload_dev,
                           int npay, int32_t* best_idx_dev, int32_t* best_count_dev, double* payload_out_dev,
                           int32_t* status_dev);

#ifdef __cplusplus
}
#endif
#endif /* RG_B200_H */
