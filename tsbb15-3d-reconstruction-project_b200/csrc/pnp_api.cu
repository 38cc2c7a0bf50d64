// Host orchestration + C ABI of the PnP-RANSAC path and of the general-N single-call solvers.
#include "pnp_kernels.cuh"
#include "tall.cuh"
#include "plan.cuh"

namespace rg {

struct ScoreState;                                   // f_api.cu (same translation unit)
int score_state_layout(Ctx* c, int P, long long Htot, int bbox_words, ScoreState& s, long long Ctot);
FlagList flag_list_for(Ctx* c, const ScoreState& s, double evals, int* rc_out);
int fixup_grid(const Ctx* c, double evals);

static int pnp_solve_launch(Ctx* c, cudaStream_t st, const double* X, const double* y, const int* idx, const FPlan& plan,
                            int n, const PnpFrame* fr) {
    const int H = (int)plan.Htot;
    if (H == 0) return RG_OK;
    const int gpb = kJacobiThreads / 16;
    const int grid = ceil_div(H, gpb);
    const PairInfo* pi = (const PairInfo*)c->pair_info.ptr;
    double* pose64 = (double*)c->pose64.ptr;
    Pose32* pose32 = (Pose32*)c->pose32.ptr;
    unsigned char* flags = (unsigned char*)c->flags.ptr;
    if (c->opt_pnp_solver == 0) {                    // default: six lanes per hypothesis, Householder QR + row Jacobi in shared memory
        if (!c->pnp_rows_attr_set) {
            RG_CUDA(cudaFuncSetAttribute(pnp_solve_rows<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rows_smem<6>()));
            RG_CUDA(cudaFuncSetAttribute(pnp_solve_rows<7>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rows_smem<7>()));
            RG_CUDA(cudaFuncSetAttribute(pnp_solve_rows<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rows_smem<8>()));
            c->pnp_rows_attr_set = true;             // per context = per device
        }
        const int g2 = ceil_div(H, kRowsHypPerBlock);
        switch (n) {
            case 6: pnp_solve_rows<6><<<g2, kRowsThreads, rows_smem<6>(), st>>>(X, y, idx, pi, plan.P, H, fr, pose64, pose32, flags); break;
            case 7: pnp_solve_rows<7><<<g2, kRowsThreads, rows_smem<7>(), st>>>(X, y, idx, pi, plan.P, H, fr, pose64, pose32, flags); break;
            case 8: pnp_solve_rows<8><<<g2, kRowsThreads, rows_smem<8>(), st>>>(X, y, idx, pi, plan.P, H, fr, pose64, pose32, flags); break;
            default: set_error("invalid argument: PnP sample size n must be 6, 7 or 8"); return RG_ERR_ARG;
        }
    } else {
        switch (n) {
            case 6: pnp_solve_jacobi<6><<<grid, kJacobiThreads, 0, st>>>(X, y, idx, pi, plan.P, H, fr, pose64, pose32, flags); break;
            case 7: pnp_solve_jacobi<7><<<grid, kJacobiThreads, 0, st>>>(X, y, idx, pi, plan.P, H, fr, pose64, pose32, flags); break;
            case 8: pnp_solve_jacobi<8><<<grid, kJacobiThreads, 0, st>>>(X, y, idx, pi, plan.P, H, fr, pose64, pose32, flags); break;
            default: set_error("invalid argument: PnP sample size n must be 6, 7 or 8"); return RG_ERR_ARG;
        }
    }
    c->last_stats[7] += 1;
    RG_CUDA(cudaGetLastError());
    return RG_OK;
}

// per-view frame + packed FP32 points of the voting correspondences
static int pnp_prepare(Ctx* c, cudaStream_t st, const double* X, const double* y, const FPlan& plan, double thr2,
                       PnpFrame** fr_out) {
    const int V = plan.P;
    int rc;
    const size_t bbox_bytes = ((sizeof(int) * 10 * (size_t)V + 63) / 64) * 64;
    if ((rc = ensure(c->bbox, bbox_bytes + sizeof(PnpFrame) * (size_t)V))) return rc;
    if ((rc = ensure(c->X32, sizeof(float4) * 3 * (size_t)std::max<long long>(plan.N32tot / 2, 1)))) return rc;
    int* bbox = (int*)c->bbox.ptr;
    PnpFrame* fr = (PnpFrame*)((char*)c->bbox.ptr + bbox_bytes);
    const PairInfo* pi = (const PairInfo*)c->pair_info.ptr;
    pnp_bbox_init<<<ceil_div(V * 10, 256), 256, 0, st>>>(bbox, V);
    const int nbx = std::max(1, std::min(c->sm_count * 2, ceil_div(plan.maxN, 1024)));
    pnp_bbox<<<dim3(nbx, V), 256, 0, st>>>(X, y, pi, bbox);
    pnp_frame<<<ceil_div(V, 128), 128, 0, st>>>(fr, bbox, V, thr2);
    const int nbn = std::max(1, std::min(c->sm_count * 4, ceil_div(plan.maxN / 2 + kSub, 256)));
    pnp_normalise<<<dim3(nbn, V), 256, 0, st>>>(X, y, pi, fr, (float4*)c->X32.ptr);
    c->last_stats[7] += 4;
    RG_CUDA(cudaGetLastError());
    *fr_out = fr;
    return RG_OK;
}

static int pnp_workspace(Ctx* c, const FPlan& plan) {
    int rc;
    const size_t H = (size_t)std::max<long long>(plan.Htot, 1);
    if ((rc = ensure(c->pose64, sizeof(double) * 12 * H))) return rc;
    if ((rc = ensure(c->pose32, sizeof(Pose32) * H))) return rc;
    if ((rc = ensure(c->flags, H))) return rc;
    if ((rc = ensure(c->stats, sizeof(unsigned long long) * 8))) return rc;
    if ((rc = ensure(c->best, sizeof(int2) * (size_t)std::max(plan.P, 1)))) return rc;
    if ((rc = ensure_pinned(c->h_stats, sizeof(unsigned long long) * 8))) return rc;
    c->prep_pts = nullptr;                            // the F path's prepared points do not survive a PnP call's PairInfo table
    return RG_OK;
}

static int pnp_score_launch(Ctx* c, cudaStream_t st, const FPlan& plan, const double* X, const double* y, double thr2,
                            int score_path) {
    ScoreState s;
    int rc = score_state_layout(c, plan.P, plan.Htot, 0, s);
    if (rc) return rc;
    unsigned long long* stats = (unsigned long long*)c->stats.ptr;
    RG_CUDA(cudaMemsetAsync(c->state.ptr, 0, s.bytes, st));     // counts + work counter + flag-list size + overflow marks
    RG_CUDA(cudaMemsetAsync(stats, 0, sizeof(unsigned long long) * 8, st));
    if (plan.Htot == 0 || (score_path == SCORE_FP32_GUARDED && plan.n_items == 0)) {
        prof_mark(c, st, 3);
        return RG_OK;
    }
    PairInfo* pi = (PairInfo*)c->pair_info.ptr;
    if (score_path == SCORE_FP32_GUARDED) {
        int bps = 1;
        if ((rc = score_blocks_per_sm<PnpPolicy>(&bps))) return rc;
        FlagList fl = flag_list_for(c, s, plan.evals, &rc);
        if (rc) return rc;
        constexpr size_t smem = score_smem_bytes<PnpPolicy>();
        const int grid = std::min(plan.n_items, c->sm_count * bps);
        score_packed<PnpPolicy><<<grid, kScoreThreads, smem, st>>>((const float4*)c->X32.ptr, (const Pose32*)c->pose32.ptr, pi,
                                                                  plan.P, plan.n_items, s.counts, fl, s.work);
        prof_mark(c, st, 3);
        PnpFix::Params fp{(const float4*)c->X32.ptr, X, y, (const Pose32*)c->pose32.ptr, (const double*)c->pose64.ptr,
                          pi, plan.P, thr2};
        fixup_list<PnpFix><<<fixup_grid(c, plan.evals), 256, 0, st>>>(fp, fl, (int)plan.Htot, s.counts, stats);
        c->last_stats[7] += 2;
    } else {
        const int zs = std::max(1, std::min(64, ceil_div(plan.maxN, 2048)));
        pnp_score_fp64<<<dim3(std::max(1, ceil_div(plan.maxH, 128)), plan.P, zs), 128, 0, st>>>(
            X, y, pi, (const double*)c->pose64.ptr, thr2, s.counts);
        prof_mark(c, st, 3);
        c->last_stats[7] += 1;
    }
    RG_CUDA(cudaGetLastError());
    return RG_OK;
}

// views batched in CSR form; n_vote (host, optional) = per-view number of leading correspondences that vote
static int pnp_ransac_dev(Ctx* c, cudaStream_t st, int V, const double* X, const double* y, const int* view_off,
                          const int* n_vote, const int* idx, const int* hyp_off, int n, double thr2, int score_path,
                          int* best_idx, int* best_count, double* Rt, unsigned char* mask, int hyp_first = 0,
                          unsigned long long* keys = nullptr) {
    RG_CHECK_ARG(n >= 6 && n <= 8, "PnP sample size n must be 6, 7 or 8 (DLT needs m >= 6)");
    RG_CHECK_ARG(thr2 >= 0.0 && std::isfinite(thr2), "thr2 must be finite and >= 0");
    RG_CHECK_ARG(score_path == SCORE_FP32_GUARDED || score_path == SCORE_FP64, "unknown scoring path");
    RG_CUDA(cudaSetDevice(c->device));
    FPlan plan;
    int bps = 1, rc = score_blocks_per_sm<PnpPolicy>(&bps);
    if (rc) return rc;
    if ((rc = f_plan(c, st, V, view_off, hyp_off, plan, bps, n_vote, hyp_first))) return rc;
    for (int v = 0; v < V; ++v)
        RG_CHECK_ARG(hyp_off[v + 1] == hyp_off[v] || view_off[v + 1] - view_off[v] >= n, "a view with hypotheses needs at least n correspondences");
    if ((rc = pnp_workspace(c, plan))) return rc;
    c->last_stats[7] = 0;
    c->last_passes = 1;
    if (V == 0) return RG_OK;
    // a zero threshold makes the FP32 frame singular: score such calls in FP64 only
    if (!(thr2 > 0.0)) score_path = SCORE_FP64;
    PnpFrame* fr = nullptr;
    prof_mark(c, st, 0);
    if ((rc = pnp_prepare(c, st, X, y, plan, thr2 > 0.0 ? thr2 : 1.0, &fr))) return rc;
    prof_mark(c, st, 1);
    if ((rc = pnp_solve_launch(c, st, X, y, idx, plan, n, fr))) return rc;
    prof_mark(c, st, 2);
    if ((rc = pnp_score_launch(c, st, plan, X, y, thr2, score_path))) return rc;
    prof_mark(c, st, 4);
    int2* best = (int2*)c->best.ptr;
    const PairInfo* pi = (const PairInfo*)c->pair_info.ptr;
    if (mask == nullptr) {                            // nothing follows the argmax: it publishes the winning poses itself
        argmax_counts<<<V, 256, 0, st>>>((const int*)c->counts_ptr, pi, best, (const unsigned char*)c->flags.ptr,
                                         (unsigned long long*)c->stats.ptr, keys, (const double*)c->pose64.ptr, 12, Rt, best_idx,
                                         best_count);
        c->last_stats[7] += 1;
    } else {
        argmax_counts<<<V, 256, 0, st>>>((const int*)c->counts_ptr, pi, best, (const unsigned char*)c->flags.ptr,
                                         (unsigned long long*)c->stats.ptr, keys);
        const int nbx = std::max(1, std::min(c->sm_count * 4, ceil_div(std::max(plan.maxN, 1), 256)));
        pnp_finish<<<dim3(nbx, V), 256, 0, st>>>(X, y, pi, (const double*)c->pose64.ptr, best, thr2, mask, Rt, best_idx,
                                                best_count);
        c->last_stats[7] += 2;
    }
    prof_mark(c, st, 5);
    RG_CUDA(cudaGetLastError());
    RG_CUDA(cudaMemcpyAsync(c->h_stats.ptr, c->stats.ptr, sizeof(unsigned long long) * 8, cudaMemcpyDeviceToHost, st));
    return RG_OK;
}

// reduce a tall design matrix to its packed triangular factor; returns the device pointer of the final factor
template <int COLS, class Gen>
static int tsqr_reduce(Ctx* c, cudaStream_t st, Gen gen, int nrows, double** R_final) {
    constexpr int SZ = PackedR<COLS>::SIZE;
    int T = std::max(1, std::min(8192, ceil_div(nrows, 64)));
    int rc;
    if ((rc = ensure(c->d_out_c, sizeof(double) * SZ * ((size_t)T + (size_t)ceil_div(T, 8) + 8)))) return rc;
    double* bufA = (double*)c->d_out_c.ptr;
    double* bufB = bufA + (size_t)SZ * T;
    tsqr_stage<COLS, Gen><<<ceil_div(T, 64), 64, 0, st>>>(gen, nrows, ceil_div(nrows, T), T, bufA);
    c->last_stats[7] += 1;
    double* cur = bufA;
    double* nxt = bufB;
    while (T > 1) {
        const int T2 = ceil_div(T, 8);
        PackedRows<COLS> pr{cur};
        tsqr_stage<COLS, PackedRows<COLS>><<<ceil_div(T2, 64), 64, 0, st>>>(pr, T * COLS, 8 * COLS, T2, nxt);
        c->last_stats[7] += 1;
        std::swap(cur, nxt);
        T = T2;
    }
    RG_CUDA(cudaGetLastError());
    *R_final = cur;
    return RG_OK;
}

}  // namespace rg

using namespace rg;

extern "C" {

int rg_pnp_ransac_batched_dev(void* ctx, void* stream, int V, const double* X_dev, const double* y_dev,
                              const int* view_off_host, const int* n_vote_host, const int* idx_dev, const int* hyp_off_host,
                              int n, double thr2, int score_path, int* best_idx_dev, int* best_count_dev, double* Rt_dev,
                              unsigned char* mask_dev) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(V >= 0 && view_off_host && hyp_off_host, "bad view table");
    RG_CHECK_ARG(best_idx_dev && best_count_dev && Rt_dev, "output pointers are null");
    return pnp_ransac_dev((Ctx*)ctx, (cudaStream_t)stream, V, X_dev, y_dev, view_off_host, n_vote_host, idx_dev,
                          hyp_off_host, n, thr2, score_path, best_idx_dev, best_count_dev, Rt_dev, mask_dev);
}

// hypothesis-split mode: this rank's hypotheses are [hyp_index_base, hyp_index_base + H_v) of every view; key_dev (V, optional)
// receives the cross-GPU argmax keys (count << 32 | ~global index)
int rg_pnp_ransac_batched_dev2(void* ctx, void* stream, int V, const double* X_dev, const double* y_dev,
                               const int* view_off_host, const int* n_vote_host, const int* idx_dev, const int* hyp_off_host,
                               int n, double thr2, int score_path, int hyp_index_base, int* best_idx_dev, int* best_count_dev,
                               double* Rt_dev, unsigned char* mask_dev, unsigned long long* key_dev) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(V >= 0 && view_off_host && hyp_off_host && hyp_index_base >= 0, "bad view table");
    RG_CHECK_ARG(best_idx_dev && best_count_dev && Rt_dev, "output pointers are null");
    return pnp_ransac_dev((Ctx*)ctx, (cudaStream_t)stream, V, X_dev, y_dev, view_off_host, n_vote_host, idx_dev,
                          hyp_off_host, n, thr2, score_path, best_idx_dev, best_count_dev, Rt_dev, mask_dev, hyp_index_base,
                          key_dev);
}

int rg_pnp_ransac_dev(void* ctx, void* stream, int N, int N_sel, const double* X_dev, const double* y_dev, int H, int n,
                      const int* idx_dev, double thr2, int score_path, int* best_idx_dev, int* best_count_dev, double* Rt_dev,
                      unsigned char* mask_dev) {
    RG_CHECK_ARG(N >= 0 && H >= 0, "negative size");
    const int view_off[2] = {0, N}, hyp_off[2] = {0, H}, vote[1] = {N_sel};
    return rg_pnp_ransac_batched_dev(ctx, stream, 1, X_dev, y_dev, view_off, vote, idx_dev, hyp_off, n, thr2, score_path,
                                     best_idx_dev, best_count_dev, Rt_dev, mask_dev);
}

int rg_pnp_ransac_batched_host(void* ctx, void* stream, int V, const double* X, const double* y, const int* view_off,
                               const int* n_vote, const int* idx, const int* hyp_off, int n, double thr2, int score_path,
                               int* best_idx, int* best_count, double* Rt, unsigned char* mask, int* counts, double* poses,
                               unsigned char* flags) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(V >= 0 && view_off && hyp_off && n >= 6 && n <= 8, "bad view table / sample size (n must be 6, 7 or 8)");
    RG_CHECK_ARG(best_idx && best_count && Rt, "output pointers are null");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    if (V == 0) return RG_OK;
    const size_t N = (size_t)view_off[V], H = (size_t)hyp_off[V];
    RG_CHECK_ARG((N == 0 || (X && y)) && (H == 0 || idx), "input pointers are null");
    int rc;
    if ((rc = ensure(c->d_in_a, sizeof(double) * 3 * std::max<size_t>(N, 1)))) return rc;
    if ((rc = ensure(c->d_in_c, sizeof(double) * 2 * std::max<size_t>(N, 1)))) return rc;
    if ((rc = ensure(c->d_in_b, sizeof(int) * (size_t)n * std::max<size_t>(H, 1)))) return rc;
    if ((rc = ensure(c->d_out_a, sizeof(int) * 2 * (size_t)V))) return rc;
    if ((rc = ensure(c->d_out_b, sizeof(double) * 12 * (size_t)V))) return rc;
    if (mask && (rc = ensure(c->d_out_d, std::max<size_t>(N, 1)))) return rc;
    if (N) {
        RG_CUDA(cudaMemcpyAsync(c->d_in_a.ptr, X, sizeof(double) * 3 * N, cudaMemcpyHostToDevice, st));
        RG_CUDA(cudaMemcpyAsync(c->d_in_c.ptr, y, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, st));
    }
    if (H) RG_CUDA(cudaMemcpyAsync(c->d_in_b.ptr, idx, sizeof(int) * (size_t)n * H, cudaMemcpyHostToDevice, st));
    int* d_i = (int*)c->d_out_a.ptr;
    rc = pnp_ransac_dev(c, st, V, (const double*)c->d_in_a.ptr, (const double*)c->d_in_c.ptr, view_off, n_vote,
                        (const int*)c->d_in_b.ptr, hyp_off, n, thr2, score_path, d_i, d_i + V, (double*)c->d_out_b.ptr,
                        mask ? (unsigned char*)c->d_out_d.ptr : nullptr);
    if (rc) return rc;
    RG_CUDA(cudaMemcpyAsync(best_idx, d_i, sizeof(int) * (size_t)V, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaMemcpyAsync(best_count, d_i + V, sizeof(int) * (size_t)V, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaMemcpyAsync(Rt, c->d_out_b.ptr, sizeof(double) * 12 * (size_t)V, cudaMemcpyDeviceToHost, st));
    if (mask && N) RG_CUDA(cudaMemcpyAsync(mask, c->d_out_d.ptr, N, cudaMemcpyDeviceToHost, st));
    if (counts && H) RG_CUDA(cudaMemcpyAsync(counts, c->counts_ptr, sizeof(int) * H, cudaMemcpyDeviceToHost, st));
    if (poses && H) RG_CUDA(cudaMemcpyAsync(poses, c->pose64.ptr, sizeof(double) * 12 * H, cudaMemcpyDeviceToHost, st));
    if (flags && H) RG_CUDA(cudaMemcpyAsync(flags, c->flags.ptr, H, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaStreamSynchronize(st));
    // sample indices are validated where they are read (the solver clamps them and sets flag bit 2): no host pass over idx
    if (c->h_stats.ptr && ((const unsigned long long*)c->h_stats.ptr)[4] != 0) {
        set_error("invalid argument: %llu hypotheses have a sample index outside [0, N) of their view",
                  ((const unsigned long long*)c->h_stats.ptr)[4]);
        return RG_ERR_ARG;
    }
    return RG_OK;
}

int rg_pnp_ransac_host(void* ctx, void* stream, int N, int N_sel, const double* X, const double* y, int H, int n,
                       const int* idx, double thr2, int score_path, int* best_idx, int* best_count, double* R, double* t,
                       unsigned char* mask, int* counts, double* poses, unsigned char* flags) {
    RG_CHECK_ARG(N >= 0 && H >= 0, "negative size");
    RG_CHECK_ARG(R && t, "output pointers are null");
    const int view_off[2] = {0, N}, hyp_off[2] = {0, H}, vote[1] = {N_sel};
    double Rt[12];
    int rc = rg_pnp_ransac_batched_host(ctx, stream, 1, X, y, view_off, vote, idx, hyp_off, n, thr2, score_path, best_idx,
                                        best_count, Rt, mask, counts, poses, flags);
    if (rc) return rc;
    for (int k = 0; k < 9; ++k) R[k] = Rt[k];
    for (int k = 0; k < 3; ++k) t[k] = Rt[9 + k];
    return RG_OK;
}

int rg_pnp_score_count_host(void* ctx, void* stream, int N, const double* X, const double* y, int H, const double* poses,
                            double thr2, int score_path, int* counts) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(N >= 0 && H >= 0 && counts, "bad sizes / null output");
    RG_CHECK_ARG(thr2 >= 0.0 && std::isfinite(thr2), "thr2 must be finite and >= 0");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    if (H == 0) return RG_OK;
    RG_CHECK_ARG(poses && (N == 0 || (X && y)), "input pointers are null");
    const int pair_off[2] = {0, N}, hyp_off[2] = {0, H};
    FPlan plan;
    int bps = 1, rc = score_blocks_per_sm<PnpPolicy>(&bps);
    if (rc) return rc;
    if ((rc = f_plan(c, st, 1, pair_off, hyp_off, plan, bps))) return rc;
    if ((rc = pnp_workspace(c, plan))) return rc;
    if ((rc = ensure(c->d_in_a, sizeof(double) * 3 * std::max<size_t>((size_t)N, 1)))) return rc;
    if ((rc = ensure(c->d_in_c, sizeof(double) * 2 * std::max<size_t>((size_t)N, 1)))) return rc;
    if (N) {
        RG_CUDA(cudaMemcpyAsync(c->d_in_a.ptr, X, sizeof(double) * 3 * (size_t)N, cudaMemcpyHostToDevice, st));
        RG_CUDA(cudaMemcpyAsync(c->d_in_c.ptr, y, sizeof(double) * 2 * (size_t)N, cudaMemcpyHostToDevice, st));
    }
    RG_CUDA(cudaMemcpyAsync(c->pose64.ptr, poses, sizeof(double) * 12 * (size_t)H, cudaMemcpyHostToDevice, st));
    c->last_stats[7] = 0;
    if (!(thr2 > 0.0)) score_path = SCORE_FP64;
    PnpFrame* fr = nullptr;
    const double* dX = (const double*)c->d_in_a.ptr;
    const double* dy = (const double*)c->d_in_c.ptr;
    if ((rc = pnp_prepare(c, st, dX, dy, plan, thr2 > 0.0 ? thr2 : 1.0, &fr))) return rc;
    pnp_make_pose32<<<ceil_div(H, 256), 256, 0, st>>>((const double*)c->pose64.ptr, (const PairInfo*)c->pair_info.ptr, 1, H, fr,
                                                      (Pose32*)c->pose32.ptr);
    c->last_stats[7] += 1;
    if ((rc = pnp_score_launch(c, st, plan, dX, dy, thr2, score_path))) return rc;
    RG_CUDA(cudaMemcpyAsync(c->h_stats.ptr, c->stats.ptr, sizeof(unsigned long long) * 8, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaMemcpyAsync(counts, c->counts_ptr, sizeof(int) * (size_t)H, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaStreamSynchronize(st));
    return RG_OK;
}

int rg_pnp_minimize_host(void* ctx, void* stream, int m, const double* X, const double* y, double* R, double* t) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(m >= 6, "pnp_minimize needs m >= 6 correspondences");
    RG_CHECK_ARG(X && y && R && t, "null buffers");
    RG_CHECK_ARG((long long)m * 3 < (1ll << 31), "too many correspondences");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    int rc;
    if ((rc = ensure(c->d_in_a, sizeof(double) * 3 * (size_t)m))) return rc;
    if ((rc = ensure(c->d_in_c, sizeof(double) * 2 * (size_t)m))) return rc;
    if ((rc = ensure(c->d_out_b, sizeof(double) * 16))) return rc;
    RG_CUDA(cudaMemcpyAsync(c->d_in_a.ptr, X, sizeof(double) * 3 * (size_t)m, cudaMemcpyHostToDevice, st));
    RG_CUDA(cudaMemcpyAsync(c->d_in_c.ptr, y, sizeof(double) * 2 * (size_t)m, cudaMemcpyHostToDevice, st));
    c->last_stats[7] = 0;
    PnpRows gen{(const double*)c->d_in_a.ptr, (const double*)c->d_in_c.ptr};
    double* Rf = nullptr;
    if ((rc = tsqr_reduce<12, PnpRows>(c, st, gen, 3 * m, &Rf))) return rc;
    pnp_min_finish<<<1, 32, 0, st>>>(Rf, (double*)c->d_out_b.ptr);
    c->last_stats[7] += 1;
    RG_CUDA(cudaGetLastError());
    RG_CUDA(cudaMemcpyAsync(R, c->d_out_b.ptr, sizeof(double) * 9, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaMemcpyAsync(t, (double*)c->d_out_b.ptr + 9, sizeof(double) * 3, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaStreamSynchronize(st));
    return RG_OK;
}

int rg_fmatrix_stls_host(void* ctx, void* stream, int N, const double* pl, const double* pr, double* F9) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(N >= 8, "fmatrix_stls needs N >= 8 correspondences");
    RG_CHECK_ARG(pl && pr && F9, "null buffers");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    int rc;
    if ((rc = ensure(c->d_in_a, sizeof(double) * (4 * (size_t)N + 32)))) return rc;
    double* d = (double*)c->d_in_a.ptr;
    double* dpl = d + 32;
    double* dpr = dpl + 2 * (size_t)N;
    RG_CUDA(cudaMemcpyAsync(dpl, pl, sizeof(double) * 2 * (size_t)N, cudaMemcpyHostToDevice, st));
    RG_CUDA(cudaMemcpyAsync(dpr, pr, sizeof(double) * 2 * (size_t)N, cudaMemcpyHostToDevice, st));
    c->last_stats[7] = 0;
    stls_stats<<<1, 256, 0, st>>>(dpl, dpr, N, d);
    c->last_stats[7] += 1;
    StlsRows gen{dpl, dpr, d, N};
    double* Rf = nullptr;
    if ((rc = tsqr_reduce<9, StlsRows>(c, st, gen, N, &Rf))) return rc;
    stls_finish<<<1, 32, 0, st>>>(Rf, d, d + 16);
    c->last_stats[7] += 1;
    RG_CUDA(cudaGetLastError());
    RG_CUDA(cudaMemcpyAsync(F9, d + 16, sizeof(double) * 9, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaStreamSynchronize(st));
    return RG_OK;
}

}  // extern "C"
