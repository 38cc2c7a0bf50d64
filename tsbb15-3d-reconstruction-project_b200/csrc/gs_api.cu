// Host orchestration + C ABI of the device-resident gold-standard refinement (SURVEY.md section 8f row N4).
#include "gs_kernels.cuh"
#include "plan.cuh"

namespace rg {

// the kernels that depend on the loss (gs_rho / gs_blocks_w inside them)
struct GsLossKernels {
    decltype(&gs_fused<LOSS_LINEAR>) fused;
    decltype(&gs_accumulate<LOSS_LINEAR>) accumulate;
    decltype(&gs_trial<LOSS_LINEAR>) trial;
};

template <int L>
static GsLossKernels gs_loss_kernels() { return {gs_fused<L>, gs_accumulate<L>, gs_trial<L>}; }

static bool gs_loss_kernels(int loss, GsLossKernels& k) {
    switch (loss) {
        case LOSS_LINEAR: k = gs_loss_kernels<LOSS_LINEAR>(); return true;
        case LOSS_SOFT_L1: k = gs_loss_kernels<LOSS_SOFT_L1>(); return true;
        case LOSS_HUBER: k = gs_loss_kernels<LOSS_HUBER>(); return true;
        case LOSS_CAUCHY: k = gs_loss_kernels<LOSS_CAUCHY>(); return true;
        case LOSS_ARCTAN: k = gs_loss_kernels<LOSS_ARCTAN>(); return true;
        default: return false;
    }
}

// loss (LOSS_*) and f_scale = C (pixels, the units of pts64): every scalar residual f contributes C^2 rho((f / C)^2) to
// twice the cost.
static int gold_standard_dev(Ctx* c, cudaStream_t st, int P, const double* pts64, const int* pair_off, const double* F0,
                             const unsigned char* mask, int max_iter, double ftol, int loss, double f_scale, double* F_gold,
                             double* cost, int* iters, int* status, double* X_out, bool host_paced) {
    RG_CHECK_ARG(P >= 0 && pair_off != nullptr, "bad pair table");
    RG_CHECK_ARG(pair_off[0] == 0, "pair_off must start at 0");
    for (int p = 0; p < P; ++p) RG_CHECK_ARG(pair_off[p + 1] >= pair_off[p], "pair_off must be non-decreasing");
    RG_CHECK_ARG(max_iter >= 0 && max_iter <= 10000, "max_iter must be in [0, 10000]");
    RG_CHECK_ARG(ftol >= 0.0 && std::isfinite(ftol), "ftol must be finite and >= 0");
    GsLossKernels kern;
    RG_CHECK_ARG(gs_loss_kernels(loss, kern), "loss must be one of RG_LOSS_LINEAR .. RG_LOSS_ARCTAN");
    const double ic = 1.0 / f_scale, c2 = f_scale * f_scale;
    RG_CHECK_ARG(std::isfinite(f_scale) && f_scale > 0.0 && std::isfinite(ic) && std::isfinite(c2) && c2 > 0.0,
                 "f_scale must be finite and > 0 (with a finite, non-zero square)");
    RG_CUDA(cudaSetDevice(c->device));
    c->last_stats[7] = 0;
    if (P == 0) return RG_OK;
    const size_t N = (size_t)pair_off[P], p = (size_t)P;
    RG_CHECK_ARG(F0 && F_gold && (N == 0 || pts64), "null buffers");
    int maxN = 0;
    for (int q = 0; q < P; ++q) maxN = std::max(maxN, pair_off[q + 1] - pair_off[q]);
    // workspace: GsPair[P] | sums[P x kGsSums] | C1, C2 (P x 12) | x1n, x2n (N double2) | Xcur, Xtrial (3N) | pair_off
    const size_t bytes = sizeof(GsPair) * p + sizeof(double) * (kGsSums * p + 24 * p + 4 * N + 6 * N + 2) +
                         sizeof(int) * (p + 1 + (size_t)max_iter) + 64;
    int rc;
    if ((rc = ensure(c->gs_ws, bytes))) return rc;
    char* w = (char*)c->gs_ws.ptr;
    GsPair* gp = (GsPair*)w;                       w += sizeof(GsPair) * p;
    w = (char*)(((uintptr_t)w + 15) & ~(uintptr_t)15);
    double2* x1n = (double2*)w;                    w += sizeof(double2) * N;
    double2* x2n = (double2*)w;                    w += sizeof(double2) * N;
    double* sums = (double*)w;                     w += sizeof(double) * kGsSums * p;
    double* C1 = (double*)w;                       w += sizeof(double) * 12 * p;
    double* C2 = (double*)w;                       w += sizeof(double) * 12 * p;
    double* Xws = (double*)w;                      w += sizeof(double) * 3 * N;
    double* Xtrial = (double*)w;                   w += sizeof(double) * 3 * N;
    int* doff = (int*)w;                           w += sizeof(int) * (p + 1);
    int* active = (int*)w;                         // pairs still running after iteration it (host-paced loop)
    double* Xcur = X_out ? X_out : Xws;

    gs_init<<<ceil_div(P, 64), 64, 0, st>>>(F0, P, 1e-3, gp, C1, C2);
    RG_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * kGsSums * p, st));
    int launches = 1;
    if (N) {
        Mat3 I3;
        for (int k = 0; k < 9; ++k) I3.m[k] = (k % 4 == 0) ? 1.0 : 0.0;
        tv_normalise<<<ceil_div((long long)N, 256), 256, 0, st>>>((const double4*)pts64, mask, (int)N, I3, x1n, x2n);
        RG_CUDA(cudaGetLastError());
        // starting points: lab3.triangulate_optimal of every inlier with the cameras of lab3.fmatrix_cameras (fun.py:345-352)
        if ((rc = triangulate_dev(c, st, P, C1, C2, pair_off, (const double*)x1n, (const double*)x2n, TRI_OPTIMAL, Xcur)))
            return rc;
        launches += 1 + (int)c->last_stats[7];
        RG_CUDA(cudaEventSynchronize(c->staging_free[0]));
        if ((rc = ensure_pinned(c->h_stage[0], sizeof(int) * (p + 1)))) return rc;
        memcpy(c->h_stage[0].ptr, pair_off, sizeof(int) * (p + 1));
        RG_CUDA(cudaMemcpyAsync(doff, c->h_stage[0].ptr, sizeof(int) * (p + 1), cudaMemcpyHostToDevice, st));
        RG_CUDA(cudaEventRecord(c->staging_free[0], st));
        if (maxN <= kGsFusedMaxPts && !c->opt_gs_multi) {
            // small pairs: the whole LM loop of a pair in one CTA, one launch (gs_fused)
            kern.fused<<<P, kGsFusedThreads, 0, st>>>((const double4*)pts64, mask, doff, gp, Xcur, Xtrial, C1, ftol, max_iter, ic,
                                                          c2);
            launches += 1;
            RG_CUDA(cudaGetLastError());
        } else {
            const int nbx = std::max(1, std::min(32, ceil_div(maxN, kGsThreads * 4)));
            const dim3 grid(nbx, P);
            // host_paced (the host-buffer entry point, which ends with a synchronisation anyway): the number of pairs still
            // running is copied to pinned memory after every iteration and the enqueue loop stays at most two iterations
            // ahead of the device: it stops two iterations after the last pair converged instead of enqueueing 4 x max_iter
            // launches that return at once.
            volatile int* h_act = nullptr;
            if (host_paced && max_iter > 2) {
                if ((rc = ensure_pinned(c->h_ba_flags, sizeof(int) * (size_t)max_iter))) return rc;
                h_act = (volatile int*)c->h_ba_flags.ptr;
                for (int i = 0; i < 2; ++i)
                    if (!c->ba_iter_ev[i]) RG_CUDA(cudaEventCreateWithFlags(&c->ba_iter_ev[i], cudaEventDisableTiming));
                RG_CUDA(cudaMemsetAsync(active, 0, sizeof(int) * (size_t)max_iter, st));
            }
            for (int it = 0; it < max_iter; ++it) {
                if (h_act && it >= 2) {
                    RG_CUDA(cudaEventSynchronize(c->ba_iter_ev[it & 1]));      // iteration it - 2 has finished
                    if (h_act[it - 2] == 0) break;
                }
                kern.accumulate<<<grid, kGsThreads, 0, st>>>((const double4*)pts64, mask, doff, gp, Xcur, Xtrial, sums, ic, c2);
                gs_solve<<<ceil_div(P, kGsSolveWarps), 32 * kGsSolveWarps, 0, st>>>(gp, sums, P);
                kern.trial<<<grid, kGsThreads, 0, st>>>((const double4*)pts64, mask, doff, gp, Xcur, Xtrial, ic, c2);
                gs_accept<<<ceil_div(P, 32), 32, 0, st>>>(gp, sums, P, ftol, max_iter, h_act ? active + it : nullptr);
                launches += 4;
                if (h_act) {
                    RG_CUDA(cudaMemcpyAsync((void*)&h_act[it], active + it, sizeof(int), cudaMemcpyDeviceToHost, st));
                    RG_CUDA(cudaEventRecord(c->ba_iter_ev[it & 1], st));
                }
            }
            RG_CUDA(cudaGetLastError());
            gs_finish<<<grid, kGsThreads, 0, st>>>(doff, gp, Xcur, Xtrial, C1);
            launches += 1;
        }
    }
    // F_gold = lab3.fmatrix_from_cameras(C1, [I | 0])   (fun.py:368)
    PairGeom* G = nullptr;
    {
        const size_t gbytes = sizeof(PairGeom) * p;
        if ((rc = ensure(c->geom, gbytes + sizeof(int) * (p + 1)))) return rc;
        G = (PairGeom*)c->geom.ptr;
        geom_prepare<<<ceil_div(P, 64), 64, 0, st>>>(C1, C2, P, G);
        geom_export_F<<<ceil_div((long long)P * 9, 256), 256, 0, st>>>(G, P, F_gold);
        gs_export<<<ceil_div(P, 64), 64, 0, st>>>(gp, P, cost, iters, status);
        launches += 3;
    }
    RG_CUDA(cudaGetLastError());
    c->last_stats[7] = launches;
    return RG_OK;
}

}  // namespace rg

using namespace rg;

extern "C" {

int rg_gold_standard_dev2(void* ctx, void* stream, int P, const double* pts64_dev, const int32_t* pair_off_host,
                          const double* F0_dev, const unsigned char* mask_dev, int max_iter, double ftol, int loss, double f_scale,
                          double* F_gold_dev, double* cost_dev, int32_t* iters_dev, int32_t* status_dev, double* X_dev) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    return gold_standard_dev((Ctx*)ctx, (cudaStream_t)stream, P, pts64_dev, pair_off_host, F0_dev, mask_dev, max_iter, ftol, loss,
                             f_scale, F_gold_dev, cost_dev, iters_dev, status_dev, X_dev, false);
}

int rg_gold_standard_dev(void* ctx, void* stream, int P, const double* pts64_dev, const int32_t* pair_off_host,
                         const double* F0_dev, const unsigned char* mask_dev, int max_iter, double ftol, double* F_gold_dev,
                         double* cost_dev, int32_t* iters_dev, int32_t* status_dev, double* X_dev) {
    return rg_gold_standard_dev2(ctx, stream, P, pts64_dev, pair_off_host, F0_dev, mask_dev, max_iter, ftol, LOSS_LINEAR, 1.0,
                                 F_gold_dev, cost_dev, iters_dev, status_dev, X_dev);
}

int rg_gold_standard_host2(void* ctx, void* stream, int P, const double* pts64, const int32_t* pair_off, const double* F0,
                           const unsigned char* mask, int max_iter, double ftol, int loss, double f_scale, double* F_gold,
                           double* cost, int32_t* iters, int32_t* status, double* X) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(P >= 0 && pair_off != nullptr, "bad pair table");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    if (P == 0) return RG_OK;
    RG_CHECK_ARG(pair_off[0] == 0 && pair_off[P] >= 0, "bad pair table");
    const size_t N = (size_t)pair_off[P], p = (size_t)P;
    RG_CHECK_ARG(F0 && F_gold && (N == 0 || pts64), "null buffers");
    int rc;
    if ((rc = ensure(c->d_in_a, sizeof(double) * 4 * std::max<size_t>(N, 1)))) return rc;
    if ((rc = ensure(c->d_in_b, sizeof(double) * 9 * p))) return rc;
    if ((rc = ensure(c->d_in_c, std::max<size_t>(N, 1)))) return rc;
    if ((rc = ensure(c->d_out_b, sizeof(double) * (9 * p + p + 3 * std::max<size_t>(N, 1)) + sizeof(int) * 2 * p))) return rc;
    if (N) RG_CUDA(cudaMemcpyAsync(c->d_in_a.ptr, pts64, sizeof(double) * 4 * N, cudaMemcpyHostToDevice, st));
    RG_CUDA(cudaMemcpyAsync(c->d_in_b.ptr, F0, sizeof(double) * 9 * p, cudaMemcpyHostToDevice, st));
    if (mask && N) RG_CUDA(cudaMemcpyAsync(c->d_in_c.ptr, mask, N, cudaMemcpyHostToDevice, st));
    double* dF = (double*)c->d_out_b.ptr;
    double* dcost = dF + 9 * p;
    double* dX = dcost + p;
    int* dit = (int*)(dX + 3 * std::max<size_t>(N, 1));
    int* dst = dit + p;
    rc = gold_standard_dev(c, st, P, (const double*)c->d_in_a.ptr, pair_off, (const double*)c->d_in_b.ptr,
                           (mask && N) ? (const unsigned char*)c->d_in_c.ptr : nullptr, max_iter, ftol, loss, f_scale, dF, dcost,
                           dit, dst, dX, true);
    if (rc) return rc;
    RG_CUDA(cudaMemcpyAsync(F_gold, dF, sizeof(double) * 9 * p, cudaMemcpyDeviceToHost, st));
    if (cost) RG_CUDA(cudaMemcpyAsync(cost, dcost, sizeof(double) * p, cudaMemcpyDeviceToHost, st));
    if (iters) RG_CUDA(cudaMemcpyAsync(iters, dit, sizeof(int) * p, cudaMemcpyDeviceToHost, st));
    if (status) RG_CUDA(cudaMemcpyAsync(status, dst, sizeof(int) * p, cudaMemcpyDeviceToHost, st));
    if (X && N) RG_CUDA(cudaMemcpyAsync(X, dX, sizeof(double) * 3 * N, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaStreamSynchronize(st));
    return RG_OK;
}

int rg_gold_standard_host(void* ctx, void* stream, int P, const double* pts64, const int32_t* pair_off, const double* F0,
                          const unsigned char* mask, int max_iter, double ftol, double* F_gold, double* cost, int32_t* iters,
                          int32_t* status, double* X) {
    return rg_gold_standard_host2(ctx, stream, P, pts64, pair_off, F0, mask, max_iter, ftol, LOSS_LINEAR, 1.0, F_gold, cost,
                                  iters, status, X);
}

int rg_fmatrix_residuals_gs_host(void* ctx, void* stream, int N, const double* params, const double* pl, const double* pr,
                                 double* out) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(N >= 0, "negative size");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    if (N == 0) return RG_OK;
    RG_CHECK_ARG(params && pl && pr && out, "null buffers");
    const size_t n = (size_t)N;
    int rc;
    if ((rc = ensure(c->d_in_a, sizeof(double) * (12 + 3 * n + 4 * n)))) return rc;
    if ((rc = ensure(c->d_out_b, sizeof(double) * 4 * n))) return rc;
    double* dp = (double*)c->d_in_a.ptr;
    double* dpl = dp + 12 + 3 * n;
    double* dpr = dpl + 2 * n;
    RG_CUDA(cudaMemcpyAsync(dp, params, sizeof(double) * (12 + 3 * n), cudaMemcpyHostToDevice, st));
    RG_CUDA(cudaMemcpyAsync(dpl, pl, sizeof(double) * 2 * n, cudaMemcpyHostToDevice, st));
    RG_CUDA(cudaMemcpyAsync(dpr, pr, sizeof(double) * 2 * n, cudaMemcpyHostToDevice, st));
    gs_residuals<<<std::max(1, std::min(c->sm_count * 4, ceil_div(N, 256))), 256, 0, st>>>(dp, dpl, dpr, N, (double*)c->d_out_b.ptr);
    c->last_stats[7] = 1;
    RG_CUDA(cudaGetLastError());
    RG_CUDA(cudaMemcpyAsync(out, c->d_out_b.ptr, sizeof(double) * 4 * n, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaStreamSynchronize(st));
    return RG_OK;
}

}  // extern "C"
