// Host orchestration + C ABI of the refinement of PnP poses (DESIGN.md section 4.7).
#include "pnp_refine_kernels.cuh"

namespace rg {

// V views in CSR form (view_off host); Rt (V x 12, device) refined in place.  K_host: V x 9 row-major on the HOST (or
// NULL): validated here, only W = K[:2, :2] is uploaded.  host_paced: see gold_standard_dev.
static int pnp_refine_dev(Ctx* c, cudaStream_t st, int V, const double* X, const double* y, const int* view_off,
                          const double* K_host, const unsigned char* mask, double* Rt, int max_iter, double ftol, int rounds,
                          double thr2, unsigned char* mask_out, double* cost, int* iters, int* status, bool host_paced) {
    RG_CHECK_ARG(V >= 0 && view_off != nullptr, "bad view table");
    RG_CHECK_ARG(view_off[0] == 0, "view_off must start at 0");
    for (int v = 0; v < V; ++v) RG_CHECK_ARG(view_off[v + 1] >= view_off[v], "view_off must be non-decreasing");
    RG_CHECK_ARG(max_iter >= 0 && max_iter <= 10000, "max_iter must be in [0, 10000]");
    RG_CHECK_ARG(ftol >= 0.0 && std::isfinite(ftol), "ftol must be finite and >= 0");
    RG_CHECK_ARG(rounds >= 1 && rounds <= 100, "rounds must be in [1, 100]");
    const bool rescore = rounds > 1 || mask_out != nullptr;
    RG_CHECK_ARG(!rescore || (thr2 >= 0.0 && std::isfinite(thr2)), "thr2 must be finite and >= 0 when rounds > 1 or mask_out is given");
    std::vector<double> W3;
    if (K_host) {
        W3.resize(3 * (size_t)std::max(V, 1));
        for (int v = 0; v < V; ++v) {
            const double* K = K_host + 9 * (size_t)v;
            RG_CHECK_ARG(K[3] == 0.0 && K[6] == 0.0 && K[7] == 0.0 && K[8] == 1.0,
                         "K must have K[1][0] == 0 and bottom row (0, 0, 1)");
            RG_CHECK_ARG(std::isfinite(K[0]) && std::isfinite(K[1]) && std::isfinite(K[4]), "K must be finite");
            W3[3 * v] = K[0]; W3[3 * v + 1] = K[1]; W3[3 * v + 2] = K[4];
        }
    }
    RG_CUDA(cudaSetDevice(c->device));
    c->last_stats[7] = 0;
    if (V == 0) return RG_OK;
    const size_t N = (size_t)view_off[V];
    RG_CHECK_ARG(Rt && (N == 0 || (X && y)), "null buffers");
    int maxN = 0;
    for (int v = 0; v < V; ++v) maxN = std::max(maxN, view_off[v + 1] - view_off[v]);
    const bool fused = maxN <= kPrFusedMaxPts && !c->opt_pr_multi;
    const int nb = fused ? 1 : std::max(1, std::min(2 * c->sm_count, ceil_div(maxN, kPrThreads * 8)));
    const bool tmp_mask = rescore && mask_out == nullptr;
    // workspace: PrView[V] | partials (V x nb x 32) | W (3V) | view_off (V+1) | active (max_iter) | consensus mask (N)
    const size_t bytes = sizeof(PrView) * (size_t)V + sizeof(double) * ((fused ? 0 : (size_t)V * nb * kPrStride) + 3 * (size_t)V) +
                         sizeof(int) * ((size_t)V + 1 + (size_t)max_iter) + (tmp_mask ? N : 0) + 64;
    int rc;
    if ((rc = ensure(c->pr_ws, bytes))) return rc;
    char* w = (char*)c->pr_ws.ptr;
    PrView* gv = (PrView*)w;                       w += sizeof(PrView) * (size_t)V;
    double* part = (double*)w;                     w += sizeof(double) * (fused ? 0 : (size_t)V * nb * kPrStride);
    double* dW = (double*)w;                       w += sizeof(double) * 3 * (size_t)V;
    int* doff = (int*)w;                           w += sizeof(int) * ((size_t)V + 1);
    int* active = (int*)w;                         w += sizeof(int) * (size_t)max_iter;
    unsigned char* cmask = tmp_mask ? (unsigned char*)w : mask_out;
    // pageable sources: cudaMemcpyAsync stages them before it returns, so these host vectors may go out of scope
    RG_CUDA(cudaMemcpyAsync(doff, view_off, sizeof(int) * ((size_t)V + 1), cudaMemcpyHostToDevice, st));
    if (K_host) RG_CUDA(cudaMemcpyAsync(dW, W3.data(), sizeof(double) * 3 * (size_t)V, cudaMemcpyHostToDevice, st));
    const double* W = K_host ? dW : nullptr;
    volatile int* h_act = nullptr;
    if (!fused && host_paced && max_iter > 2) {
        if ((rc = ensure_pinned(c->h_pr_flags, sizeof(int) * (size_t)max_iter))) return rc;
        h_act = (volatile int*)c->h_pr_flags.ptr;
        for (int i = 0; i < 2; ++i)
            if (!c->pr_iter_ev[i]) RG_CUDA(cudaEventCreateWithFlags(&c->pr_iter_ev[i], cudaEventDisableTiming));
    }
    int launches = 0;
    for (int r = 0; r < rounds; ++r) {
        const unsigned char* sel = r == 0 ? mask : cmask;
        pnp_refine_init<<<ceil_div(V, 64), 64, 0, st>>>(Rt, V, gv);
        launches += 1;
        if (fused) {
            pnp_refine_fused<<<V, kPrThreads, 0, st>>>(X, y, doff, W, sel, gv, max_iter, ftol);
            launches += 1;
        } else {
            const dim3 grid(nb, V);
            pnp_refine_pass<<<grid, kPrThreads, 0, st>>>(X, y, doff, W, sel, gv, part);
            pnp_refine_step<<<V, kPrThreads, 0, st>>>(gv, part, nb, 1, max_iter, ftol, nullptr);
            launches += 2;
            // host_paced (the host-buffer entry point, which synchronises anyway): the enqueue stays at most two
            // iterations ahead of the device and stops two iterations after the last view finished
            if (h_act) RG_CUDA(cudaMemsetAsync(active, 0, sizeof(int) * (size_t)max_iter, st));
            for (int it = 0; it < max_iter; ++it) {
                if (h_act && it >= 2) {
                    RG_CUDA(cudaEventSynchronize(c->pr_iter_ev[it & 1]));      // iteration it - 2 has finished
                    if (h_act[it - 2] == 0) break;
                }
                pnp_refine_pass<<<grid, kPrThreads, 0, st>>>(X, y, doff, W, sel, gv, part);
                pnp_refine_step<<<V, kPrThreads, 0, st>>>(gv, part, nb, 0, max_iter, ftol, h_act ? active + it : nullptr);
                launches += 2;
                if (h_act) {
                    RG_CUDA(cudaMemcpyAsync((void*)&h_act[it], active + it, sizeof(int), cudaMemcpyDeviceToHost, st));
                    RG_CUDA(cudaEventRecord(c->pr_iter_ev[it & 1], st));
                }
            }
        }
        pnp_refine_export<<<ceil_div(V, 64), 64, 0, st>>>(gv, V, Rt, cost, iters, status);
        launches += 1;
        if (rescore && N) {
            const int nbx = std::max(1, std::min(c->sm_count * 4, ceil_div(maxN, 256)));
            pnp_refine_consensus<<<dim3(nbx, V), 256, 0, st>>>(X, y, doff, gv, thr2, cmask);
            launches += 1;
        }
        RG_CUDA(cudaGetLastError());
    }
    c->last_stats[7] = launches;
    return RG_OK;
}

}  // namespace rg

using namespace rg;

extern "C" {

int rg_pnp_refine_dev(void* ctx, void* stream, int V, const double* X_dev, const double* y_dev, const int32_t* view_off_host,
                      const double* K_host, const unsigned char* mask_dev, double* Rt_dev, int max_iter, double ftol,
                      int rounds, double thr2, unsigned char* mask_out_dev, double* cost_dev, int32_t* iters_dev,
                      int32_t* status_dev) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    return pnp_refine_dev((Ctx*)ctx, (cudaStream_t)stream, V, X_dev, y_dev, view_off_host, K_host, mask_dev, Rt_dev, max_iter,
                          ftol, rounds, thr2, mask_out_dev, cost_dev, iters_dev, status_dev, false);
}

int rg_pnp_refine_host(void* ctx, void* stream, int V, const double* X, const double* y, const int32_t* view_off,
                       const double* K, const unsigned char* mask, double* Rt, int max_iter, double ftol, int rounds,
                       double thr2, unsigned char* mask_out, double* cost, int32_t* iters, int32_t* status) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(V >= 0 && view_off != nullptr, "bad view table");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    if (V == 0) return RG_OK;
    RG_CHECK_ARG(view_off[0] == 0 && view_off[V] >= 0, "bad view table");
    const size_t N = (size_t)view_off[V], v = (size_t)V;
    RG_CHECK_ARG(Rt && (N == 0 || (X && y)), "null buffers");
    const size_t n1 = std::max<size_t>(N, 1);
    int rc;
    if ((rc = ensure(c->d_in_a, sizeof(double) * 3 * n1))) return rc;
    if ((rc = ensure(c->d_in_c, sizeof(double) * 2 * n1))) return rc;
    if ((rc = ensure(c->d_in_b, 2 * n1))) return rc;                       // input mask | output mask
    if ((rc = ensure(c->d_out_b, sizeof(double) * 13 * v + sizeof(int) * 2 * v))) return rc;
    double* dRt = (double*)c->d_out_b.ptr;
    double* dcost = dRt + 12 * v;
    int* dit = (int*)(dcost + v);
    int* dst = dit + v;
    unsigned char* dmask = (unsigned char*)c->d_in_b.ptr;
    unsigned char* dmask_out = dmask + n1;
    if (N) {
        RG_CUDA(cudaMemcpyAsync(c->d_in_a.ptr, X, sizeof(double) * 3 * N, cudaMemcpyHostToDevice, st));
        RG_CUDA(cudaMemcpyAsync(c->d_in_c.ptr, y, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, st));
        if (mask) RG_CUDA(cudaMemcpyAsync(dmask, mask, N, cudaMemcpyHostToDevice, st));
    }
    RG_CUDA(cudaMemcpyAsync(dRt, Rt, sizeof(double) * 12 * v, cudaMemcpyHostToDevice, st));
    rc = pnp_refine_dev(c, st, V, (const double*)c->d_in_a.ptr, (const double*)c->d_in_c.ptr, view_off, K,
                        (mask && N) ? dmask : nullptr, dRt, max_iter, ftol, rounds, thr2, mask_out ? dmask_out : nullptr, dcost,
                        dit, dst, true);
    if (rc) return rc;
    RG_CUDA(cudaMemcpyAsync(Rt, dRt, sizeof(double) * 12 * v, cudaMemcpyDeviceToHost, st));
    if (cost) RG_CUDA(cudaMemcpyAsync(cost, dcost, sizeof(double) * v, cudaMemcpyDeviceToHost, st));
    if (iters) RG_CUDA(cudaMemcpyAsync(iters, dit, sizeof(int) * v, cudaMemcpyDeviceToHost, st));
    if (status) RG_CUDA(cudaMemcpyAsync(status, dst, sizeof(int) * v, cudaMemcpyDeviceToHost, st));
    if (mask_out && N) RG_CUDA(cudaMemcpyAsync(mask_out, dmask_out, N, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaStreamSynchronize(st));
    return RG_OK;
}

}  // extern "C"
