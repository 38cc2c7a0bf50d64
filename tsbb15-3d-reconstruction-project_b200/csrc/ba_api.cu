// Host orchestration + C ABI of the device-resident bundle adjustment (SURVEY.md section 8f row N4, multi-view half).
#include "ba_kernels.cuh"
#include "plan.cuh"
#include <vector>

namespace rg {

// the caller's uv array is only guaranteed 8-byte aligned: scalar loads
__global__ void __launch_bounds__(256) ba_gather_uv(const double* __restrict__ uv, const int* __restrict__ perm, int nO,
                                                    double2* __restrict__ out) {
    for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < nO; s += gridDim.x * blockDim.x) {
        const size_t o = (size_t)perm[s];
        out[s] = make_double2(uv[2 * o], uv[2 * o + 1]);
    }
}

static inline char* align16(char* w) { return (char*)(((uintptr_t)w + 15) & ~(uintptr_t)15); }

// the kernels that depend on the loss (ba_points, ba_trial: rho and its weights; ba_blocks: the record layout)
struct BaLossKernels {
    decltype(&ba_points<LOSS_LINEAR>) points;
    decltype(&ba_trial<LOSS_LINEAR>) trial;
    decltype(&ba_blocks<false>) blocks;
};

template <int L>
static BaLossKernels ba_loss_kernels() { return {ba_points<L>, ba_trial<L>, ba_blocks<L != LOSS_LINEAR>}; }

static bool ba_loss_kernels(int loss, BaLossKernels& k) {
    switch (loss) {
        case LOSS_LINEAR: k = ba_loss_kernels<LOSS_LINEAR>(); return true;
        case LOSS_SOFT_L1: k = ba_loss_kernels<LOSS_SOFT_L1>(); return true;
        case LOSS_HUBER: k = ba_loss_kernels<LOSS_HUBER>(); return true;
        case LOSS_CAUCHY: k = ba_loss_kernels<LOSS_CAUCHY>(); return true;
        case LOSS_ARCTAN: k = ba_loss_kernels<LOSS_ARCTAN>(); return true;
        default: return false;
    }
}

// cams_dev (nC x 12) and pts_dev (nP x 3) are refined in place; uv_dev (nO x 2) in the caller's observation order;
// cam_idx / pt_idx are HOST arrays (table bookkeeping lives on the host in the reference too).  loss (LOSS_*) and
// f_scale = C: every residual component f contributes C^2 rho((f / C)^2) to twice the cost.
static int bundle_adjust_dev(Ctx* c, cudaStream_t st, int nC, int nP, int nO, double* cams, double* pts, const double* uv,
                             const int* cam_idx, const int* pt_idx, int n_fixed, int max_iter, double ftol, int loss,
                             double f_scale, double* cost, int* iters, int* status, bool host_paced) {
    RG_CHECK_ARG(nC >= 0 && nP >= 0 && nO >= 0, "negative size");
    RG_CHECK_ARG(n_fixed >= 0, "n_fixed must be >= 0");
    RG_CHECK_ARG(max_iter >= 0 && max_iter <= 10000, "max_iter must be in [0, 10000]");
    RG_CHECK_ARG(ftol >= 0.0 && std::isfinite(ftol), "ftol must be finite and >= 0");
    BaLossKernels kern;
    RG_CHECK_ARG(ba_loss_kernels(loss, kern), "loss must be one of RG_LOSS_LINEAR .. RG_LOSS_ARCTAN");
    const double ic = 1.0 / f_scale, c2 = f_scale * f_scale;
    RG_CHECK_ARG(std::isfinite(f_scale) && f_scale > 0.0 && std::isfinite(ic) && std::isfinite(c2) && c2 > 0.0,
                 "f_scale must be finite and > 0 (with a finite, non-zero square)");
    RG_CHECK_ARG(nO == 0 || (cam_idx && pt_idx && uv), "null observation table");
    RG_CHECK_ARG((nC == 0 || cams) && (nP == 0 || pts), "null parameter buffers");
    const int nF = std::max(0, nC - n_fixed);
    if (nF > kBaMaxFree) {
        set_error("invalid argument: %d free views; the dense reduced camera system supports at most %d", nF, kBaMaxFree);
        return RG_ERR_ARG;
    }
    for (int o = 0; o < nO; ++o)
        RG_CHECK_ARG(cam_idx[o] >= 0 && cam_idx[o] < nC && pt_idx[o] >= 0 && pt_idx[o] < nP, "observation index out of range");
    RG_CUDA(cudaSetDevice(c->device));
    c->last_stats[7] = 0;

    // ---- host: observations sorted by point (stable), CSR by point and by view -------------------------------------
    const size_t n_int_base = (size_t)4 * nO + (size_t)nP + 1 + (size_t)nC + 1;
    const size_t n_int = n_int_base;
    RG_CUDA(cudaEventSynchronize(c->staging_free[0]));
    int rc;
    if ((rc = ensure_pinned(c->h_stage[0], sizeof(int) * n_int))) return rc;
    int* h = (int*)c->h_stage[0].ptr;
    int* h_perm = h;                     // sorted position -> caller's observation index
    int* h_ocam = h_perm + nO;           // view of the sorted observation
    int* h_opt = h_ocam + nO;            // point of the sorted observation
    int* h_cam_obs = h_opt + nO;         // sorted positions grouped by view
    int* h_pt_off = h_cam_obs + nO;      // nP + 1
    int* h_cam_off = h_pt_off + nP + 1;  // nC + 1
    for (int j = 0; j <= nP; ++j) h_pt_off[j] = 0;
    for (int k = 0; k <= nC; ++k) h_cam_off[k] = 0;
    for (int o = 0; o < nO; ++o) { h_pt_off[pt_idx[o] + 1]++; h_cam_off[cam_idx[o] + 1]++; }
    for (int j = 0; j < nP; ++j) h_pt_off[j + 1] += h_pt_off[j];
    for (int k = 0; k < nC; ++k) h_cam_off[k + 1] += h_cam_off[k];
    {
        std::vector<int> fill(std::max(nP, nC) + 1);
        for (int j = 0; j < nP; ++j) fill[j] = h_pt_off[j];
        for (int o = 0; o < nO; ++o) {
            const int s = fill[pt_idx[o]]++;
            h_perm[s] = o; h_ocam[s] = cam_idx[o]; h_opt[s] = pt_idx[o];
        }
        for (int k = 0; k < nC; ++k) fill[k] = h_cam_off[k];
        for (int s = 0; s < nO; ++s) h_cam_obs[fill[h_ocam[s]]++] = s;
    }

    // blocks (kf, lf <= kf) of the reduced camera system with at least one common point (all diagonal blocks included)
    const int nFh = std::max(0, nC - n_fixed);
    std::vector<int2> blist;
    {
        const int words = (nC + 63) / 64;
        std::vector<unsigned long long> cov((size_t)nC * words, 0ull), tm(words);
        for (int j = 0; j < nP; ++j) {
            const int a = h_pt_off[j], b = h_pt_off[j + 1];
            if (b - a < 2) continue;
            std::fill(tm.begin(), tm.end(), 0ull);
            for (int s = a; s < b; ++s) tm[h_ocam[s] >> 6] |= 1ull << (h_ocam[s] & 63);
            for (int s = a; s < b; ++s) {
                unsigned long long* row = &cov[(size_t)h_ocam[s] * words];
                for (int w = 0; w < words; ++w) row[w] |= tm[w];
            }
        }
        for (int kf = 0; kf < nFh; ++kf)
            for (int lf = 0; lf <= kf; ++lf) {
                const int k = n_fixed + kf, l = n_fixed + lf;
                if (kf == lf || ((cov[(size_t)k * words + (l >> 6)] >> (l & 63)) & 1ull)) blist.push_back(make_int2(kf, lf));
            }
    }
    const size_t n_blocks = blist.size();
    // work items of ba_blocks: a block whose view has many observations is split into segments of kBaSegChunks chunks
    const int seg_len = kBaSegChunks * kBaBlockThreads;
    size_t n_items = 0;
    bool any_split = false;
    for (size_t i = 0; i < n_blocks; ++i) {
        const int k = n_fixed + blist[i].x;
        const int nseg = std::max(1, ceil_div(h_cam_off[k + 1] - h_cam_off[k], seg_len));
        n_items += (size_t)nseg;
        any_split = any_split || nseg > 1;
    }
    const size_t item_ints = 4 * n_items + n_blocks + 8;
    if ((rc = ensure_pinned(c->h_ba_items, sizeof(int) * item_ints))) return rc;
    int* h_items = (int*)c->h_ba_items.ptr;                        // int4 per item, then first item of every block
    int* h_first = h_items + 4 * n_items;
    {
        size_t it = 0;
        for (size_t i = 0; i < n_blocks; ++i) {
            const int k = n_fixed + blist[i].x;
            const int nseg = std::max(1, ceil_div(h_cam_off[k + 1] - h_cam_off[k], seg_len));
            h_first[i] = (int)it;
            for (int sgm = 0; sgm < nseg; ++sgm, ++it) {
                h_items[4 * it] = blist[i].x; h_items[4 * it + 1] = blist[i].y; h_items[4 * it + 2] = sgm; h_items[4 * it + 3] = nseg;
            }
        }
    }
    const bool sparse_blocks = n_blocks < (size_t)nFh * (nFh + 1) / 2;

    // ---- workspace ---------------------------------------------------------------------------------------------------
    const int n = 12 * nF;
    const int nparts = std::max(1, std::min(1024, ceil_div(std::max(nP, 1), kBaPointThreads / kBaPointLanes)));
    const size_t s_elems = (size_t)(n + 1) * (size_t)std::max(n, 1);
    const size_t bytes = sizeof(BaState) + 64 + sizeof(double) * ((size_t)12 * std::max(nC, 1) + (size_t)3 * nP + (size_t)2 * nO +
                                                                  (size_t)12 * nP + (size_t)kBaLin * nO + (any_split ? (size_t)kBaPart * n_items : 0) + s_elems + (size_t)24 * (n + 1) + (size_t)n + (size_t)3 * nparts + 8) +
                         sizeof(int) * (n_int + nparts + 8 + item_ints) + 256;
    if ((rc = ensure(c->ba_ws, bytes))) return rc;
    char* w = (char*)c->ba_ws.ptr;
    BaState* bs = (BaState*)w;                     w = align16(w + sizeof(BaState));
    double2* uvS = (double2*)w;                    w += sizeof(double2) * nO;
    double* dC = (double*)w;                       w += sizeof(double) * 12 * std::max(nC, 1);
    double* Xtrial = (double*)w;                   w += sizeof(double) * 3 * nP;
    double* pblk = (double*)w;                     w += sizeof(double) * 12 * nP;
    w = align16(w) + 16;                           w = (char*)(((uintptr_t)w + 31) & ~(uintptr_t)31);
    double* lin = (double*)w;                      w += sizeof(double) * kBaLin * nO;       // per-observation linearisation
    double* part = (double*)w;                     w += sizeof(double) * (any_split ? (size_t)kBaPart * n_items : 0);
    double* S = (double*)w;                        w += sizeof(double) * s_elems;
    double* Pg = (double*)w;                       w += sizeof(double) * 24 * (n + 1);      // published panels (double buffer)
    double* dinv = (double*)w;                     w += sizeof(double) * n;                 // reciprocal diagonal (L2 variant)
    double* cost_part = (double*)w;                w += sizeof(double) * nparts;
    double* trial_part = (double*)w;               w += sizeof(double) * nparts;
    double* obs2_part = (double*)w;                w += sizeof(double) * nparts;
    int* d_int = (int*)w;                          w += sizeof(int) * n_int;
    w = align16(w);
    int* d_items_raw = (int*)w;                    w += sizeof(int) * item_ints;
    int* bad_part = (int*)w;
    const int4* d_items = (const int4*)d_items_raw;
    const int* d_first = d_items_raw + 4 * n_items;
    int* d_perm = d_int;
    int* d_ocam = d_perm + nO;
    int* d_opt = d_ocam + nO;
    int* d_cam_obs = d_opt + nO;
    int* d_pt_off = d_cam_obs + nO;
    int* d_cam_off = d_pt_off + nP + 1;

    RG_CUDA(cudaMemcpyAsync(d_int, h, sizeof(int) * n_int, cudaMemcpyHostToDevice, st));
    if (n_items) RG_CUDA(cudaMemcpyAsync(d_items_raw, h_items, sizeof(int) * item_ints, cudaMemcpyHostToDevice, st));
    RG_CUDA(cudaEventRecord(c->staging_free[0], st));
    RG_CUDA(cudaMemsetAsync(dC, 0, sizeof(double) * 12 * std::max(nC, 1), st));
    int launches = 0;
    ba_init<<<1, 1, 0, st>>>(bs, 1e-3);
    ++launches;
    if (nO) {
        ba_gather_uv<<<std::max(1, std::min(c->sm_count * 4, ceil_div(nO, 256))), 256, 0, st>>>(uv, d_perm, nO, uvS);
        ++launches;
    }
    RG_CUDA(cudaGetLastError());

    // cluster launch of the factorisation
    int cluster = c->opt_ba_cluster > 0 ? c->opt_ba_cluster : 8;
    constexpr size_t kSmemMax = 226 * 1024;         // 227 KB per CTA minus the kernels' static shared memory
    // the cluster-resident factorisation when the matrix fits in the cluster's shared memory (option 4 = 1: L2 variant)
    const bool dsmem = nF > 0 && !c->opt_ba_l2 && sizeof(double) * ba_dsmem_doubles(nF, cluster) <= kSmemMax;
    const size_t smem = dsmem ? sizeof(double) * ba_dsmem_doubles(nF, cluster) : sizeof(double) * (kBaSolveFixed + (size_t)12 * (n + 1));
    if (nF > 0 && !c->ba_attr_set) {
        RG_CUDA(cudaFuncSetAttribute(ba_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
        RG_CUDA(cudaFuncSetAttribute(ba_solve_dsmem, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
        c->ba_attr_set = true;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.gridDim = dim3(cluster); cfg.blockDim = dim3(kBaSolveThreads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cfg.attrs = attr; cfg.numAttrs = 1;

    // host_paced (the host-buffer entry point, which ends with a synchronisation anyway): the solver's `done` flag is
    // copied to pinned memory after every iteration and the enqueue loop stays at most two iterations ahead of the
    // device, so that it stops two iterations after convergence instead of enqueueing max_iter x 5 empty launches.
    volatile int* h_flags = nullptr;
    if (host_paced && max_iter > 2) {
        if ((rc = ensure_pinned(c->h_ba_flags, sizeof(int) * (size_t)max_iter))) return rc;
        h_flags = (volatile int*)c->h_ba_flags.ptr;
        for (int i = 0; i < 2; ++i)
            if (!c->ba_iter_ev[i]) RG_CUDA(cudaEventCreateWithFlags(&c->ba_iter_ev[i], cudaEventDisableTiming));
    }
    for (int it = 0; it < max_iter; ++it) {
        if (h_flags && it >= 2) {
            RG_CUDA(cudaEventSynchronize(c->ba_iter_ev[it & 1]));          // iteration it - 2 has finished
            if (h_flags[it - 2]) break;
        }
        kern.points<<<nparts, kBaPointThreads, 0, st>>>(bs, cams, pts, Xtrial, uvS, d_ocam, d_pt_off, nP, pblk, cost_part, bad_part,
                                                          obs2_part, lin, ic, c2);
        if (nF > 0) {
            if (sparse_blocks) RG_CUDA(cudaMemsetAsync(S, 0, sizeof(double) * s_elems, st));   // blocks without a common point
            kern.blocks<<<(unsigned)n_items, kBaBlockThreads, 0, st>>>(bs, d_items, part, pts, lin, d_ocam, d_opt, d_pt_off, d_cam_off,
                                                                      d_cam_obs, pblk, n_fixed, nF, S);
            if (any_split) {
                ba_blocks_reduce<<<(unsigned)n_blocks, kBaBlockThreads, 0, st>>>(bs, d_items, d_first, (int)n_blocks, part, nF, S);
                ++launches;
            }
            if (dsmem) RG_CUDA(cudaLaunchKernelEx(&cfg, ba_solve_dsmem, bs, (const double*)S, Pg, n_fixed, nF, dC));
            else RG_CUDA(cudaLaunchKernelEx(&cfg, ba_solve, bs, S, dinv, n_fixed, nF, dC));
        } else {
            ba_solve_none<<<1, 1, 0, st>>>(bs);
        }
        kern.trial<<<nparts, kBaPointThreads, 0, st>>>(bs, cams, dC, pts, Xtrial, uvS, d_ocam, d_pt_off, nP, pblk, lin, trial_part,
                                                         ic, c2);
        ba_accept<<<1, 256, 0, st>>>(bs, cams, dC, nC, cost_part, trial_part, bad_part, obs2_part, nparts, ftol, max_iter);
        launches += nF > 0 ? 5 : 4;
        if (h_flags) {
            RG_CUDA(cudaMemcpyAsync((void*)&h_flags[it], &bs->done, sizeof(int), cudaMemcpyDeviceToHost, st));
            RG_CUDA(cudaEventRecord(c->ba_iter_ev[it & 1], st));
        }
    }
    if (max_iter == 0) {
        kern.points<<<nparts, kBaPointThreads, 0, st>>>(bs, cams, pts, Xtrial, uvS, d_ocam, d_pt_off, nP, pblk, cost_part, bad_part,
                                                          obs2_part, lin, ic, c2);
        ba_cost_only<<<1, 1, 0, st>>>(bs, cost_part, nparts);
        launches += 2;
    }
    ba_finish<<<std::max(1, std::min(c->sm_count, ceil_div(3 * std::max(nP, 1), 256))), 256, 0, st>>>(bs, pts, Xtrial, nP, cost, iters,
                                                                                                    status);
    ++launches;
    RG_CUDA(cudaGetLastError());
    c->last_stats[7] = launches;
    return RG_OK;
}

}  // namespace rg

using namespace rg;

extern "C" {

int rg_bundle_adjust_dev2(void* ctx, void* stream, int n_views, int n_points, int n_obs, double* cams_dev, double* pts_dev,
                          const double* uv_dev, const int32_t* cam_idx_host, const int32_t* pt_idx_host, int n_fixed, int max_iter,
                          double ftol, int loss, double f_scale, double* cost_dev, int32_t* iters_dev, int32_t* status_dev) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    return bundle_adjust_dev((Ctx*)ctx, (cudaStream_t)stream, n_views, n_points, n_obs, cams_dev, pts_dev, uv_dev, cam_idx_host,
                             pt_idx_host, n_fixed, max_iter, ftol, loss, f_scale, cost_dev, iters_dev, status_dev, false);
}

int rg_bundle_adjust_dev(void* ctx, void* stream, int n_views, int n_points, int n_obs, double* cams_dev, double* pts_dev,
                         const double* uv_dev, const int32_t* cam_idx_host, const int32_t* pt_idx_host, int n_fixed, int max_iter,
                         double ftol, double* cost_dev, int32_t* iters_dev, int32_t* status_dev) {
    return rg_bundle_adjust_dev2(ctx, stream, n_views, n_points, n_obs, cams_dev, pts_dev, uv_dev, cam_idx_host, pt_idx_host,
                                 n_fixed, max_iter, ftol, LOSS_LINEAR, 1.0, cost_dev, iters_dev, status_dev);
}

int rg_bundle_adjust_host2(void* ctx, void* stream, int n_views, int n_points, int n_obs, double* cams, double* pts,
                           const double* uv, const int32_t* cam_idx, const int32_t* pt_idx, int n_fixed, int max_iter, double ftol,
                           int loss, double f_scale, double* cost, int32_t* iters, int32_t* status) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(n_views >= 0 && n_points >= 0 && n_obs >= 0, "negative size");
    RG_CHECK_ARG((n_views == 0 || cams) && (n_points == 0 || pts) && (n_obs == 0 || uv), "null buffers");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    const size_t nc = (size_t)n_views, np = (size_t)n_points, no = (size_t)n_obs;
    int rc;
    if ((rc = ensure(c->d_in_a, sizeof(double) * (12 * nc + 3 * np + 2 * no + 2) + sizeof(int) * 4))) return rc;
    double* dcam = (double*)c->d_in_a.ptr;
    double* dpts = dcam + 12 * nc;
    double* duv = dpts + 3 * np;
    double* dcost = duv + 2 * no;
    int* dit = (int*)(dcost + 1);
    if (nc) RG_CUDA(cudaMemcpyAsync(dcam, cams, sizeof(double) * 12 * nc, cudaMemcpyHostToDevice, st));
    if (np) RG_CUDA(cudaMemcpyAsync(dpts, pts, sizeof(double) * 3 * np, cudaMemcpyHostToDevice, st));
    if (no) RG_CUDA(cudaMemcpyAsync(duv, uv, sizeof(double) * 2 * no, cudaMemcpyHostToDevice, st));
    rc = bundle_adjust_dev(c, st, n_views, n_points, n_obs, dcam, dpts, duv, cam_idx, pt_idx, n_fixed, max_iter, ftol, loss, f_scale,
                           dcost, dit, dit + 1, true);
    if (rc) return rc;
    if (nc) RG_CUDA(cudaMemcpyAsync(cams, dcam, sizeof(double) * 12 * nc, cudaMemcpyDeviceToHost, st));
    if (np) RG_CUDA(cudaMemcpyAsync(pts, dpts, sizeof(double) * 3 * np, cudaMemcpyDeviceToHost, st));
    if (cost) RG_CUDA(cudaMemcpyAsync(cost, dcost, sizeof(double), cudaMemcpyDeviceToHost, st));
    if (iters) RG_CUDA(cudaMemcpyAsync(iters, dit, sizeof(int), cudaMemcpyDeviceToHost, st));
    if (status) RG_CUDA(cudaMemcpyAsync(status, dit + 1, sizeof(int), cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaStreamSynchronize(st));
    return RG_OK;
}

int rg_bundle_adjust_host(void* ctx, void* stream, int n_views, int n_points, int n_obs, double* cams, double* pts,
                          const double* uv, const int32_t* cam_idx, const int32_t* pt_idx, int n_fixed, int max_iter, double ftol,
                          double* cost, int32_t* iters, int32_t* status) {
    return rg_bundle_adjust_host2(ctx, stream, n_views, n_points, n_obs, cams, pts, uv, cam_idx, pt_idx, n_fixed, max_iter, ftol,
                                  LOSS_LINEAR, 1.0, cost, iters, status);
}

#ifdef RG_BA_PROF
/* experiment builds only (-DRG_BA_PROF): summed clock64 ticks of the phases of ba_solve_dsmem as seen by CTA 0 */
int rg_ba_prof_read(long long* out16) {
    RG_CUDA(cudaMemcpyFromSymbol(out16, g_ba_prof, sizeof(long long) * 16));
    long long z[16] = {0};
    RG_CUDA(cudaMemcpyToSymbol(g_ba_prof, z, sizeof(z)));
    return RG_OK;
}
#endif

int rg_ba_residuals_host(void* ctx, void* stream, int n_views, int n_points, int n_obs, const double* x, const double* u,
                         const double* v, const int32_t* cam_idx, const int32_t* pt_idx, double* out) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    RG_CHECK_ARG(n_views >= 0 && n_points >= 0 && n_obs >= 0, "negative size");
    Ctx* c = (Ctx*)ctx;
    cudaStream_t st = (cudaStream_t)stream;
    RG_CUDA(cudaSetDevice(c->device));
    if (n_obs == 0) return RG_OK;
    RG_CHECK_ARG(x && u && v && cam_idx && pt_idx && out, "null buffers");
    for (int o = 0; o < n_obs; ++o)
        RG_CHECK_ARG(cam_idx[o] >= 0 && cam_idx[o] < n_views && pt_idx[o] >= 0 && pt_idx[o] < n_points,
                     "observation index out of range");
    const size_t nx = (size_t)12 * n_views + (size_t)3 * n_points, no = (size_t)n_obs;
    int rc;
    if ((rc = ensure(c->d_in_a, sizeof(double) * (nx + 2 * no) + sizeof(int) * 2 * no))) return rc;
    if ((rc = ensure(c->d_out_b, sizeof(double) * 2 * no))) return rc;
    double* dx = (double*)c->d_in_a.ptr;
    double* du = dx + nx;
    double* dv = du + no;
    int* dci = (int*)(dv + no);
    int* dpi = dci + no;
    RG_CUDA(cudaMemcpyAsync(dx, x, sizeof(double) * nx, cudaMemcpyHostToDevice, st));
    RG_CUDA(cudaMemcpyAsync(du, u, sizeof(double) * no, cudaMemcpyHostToDevice, st));
    RG_CUDA(cudaMemcpyAsync(dv, v, sizeof(double) * no, cudaMemcpyHostToDevice, st));
    RG_CUDA(cudaMemcpyAsync(dci, cam_idx, sizeof(int) * no, cudaMemcpyHostToDevice, st));
    RG_CUDA(cudaMemcpyAsync(dpi, pt_idx, sizeof(int) * no, cudaMemcpyHostToDevice, st));
    ba_residuals<<<std::max(1, std::min(c->sm_count * 4, ceil_div(n_obs, 256))), 256, 0, st>>>(dx, n_views, du, dv, dci, dpi, n_obs,
                                                                                              (double*)c->d_out_b.ptr);
    c->last_stats[7] = 1;
    RG_CUDA(cudaGetLastError());
    RG_CUDA(cudaMemcpyAsync(out, c->d_out_b.ptr, sizeof(double) * 2 * no, cudaMemcpyDeviceToHost, st));
    RG_CUDA(cudaStreamSynchronize(st));
    return RG_OK;
}

}  // extern "C"
