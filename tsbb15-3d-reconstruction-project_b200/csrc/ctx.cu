// Context / error plumbing of librg_b200.so.
#include "common.cuh"
#include <cstdarg>
#include <mutex>

namespace rg {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int ensure(Buffer& b, size_t bytes) {
    if (bytes <= b.cap) return RG_OK;
    size_t want = bytes + bytes / 4 + 256;       // head-room: ragged batches do not realloc every call
    if (b.ptr) {
        RG_CUDA(cudaFree(b.ptr));
        b.ptr = nullptr;
        b.cap = 0;
    }
    RG_CUDA(cudaMalloc(&b.ptr, want));
    b.cap = want;
    return RG_OK;
}

int ensure_pinned(Buffer& b, size_t bytes) {
    if (bytes <= b.cap) return RG_OK;
    size_t want = bytes + bytes / 4 + 256;
    if (b.ptr) {
        RG_CUDA(cudaFreeHost(b.ptr));
        b.ptr = nullptr;
        b.cap = 0;
    }
    RG_CUDA(cudaMallocHost(&b.ptr, want));
    b.cap = want;
    return RG_OK;
}

void release(Buffer& b) {
    if (b.ptr) cudaFree(b.ptr);
    b.ptr = nullptr;
    b.cap = 0;
}

// boundary 0 opens a pass (dropped, together with the pass's other boundaries, once the ring is full); boundaries
// 1..kProfPhases close the phases.  prof_masks[] remembers which boundaries of a pass were recorded, so a pass that
// failed half-way is skipped by rg_get_profile instead of pairing events of different passes.
int prof_begin(Ctx* c) {
    if (!c->opt_profile || !c->prof_ev) return -1;
    c->prof_open = c->prof_calls < Ctx::kProfRing;
    if (!c->prof_open) return -1;
    c->prof_masks[c->prof_calls] = 0u;
    return c->prof_calls++;
}

void prof_mark_at(Ctx* c, cudaStream_t st, int call, int boundary) {
    if (!c->opt_profile || !c->prof_ev) return;
    if (call < 0 || call >= Ctx::kProfRing || boundary < 0 || boundary >= Ctx::kProfEvents) return;
    if (cudaEventRecord(c->prof_ev[call * Ctx::kProfEvents + boundary], st) == cudaSuccess)
        c->prof_masks[call] |= 1u << boundary;
}

void prof_mark(Ctx* c, cudaStream_t st, int boundary) {
    if (boundary == 0) c->prof_cur = prof_begin(c);
    prof_mark_at(c, st, c->prof_cur, boundary);
}

void release_pinned(Buffer& b) {
    if (b.ptr) cudaFreeHost(b.ptr);
    b.ptr = nullptr;
    b.cap = 0;
}

}  // namespace rg

using namespace rg;

extern "C" {

const char* rg_last_error(void) { return g_err; }

int rg_abi_version(void) { return 1; }

int rg_init(int device, void** out_ctx) {
    RG_CHECK_ARG(out_ctx != nullptr, "out_ctx is null");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        set_error("no CUDA device visible (%s); this library has no CPU fallback",
                  e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return RG_ERR_NO_DEVICE;
    }
    RG_CHECK_ARG(device >= 0 && device < n, "device index out of range");
    cudaDeviceProp prop;
    RG_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("device %d is sm_%d%d; librg_b200 is built for sm_100a only", device, prop.major, prop.minor);
        return RG_ERR_NO_DEVICE;
    }
    RG_CUDA(cudaSetDevice(device));
    Ctx* c = new Ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    if (getenv("RG_NOPIPE")) c->opt_pipeline = 0;              // experiment hook (tools/r2_pipe_sweep.sh); rg_set_option(ctx, 10, v) is the API
    for (int i = 0; i < 2; ++i) RG_CUDA(cudaEventCreateWithFlags(&c->staging_free[i], cudaEventDisableTiming));
    *out_ctx = c;
    return RG_OK;
}

int rg_shutdown(void* ctx) {
    if (!ctx) return RG_OK;
    Ctx* c = (Ctx*)ctx;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (Buffer* b : {&c->pair_info, &c->pair_frame, &c->state, &c->bbox, &c->pts32, &c->F64, &c->hyp32, &c->flags,
                      &c->flag_list, &c->stats, &c->best, &c->tie_stats, &c->d_in_a, &c->d_in_b, &c->d_in_c, &c->geom, &c->geom_ws, &c->gs_ws, &c->ba_ws, &c->pr_ws, &c->d_out_a, &c->d_out_b,
                      &c->d_out_c, &c->d_out_d, &c->pose64, &c->pose32, &c->X32, &c->bnd, &c->bnd_stats})
        release(*b);
    for (Ctx::PassSet& o : c->spare)
        for (Buffer* b : {&o.pair_info, &o.pair_frame, &o.state, &o.pts32, &o.F64, &o.hyp32, &o.flags, &o.flag_list, &o.best,
                          &o.tie_stats, &o.bnd})
            release(*b);
    for (int i = 0; i < Ctx::kPassSets; ++i) {
        if (c->head_done[i]) cudaEventDestroy(c->head_done[i]);
        if (c->score_done[i]) cudaEventDestroy(c->score_done[i]);
        if (c->cand_done[i]) cudaEventDestroy(c->cand_done[i]);
        if (c->sweep_done[i]) cudaEventDestroy(c->sweep_done[i]);
    }
    if (c->tail_done) cudaEventDestroy(c->tail_done);
    if (c->pipe_gate) cudaEventDestroy(c->pipe_gate);
    if (c->tail_stream) cudaStreamDestroy(c->tail_stream);
    if (c->pass_stream) cudaStreamDestroy(c->pass_stream);
    release_pinned(c->h_stage[0]);
    release_pinned(c->h_stage[1]);
    release_pinned(c->h_stats);
    release_pinned(c->h_ba_flags);
    release_pinned(c->h_ba_items);
    release_pinned(c->h_pr_flags);
    for (int i = 0; i < 2; ++i) {
        if (c->ba_iter_ev[i]) cudaEventDestroy(c->ba_iter_ev[i]);
        if (c->pr_iter_ev[i]) cudaEventDestroy(c->pr_iter_ev[i]);
    }
    if (c->prof_ev) {
        for (int i = 0; i < Ctx::kProfRing * Ctx::kProfEvents; ++i) cudaEventDestroy(c->prof_ev[i]);
        delete[] c->prof_ev;
    }
    for (int i = 0; i < 2; ++i)
        if (c->staging_free[i]) cudaEventDestroy(c->staging_free[i]);
    if (c->copy_gate) cudaEventDestroy(c->copy_gate);
    for (cudaEvent_t e : c->pass_ready) cudaEventDestroy(e);
    for (cudaEvent_t e : c->pass_done) cudaEventDestroy(e);
    if (c->d2h_done) cudaEventDestroy(c->d2h_done);
    if (c->d2h_stream) cudaStreamDestroy(c->d2h_stream);
    for (int i = 0; i < 4; ++i)
        if (c->rate_ev[i]) cudaEventDestroy(c->rate_ev[i]);
    p2p_release(c);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    delete c;
    return RG_OK;
}

// page-locked host memory for callers that build their input batches in place (uploads from pageable memory are staged
// by the driver at a fraction of the link rate); freed with rg_host_free
int rg_host_alloc(size_t bytes, void** out) {
    RG_CHECK_ARG(out != nullptr, "out is null");
    *out = nullptr;
    RG_CUDA(cudaMallocHost(out, bytes > 0 ? bytes : 1));
    return RG_OK;
}

int rg_host_free(void* p) {
    if (p) RG_CUDA(cudaFreeHost(p));
    return RG_OK;
}

int rg_device_sm_count(void* ctx) { return ctx ? ((Ctx*)ctx)->sm_count : 0; }

// option 1: phase profiling (CUDA events on the launching stream around the phases of every RANSAC call)
// option 2: number of sub-batches of rg_f_ransac_host (0 = automatic): uploads overlap the previous sub-batch's kernels
// option 3: thread-block cluster size of the bundle-adjustment Cholesky (0 = default 8; 1, 2, 4, 8)
// option 4: 1 = factorise the bundle-adjustment camera system in L2 even when it fits in distributed shared memory
// option 5: 1 = gold-standard refinement always on the multi-kernel path (default: pairs of <= 4096 points run the whole
//           Levenberg-Marquardt loop in one CTA, one launch)
// option 6: hypothesis x correspondence evaluations per pass of a large RANSAC batch (0 = default 2.7e10)
// option 7: PnP minimal-sample solver: 0 = Givens QR + row Jacobi, thread per hypothesis (default); 1 = 16-lane group Jacobi
// option 8: test hook: capacity of the guard-band flag list in records (0 = automatic); a tiny value forces the FP64 recount
// option 10: 1 (default) = in F calls of several passes the fix-up / selection / mask kernels of pass k run on a second
//           stream while pass k+1 is solved and scored (two sets of per-pass workspaces); 0 = strictly one after the other
// option 11: 1 = refinement of PnP poses always on the multi-CTA path (default: views of <= 4096 correspondences run the whole
//           Levenberg-Marquardt loop in one CTA, one launch per round); test hook comparing the two paths
// option 12: 1 (default) = F calls that want no per-hypothesis counts run the bounded sweep (bounded.cuh: hypotheses that
//           provably cannot reach their pair's maximum are not scored in full; results are those of the full sweep);
//           0 = every hypothesis against every correspondence
// option 13: prefix share rho of the bounded sweep in thousandths, in [1, 1000] (default 450)
// option 14: candidates per pair of the bounded sweep, in [1, 65536] (default 512)
// option 15: prefix stage of the bounded sweep: 1 (default) = bound-only scorer (upper-bound counts, no fix-up; the
//           candidates are then scored over the whole pair), 0 = guarded scorer + fix-up (exact prefix counts)
// option 9: guard-band safety factor x 1000 (default 1000 = the proven FP32 rounding bound); larger values keep every result
//           exact and only send more evaluations to the FP64 recheck — used to MEASURE what a less accurate scorer
//           (tensor-core split-precision accumulation) would cost in fix-up time
int rg_set_option(void* ctx, int option, long long value) {
    RG_CHECK_ARG(ctx != nullptr, "ctx is null");
    Ctx* c = (Ctx*)ctx;
    if (option == 1) {
        c->opt_profile = value != 0;
        c->prof_calls = 0;
        c->prof_open = false;
        c->prof_cur = -1;
        if (c->opt_profile && !c->prof_ev) {
            const int n = Ctx::kProfRing * Ctx::kProfEvents;
            c->prof_ev = new cudaEvent_t[n];
            for (int i = 0; i < n; ++i) RG_CUDA(cudaEventCreate(&c->prof_ev[i]));
        }
        return RG_OK;
    }
    if (option == 2) {
        if (value < 0 || value > Ctx::kMaxSlices) {
            set_error("invalid argument: option 2 (host sub-batches) must be in [0, %d]", Ctx::kMaxSlices);
            return RG_ERR_ARG;
        }
        c->opt_host_slices = (int)value;
        return RG_OK;
    }
    if (option == 3) {
        if (!(value == 0 || value == 1 || value == 2 || value == 4 || value == 8)) {
            set_error("invalid argument: option 3 (cluster size of the bundle-adjustment factorisation) must be 0, 1, 2, 4 or 8");
            return RG_ERR_ARG;
        }
        c->opt_ba_cluster = (int)value;
        return RG_OK;
    }
    if (option == 4) {
        c->opt_ba_l2 = value != 0;
        return RG_OK;
    }
    if (option == 5) {
        c->opt_gs_multi = value != 0;
        return RG_OK;
    }
    if (option == 6) {
        if (value < 0) { set_error("invalid argument: option 6 (evaluations per pass) must be >= 0"); return RG_ERR_ARG; }
        c->opt_pass_evals = value;
        return RG_OK;
    }
    if (option == 7) {
        if (value != 0 && value != 1) { set_error("invalid argument: option 7 (PnP minimal solver) must be 0 or 1"); return RG_ERR_ARG; }
        c->opt_pnp_solver = (int)value;
        return RG_OK;
    }
    if (option == 9) {
        if (value < 1000 || value > 100000000ll) { set_error("invalid argument: option 9 (guard-band factor x 1000) must be in [1000, 1e8]"); return RG_ERR_ARG; }
        c->opt_band_scale = (double)value / 1000.0;
        c->prep_pts = nullptr;
        return RG_OK;
    }
    if (option == 10) {
        if (value != 0 && value != 1) { set_error("invalid argument: option 10 (pass pipelining) must be 0 or 1"); return RG_ERR_ARG; }
        c->opt_pipeline = (int)value;
        return RG_OK;
    }
    if (option == 11) {
        if (value != 0 && value != 1) { set_error("invalid argument: option 11 (PnP refinement path) must be 0 or 1"); return RG_ERR_ARG; }
        c->opt_pr_multi = (int)value;
        return RG_OK;
    }
    if (option == 12) {
        if (value != 0 && value != 1) { set_error("invalid argument: option 12 (bounded sweep) must be 0 or 1"); return RG_ERR_ARG; }
        c->opt_bounded = (int)value;
        return RG_OK;
    }
    if (option == 13) {
        if (value < 1 || value > 1000) { set_error("invalid argument: option 13 (prefix share x 1000) must be in [1, 1000]"); return RG_ERR_ARG; }
        c->opt_rho_milli = (int)value;
        return RG_OK;
    }
    if (option == 14) {
        if (value < 1 || value > 65536) { set_error("invalid argument: option 14 (candidates per pair) must be in [1, 65536]"); return RG_ERR_ARG; }
        c->opt_bounded_k = (int)value;
        return RG_OK;
    }
    if (option == 15) {
        if (value != 0 && value != 1) { set_error("invalid argument: option 15 (bound-only prefix stage) must be 0 or 1"); return RG_ERR_ARG; }
        c->opt_bound_prefix = (int)value;
        return RG_OK;
    }
    if (option == 16) {
        if (value < 1 || value > 1000) { set_error("invalid argument: option 16 (stage-A prefix share x 1000) must be in [1, 1000]"); return RG_ERR_ARG; }
        c->opt_rho0_milli = (int)value;
        return RG_OK;
    }
    if (option == 8) {
        if (value < 0 || value > 1000000000ll) { set_error("invalid argument: option 8 (flag list capacity) must be in [0, 1e9]"); return RG_ERR_ARG; }
        c->opt_list_cap = value;
        return RG_OK;
    }
    set_error("invalid argument: unknown option %d", option);
    return RG_ERR_ARG;
}

// Phase times of the calls made since profiling was switched on / last read (option 1): out_ms[0..4] = summed
// milliseconds of {prepare, solve, score kernel, fixup + repair, select}, *out_calls = number of calls covered.
// A pass of the bounded sweep has three or four scorer launches: its score phase is their sum; its fixup phase runs from the
// end of prefix stage A to the chosen candidates, and its select phase from there to the end of its tail.
// Synchronises the stream; resets the ring.
int rg_get_profile(void* ctx, void* stream, double* out_ms5, int* out_calls) {
    RG_CHECK_ARG(ctx != nullptr && out_ms5 != nullptr && out_calls != nullptr, "null argument");
    Ctx* c = (Ctx*)ctx;
    RG_CUDA(cudaSetDevice(c->device));
    RG_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    for (int k = 0; k < Ctx::kProfPhases; ++k) out_ms5[k] = 0.0;
    *out_calls = c->prof_calls;
    int complete = 0;
    for (int call = 0; call < c->prof_calls; ++call) {
        const unsigned need = (1u << (Ctx::kProfPhases + 1)) - 1u;
        if ((c->prof_masks[call] & need) != need) continue;                             // pass aborted between two boundaries
        cudaEvent_t* e = c->prof_ev + call * Ctx::kProfEvents;
        const bool own_start = (c->prof_masks[call] >> Ctx::kProfScoreStart) & 1u;     // the scorer's own start was recorded
        for (int k = 0; k < Ctx::kProfPhases; ++k) {
            float ms = 0.f;
            RG_CUDA(cudaEventElapsedTime(&ms, (k == 2 && own_start) ? e[Ctx::kProfScoreStart] : e[k], e[k + 1]));
            out_ms5[k] += ms;
        }
        for (int b = Ctx::kProfSweep; b + 1 < Ctx::kProfEvents; b += 2) {   // the bounded sweep's later scorer launches
            if (((c->prof_masks[call] >> b) & 3u) != 3u) continue;
            float ms = 0.f;
            RG_CUDA(cudaEventElapsedTime(&ms, e[b], e[b + 1]));
            out_ms5[2] += ms;
        }
        ++complete;
    }
    *out_calls = complete;
    c->prof_calls = 0;
    c->prof_open = false;
    c->prof_cur = -1;
    return RG_OK;
}

}  // extern "C"
