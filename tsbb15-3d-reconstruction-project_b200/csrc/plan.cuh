// Host-side work planning shared by the F and PnP entry points.
#pragma once
#include "score_core.cuh"
#include <algorithm>
#include <cstdlib>

namespace rg {


inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// Fill the PairInfo table (integer part) on the host and upload it.  Work items of the packed scorer:
// item = (pair, kHypPerBlock-hypothesis block, contiguous range of kSub-point groups), claimed dynamically by the persistent grid.
// resident blocks per SM of a persistent scorer instantiation (queried once; also sets the dynamic smem attribute)
// (cached per DEVICE: cudaFuncSetAttribute is a per-device function attribute, and one process may drive several GPUs)
template <class Pol>
inline int score_blocks_per_sm(int* out) {
    static int cached[64] = {0};
    int dev = 0;
    RG_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) { set_error("device ordinal %d out of range", dev); return RG_ERR_ARG; }
    if (cached[dev] == 0) {
        constexpr size_t smem = score_smem_bytes<Pol>();
        RG_CUDA(cudaFuncSetAttribute(score_packed<Pol>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int n = 0;
        RG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, score_packed<Pol>, kScoreThreads, smem));
        cached[dev] = n < 1 ? 1 : n;
    }
    *out = cached[dev];
    return RG_OK;
}

// The per-pass PairInfo table travels host -> device through a KERNEL that reads the page-locked staging buffer (mapped under
// unified addressing), not through cudaMemcpyAsync: a copy-engine transfer queues behind every upload submitted before it,
// and the host-buffer entry point submits gigabytes of uploads ahead of the passes — the 3 KB table of pass 0 then waited for
// the whole batch's upload and nothing overlapped (measured: config 5 end to end 1237 ms against 1115 ms device resident,
// the difference being exactly the 6.5 GB upload).
__global__ void stage_fetch(const int4* __restrict__ host_mapped, int4* __restrict__ dev, int n16) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n16) dev[i] = host_mapped[i];
}

// Work items of one table: every entry has pt/n/hyp/H and its group window [g_base, g_end) set; fills item_off / nsplit /
// groups_per_split and returns the number of items (-1: too many).
inline long long plan_items(const Ctx* c, PairInfo* pi, int P, int blocks_per_sm) {
    long long unit_total = 0;      // work in units of (hypothesis block x point group)
    for (int p = 0; p < P; ++p) unit_total += (long long)ceil_div(pi[p].H, kHypPerBlock) * (pi[p].g_end - pi[p].g_base);
    const long long grid = (long long)c->sm_count * blocks_per_sm;
    // Items are claimed dynamically, so what matters is (a) enough items per resident block that the tail is short and
    // (b), for SMALL batches (one pair split over GPUs: a few hundred items), an item count that fills whole rounds of the
    // grid: 784 equal items on 592 resident blocks take two rounds (66 % busy), 592 take one.  Aim for ~kItemsPerBlock
    // items per block, never below 16 groups (128 points) per item, then search the neighbourhood of that size for the
    // split whose rounded-up rounds waste the least (uniform batches; ragged ones take the target as is).  Since the
    // guard-band flags went from a bitmap to a list, item boundaries may fall on any group.
    static const long long kItemsPerBlock = [] {
        const char* e = getenv("RG_ITEMS_PER_BLOCK");
        const long long v = e ? atoll(e) : 0;
        return v > 0 ? v : 24ll;              // measured on B200, config-5 batch: 8 -> 4.17 ms, 24 -> 4.07 ms, 48 -> 4.07 ms
    }();
    long long gps_target = std::max<long long>(64, unit_total / std::max<long long>(1, grid * kItemsPerBlock));
    bool uniform = P > 0;
    for (int p = 1; p < P; ++p)
        uniform = uniform && pi[p].g_end - pi[p].g_base == pi[0].g_end - pi[0].g_base && pi[p].H == pi[0].H;
    if (uniform && pi[0].g_end > pi[0].g_base && pi[0].H > 0) {
        const long long ng = pi[0].g_end - pi[0].g_base;
        const long long hb_total = (long long)P * ceil_div(pi[0].H, kHypPerBlock);
        // large batches keep >= kItemsPerBlock items per block (the dynamic tail is half an item); a batch so small that the
        // target sits on its floor may also use fewer, larger items when that fills the grid's rounds better
        const bool small = gps_target == 64;
        // (upper end 4 x the floor: with 256-hypothesis items one rank's share of a split pair fills ONE round of the
        //  592-block grid at 169 groups per item — 0.614 -> 0.572 / 0.326 -> 0.323 / 0.186 -> 0.182 ms for the 1/2, 1/4, 1/8
        //  shares of config 3, profiles/r02_split_gps_sweep.txt)
        const long long lo = std::max<long long>(16, gps_target / 2), hi = std::min<long long>(ng, small ? gps_target * 4 : gps_target);
        double best_cost = 1e300;
        long long best_gps = std::min<long long>(ng, gps_target);
        for (long long gps = lo; gps <= hi; ++gps) {
            const long long items = hb_total * ceil_div(ng, gps);
            const long long rounds = (items + grid - 1) / grid;
            // makespan in group-units per block (+ a per-item cost of ~6 groups: hypothesis reload, claim, count atomics)
            const double cost = (double)rounds * (double)(gps + 6);
            if (cost < best_cost * (1.0 - 1e-9)) { best_cost = cost; best_gps = gps; }
        }
        gps_target = best_gps;
    }
    {   // experiment hook: RG_FORCE_GPS=<groups per item> overrides the planner (tools/r2_eighth_probe.py sweeps it)
        static const long long forced = [] { const char* e = getenv("RG_FORCE_GPS"); return e ? atoll(e) : 0ll; }();
        if (forced > 0) gps_target = forced;
    }
    long long item_off = 0;
    for (int p = 0; p < P; ++p) {
        PairInfo& o = pi[p];
        const int ng = o.g_end - o.g_base;
        const int nhb = ceil_div(o.H, kHypPerBlock);
        o.item_off = (int)item_off;
        if (ng == 0 || nhb == 0) { o.nsplit = 1; o.groups_per_split = 0; continue; }     // contributes no items
        int gps = (int)std::min<long long>(ng, gps_target);
        int ns = ceil_div(ng, gps);
        gps = ceil_div(ng, ns);
        ns = ceil_div(ng, gps);
        o.nsplit = ns;
        o.groups_per_split = gps;
        item_off += (long long)nhb * ns;
    }
    // (pairs without items share their item_off with the next pair; decode_item takes the LAST pair whose
    //  item_off <= item, which is never an empty one)
    return item_off < (1ll << 31) ? item_off : -1;
}

// Prefix window of the bounded sweep: ceil(rho * G) groups rounded up to whole 32-group flag words, at most G.
inline int bounded_prefix_groups(int G, int rho_milli) {
    const long long g = ((long long)G * rho_milli + 999) / 1000;
    return (int)std::min<long long>(G, (g + 31) / 32 * 32);
}

// bounded_k > 0: the bounded sweep's four tables (bounded.cuh) go into pair_info as [prefix stage A | candidate stage |
// fallback template | stage-B template], P entries each; stage A's table is also the pass's main table (solver, selection,
// masks).  bound_prefix: the prefix stages count an upper bound only, so the candidate and fallback stages cover the whole
// pair, and stage A stops at rho0 (rho0_milli) when that is shorter than rho; stage B covers the rest of the prefix.
inline int f_plan(Ctx* c, cudaStream_t st, int P, const int* pair_off, const int* hyp_off, FPlan& plan, int blocks_per_sm,
                  const int* n_vote = nullptr /* PnP: per-view number of voting correspondences (<= view size) */,
                  int hyp_first = 0 /* hypothesis-split mode: global index of this rank's first hypothesis */,
                  int bounded_k = 0, int rho_milli = 0, bool bound_prefix = false, int rho0_milli = 0) {
    RG_CHECK_ARG(P >= 0 && P <= 65535, "number of pairs must be in [0, 65535]");
    RG_CHECK_ARG(pair_off != nullptr && hyp_off != nullptr, "offset arrays are null");
    RG_CHECK_ARG(pair_off[0] == 0 && hyp_off[0] == 0, "offset arrays must start at 0");
    plan = FPlan();
    plan.P = P;
    if (P == 0) return RG_OK;
    for (int p = 0; p < P; ++p) {
        RG_CHECK_ARG(pair_off[p + 1] >= pair_off[p] && hyp_off[p + 1] >= hyp_off[p], "offset arrays must be non-decreasing");
    }
    // A call that repeats the previous call's tables (hypothesis-split mode: same pair, same block, call after call) finds
    // its PairInfo table still on the device: no staging, no upload, no host synchronisation — which also makes the whole
    // launch chain capturable in a CUDA graph.
    unsigned long long hsh = 1469598103934665603ull;
    auto mix = [&hsh](unsigned v) { hsh ^= v; hsh *= 1099511628211ull; };
    for (int p = 0; p <= P; ++p) { mix((unsigned)pair_off[p]); mix((unsigned)hyp_off[p]); }
    if (n_vote) for (int p = 0; p < P; ++p) mix((unsigned)n_vote[p]);
    mix((unsigned)hyp_first); mix((unsigned)blocks_per_sm); mix(n_vote ? 1u : 0u); mix((unsigned)P);
    mix((unsigned)bounded_k); mix((unsigned)rho_milli); mix(bound_prefix ? 1u : 0u); mix((unsigned)rho0_milli);
    if (c->plan_valid && c->plan_hash == hsh && c->plan_cached.P == P && c->pair_info.ptr == c->plan_table) {
        plan = c->plan_cached;
        return RG_OK;
    }
    c->plan_valid = false;
    const int n_tables = bounded_k > 0 ? 4 : 1;
    const int turn = c->stage_turn;       // double-buffered staging: planning pass k+1 does not wait for pass k's kernels
    c->stage_turn ^= 1;
    int rc = ensure_pinned(c->h_stage[turn], sizeof(PairInfo) * (size_t)P * n_tables);
    if (rc) return rc;
    RG_CUDA(cudaEventSynchronize(c->staging_free[turn]));
    PairInfo* pi = (PairInfo*)c->h_stage[turn].ptr;

    long long off32 = 0;
    for (int p = 0; p < P; ++p) {
        PairInfo& o = pi[p];
        memset(&o, 0, sizeof(o));
        o.pt_off = pair_off[p];
        o.n_all = pair_off[p + 1] - pair_off[p];
        o.n = n_vote ? n_vote[p] : o.n_all;
        RG_CHECK_ARG(o.n >= 0 && o.n <= o.n_all, "voting count must be in [0, view size]");
        o.hyp_off = hyp_off[p];
        o.H = hyp_off[p + 1] - hyp_off[p];
        o.hyp_first = hyp_first;
        o.n_pad = ((o.n + kSub - 1) / kSub) * kSub;
        o.pt_off32 = (int)off32;
        o.g_base = 0;
        o.g_end = o.n_pad / kSub;
        off32 += o.n_pad;
        plan.maxN = std::max(plan.maxN, o.n);
        plan.maxH = std::max(plan.maxH, o.H);
        plan.evals += (double)o.n * (double)o.H;
    }
    RG_CHECK_ARG(off32 < (1ll << 31) && (long long)hyp_off[P] * 9 < (1ll << 40), "batch too large for 32-bit offsets");
    plan.Ntot = pair_off[P];
    plan.Htot = hyp_off[P];
    plan.N32tot = off32;
    if (bounded_k > 0) {
        // prefix stage A: every hypothesis over groups [0, gA0); candidate stage: min(K, H) compact records per pair over
        // [gA, G) ([0, G) after a bound-only prefix); fallback template: every hypothesis over the same window as the
        // candidates (bnd_live_plan keeps the marked pairs' items); stage-B template: room for the H - min(K, H)
        // non-candidates over [gA0, gA) (bnd_live_plan keeps the items of those bnd_extend gathered)
        PairInfo* pc = pi + P;
        PairInfo* pf = pi + 2 * (size_t)P;
        PairInfo* pb = pi + 3 * (size_t)P;
        plan.bounded = true;
        plan.bound_prefix = bound_prefix;
        plan.K = bounded_k;
        plan.evals = 0.0;
        long long coff = 0, boff = 0;
        for (int p = 0; p < P; ++p) {
            PairInfo& o = pi[p];
            const int G = o.g_end, gA = bounded_prefix_groups(G, rho_milli);
            const int gA0 = bound_prefix ? std::min(gA, bounded_prefix_groups(G, rho0_milli)) : gA;
            const int kA = std::min(o.n, gA * kSub);              // real correspondences of the prefix
            o.g_end = gA;
            pf[p] = o;
            pf[p].g_base = bound_prefix ? 0 : gA; pf[p].g_end = G;
            pc[p] = pf[p];
            pc[p].hyp_off = (int)coff;
            pc[p].H = std::min(o.H, bounded_k);
            coff += pc[p].H;
            pb[p] = o;
            pb[p].g_base = gA0;
            pb[p].hyp_off = (int)boff;
            pb[p].H = o.H - pc[p].H;
            boff += pb[p].H;
            o.g_end = gA0;
            const int rest = bound_prefix ? o.n : o.n - kA;          // real correspondences of the later stages' window
            plan.evals += (double)std::min(o.n, gA0 * kSub) * (double)o.H;
            plan.evals_c += (double)rest * (double)pc[p].H;
            plan.evals_f += (double)rest * (double)o.H;
        }
        plan.Ctot = coff;
        plan.Btot = boff;
        const long long nc = plan_items(c, pc, P, blocks_per_sm), nf = plan_items(c, pf, P, blocks_per_sm),
                        nb = plan_items(c, pb, P, blocks_per_sm);
        RG_CHECK_ARG(nc >= 0 && nf >= 0 && nb >= 0, "too many scorer work items");
        plan.n_items_c = (int)nc;
        plan.n_items_f = (int)nf;
        plan.n_items_b = (int)nb;
    }
    const long long n_items = plan_items(c, pi, P, blocks_per_sm);
    RG_CHECK_ARG(n_items >= 0, "too many scorer work items");
    plan.n_items = (int)n_items;
    rc = ensure(c->pair_info, sizeof(PairInfo) * (size_t)P * n_tables);
    if (rc) return rc;
    static_assert(sizeof(PairInfo) % 16 == 0, "PairInfo is copied as int4");
    const int n16 = (int)(sizeof(PairInfo) / 16) * P * n_tables;
    stage_fetch<<<(n16 + 255) / 256, 256, 0, st>>>((const int4*)pi, (int4*)c->pair_info.ptr, n16);
    RG_CUDA(cudaGetLastError());
    RG_CUDA(cudaEventRecord(c->staging_free[turn], st));
    c->plan_cached = plan;
    c->plan_hash = hsh;
    c->plan_table = c->pair_info.ptr;
    c->plan_valid = true;
    return RG_OK;
}


}  // namespace rg
