// Bounded sweep of the F path: score every hypothesis on a prefix of each pair's correspondences, finish only the best
// prefix scores, and prove that no other hypothesis can reach the pair's maximum.
//
// Per pass, after the head (memset, prepare, solve):
//   prefix stage A   every hypothesis x groups [0, gA0) (the main table's window): counts[h] = c^0(h) >= the exact count over
//                    the first k0 = min(n, gA0 * kSub) correspondences.  Option 15 = 1 (default): score_packed<EpiBoundPolicy>,
//                    an upper bound with no fix-up; option 15 = 0: score_packed<EpiPolicy> + fix-up, exact counts.
//   bnd_select       per pair the K hypotheses with the largest (c^0, -index), gathered into compact Hyp32 records + map
//   candidate stage  score_packed over the compact records + fix-up (map: compact -> global index), over [gA, G) after an
//                    exact prefix (sfx_c[j] = exact count over the other n - k correspondences) or over [0, G) after a
//                    bound-only prefix (sfx_c[j] = exact full count)
//   bnd_extend       L = the candidates' largest full count.  S = the non-candidates with c^0(h) + (n - k0) >= L.  Since
//                    c^(h) >= c^0(h), a member with c^0(h) + (n - k) >= L already fails the test below: such a pair is
//                    marked here and skips stage B (with gA0 = gA every member of S does).  Otherwise S is gathered into
//                    compact records + map; bnd_live_plan turns the stage-B template into their live item table.
//   prefix stage B   score_packed<EpiBoundPolicy> over S x groups [gA0, gA) (bound-only prefix only; with an exact prefix,
//                    or rho0 >= rho, gA0 = gA and the stage has no items), item count read from the device
//   bnd_check        adds the stage-B counts into counts: c^(h) = c^0(h) + c^B(h) for h in S, the bound over the first
//                    k = min(n, gA * kSub) correspondences, bit for bit what a one-step prefix over [0, gA) counts.  A
//                    non-candidate's full count is at most c^(h) + (n - k); if that is below L it can never be the maximum
//                    nor tie with it.  Outside S, c^0(h) + (n - k) <= c^0(h) + (n - k0) < L, so only members of S can fail
//                    the test.  Pairs where one does are marked; the others get the candidates' full counts written into counts.
//   bnd_live_plan    the fallback table: the marked pairs' items over the candidates' window for EVERY hypothesis (usually none)
//   fallback stage   score_packed with the item count read from the device + fix-up into sfx_f; bnd_merge adds sfx_f to the
//                    marked pairs' prefix counts (or writes it, after a bound-only prefix): full counts for every hypothesis.
// In an unmarked pair a hypothesis that was not fully scored keeps c^0(h) or c^(h), both < L <= max, and has
// full(h) < L, so argmax_counts' first maximum, the tie replay over the hypotheses with count == max and the winner's mask
// are those of a full sweep.
#pragma once
#include "score_core.cuh"

namespace rg {

// one 256-thread block fits beside the four resident scorer blocks of an SM (bnd_select runs beside the next pass's scorer)
constexpr int kSelectThreads = 256;

// exclusive prefix of `v` over the block (in thread order) and the block total; every thread calls it
__device__ __forceinline__ int block_excl_scan(int v, int* s_warp, int& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    __syncthreads();
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int before = 0;
    total = 0;
    for (int w = 0; w < nw; ++w) {
        const int t = s_warp[w];
        if (w < warp) before += t;
        total += t;
    }
    return before + incl - v;
}

// Copies, in index order, the records of the pair's hypotheses h < H with take(h, v, eq, rank) to out / map (v = cnt[h];
// eq = v == tie, rank = hypotheses before h with v == tie) and returns how many it took; out / map hold `cap` records.
// Every thread calls it.
template <class Take>
__device__ __forceinline__ int gather_hyp(const int* __restrict__ cnt, int H, int hyp_off, int tie,
                                          const Hyp32* __restrict__ hyp32, Hyp32* __restrict__ out, int* __restrict__ map,
                                          int cap, int* s_warp, Take take) {
    int taken = 0, ties = 0;
    for (int base = 0; base < H; base += blockDim.x) {
        const int h = base + threadIdx.x;
        const int v = h < H ? cnt[h] : -2;
        const bool eq = h < H && v == tie;
        int tot_eq = 0, tot_sel = 0;
        const int eq_before = block_excl_scan(eq ? 1 : 0, s_warp, tot_eq);
        const bool is_sel = h < H && take(h, v, eq, ties + eq_before);
        const int pos = taken + block_excl_scan(is_sel ? 1 : 0, s_warp, tot_sel);
        if (is_sel) {
            RG_ASSERT(pos < cap);
            out[pos] = hyp32[hyp_off + h];
            map[pos] = hyp_off + h;
        }
        taken += tot_sel;
        ties += tot_eq;
    }
    return taken;
}

// One CTA per pair: the candidates are the min(K, H) hypotheses with the largest (c_A, -index), stored in index order.
// sel[p] = {T, last, n_sel, L}: a hypothesis is a candidate iff c_A > T or (c_A == T and index <= last); T = -1 when every
// hypothesis is one.  L (the candidates' largest full count) is filled in by bnd_extend.
__global__ void __launch_bounds__(kSelectThreads) bnd_select(const int* __restrict__ counts, const PairInfo* __restrict__ pi,
                                                              const PairInfo* __restrict__ pc, const Hyp32* __restrict__ hyp32,
                                                              Hyp32* __restrict__ hypc, int* __restrict__ map,
                                                              int4* __restrict__ sel) {
    __shared__ int hist[256];
    __shared__ int s_warp[32];
    __shared__ int s_bin, s_k, s_last;
    const int p = blockIdx.x;
    const PairInfo info = pi[p];
    const int Kp = pc[p].H, cbase = pc[p].hyp_off;
    const int* cnt = counts + info.hyp_off;
    int T = -1, need = 0;
    if (Kp < info.H) {
        // radix select of the Kp-th largest count, 8 bits at a time from the top
        unsigned prefix = 0u, mask = 0u;
        int k = Kp;
        for (int shift = 24; shift >= 0; shift -= 8) {
            for (int b = threadIdx.x; b < 256; b += blockDim.x) hist[b] = 0;
            __syncthreads();
            for (int h = threadIdx.x; h < info.H; h += blockDim.x) {
                const unsigned v = (unsigned)cnt[h];
                if ((v & mask) == prefix) atomicAdd(&hist[(v >> shift) & 255u], 1);
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                int cum = 0, b = 255;
                for (; b > 0 && cum + hist[b] < k; --b) cum += hist[b];
                s_bin = b;
                s_k = k - cum;
            }
            __syncthreads();
            prefix |= (unsigned)s_bin << shift;
            mask |= 255u << shift;
            k = s_k;
            __syncthreads();
        }
        T = (int)prefix;
        need = k;                      // candidates among the hypotheses with c_A == T (the first `need` in index order)
    }
    if (threadIdx.x == 0) s_last = -1;
    const int taken = gather_hyp(cnt, info.H, info.hyp_off, T, hyp32, hypc + cbase, map + cbase, Kp, s_warp,
                                 [&](int h, int v, bool eq, int rank) {
                                     const bool take = v > T || (eq && rank < need);
                                     if (take && eq) atomicMax(&s_last, h);
                                     return take;
                                 });
    __syncthreads();
    if (threadIdx.x == 0) {
        RG_ASSERT(taken == Kp);
        sel[p] = make_int4(T, s_last, taken, 0);
    }
}

__device__ __forceinline__ int block_reduce_max(int v, int* s) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = v;
    __syncthreads();
    int r = s[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) r = max(r, s[w]);
    return r;
}

// One CTA per pair, after the candidate stage's fix-up.  exact_prefix: counts hold exact prefix counts and sfx_c suffix
// counts; otherwise counts hold upper bounds of the prefix counts and sfx_c full counts.  pb: the stage-B template (window
// [gA0, gA), room for H - K records at hyp_off).  Stores L in sel[p].w.  A pair whose fallback is already certain gets
// mark[p] = H and n_s[p] = 0; otherwise S (non-candidates with c^0 + (n - k0) >= L) is gathered into hypb / mapb at
// pb[p].hyp_off, n_s[p] = |S| and stats[3] += |S| * (k - k0): the evaluations of stage B.
__global__ void __launch_bounds__(256) bnd_extend(const int* __restrict__ counts, const int* __restrict__ sfx_c,
                                                   const int* __restrict__ map, const PairInfo* __restrict__ pi,
                                                   const PairInfo* __restrict__ pc, const PairInfo* __restrict__ pb,
                                                   const Hyp32* __restrict__ hyp32, int4* __restrict__ sel,
                                                   Hyp32* __restrict__ hypb, int* __restrict__ mapb, int* __restrict__ n_s,
                                                   int* __restrict__ mark, unsigned long long* __restrict__ stats,
                                                   bool exact_prefix) {
    __shared__ int s_red[32];
    const int p = blockIdx.x;
    const PairInfo info = pi[p], b = pb[p];
    const int Kp = pc[p].H, cbase = pc[p].hyp_off;
    const int4 sl = sel[p];
    const int k0 = min(info.n, b.g_base * kSub), k = min(info.n, b.g_end * kSub);
    int L = 0;
    for (int j = threadIdx.x; j < Kp; j += blockDim.x)
        L = max(L, (exact_prefix ? counts[map[cbase + j]] : 0) + sfx_c[cbase + j]);
    L = block_reduce_max(L, s_red);
    const int rest0 = info.n - k0, rest = info.n - k;
    const int* cnt = counts + info.hyp_off;
    int sure = 0;
    for (int h = threadIdx.x; h < info.H; h += blockDim.x) {
        const int v = cnt[h];
        const bool cand = v > sl.x || (v == sl.x && h <= sl.y);
        sure |= (!cand && (long long)v + rest >= (long long)L) ? 1 : 0;
    }
    sure = block_reduce_max(sure, s_red);
    if (sure) {
        if (threadIdx.x == 0) {
            sel[p].w = L;
            mark[p] = info.H;
            n_s[p] = 0;
        }
        return;
    }
    // (k == k0: every member of S would have been a certain escapee, so S is empty)
    const int ns = k == k0 ? 0
                           : gather_hyp(cnt, info.H, info.hyp_off, -1, hyp32, hypb + b.hyp_off, mapb + b.hyp_off, b.H, s_red,
                                        [&](int h, int v, bool, int) {
                                            const bool cand = v > sl.x || (v == sl.x && h <= sl.y);
                                            return !cand && (long long)v + rest0 >= (long long)L;
                                        });
    if (threadIdx.x == 0) {
        RG_ASSERT(ns <= b.H);
        sel[p].w = L;
        n_s[p] = ns;
        if (ns && k > k0) atomicAdd(&stats[3], (unsigned long long)ns * (unsigned long long)(k - k0));
    }
}

// One CTA per pair, after stage B.  stats: [0] fallback evaluations, [1] hypotheses not fully scored, [2] pairs that fell
// back.  Adds stage B's counts (cnt_b, compact like S) into counts, then marks the pair (mark[p] = H: every hypothesis is
// live in the fallback) when a member of S has c^(h) + (n - k) >= L (>=: a tie with the maximum must be scored too), or
// keeps the mark bnd_extend set.
__global__ void __launch_bounds__(256) bnd_check(int* __restrict__ counts, const int* __restrict__ sfx_c,
                                                  const int* __restrict__ map, const int* __restrict__ cnt_b,
                                                  const int* __restrict__ mapb, const int* __restrict__ n_s,
                                                  const PairInfo* __restrict__ pi, const PairInfo* __restrict__ pc,
                                                  const PairInfo* __restrict__ pb, const int4* __restrict__ sel,
                                                  int* __restrict__ mark, unsigned long long* __restrict__ stats,
                                                  bool exact_prefix) {
    __shared__ int s_red[8];
    const int p = blockIdx.x;
    const PairInfo info = pi[p];
    const int Kp = pc[p].H, cbase = pc[p].hyp_off, bbase = pb[p].hyp_off;
    const int L = sel[p].w;
    const int rest = info.n - min(info.n, pb[p].g_end * kSub);     // correspondences outside the prefix [0, gA)
    int esc = mark[p] != 0;
    for (int j = threadIdx.x; j < n_s[p]; j += blockDim.x) {
        const int h = mapb[bbase + j];
        const int v = counts[h] + cnt_b[bbase + j];
        counts[h] = v;
        esc |= ((long long)v + rest >= (long long)L) ? 1 : 0;
    }
    esc = block_reduce_max(esc, s_red);
    if (esc) {
        if (threadIdx.x == 0) {
            mark[p] = info.H;
            atomicAdd(&stats[0], (unsigned long long)info.H * (unsigned long long)(exact_prefix ? rest : info.n));
            atomicAdd(&stats[2], 1ull);
        }
        return;
    }
    for (int j = threadIdx.x; j < Kp; j += blockDim.x)
        counts[map[cbase + j]] = (exact_prefix ? counts[map[cbase + j]] : 0) + sfx_c[cbase + j];
    if (threadIdx.x == 0 && info.H > Kp) atomicAdd(&stats[1], (unsigned long long)(info.H - Kp));
}

// One CTA: the live table of a stage whose hypotheses are chosen on the device = the template with H = live[p] (the stage-B
// records of S, or every hypothesis of a marked pair in the fallback) and the items of the other hypothesis blocks
// removed; *n_items = their total.
__global__ void __launch_bounds__(kSelectThreads) bnd_live_plan(const PairInfo* __restrict__ tmpl, const int* __restrict__ live,
                                                                 int P, PairInfo* __restrict__ out, int* __restrict__ n_items) {
    __shared__ int s_warp[32];
    int run = 0;
    for (int base = 0; base < P; base += blockDim.x) {
        const int p = base + threadIdx.x;
        int items = 0;
        PairInfo o;
        if (p < P) {
            o = tmpl[p];
            o.H = live[p];
            RG_ASSERT(o.H >= 0 && o.H <= tmpl[p].H);
            if (o.groups_per_split > 0) items = (o.H + kHypPerBlock - 1) / kHypPerBlock * o.nsplit;
        }
        int tot = 0;
        const int before = block_excl_scan(items, s_warp, tot);
        if (p < P) {
            o.item_off = run + before;
            out[p] = o;
        }
        run += tot;
    }
    if (threadIdx.x == 0) *n_items = run;
}

// One CTA per pair: marked pairs add the fallback's suffix counts to the exact prefix counts, or take the fallback's full
// counts after a bound-only prefix
__global__ void __launch_bounds__(256) bnd_merge(int* __restrict__ counts, const int* __restrict__ sfx_f,
                                                  const PairInfo* __restrict__ pi, const int* __restrict__ mark,
                                                  bool exact_prefix) {
    const int p = blockIdx.x;
    if (!mark[p]) return;
    const PairInfo info = pi[p];
    for (int h = threadIdx.x; h < info.H; h += blockDim.x)
        counts[info.hyp_off + h] = (exact_prefix ? counts[info.hyp_off + h] : 0) + sfx_f[info.hyp_off + h];
}

}  // namespace rg
