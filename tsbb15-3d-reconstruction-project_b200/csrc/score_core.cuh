// Generic persistent FP32 scorer skeleton shared by the F path (epipolar criterion) and the PnP path (reprojection
// criterion).  A policy supplies the packed point layout, the hypothesis record and the two-point evaluation.
#pragma once
#include "common.cuh"

namespace rg {

#ifndef RG_SCORE_BLOCKS
#define RG_SCORE_BLOCKS 4      // 128 threads x 4 blocks: 2 stages x (8 KB points + 16 KB hypothesis records) per block, <= 128 registers
#endif
#ifndef RG_EPI_CHUNK
#define RG_EPI_CHUNK 512
#endif
#ifndef RG_SCORE_THREADS
#define RG_SCORE_THREADS 128      // 4 warps per barrier domain: 128 x 4 blocks beats 256 x 2 by 1.7 % (profiles/r02_variant_sweep_rot.txt)
#endif
#ifndef RG_HPT
#define RG_HPT 2
#endif
#ifndef RG_PAIR_UNROLL
#define RG_PAIR_UNROLL 4          // point pairs of a flag group evaluated per unrolled loop body (kSub / 2 = all)
#endif
constexpr int kScoreThreads = RG_SCORE_THREADS;
constexpr int kScoreBlocksPerSM = RG_SCORE_BLOCKS;
constexpr int kHypPerThread = RG_HPT;
constexpr int kHypPerBlock  = kScoreThreads * kHypPerThread;   // 256 hypotheses per work item
constexpr int kStages       = 2;
constexpr int kPairUnroll   = RG_PAIR_UNROLL;

// packed FMA with scalar operands broadcast inside the instruction (SASS: FFMA2 Rd, Rs.F32, Rb.F32x2, ...).  Building the
// {s, s} pair inside the asm block keeps the coefficient in ONE register: a duplicated pair would cost a second
// register-file read per use, and the scorer is bound by register-file read ports (DESIGN.md, "scorer").
__device__ __forceinline__ float2 ffma2_sbc(float s, float2 b, float2 c) {          // {s,s} * b + c
    float2 d;
    asm("{\n.reg .b64 ts, tb, tc, td;\nmov.b64 ts, {%2, %2};\nmov.b64 tb, {%3, %4};\nmov.b64 tc, {%5, %6};\n"
        "fma.rn.f32x2 td, ts, tb, tc;\nmov.b64 {%0, %1}, td;\n}"
        : "=f"(d.x), "=f"(d.y) : "f"(s), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
}
__device__ __forceinline__ float2 ffma2_sbs(float s, float2 b, float c) {           // {s,s} * b + {c,c}
    float2 d;
    asm("{\n.reg .b64 ts, tb, tc, td;\nmov.b64 ts, {%2, %2};\nmov.b64 tb, {%3, %4};\nmov.b64 tc, {%5, %5};\n"
        "fma.rn.f32x2 td, ts, tb, tc;\nmov.b64 {%0, %1}, td;\n}"
        : "=f"(d.x), "=f"(d.y) : "f"(s), "f"(b.x), "f"(b.y), "f"(c));
    return d;
}

struct ScoreItem {
    int pair, h_base, H_end;        // hypotheses [h_base, min(h_base + kHypPerBlock, H_end)) (global indices)
    int g0, g1;                     // kSub-point groups [g0, g1) of the pair (inside its window [g_base, g_end))
};

__device__ __forceinline__ ScoreItem decode_item(const PairInfo* __restrict__ pi, int P, int item) {
    int lo = 0, hi = P;
    while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (pi[mid].item_off <= item) lo = mid; else hi = mid; }
    const PairInfo& info = pi[lo];
    const int local = item - info.item_off;
    RG_ASSERT(lo >= 0 && lo < P && local >= 0 && info.nsplit >= 1 && info.groups_per_split >= 1);
    const int hb = local / info.nsplit;
    const int sp = local - hb * info.nsplit;
    ScoreItem it;
    it.pair = lo;
    it.h_base = info.hyp_off + hb * kHypPerBlock;
    it.H_end = info.hyp_off + info.H;
    it.g0 = min(info.g_base + sp * info.groups_per_split, info.g_end);
    it.g1 = min(it.g0 + info.groups_per_split, info.g_end);
    RG_ASSERT(it.g0 < it.g1 && it.h_base < it.H_end && it.h_base >= info.hyp_off);
    return it;
}

// Guard-band bookkeeping: one flag per (hypothesis, kSub-point group) = "the FP32 result of at least one evaluation of this
// group lies inside the rounding band of this hypothesis"; the fix-up kernel re-evaluates exactly those groups in FP64.
// Round 1 kept the flags in a bitmap (1 bit per hypothesis and group: 102 MB written by the scorer and scanned by the
// fix-up for a 16-pair batch although only 0.36 % of the bits are set).  Now a thread collects the 32 flags of 256
// consecutive correspondences in a register and, once per such word, the warp appends its set flags as dense
// (hypothesis, group) records to ONE global list (warp-aggregated: REDUX + prefix + one atomicAdd per warp and word, outside
// the evaluation loop).  If the list is full the hypothesis is marked in `ovf` and recounted entirely in FP64 by the fix-up
// kernel, so adversarial inputs (everything on the threshold) degrade to the FP64 path instead of failing (the slots such
// an append had reserved inside the list are filled with sentinel records).
struct FlagList {
    int2* rec;                 // {global hypothesis index, group index inside the pair}
    unsigned* n;               // records appended so far (may exceed cap: the excess was not stored)
    unsigned cap;
    unsigned char* ovf;        // per hypothesis: 1 = some records of this hypothesis were dropped
};

// all 32 lanes call this (fl = 0 for lanes with nothing to append)
__device__ __forceinline__ void flag_append(const FlagList& L, unsigned fl, int h, int group_base) {
    const unsigned full = 0xffffffffu;
    const int nb = __popc(fl);
    const int tot = __reduce_add_sync(full, nb);
    if (tot == 0) return;
    const int lane = threadIdx.x & 31;
    int incl = nb;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(full, incl, o);
        if (lane >= o) incl += v;
    }
    unsigned base = 0u;
    if (lane == 0) base = atomicAdd(L.n, (unsigned)tot);
    base = __shfl_sync(full, base, 0);
    if (nb == 0) return;
    unsigned pos = base + (unsigned)(incl - nb);
    if (base + (unsigned)tot > L.cap || base + (unsigned)tot < base) {      // list full: FP64 recount of this hypothesis
        L.ovf[h] = 1;
        // the part of [base, base + tot) that lies inside the list is counted as present by the fix-up (it reads
        // min(n, cap) records): fill it with sentinels, or it would re-apply whatever an earlier call left there
        for (int k = 0; k < nb; ++k)
            if (pos + (unsigned)k < L.cap && base + (unsigned)tot >= base) L.rec[pos + k] = make_int2(-1, -1);
        return;
    }
    while (fl) {
        const int b = __ffs(fl) - 1;
        fl &= fl - 1;
        RG_ASSERT(pos < L.cap && h >= 0 && group_base + b >= 0);
        L.rec[pos++] = make_int2(h, group_base + b);
    }
}

// Policy requirements:
//   typedef Rec;                       hypothesis record in global/shared memory (sizeof % 16 == 0)
//   typedef Regs;                      hypothesis in registers
//   static constexpr bool kBoundOnly;  true: evalN(H, pair, cnt) counts an upper bound and the guard-band bookkeeping
//                                      (min|q|, flags, list appends) is compiled out; the counts need no fix-up
//   static constexpr int kVec4PerPair; float4 per packed point pair
//   static constexpr int kChunkPts;    points per shared-memory stage
//   static void load(const Rec* sh, int slot, bool valid, Regs&, float& G);
//   template <int K> static void evalN(const Regs (&H)[K], const float4* pair, unsigned (&cnt)[K], float (&minabs)[K]);
template <class Pol>
struct __align__(128) ScoreStage {
    float4 pts[Pol::kChunkPts / 2 * Pol::kVec4PerPair];
    typename Pol::Rec hyp[kHypPerBlock];
};
template <class Pol>
constexpr size_t score_smem_bytes() { return kStages * sizeof(ScoreStage<Pol>) + 64; }

// persistent block: first item blockIdx.x, then items claimed from a global counter (dynamic: with static round-robin a
// batch whose item count is not a multiple of the grid leaves most SMs idle during the last round); every item = kHypPerBlock
// hypotheses x a contiguous range of kSub-point groups of one pair.  Host guarantees every item has >= 1 group and >= 1
// hypothesis; *work_counter is 0 at launch.  n_items_dev (optional): the item count is read from the device instead (a stage
// whose size is decided on the device — the bounded sweep's fallback — is queued at full grid and usually has no items).
// Points and (at the first chunk of an item) hypothesis records arrive by 1-D bulk TMA on one mbarrier per stage;
// the next chunk / next item is always in flight while the current one is being scored.
template <class Pol>
__global__ void __launch_bounds__(kScoreThreads, kScoreBlocksPerSM)
score_packed(const float4* __restrict__ pts32, const typename Pol::Rec* __restrict__ hyp32,
             const PairInfo* __restrict__ pi, int P, int n_items, int* __restrict__ counts,
             FlagList flist, int* __restrict__ work_counter, const int* __restrict__ n_items_dev = nullptr) {
    __shared__ int s_next;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    ScoreStage<Pol>* st = reinterpret_cast<ScoreStage<Pol>*>(smem_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + kStages * sizeof(ScoreStage<Pol>));
    constexpr int kChunkPts = Pol::kChunkPts;
    constexpr uint32_t kPtBytes = Pol::kVec4PerPair * 8;        // bytes per point in the packed layout
    constexpr int kV = Pol::kVec4PerPair;

    const int tid = threadIdx.x;
    int item = blockIdx.x;
    if (n_items_dev != nullptr) n_items = *n_items_dev;
    if (item >= n_items) return;
    if (tid == 0) {
        mbar_init(&full[0], 1);
        mbar_init(&full[1], 1);
        fence_mbar_init();
    }
    __syncthreads();

    uint32_t phases = 0u;
    int stage = 0;

    ScoreItem cur = decode_item(pi, P, item);
    // packed points of the pair: kV float4 per point pair
    const float4* cur_src = pts32 + (size_t)(pi[cur.pair].pt_off32 / 2) * kV;
    if (tid == 0) {
        const uint32_t nb = (uint32_t)min((cur.g1 - cur.g0) * kSub, kChunkPts) * kPtBytes;
        const uint32_t hb = (uint32_t)min(kHypPerBlock, cur.H_end - cur.h_base) * (uint32_t)sizeof(typename Pol::Rec);
        RG_ASSERT(nb > 0 && nb <= sizeof(st[0].pts) && hb > 0 && hb <= sizeof(st[0].hyp) && nb % 16 == 0 && hb % 16 == 0);
        mbar_expect_tx(&full[0], nb + hb);
        tma_load_1d(st[0].pts, cur_src + (size_t)cur.g0 * (kSub / 2) * kV, nb, &full[0]);
        tma_load_1d(st[0].hyp, hyp32 + cur.h_base, hb, &full[0]);
    }

    while (true) {
        // claim the following item now: its first chunk and hypotheses are prefetched during the last chunk of this one
        if (tid == 0) s_next = (int)gridDim.x + atomicAdd(work_counter, 1);
        __syncthreads();                  // (the previous value was read by everybody before the last chunk's barrier)
        const int next_item = s_next;
        const bool has_next = next_item < n_items;
        ScoreItem nxt = cur;
        const float4* nxt_src = cur_src;
        if (has_next) {
            nxt = decode_item(pi, P, next_item);
            nxt_src = pts32 + (size_t)(pi[nxt.pair].pt_off32 / 2) * kV;
        }
        typename Pol::Regs Hy[kHypPerThread];
        float G[kHypPerThread];
        unsigned cnt[kHypPerThread];
        int hid[kHypPerThread];
#pragma unroll
        for (int k = 0; k < kHypPerThread; ++k) {
            G[k] = 0.f; cnt[k] = 0u;
            hid[k] = cur.h_base + k * kScoreThreads + tid;
        }

        const int total_pts = (cur.g1 - cur.g0) * kSub;
        for (int done = 0; done < total_pts; done += kChunkPts) {
            const int npts = min(total_pts - done, kChunkPts);
            // prefetch the following chunk (of this item, or the first chunk + hypotheses of the next item)
            if (tid == 0) {
                const int s2 = stage ^ 1;
                if (done + kChunkPts < total_pts) {
                    const uint32_t nb = (uint32_t)min(total_pts - done - kChunkPts, kChunkPts) * kPtBytes;
                    mbar_expect_tx(&full[s2], nb);
                    tma_load_1d(st[s2].pts, cur_src + (size_t)(cur.g0 * kSub + done + kChunkPts) / 2 * kV, nb, &full[s2]);
                } else if (has_next) {
                    const uint32_t nb = (uint32_t)min((nxt.g1 - nxt.g0) * kSub, kChunkPts) * kPtBytes;
                    const uint32_t hb =
                        (uint32_t)min(kHypPerBlock, nxt.H_end - nxt.h_base) * (uint32_t)sizeof(typename Pol::Rec);
                    mbar_expect_tx(&full[s2], nb + hb);
                    tma_load_1d(st[s2].pts, nxt_src + (size_t)nxt.g0 * (kSub / 2) * kV, nb, &full[s2]);
                    tma_load_1d(st[s2].hyp, hyp32 + nxt.h_base, hb, &full[s2]);
                }
            }
            mbar_wait(&full[stage], (phases >> stage) & 1u);
            phases ^= 1u << stage;

            if (done == 0) {
#pragma unroll
                for (int k = 0; k < kHypPerThread; ++k)
                    Pol::load(st[stage].hyp, k * kScoreThreads + tid, hid[k] < cur.H_end, Hy[k], G[k]);
            }
            const float4* sp = st[stage].pts;
            if constexpr (Pol::kBoundOnly) {           // upper-bound counts only: no min|q|, no flags, no list
#pragma unroll kPairUnroll
                for (int j = 0; j < npts / 2; ++j) Pol::template evalN<kHypPerThread>(Hy, sp + j * kV, cnt);
            } else {
                // chunk = whole flag words (32 flag groups of kSub points each), except the last word of an item
                const int ngr = npts / kSub;
                const int gfirst = cur.g0 + done / kSub;
                for (int wq = 0; wq * 32 < ngr; ++wq) {
                    const int ng = min(32, ngr - wq * 32);
                    unsigned flag[kHypPerThread];
#pragma unroll
                    for (int k = 0; k < kHypPerThread; ++k) flag[k] = 0u;
                    const float4* wp = sp + wq * 32 * (kSub / 2) * kV;
                    for (int g = 0; g < ng; ++g) {
                        float ma[kHypPerThread];
#pragma unroll
                        for (int k = 0; k < kHypPerThread; ++k) ma[k] = INFINITY;
                        const float4* gp = wp + g * (kSub / 2) * kV;
#pragma unroll kPairUnroll
                        for (int j = 0; j < kSub / 2; ++j) Pol::template evalN<kHypPerThread>(Hy, gp + j * kV, cnt, ma);
                        const unsigned bit = 1u << g;             // uniform: the shift stays in the uniform datapath
#pragma unroll
                        for (int k = 0; k < kHypPerThread; ++k)   // (NaN: no flag) FSETP + predicated LOP3; plain C++ compiles to FSETP + SEL + SHF + LOP3
                            asm("{\n.reg .pred p;\nsetp.le.f32 p, %1, %2;\n@p or.b32 %0, %0, %3;\n}"
                                : "+r"(flag[k]) : "f"(ma[k]), "f"(G[k]), "r"(bit));
                    }
#pragma unroll
                    for (int k = 0; k < kHypPerThread; ++k)
                        flag_append(flist, hid[k] < cur.H_end ? flag[k] : 0u, hid[k], gfirst + wq * 32);
                }
            }
            __syncthreads();          // everyone is done with this stage before it is refilled
            stage ^= 1;
        }
#pragma unroll
        for (int k = 0; k < kHypPerThread; ++k)
            if (hid[k] < cur.H_end && cnt[k]) atomicAdd(&counts[hid[k]], (int)cnt[k]);
        if (!has_next) break;
        item = next_item;
        cur = nxt;
        cur_src = nxt_src;
    }
}

// FP64 fix-up.  Two levels of warp compaction keep all 32 lanes busy although only ~1 in 8 evaluations of a flagged group
// is inside the band:
//   level 1  one lane per record of the flag list: re-evaluate the group's kSub correspondences in FP32 (bit-identical
//            op sequence) -> band mask + FP32 decisions;
//   level 2  queue the band evaluations; one lane per evaluation applies the reference formula in FP64 and corrects
//            counts[h] by (exact decision - FP32 decision).
// Hypotheses marked in flist.ovf (list overflow) are recounted in FP64 first, over the correspondences of the pair's scored
// window [g_base, g_end) (the whole pair in a full sweep): counts[h] then holds the exact count over that window.
// stats: [0] flagged groups, [1] band evaluations, [2] changed decisions, [3] hypotheses recounted after a list overflow.
//   Fix::pair_of(params, h)                                       pair / view of a global hypothesis index
//   Fix::n_points(params, aux)                                    voting correspondences of that pair / view
//   Fix::scan(params, h, group, aux, band, sign)                  FP32 pass over one group (bit k = correspondence k)
//   Fix::exact(params, h, i, aux)                                 FP64 decision for correspondence i of the pair/view
template <class Fix>
__global__ void __launch_bounds__(256) fixup_list(typename Fix::Params prm, FlagList flist, int Htot,
                                                   int* __restrict__ counts, unsigned long long* __restrict__ stats) {
    __shared__ int4 queue2[8][64];
    __shared__ int s_red[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int4* q2 = queue2[warp];
    int q2n = 0;
    unsigned long long n_groups = 0, n_band = 0, n_flip = 0;
    const unsigned lt = (1u << lane) - 1u;
    const unsigned full = 0xffffffffu;
    const unsigned n_rec_raw = *flist.n;
    const unsigned n_rec = n_rec_raw < flist.cap ? n_rec_raw : flist.cap;

    if (n_rec_raw > flist.cap) {                       // rare: some hypotheses lost records -> exact recount (block per hypothesis)
        for (int h = blockIdx.x; h < Htot; h += gridDim.x) {
            if (!flist.ovf[h]) continue;               // uniform per block
            const int aux = Fix::pair_of(prm, h);
            const int n = Fix::n_points(prm, aux);
            const int i1 = min(n, prm.pi[aux].g_end * kSub);
            int c = 0;
            for (int i = min(n, prm.pi[aux].g_base * kSub) + (int)threadIdx.x; i < i1; i += blockDim.x) c += Fix::exact(prm, h, i, aux);
            c = __reduce_add_sync(full, c);
            __syncthreads();
            if (lane == 0) s_red[warp] = c;
            __syncthreads();
            if (threadIdx.x == 0) {
                int t = 0;
                for (int w = 0; w < 8; ++w) t += s_red[w];
                counts[h] = t;
                atomicAdd(&stats[3], 1ull);
            }
        }
    }

    auto drain2 = [&](int n) {                      // lanes < n: one band evaluation each, FP64
        if (lane < n) {
            const int4 e = q2[lane];
            RG_ASSERT(e.y >= 0 && e.y < Fix::n_points(prm, e.z) && (e.w == 0 || e.w == 1));
            const int d = Fix::exact(prm, e.x, e.y, e.z) - e.w;
            if (d) { atomicAdd(&counts[e.x], d); n_flip += 1; }
            n_band += 1;
        }
        __syncwarp();
    };
    auto push2 = [&](bool has, int4 rec) {          // warp-collective append to the level-2 queue
        const unsigned m = __ballot_sync(full, has);
        if (has) q2[q2n + __popc(m & lt)] = rec;
        q2n += __popc(m);
        __syncwarp();
        if (q2n >= 32) {
            drain2(32);
            const int rest = q2n - 32;
            int4 mv = make_int4(0, 0, 0, 0);
            if (lane < rest) mv = q2[32 + lane];
            __syncwarp();
            if (lane < rest) q2[lane] = mv;
            __syncwarp();
            q2n = rest;
        }
    };

    const unsigned stride = gridDim.x * blockDim.x;
    for (unsigned base = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n_rec; base += stride) {
        const unsigned i = base + lane;
        unsigned band = 0u, sign = 0u;
        int2 r = make_int2(0, 0);
        int aux = 0;
        if (i < n_rec) {
            r = flist.rec[i];
            RG_ASSERT(r.x >= -1 && r.x < Htot && (r.x < 0 || r.y >= 0));
            if (r.x >= 0 && !flist.ovf[r.x]) {
                aux = Fix::pair_of(prm, r.x);
                RG_ASSERT(r.y * kSub < Fix::n_points(prm, aux) + kSub);
                Fix::scan(prm, r.x, r.y, aux, band, sign);
                n_groups += 1;
            }
        }
        while (__any_sync(full, band != 0u)) {
            const bool has = band != 0u;
            int k = 0;
            if (has) { k = __ffs(band) - 1; band &= band - 1; }
            push2(has, make_int4(r.x, r.y * kSub + k, aux, (int)((sign >> k) & 1u)));
        }
    }
    drain2(q2n);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n_groups += __shfl_xor_sync(full, n_groups, o);
        n_band += __shfl_xor_sync(full, n_band, o);
        n_flip += __shfl_xor_sync(full, n_flip, o);
    }
    // one set of atomics per BLOCK (the three statistics words are shared by the whole grid)
    __shared__ unsigned long long s_stat[3][8];
    if (lane == 0) { s_stat[0][warp] = n_groups; s_stat[1][warp] = n_band; s_stat[2][warp] = n_flip; }
    __syncthreads();
    if (threadIdx.x < 3) {
        unsigned long long t = 0;
        for (int w = 0; w < 8; ++w) t += s_stat[threadIdx.x][w];
        if (t) atomicAdd(&stats[threadIdx.x], t);
    }
}

// best[p] = {index inside the pair of the first hypothesis with the largest count (-1 if that count is 0), count}
// flags / stats (optional): hypotheses whose flag byte has bit 2 set (sample index out of range) are counted in stats[4]
// model / best_model / best_idx / best_count (optional): also publish the winner (its F or R|t, model_len doubles per
// hypothesis) — saves the separate finish kernel when no inlier mask is wanted (hypothesis-split mode)
// keys (optional): the cross-GPU argmax key of the pair, (count << 32) | (0xFFFFFFFF - (hyp_first + index)), 0 when no
// hypothesis of this rank has an inlier — what rg_argmax_pack_dev computed with a separate launch in round 1
__global__ void __launch_bounds__(256) argmax_counts(const int* __restrict__ counts, const PairInfo* __restrict__ pi,
                                                      int2* __restrict__ best, const unsigned char* __restrict__ flags,
                                                      unsigned long long* __restrict__ stats,
                                                      unsigned long long* __restrict__ keys,
                                                      const double* __restrict__ model = nullptr, int model_len = 0,
                                                      double* __restrict__ best_model = nullptr,
                                                      int* __restrict__ best_idx = nullptr, int* __restrict__ best_count = nullptr) {
    __shared__ unsigned long long sk[8];
    __shared__ int s_win;
    const int p = blockIdx.x;
    const PairInfo info = pi[p];
    unsigned long long key = 0ull;
    unsigned bad = 0u;
    // four independent loads in flight per thread: with one pair per call (hypothesis-split mode) this single block is on
    // the critical path and was a chain of dependent L2 round trips
    for (int h0 = threadIdx.x; h0 < info.H; h0 += 4 * blockDim.x) {
        int cv[4];
        unsigned fv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int h = h0 + u * blockDim.x;
            cv[u] = h < info.H ? counts[info.hyp_off + h] : 0;
            fv[u] = (flags != nullptr && h < info.H) ? flags[info.hyp_off + h] : 0u;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int h = h0 + u * blockDim.x;
            if (h < info.H) {
                const unsigned long long k =
                    ((unsigned long long)(unsigned)cv[u] << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)h);
                key = k > key ? k : key;
                bad += (fv[u] >> 2) & 1u;
            }
        }
    }
    if (stats != nullptr && bad) atomicAdd(&stats[4], (unsigned long long)bad);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
        key = other > key ? other : key;
    }
    if ((threadIdx.x & 31) == 0) sk[threadIdx.x >> 5] = key;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) key = sk[w] > key ? sk[w] : key;
        const int cnt = (int)(key >> 32);
        const int idx = cnt > 0 ? (int)(0xFFFFFFFFu - (unsigned)(key & 0xFFFFFFFFull)) : -1;
        best[p] = make_int2(idx, cnt);
        if (keys != nullptr)
            keys[p] = idx >= 0 ? (((unsigned long long)(unsigned)cnt << 32) |
                                  (unsigned long long)(0xFFFFFFFFu - (unsigned)(info.hyp_first + idx)))
                               : 0ull;
        if (best_idx != nullptr) { best_idx[p] = idx; best_count[p] = cnt; }
        s_win = idx;
    }
    if (best_model != nullptr) {
        __syncthreads();
        const int w = s_win;
        if ((int)threadIdx.x < model_len)
            best_model[(size_t)p * model_len + threadIdx.x] =
                w >= 0 ? model[(size_t)(info.hyp_off + w) * model_len + threadIdx.x] : __longlong_as_double(0x7FF8000000000000ll);
    }
}

}  // namespace rg
