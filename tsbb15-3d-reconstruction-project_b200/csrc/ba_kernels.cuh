// Bundle adjustment on the device (SURVEY.md section 8f row N4, the multi-view half): the minimisation that
// tables.Tables.BundleAdjustment2 (tables.py:260-333) hands to SciPy's least_squares —
//   minimise  sum_o |u_o - c1.x / c3.x|^2 + |v_o - c2.x / c3.x|^2      (EpsilonBA, tables.py:266-296)
// over all 12 entries of every 3x4 camera matrix except the first view's (its Jacobian columns are cleared in
// sparsity_mask, tables.py:376) and all 3-D points.  The reference: trust-region reflective, finite-difference
// Jacobian through a Python loop over the observation table, ftol = 1e-4 (8 s for the 36-view Dino scene).
// Here: Levenberg-Marquardt with Marquardt scaling; the 3x3 point blocks are eliminated analytically (Schur
// complement), the reduced camera system (12 x free views, dense) is factorised by a blocked Cholesky that runs on one
// thread-block cluster; no host synchronisation between iterations, every reduction in a fixed order (bit-reproducible).
//
// Structure used (as in gs_kernels.cuh).  Per observation o = (view k, point j), y = C_k Xh, P2 = d proj / d y (2x3),
// Q = P2 C_k[:, :3] = d pred / d X, M = P2^T P2, T = P2^T Q:
//   J_c^T J_c = M (x) Xh Xh^T      J_c^T J_p = T (x) Xh      V_j = sum_o Q^T Q      g_j = sum_o Q^T r
// so the block (k, l) of the reduced system is   [k == l] sum_o M_o (x) XX  -  sum_{o in k, o' in l, same point}
// (T_o V_j'^-1 T_o'^T) (x) Xh Xh^T : a 3x3 matrix per pair of observations, expanded by the 4x4 outer product.
//
// Robust losses (the loss / f_scale of SciPy's least_squares): every scalar residual f contributes C^2 rho((f / C)^2) to
// twice the cost.  The linearisation is IRLS: the residual row and the Jacobian row of each component are weighted by
// w = rho'(z), i.e. every product above gets W = diag(w0, w1) between its two factors (M = P2^T W P2, T = P2^T W Q,
// V_j = sum Q^T W Q, g_j = sum Q^T W r); the gradient is exact, the normal matrix the weighted Gauss-Newton one.  M then
// has M11 != M00, and the linearisation record stores w0, w1 in place of the third entry of P2^T W r (rebuilt from the
// first two: -(u a0 + v a1)).  The loss is a template parameter; the linear instantiation is the unweighted code.
#pragma once
#include <cooperative_groups.h>
#include "gs_kernels.cuh"

namespace rg {

namespace cg = cooperative_groups;

constexpr int kBaPointThreads = 128;
constexpr int kBaPointLanes = 8;          // lanes that share one point in ba_points / ba_trial (one observation of the track each)
constexpr int kBaBlockThreads = 192;      // chunk of observations per pass; threads 0..143 own the 12x12 entries
constexpr int kBaRec = 17;                // doubles per staged observation: A (9) | X (3) | z (3) | M00, M22
constexpr int kBaRecW = 18;               // the same for a robust loss: A (9) | X (3) | z (3) | M00, M11, M22
constexpr int kBaSegChunks = 2;            // chunks of kBaBlockThreads observations per work item of ba_blocks
constexpr int kBaPart = 168;              // doubles per partial block: 144 entries | 12 rhs | 12 diagonal damping sums
constexpr int kBaLin = 16;                // doubles per observation written by ba_points: T (9) | iy^2, u, v | P2^T r (3) | pad
                                          // robust loss: T (9) | iy^2, u, v | (P2^T W r)[0..1] | w0, w1
constexpr int kBaSolveThreads = 512;
constexpr int kBaSolveFixed = 192;        // doubles at the start of ba_solve*'s dynamic shared memory: Ld (144) | Li (16) | scratch (32)
constexpr int kBaMaxFree = 170;           // free views: the 12 x (n + 1) Cholesky panel must fit in shared memory

struct BaState {                // one per problem, device resident
    double lambda, cost, cost_trial;
    int iters, done, accepted, have_cost;
    int n_bad, pad;             // observations skipped (non-finite projection) at the last linearisation
    double floor;               // cost at which the residuals are rounding noise of the observations: (64 eps)^2 sum |uv|^2 / 2
};

// one observation at (C, X): prediction, residual, the derivative factors
struct BaObs {
    double iy, u, v, r0, r1;
    double Q[2][3];
    bool ok;
};

__device__ __forceinline__ void ba_obs(const double* __restrict__ C, const double X0, const double X1, const double X2,
                                       const double mu, const double mv, BaObs& g) {
    double y[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) y[a] = C[4 * a] * X0 + C[4 * a + 1] * X1 + C[4 * a + 2] * X2 + C[4 * a + 3];
    g.iy = 1.0 / y[2];
    g.u = y[0] * g.iy;
    g.v = y[1] * g.iy;
    g.r0 = mu - g.u;
    g.r1 = mv - g.v;
    const double p02 = -g.u * g.iy, p12 = -g.v * g.iy;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        g.Q[0][c] = g.iy * C[c] + p02 * C[8 + c];
        g.Q[1][c] = g.iy * C[4 + c] + p12 * C[8 + c];
    }
    g.ok = isfinite(g.r0) && isfinite(g.r1) && isfinite(g.iy);
}

// C^2 (rho(z0) + rho(z1)) of one observation, with the weights; ic = 1 / C, c2 = C^2
template <int kLoss>
__device__ __forceinline__ double ba_robust(const BaObs& g, const double ic, const double c2, double& w0, double& w1) {
    const double s0 = g.r0 * ic, s1 = g.r1 * ic;
    double p0, p1;
    ba_rho<kLoss>(s0 * s0, p0, w0);
    ba_rho<kLoss>(s1 * s1, p1, w1);
    return c2 * (p0 + p1);
}

// T = P2^T Q with P2 = [[iy, 0, -u iy], [0, iy, -v iy]]
__device__ __forceinline__ void ba_T(const BaObs& g, double (&T)[3][3]) {
    const double p02 = -g.u * g.iy, p12 = -g.v * g.iy;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        T[0][c] = g.iy * g.Q[0][c];
        T[1][c] = g.iy * g.Q[1][c];
        T[2][c] = p02 * g.Q[0][c] + p12 * g.Q[1][c];
    }
}

// deterministic block sum (fixed shuffle tree, then warps in order); result valid in thread 0
__device__ __forceinline__ double ba_block_sum(double v, double* sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sh[w];
    __syncthreads();
    return s;
}

// ------------------------------------------------------------------------------------------------
// step 1 (kBaPointLanes lanes per point): commit an accepted trial, linearise the track, V_j, g_j, damped inverse,
// e_j = V'^-1 g_j, cost partials
// observations are stored sorted by point: the track of point j is [pt_off[j], pt_off[j+1])
// ------------------------------------------------------------------------------------------------
template <int kLoss>
__global__ void __launch_bounds__(kBaPointThreads) ba_points(BaState* __restrict__ st, const double* __restrict__ cams,
                                                             double* __restrict__ X, const double* __restrict__ Xtrial,
                                                             const double2* __restrict__ uv, const int* __restrict__ ocam,
                                                             const int* __restrict__ pt_off, int nP, double* __restrict__ pblk,
                                                             double* __restrict__ cost_part, int* __restrict__ bad_part,
                                                             double* __restrict__ obs2_part, double* __restrict__ lin,
                                                             double ic, double c2) {
    __shared__ double sh[kBaPointThreads / 32];
    if (st->done) return;
    const double lambda = st->lambda;
    const bool commit = st->accepted > 0;
    const bool first = st->have_cost == 0;                  // first linearisation: also sum |uv|^2 for the rounding floor
    double cost = 0.0, obs2 = 0.0;
    int bad = 0;
    // kBaPointLanes lanes per point: lane t of the group takes observations t, t + kBaPointLanes, ... of the track; the
    // 3x3 block and the gradient are reduced inside the group by a fixed xor-shuffle tree (reproducible)
    const int sub = threadIdx.x & (kBaPointLanes - 1);
    const int gpb = blockDim.x / kBaPointLanes;                               // groups per block
    const int npad = ((nP + gpb - 1) / gpb) * gpb;                            // whole warps stay together in the shuffles
    for (int j = blockIdx.x * gpb + threadIdx.x / kBaPointLanes; j < npad; j += gridDim.x * gpb) {
        const bool real = j < nP;
        double X0 = 0.0, X1 = 0.0, X2 = 1.0;
        if (real) {
            if (commit) {
                X0 = Xtrial[3 * (size_t)j]; X1 = Xtrial[3 * (size_t)j + 1]; X2 = Xtrial[3 * (size_t)j + 2];
                if (sub == 0) { X[3 * (size_t)j] = X0; X[3 * (size_t)j + 1] = X1; X[3 * (size_t)j + 2] = X2; }
            } else {
                X0 = X[3 * (size_t)j]; X1 = X[3 * (size_t)j + 1]; X2 = X[3 * (size_t)j + 2];
            }
        }
        double V[6] = {0, 0, 0, 0, 0, 0}, g[3] = {0, 0, 0};
        const int t0 = real ? pt_off[j] : 0, t1 = real ? pt_off[j + 1] : 0;
        for (int o = t0 + sub; o < t1; o += kBaPointLanes) {
            BaObs b;
            const double2 m = uv[o];
            ba_obs(cams + 12 * (size_t)ocam[o], X0, X1, X2, m.x, m.y, b);
            double4* lo = reinterpret_cast<double4*>(lin + kBaLin * (size_t)o);
            if (!b.ok) {                                                            // skipped everywhere: an all-zero record
                ++bad;
                const double4 z4 = make_double4(0.0, 0.0, 0.0, 0.0);
                lo[0] = z4; lo[1] = z4; lo[2] = z4; lo[3] = z4;
                continue;
            }
            if constexpr (kLoss != LOSS_LINEAR) {
                double w0, w1;
                cost += ba_robust<kLoss>(b, ic, c2, w0, w1);
                const double a0 = w0 * b.r0, a1 = w1 * b.r1;               // W r
                double T[3][3];
                ba_T(b, T);
#pragma unroll
                for (int c = 0; c < 3; ++c) {                               // P2^T W Q = P2^T W P2 C[:, :3]
                    T[0][c] *= w0;
                    T[1][c] *= w1;
                    T[2][c] = -(b.u * T[0][c] + b.v * T[1][c]);
                }
                lo[0] = make_double4(T[0][0], T[0][1], T[0][2], T[1][0]);
                lo[1] = make_double4(T[1][1], T[1][2], T[2][0], T[2][1]);
                lo[2] = make_double4(T[2][2], b.iy * b.iy, b.u, b.v);
                lo[3] = make_double4(b.iy * a0, b.iy * a1, w0, w1);
#pragma unroll
                for (int a = 0; a < 3; ++a) {
#pragma unroll
                    for (int c = a; c < 3; ++c) V[sym3(a, c)] += w0 * b.Q[0][a] * b.Q[0][c] + w1 * b.Q[1][a] * b.Q[1][c];
                    g[a] += b.Q[0][a] * a0 + b.Q[1][a] * a1;
                }
                obs2 += m.x * m.x + m.y * m.y;
                continue;
            }
            {
                double T[3][3];
                ba_T(b, T);
                lo[0] = make_double4(T[0][0], T[0][1], T[0][2], T[1][0]);
                lo[1] = make_double4(T[1][1], T[1][2], T[2][0], T[2][1]);
                lo[2] = make_double4(T[2][2], b.iy * b.iy, b.u, b.v);
                lo[3] = make_double4(b.iy * b.r0, b.iy * b.r1, -(b.u * b.r0 + b.v * b.r1) * b.iy, 0.0);   // P2^T r
            }
#pragma unroll
            for (int a = 0; a < 3; ++a) {
#pragma unroll
                for (int c = a; c < 3; ++c) V[sym3(a, c)] += b.Q[0][a] * b.Q[0][c] + b.Q[1][a] * b.Q[1][c];
                g[a] += b.Q[0][a] * b.r0 + b.Q[1][a] * b.r1;
            }
            cost += b.r0 * b.r0 + b.r1 * b.r1;
            obs2 += m.x * m.x + m.y * m.y;
        }
#pragma unroll
        for (int o = kBaPointLanes / 2; o > 0; o >>= 1) {
#pragma unroll
            for (int k = 0; k < 6; ++k) V[k] += __shfl_xor_sync(0xffffffffu, V[k], o);
#pragma unroll
            for (int k = 0; k < 3; ++k) g[k] += __shfl_xor_sync(0xffffffffu, g[k], o);
        }
        if (real && sub == 0) {
            V[0] += lambda * V[0]; V[3] += lambda * V[3]; V[5] += lambda * V[5];        // Marquardt scaling
            double Vi[6];
            if (!inv_sym3(V, Vi)) {
#pragma unroll
                for (int k = 0; k < 6; ++k) Vi[k] = 0.0;                              // unobserved / degenerate point: not moved
            }
            double* pb = pblk + 12 * (size_t)j;
#pragma unroll
            for (int k = 0; k < 6; ++k) pb[k] = Vi[k];
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                pb[6 + a] = Vi[sym3(a, 0)] * g[0] + Vi[sym3(a, 1)] * g[1] + Vi[sym3(a, 2)] * g[2];
                pb[9 + a] = g[a];
            }
        }
    }
    const double s = ba_block_sum(cost, sh);
    if (first) {
        const double s2 = ba_block_sum(obs2, sh);
        if (threadIdx.x == 0) obs2_part[blockIdx.x] = s2;
    }
    for (int o = 16; o > 0; o >>= 1) bad += __shfl_xor_sync(0xffffffffu, bad, o);
    if (threadIdx.x == 0) { cost_part[blockIdx.x] = s; bad_part[blockIdx.x] = 0; }
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && bad) atomicAdd(&bad_part[blockIdx.x], bad);          // integer: order does not matter
}

// ------------------------------------------------------------------------------------------------
// step 2 (CTA per 12x12 block (kf, lf <= kf) of the reduced camera system that has at least one common point; the list
// of such blocks comes from the host, the others stay zero): observations of view k in chunks; each thread takes one
// observation's linearisation (written by ba_points), looks through the point's track for observations in view l,
// stages A = [k == l] M - T V'^-1 T'^T and Xh in shared memory (ordered ballot compaction); then thread (r, c) adds
// A[a][a2] Xh[b] Xh[b2] over the chunk.  Row n of the matrix (leading dimension n + 1) receives the right-hand side,
// so that the factorisation performs the forward substitution as it goes.  kW: the record of a robust loss (weights w0, w1).
// ------------------------------------------------------------------------------------------------
template <bool kW>
__global__ void __launch_bounds__(kBaBlockThreads, 3) ba_blocks(const BaState* __restrict__ st, const int4* __restrict__ items,
                                                                double* __restrict__ part,
                                                                const double* __restrict__ X, const double* __restrict__ lin,
                                                                const int* __restrict__ ocam, const int* __restrict__ opt,
                                                                const int* __restrict__ pt_off, const int* __restrict__ cam_off,
                                                                const int* __restrict__ cam_obs, const double* __restrict__ pblk,
                                                                int n_fixed, int nF, double* __restrict__ S) {
    if (st->done) return;
    const int4 item = items[blockIdx.x];                    // (kf, lf, segment, segments of this block)
    const int kf = item.x, lf = item.y;
    constexpr int kRec = kW ? kBaRecW : kBaRec;
    __shared__ double rec[kBaBlockThreads * kRec];
    __shared__ int wcount[kBaBlockThreads / 32 + 1];
    const int k = n_fixed + kf, l = n_fixed + lf;
    const bool diag = kf == lf;
    const double lambda = st->lambda;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int er = tid / 12, ec = tid % 12;                 // entry of the block owned by threads 0..143
    const int ea = er >> 2, eb = er & 3, ea2 = ec >> 2, eb2 = ec & 3;
    const int rz = tid - 144;                               // threads 144..155: right-hand side entry (a, b) = (rz/4, rz%4)
    double acc = 0.0, accd = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
    const int lo = cam_off[k] + item.z * (kBaSegChunks * kBaBlockThreads);
    const int hi = min(cam_off[k + 1], lo + kBaSegChunks * kBaBlockThreads);
    for (int base = lo; base < hi; base += kBaBlockThreads) {
        const int oi = base + tid;
        bool valid = false;
        double A[9], Xh[3], z[3], m00 = 0.0, m11 = 0.0, m22 = 0.0;
        if (oi < hi) {
            const int o = cam_obs[oi], j = opt[o];
            const int t0 = pt_off[j], t1 = pt_off[j + 1];
            const double4* L = reinterpret_cast<const double4*>(lin + kBaLin * (size_t)o);
            const double4 l0 = L[0], l1 = L[1], l2 = L[2];
            const double T[3][3] = {{l0.x, l0.y, l0.z}, {l0.w, l1.x, l1.y}, {l1.z, l1.w, l2.x}};
            const double* pb = pblk + 12 * (size_t)j;
            double Vi[6], TV[3][3];
#pragma unroll
            for (int q = 0; q < 6; ++q) Vi[q] = pb[q];
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    TV[a][c] = T[a][0] * Vi[sym3(0, c)] + T[a][1] * Vi[sym3(1, c)] + T[a][2] * Vi[sym3(2, c)];
#pragma unroll
            for (int q = 0; q < 9; ++q) A[q] = 0.0;
            if (diag) {
                const double i2 = l2.y, u = l2.z, v = l2.w;
                const double4 l3 = L[3];
                double pr2 = l3.z;                                      // (P2^T W r)[2]
                if constexpr (kW) {                                     // M = P2^T W P2
                    m00 = l3.z * i2; m11 = l3.w * i2; m22 = (l3.z * u * u + l3.w * v * v) * i2;
                    A[0] = m00; A[4] = m11; A[8] = m22;
                    A[2] = A[6] = -u * m00;
                    A[5] = A[7] = -v * m11;
                    pr2 = -(u * l3.x + v * l3.y);
                } else {
                    m00 = i2; m22 = (u * u + v * v) * i2;
                    A[0] = i2; A[4] = i2; A[8] = m22;
                    A[2] = A[6] = -u * i2;
                    A[5] = A[7] = -v * i2;
                }
                const double e0 = pb[6], e1 = pb[7], e2 = pb[8];        // z = P2^T r - T e_j
                z[0] = l3.x - (T[0][0] * e0 + T[0][1] * e1 + T[0][2] * e2);
                z[1] = l3.y - (T[1][0] * e0 + T[1][1] * e1 + T[1][2] * e2);
                z[2] = pr2 - (T[2][0] * e0 + T[2][1] * e1 + T[2][2] * e2);
                valid = true;
            }
            for (int o2 = t0; o2 < t1; ++o2) {
                if (ocam[o2] != l) continue;
                const double4* L2 = reinterpret_cast<const double4*>(lin + kBaLin * (size_t)o2);
                const double4 p0 = L2[0], p1 = L2[1], p2 = L2[2];
                const double T2[3][3] = {{p0.x, p0.y, p0.z}, {p0.w, p1.x, p1.y}, {p1.z, p1.w, p2.x}};
#pragma unroll
                for (int a = 0; a < 3; ++a)
#pragma unroll
                    for (int a2 = 0; a2 < 3; ++a2)
                        A[a * 3 + a2] -= TV[a][0] * T2[a2][0] + TV[a][1] * T2[a2][1] + TV[a][2] * T2[a2][2];
                valid = true;
            }
            if (valid) { Xh[0] = X[3 * (size_t)j]; Xh[1] = X[3 * (size_t)j + 1]; Xh[2] = X[3 * (size_t)j + 2]; }
        }
        // ordered compaction of the valid observations of this chunk
        const unsigned bal = __ballot_sync(0xffffffffu, valid);
        if (lane == 0) wcount[warp] = __popc(bal);
        __syncthreads();
        int slot = __popc(bal & ((1u << lane) - 1u)), total = 0;
        for (int w = 0; w < kBaBlockThreads / 32; ++w) {
            if (w < warp) slot += wcount[w];
            total += wcount[w];
        }
        if (valid) {
            double* r = rec + slot * kRec;
#pragma unroll
            for (int q = 0; q < 9; ++q) r[q] = A[q];
            r[9] = Xh[0]; r[10] = Xh[1]; r[11] = Xh[2];
            if (diag) {
                r[12] = z[0]; r[13] = z[1]; r[14] = z[2]; r[15] = m00;
                if constexpr (kW) { r[16] = m11; r[17] = m22; }
                else r[16] = m22;
            }
        }
        __syncthreads();
        if (tid < 144) {
            const bool dd = diag && er == ec;
            const int ia = ea * 3 + ea2, ib = eb < 3 ? 9 + eb : -1, ib2 = eb2 < 3 ? 9 + eb2 : -1;
            int i = 0;
            for (; i + 4 <= total; i += 4) {                 // four independent chains (fixed order: still reproducible)
                const double* r = rec + i * kRec;
                const double xa0 = ib >= 0 ? r[ib] : 1.0, xa1 = ib >= 0 ? r[kRec + ib] : 1.0;
                const double xa2 = ib >= 0 ? r[2 * kRec + ib] : 1.0, xa3 = ib >= 0 ? r[3 * kRec + ib] : 1.0;
                const double xc0 = ib2 >= 0 ? r[ib2] : 1.0, xc1 = ib2 >= 0 ? r[kRec + ib2] : 1.0;
                const double xc2 = ib2 >= 0 ? r[2 * kRec + ib2] : 1.0, xc3 = ib2 >= 0 ? r[3 * kRec + ib2] : 1.0;
                acc = fma(r[ia] * xa0, xc0, acc);
                acc1 = fma(r[kRec + ia] * xa1, xc1, acc1);
                acc2 = fma(r[2 * kRec + ia] * xa2, xc2, acc2);
                acc3 = fma(r[3 * kRec + ia] * xa3, xc3, acc3);
                if (dd) {
                    const int im = kW ? 15 + ea : (ea < 2 ? 15 : 16);     // M_aa of the diagonal damping sum
                    accd = fma(r[im] * xa0, xa0, accd);
                    accd = fma(r[kRec + im] * xa1, xa1, accd);
                    accd = fma(r[2 * kRec + im] * xa2, xa2, accd);
                    accd = fma(r[3 * kRec + im] * xa3, xa3, accd);
                }
            }
            for (; i < total; ++i) {
                const double* r = rec + i * kRec;
                const double xb = ib >= 0 ? r[ib] : 1.0, xb2 = ib2 >= 0 ? r[ib2] : 1.0;
                acc = fma(r[ia] * xb, xb2, acc);
                if (dd) accd = fma((kW ? r[15 + ea] : (ea < 2 ? r[15] : r[16])) * xb, xb, accd);
            }
        } else if (diag && rz < 12) {
            const int za = rz >> 2, zb = rz & 3;
            for (int i = 0; i < total; ++i) {
                const double* r = rec + i * kRec;
                acc = fma(r[12 + za], zb < 3 ? r[9 + zb] : 1.0, acc);
            }
        }
        __syncthreads();
    }
    acc = (acc + acc1) + (acc2 + acc3);
    if (item.w > 1) {                                       // the block is split over several work items: partial sums
        double* p = part + (size_t)blockIdx.x * kBaPart;
        if (tid < 144) {
            p[tid] = acc;
            if (diag && er == ec) p[156 + er] = accd;
        } else if (rz < 12) {
            p[144 + rz] = diag ? acc : 0.0;
        }
        return;
    }
    const size_t ld = (size_t)12 * nF + 1;
    if (tid < 144) {
        // Marquardt damping; a parameter without any information (a view without observations) gets a unit diagonal:
        // its row and right-hand side are zero, so it simply does not move instead of making the system singular
        if (diag && er == ec) acc += accd > 0.0 ? lambda * accd : 1.0;
        S[(size_t)(12 * kf + er) + (size_t)(12 * lf + ec) * ld] = acc;
    } else if (diag && rz < 12) {
        S[(size_t)12 * nF + (size_t)(12 * kf + rz) * ld] = acc;
    }
}

// blocks that were split over several work items: sum the partials in segment order (reproducible), write the block
__global__ void __launch_bounds__(kBaBlockThreads) ba_blocks_reduce(const BaState* __restrict__ st, const int4* __restrict__ items,
                                                                    const int* __restrict__ first_item, int n_blocks,
                                                                    const double* __restrict__ part, int nF,
                                                                    double* __restrict__ S) {
    if (st->done) return;
    const int f = first_item[blockIdx.x];
    const int4 item = items[f];
    if (item.w <= 1) return;                                // written directly by ba_blocks
    const int kf = item.x, lf = item.y, tid = threadIdx.x;
    const bool diag = kf == lf;
    const size_t ld = (size_t)12 * nF + 1;
    if (tid < 144) {
        const int er = tid / 12, ec = tid % 12;
        double a = 0.0, d = 0.0;
        for (int s = 0; s < item.w; ++s) {
            a += part[(size_t)(f + s) * kBaPart + tid];
            if (diag && er == ec) d += part[(size_t)(f + s) * kBaPart + 156 + er];
        }
        if (diag && er == ec) a += d > 0.0 ? st->lambda * d : 1.0;      // see ba_blocks
        S[(size_t)(12 * kf + er) + (size_t)(12 * lf + ec) * ld] = a;
    } else if (diag && tid < 156) {
        double a = 0.0;
        for (int s = 0; s < item.w; ++s) a += part[(size_t)(f + s) * kBaPart + tid];
        S[(size_t)12 * nF + (size_t)(12 * kf + (tid - 144)) * ld] = a;
    }
}

// one panel row: x L_kk^T = a  (forward substitution with the reciprocal diagonal)
__device__ __forceinline__ void ba_panel_row(double (&x)[12], const double* Ld, const double* Li) {
#pragma unroll
    for (int c = 0; c < 12; ++c) {
        double a = x[c];
#pragma unroll
        for (int m = 0; m < c; ++m) a = fma(-x[m], Ld[c * 12 + m], a);
        x[c] = a * Li[c];
    }
}

// backward substitution of one 12-block by one thread: x_blk = L_kk^-T (y_blk - tv); L(c, m) = Lb[m * ldb + c], c >= m
__device__ __forceinline__ void ba_back12(double* yb, const double* tv, const double* Lb, const int ldb, const double* Li) {
    double v[12];
#pragma unroll
    for (int c = 0; c < 12; ++c) v[c] = yb[c] - tv[c];
#pragma unroll
    for (int c = 11; c >= 0; --c) {
        v[c] *= Li[c];
#pragma unroll
        for (int m = 0; m < c; ++m) v[m] = fma(-Lb[m * ldb + c], v[c], v[m]);
    }
#pragma unroll
    for (int c = 0; c < 12; ++c) yb[c] = v[c];
}

// ------------------------------------------------------------------------------------------------
// step 3, L2 variant (any size up to kBaMaxFree free views; one thread-block cluster): right-looking blocked Cholesky
// of the (n + 1) x n lower-trapezoidal array [S; rhs^T] (column-major, leading dimension n + 1) in global memory, panel
// width 12 = one view.  Every CTA factorises the 12x12 diagonal block and solves the whole panel redundantly into its
// own shared memory, the trailing update is split over the warps of all CTAs by column; one cluster barrier per panel.
// Row n comes out as y = L^-1 rhs; CTA 0 finishes with the backward substitution L^T x = y and writes the camera step.
// ------------------------------------------------------------------------------------------------
// (S and dinv carry data between the CTAs of the cluster across barriers: deliberately not __restrict__)
__global__ void __launch_bounds__(kBaSolveThreads) ba_solve(BaState* __restrict__ st, double* S, double* dinv, int n_fixed, int nF,
                                                            double* __restrict__ dC) {
    cg::cluster_group cluster = cg::this_cluster();
    if (st->done) return;                                   // uniform over the cluster
    extern __shared__ double sm[];
    __shared__ int fail;
    const int n = 12 * nF, ld = n + 1, rows = n + 1;
    double* Ld = sm;                                        // 12 x 12 factor of the diagonal block (row-major)
    double* Li = sm + 144;                                  // reciprocal diagonal of the block / backward partial sums
    double* cb = sm + 160;                                  // scratch of the block factorisation
    double* Pn = sm + kBaSolveFixed;                        // panel: Pn[c * rows + i]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
    const int rank = (int)cluster.block_rank(), nr = (int)cluster.num_blocks();
    if (tid == 0) fail = 0;
    __syncthreads();
    // Every CTA reads block column kb of S (diagonal block + panel) at the start of step kb, so the factor of that block
    // column may only be written back once ALL CTAs are past those reads: it is written at the start of step kb + 1
    // (after the cluster barrier), from the copies every CTA still holds in shared memory (Ld, Li, Pn).
    auto write_back = [&](const int kb) {
        const int j0 = 12 * kb;
        int pass = 0;
        for (int i = j0 + 12 + tid; i < rows; i += blockDim.x, ++pass)
            if (pass % nr == rank) {
#pragma unroll
                for (int c = 0; c < 12; ++c) __stcg(&S[(size_t)i + (size_t)(j0 + c) * ld], Pn[c * rows + i]);
            }
        if (rank == nr - 1 && tid < 144) {
            const int r = tid / 12, c = tid % 12;
            if (r >= c) __stcg(&S[(size_t)(j0 + r) + (size_t)(j0 + c) * ld], Ld[tid]);
            if (r == c) __stcg(&dinv[j0 + r], Li[r]);
        }
    };
    for (int kb = 0; kb < nF; ++kb) {
        const int j0 = 12 * kb;
        if (kb > 0) {
            write_back(kb - 1);
            __syncthreads();                                // Ld / Li / Pn are overwritten below
        }
        if (tid < 144) {
            const int r = tid / 12, c = tid % 12;
            Ld[tid] = r >= c ? __ldcg(&S[(size_t)(j0 + r) + (size_t)(j0 + c) * ld]) : 0.0;
        }
        __syncthreads();
        if (warp == 0 && !ba_chol12(Ld, Li, cb, lane) && lane == 0) fail = 1;
        __syncthreads();
        if (fail) break;                                    // identical arithmetic in every CTA: uniform decision
        for (int i = j0 + 12 + tid; i < rows; i += blockDim.x) {
            double x[12];
#pragma unroll
            for (int c = 0; c < 12; ++c) x[c] = __ldcg(&S[(size_t)i + (size_t)(j0 + c) * ld]);
            ba_panel_row(x, Ld, Li);
#pragma unroll
            for (int c = 0; c < 12; ++c) Pn[c * rows + i] = x[c];
        }
        __syncthreads();
        const int ncol = n - j0 - 12;
        for (int jj = warp * nr + rank; jj < ncol; jj += nwarp * nr) {
            const int j = j0 + 12 + jj;
            double pj[12];
#pragma unroll
            for (int c = 0; c < 12; ++c) pj[c] = Pn[c * rows + j];
            for (int i = j + lane; i < rows; i += 32) {
                double* p = &S[(size_t)i + (size_t)j * ld];
                double s = __ldcg(p);
#pragma unroll
                for (int c = 0; c < 12; ++c) s = fma(-Pn[c * rows + i], pj[c], s);
                __stcg(p, s);
            }
        }
        cluster.sync();
    }
    if (!fail && nF > 0) write_back(nF - 1);
    cluster.sync();                                         // the factor is complete in global memory
    const bool bad = fail != 0;
    if (rank != 0) return;
    // backward substitution  L^T x = y,  y = row n of the factor
    double* y = Pn;                                         // reuse: n values
    double* tv = cb;
    __syncthreads();
    if (!bad) {
        for (int i = tid; i < n; i += blockDim.x) y[i] = __ldcg(&S[(size_t)n + (size_t)i * ld]);
        __syncthreads();
        for (int kb = nF - 1; kb >= 0; --kb) {
            const int j0 = 12 * kb;
            if (tid < 144) {
                const int r = tid / 12, c = tid % 12;
                Ld[c * 12 + r] = r >= c ? __ldcg(&S[(size_t)(j0 + r) + (size_t)(j0 + c) * ld]) : 0.0;   // column-major here
                if (r == c) Li[r] = __ldcg(&dinv[j0 + r]);
            }
            if (warp < 12) {
                const int j = j0 + warp;
                double s = 0.0;
                for (int i = j0 + 12 + lane; i < n; i += 32) s = fma(__ldcg(&S[(size_t)i + (size_t)j * ld]), y[i], s);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                if (lane == 0) tv[warp] = s;
            }
            __syncthreads();
            if (tid == 0) ba_back12(y + j0, tv, Ld, 12, Li);
            __syncthreads();
        }
    }
    __shared__ int okflag;
    if (tid == 0) okflag = 1;
    __syncthreads();
    if (!bad)
        for (int i = tid; i < n; i += blockDim.x)
            if (!isfinite(y[i])) okflag = 0;
    __syncthreads();
    const bool ok = !bad && okflag;
    for (int i = tid; i < n; i += blockDim.x) dC[(size_t)12 * n_fixed + i] = ok ? y[i] : 0.0;
    if (tid == 0) st->accepted = ok ? 1 : -1;               // -1: no step could be computed -> ba_accept raises lambda
}

// ------------------------------------------------------------------------------------------------
// step 3, cluster-resident variant (used when the matrix fits): the same factorisation with the matrix held in the
// SHARED MEMORY OF THE CLUSTER.  Block column kb (12 columns, rows 12 kb .. n) lives in the shared memory of CTA
// kb % nr and never leaves it.  Per panel: the owner factorises its diagonal block (one warp, registers), solves its
// panel in place and publishes the solved panel (<= 39 KB) through a double-buffered global array (L2; pushing it with
// st.shared::cluster was measured no faster than the L2 variant: DSMEM moves ~20 B/clk per SM); one cluster barrier;
// every CTA copies the panel into its shared memory and updates the block columns it owns there, 4 x 6 elements per
// thread in registers (the update is shared-memory-bandwidth bound otherwise: 2 loads per FMA).  Look-ahead: the owner of
// the NEXT block column updates that column first, factorises it, publishes its panel and arrives at the barrier before
// it updates the rest of its columns (barrier.cluster.arrive / .wait split).  The backward
// substitution walks the owners in reverse: dot products with the local block column, 12x12 back-solve by one thread,
// the 12 new unknowns pushed to every CTA's copy of x through distributed shared memory, one barrier per block.
// Same operations in the same order as ba_solve: bit-identical results.
// Shared memory per CTA: kBaSolveFixed + npad + 12 ceil(nF / nr) + 12 (n + 1) + own block columns  doubles
// (156 KB for 35 free views on 8 CTAs).
// ------------------------------------------------------------------------------------------------
#ifdef RG_BA_PROF
__device__ long long g_ba_prof[16];
#define BA_T(k) do { if (tid == 0 && rank == 0) { long long _t = clock64(); atomicAdd((unsigned long long*)&g_ba_prof[k], (unsigned long long)(_t - t_prev)); t_prev = _t; } } while (0)
#else
#define BA_T(k) do { } while (0)
#endif

__host__ __device__ inline size_t ba_dsmem_own_elems(int nF, int nr, int rank) {
    size_t e = 0;
    for (int kb = rank; kb < nF; kb += nr) e += (size_t)12 * (size_t)(12 * nF + 1 - 12 * kb);
    return e;
}
__host__ __device__ inline size_t ba_dsmem_doubles(int nF, int nr) {
    const int n = 12 * nF, npad = (n + 1) & ~1;
    return kBaSolveFixed + (size_t)npad + 12 * (size_t)((nF + nr - 1) / nr) + 12 * (size_t)(n + 1) +
           ba_dsmem_own_elems(nF, nr, 0);                                                       // rank 0 owns the most
}

// (Pg carries the published panels between the CTAs across barriers: deliberately not __restrict__)
__global__ void __launch_bounds__(kBaSolveThreads) ba_solve_dsmem(BaState* __restrict__ st, const double* __restrict__ S,
                                                                  double* Pg, int n_fixed, int nF,
                                                                  double* __restrict__ dC) {
    cg::cluster_group cluster = cg::this_cluster();
    if (st->done) return;                                   // uniform over the cluster
    extern __shared__ double sm[];
    __shared__ int fail;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int rank = (int)cluster.block_rank(), nr = (int)cluster.num_blocks();
    const int n = 12 * nF, ld = n + 1, rows = n + 1, npad = (n + 1) & ~1;
    double* Ld = sm;                                        // 12 x 12 factor of the diagonal block (row-major)
    double* Li = sm + 144;                                  // reciprocal diagonal of the block
    double* cb = sm + 160;                                  // scratch of the block factorisation / backward partial sums
    double* y = sm + kBaSolveFixed;                         // own entries: L^-1 rhs; then x, replicated in every CTA
    double* linv = y + npad;                                // reciprocal diagonals of the own blocks, 12 per block
    double* Pn = linv + 12 * ((nF + nr - 1) / nr);          // solved panel: Pn[c * rows + i]
    double* cols = Pn + 12 * rows;                          // own block columns, each (rows - 12 kb) x 12 column-major
    if (tid == 0) fail = 0;
#ifdef RG_BA_PROF
    long long t_prev = clock64();
#endif
    {
        size_t off = 0;
        for (int kb = rank; kb < nF; kb += nr) {
            const int j0 = 12 * kb, h = rows - j0;
            for (int e = tid; e < 12 * h; e += blockDim.x) {
                const int c = e / h, r = e - c * h;
                cols[off + e] = r >= c ? S[(size_t)(j0 + r) + (size_t)(j0 + c) * ld] : 0.0;
            }
            off += (size_t)12 * h;
        }
    }
    cluster.sync();                                         // every CTA of the cluster is running: remote accesses are legal
    BA_T(0);
    size_t own_off = 0;                                     // first own block column that is not factorised yet
    int own_kb = rank;

    // the owner's part of step kb: factorise the diagonal block, solve the panel in place, publish it through L2
    auto factor_and_publish = [&](const int kb) {
        const int j0 = 12 * kb, h = rows - j0;
        double* Pgb = Pg + (size_t)(kb & 1) * 12 * rows;
        double* B = cols + own_off;
        if (tid < 144) {
            const int r = tid / 12, c = tid % 12;
            Ld[tid] = r >= c ? B[c * h + r] : 0.0;
        }
        __syncthreads();
        if (warp == 0 && !ba_chol12(Ld, Li, cb, lane) && lane < nr) *cluster.map_shared_rank(&fail, lane) = 1;
        __syncthreads();
        if (!fail) {
            if (tid < 144) {
                const int r = tid / 12, c = tid % 12;
                if (r >= c) B[c * h + r] = Ld[tid];
                if (r == c) linv[12 * (kb / nr) + r] = Li[r];
            }
            for (int r = 12 + tid; r < h; r += blockDim.x) {
                double x[12];
#pragma unroll
                for (int c = 0; c < 12; ++c) x[c] = B[c * h + r];
                ba_panel_row(x, Ld, Li);
#pragma unroll
                for (int c = 0; c < 12; ++c) {
                    B[c * h + r] = x[c];
                    __stcg(&Pgb[c * rows + j0 + r], x[c]);
                }
                if (r == h - 1) {                           // the right-hand-side row: y = L^-1 rhs, final for these 12 entries
#pragma unroll
                    for (int c = 0; c < 12; ++c) y[j0 + c] = x[c];
                }
            }
        }
        own_off += (size_t)12 * h;
        own_kb += nr;
    };

    // trailing update of the own block columns kb_first, kb_first + nr, ... (at most n_cols of them) with the panel in Pn:
    // tiles of 4 rows x 6 columns, numbered across the block columns so that every warp has work
    auto update_columns = [&](const int kb_first, const size_t off_first, const int n_cols) {
        int total = 0, ncol = 0;
        for (int kb2 = kb_first; kb2 < nF && ncol < n_cols; kb2 += nr, ++ncol) total += 2 * ((rows - 12 * kb2 + 3) >> 2);
        for (int t0 = tid; t0 < total; t0 += blockDim.x) {
            int t = t0, kb2 = kb_first;
            size_t off2 = off_first;
            for (;;) {
                const int nt = 2 * ((rows - 12 * kb2 + 3) >> 2);
                if (t < nt) break;
                t -= nt;
                off2 += (size_t)12 * (rows - 12 * kb2);
                kb2 += nr;
            }
            const int j2 = 12 * kb2, h2 = rows - j2;
            double* B2 = cols + off2;
            const int ntr = (h2 + 3) >> 2;                  // row groups: thread rows tr, tr + ntr, tr + 2 ntr, tr + 3 ntr
            const int cgp = t >= ntr ? 1 : 0, tr = t - cgp * ntr, c0 = 6 * cgp;
            int rq[4];
            bool vq[4];
            double acc[4][6];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                rq[q] = tr + q * ntr;
                vq[q] = rq[q] < h2;
                if (!vq[q]) rq[q] = h2 - 1;
#pragma unroll
                for (int k = 0; k < 6; ++k) acc[q][k] = B2[(c0 + k) * h2 + rq[q]];
            }
#pragma unroll
            for (int c = 0; c < 12; ++c) {
                const double* Pc = Pn + c * rows + j2;
                double pi[4], pj[6];
#pragma unroll
                for (int q = 0; q < 4; ++q) pi[q] = Pc[rq[q]];
#pragma unroll
                for (int k = 0; k < 6; ++k) pj[k] = Pc[c0 + k];
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int k = 0; k < 6; ++k) acc[q][k] = fma(-pi[q], pj[k], acc[q][k]);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (vq[q]) {
#pragma unroll
                    for (int k = 0; k < 6; ++k) B2[(c0 + k) * h2 + rq[q]] = acc[q][k];
                }
        }
    };

    // Look-ahead: in step kb the owner of block column kb + 1 updates that column first, factorises it and publishes
    // panel kb + 1, ARRIVES at the cluster barrier and only then updates the rest of its columns; the other CTAs arrive
    // after their own update.  The pivot chain (copy, column update, factor, panel, barrier) no longer waits for anybody's
    // bulk update.
    if (rank == 0 && nF > 0) factor_and_publish(0);
    BA_T(1);
    cluster.sync();
    for (int kb = 0; kb < nF; ++kb) {
        if (fail) break;                                    // set by the owner before its arrive: uniform after the wait
        BA_T(3);
        const int j0 = 12 * kb;
        const double* Pgb = Pg + (size_t)(kb & 1) * 12 * rows;
        if (own_kb < nF) {                                  // something left to update in this CTA
            for (int i = j0 + 12 + tid; i < rows; i += blockDim.x) {        // 12 independent L2 loads per thread
                double v[12];
#pragma unroll
                for (int c = 0; c < 12; ++c) v[c] = __ldcg(&Pgb[c * rows + i]);
#pragma unroll
                for (int c = 0; c < 12; ++c) Pn[c * rows + i] = v[c];
            }
            __syncthreads();
        }
        BA_T(4);
        if (kb + 1 < nF && rank == (kb + 1) % nr) {         // own_kb == kb + 1
            update_columns(own_kb, own_off, 1);
            __syncthreads();
            factor_and_publish(kb + 1);
            BA_T(2);
            asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
            update_columns(own_kb, own_off, 1 << 30);
            __syncthreads();
            BA_T(5);
            asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
        } else {
            update_columns(own_kb, own_off, 1 << 30);
            __syncthreads();
            BA_T(5);
            asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
            asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
        }
    }
    const bool bad = fail != 0;
    // backward substitution L^T x = y: the owners in reverse order, x replicated through distributed shared memory
    if (!bad) {
        double* tv = cb;
        for (int kb = nF - 1; kb >= 0; --kb) {
            const int j0 = 12 * kb, h = rows - j0;
            if (rank == kb % nr) {
                own_off -= (size_t)12 * h;                  // own block columns are visited in reverse
                const double* B = cols + own_off;
                if (warp < 12) {
                    double s = 0.0;
                    for (int r = 12 + lane; r < h - 1; r += 32) s = fma(B[warp * h + r], y[j0 + r], s);
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                    if (lane == 0) tv[warp] = s;
                }
                __syncthreads();
                if (tid == 0) ba_back12(y + j0, tv, B, h, linv + 12 * (kb / nr));
                __syncthreads();
                if (tid < 12 * nr) {
                    const int d = tid / 12, c = tid - 12 * d;
                    if (d != rank) cluster.map_shared_rank(y, d)[j0 + c] = y[j0 + c];
                }
            }
            cluster.sync();
        }
    }
    BA_T(6);
    if (rank != 0) return;
    __shared__ int okflag;
    if (tid == 0) okflag = 1;
    __syncthreads();
    if (!bad)
        for (int i = tid; i < n; i += blockDim.x)
            if (!isfinite(y[i])) okflag = 0;
    __syncthreads();
    const bool ok = !bad && okflag;
    for (int i = tid; i < n; i += blockDim.x) dC[(size_t)12 * n_fixed + i] = ok ? y[i] : 0.0;
    if (tid == 0) st->accepted = ok ? 1 : -1;
}

// no free view (points only): nothing to solve
__global__ void ba_solve_none(BaState* __restrict__ st) {
    if (!st->done) st->accepted = 1;
}

// ------------------------------------------------------------------------------------------------
// step 4 (kBaPointLanes lanes per point): point steps by back-substitution, trial points, trial cost partials
// ------------------------------------------------------------------------------------------------
template <int kLoss>
__global__ void __launch_bounds__(kBaPointThreads) ba_trial(const BaState* __restrict__ st, const double* __restrict__ cams,
                                                            const double* __restrict__ dC, const double* __restrict__ X,
                                                            double* __restrict__ Xtrial, const double2* __restrict__ uv,
                                                            const int* __restrict__ ocam, const int* __restrict__ pt_off, int nP,
                                                            const double* __restrict__ pblk, const double* __restrict__ lin,
                                                            double* __restrict__ trial_part, double ic, double c2) {
    __shared__ double sh[kBaPointThreads / 32];
    if (st->done || st->accepted < 0) return;
    double cost = 0.0;
    const int sub = threadIdx.x & (kBaPointLanes - 1);
    const int gpb = blockDim.x / kBaPointLanes;
    const int npad = ((nP + gpb - 1) / gpb) * gpb;
    for (int j = blockIdx.x * gpb + threadIdx.x / kBaPointLanes; j < npad; j += gridDim.x * gpb) {
        const bool real = j < nP;
        const size_t jj = real ? (size_t)j : 0;
        const double X0 = X[3 * jj], X1 = X[3 * jj + 1], X2 = X[3 * jj + 2];
        const double* pb = pblk + 12 * jj;
        double back[3] = {0, 0, 0};
        const int lo = real ? pt_off[j] : 0, hi = real ? pt_off[j + 1] : 0;
        for (int o = lo + sub; o < hi; o += kBaPointLanes) {
            const double* d = dC + 12 * (size_t)ocam[o];
            double q[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) q[a] = d[4 * a] * X0 + d[4 * a + 1] * X1 + d[4 * a + 2] * X2 + d[4 * a + 3];
            if (q[0] == 0.0 && q[1] == 0.0 && q[2] == 0.0) continue;             // fixed view
            const double4* L = reinterpret_cast<const double4*>(lin + kBaLin * (size_t)o);   // T of ba_points (zero if skipped)
            const double4 l0 = L[0], l1 = L[1];
            const double t22 = L[2].x;
            back[0] += l0.x * q[0] + l0.w * q[1] + l1.z * q[2];
            back[1] += l0.y * q[0] + l1.x * q[1] + l1.w * q[2];
            back[2] += l0.z * q[0] + l1.y * q[1] + t22 * q[2];
        }
#pragma unroll
        for (int o = kBaPointLanes / 2; o > 0; o >>= 1) {
#pragma unroll
            for (int k = 0; k < 3; ++k) back[k] += __shfl_xor_sync(0xffffffffu, back[k], o);
        }
        const double r0 = pb[9] - back[0], r1 = pb[10] - back[1], r2 = pb[11] - back[2];
        const double n0 = X0 + pb[0] * r0 + pb[1] * r1 + pb[2] * r2;
        const double n1 = X1 + pb[1] * r0 + pb[3] * r1 + pb[4] * r2;
        const double n2 = X2 + pb[2] * r0 + pb[4] * r1 + pb[5] * r2;
        if (real && sub == 0) { Xtrial[3 * jj] = n0; Xtrial[3 * jj + 1] = n1; Xtrial[3 * jj + 2] = n2; }
        for (int o = lo + sub; o < hi; o += kBaPointLanes) {
            if (lin[kBaLin * (size_t)o + 9] == 0.0) continue;                  // skipped in the linearisation: skipped here
            const size_t k = (size_t)ocam[o];
            double Cn[12];
#pragma unroll
            for (int q = 0; q < 12; ++q) Cn[q] = cams[12 * k + q] + dC[12 * k + q];
            const double2 m = uv[o];
            BaObs t;
            ba_obs(Cn, n0, n1, n2, m.x, m.y, t);
            if constexpr (kLoss != LOSS_LINEAR) {
                double w0, w1;
                cost += t.ok ? ba_robust<kLoss>(t, ic, c2, w0, w1) : INFINITY;
            } else {
                cost += t.ok ? t.r0 * t.r0 + t.r1 * t.r1 : INFINITY;
            }
        }
    }
    const double s = ba_block_sum(cost, sh);
    if (threadIdx.x == 0) trial_part[blockIdx.x] = s;
}

// ------------------------------------------------------------------------------------------------
// step 5 (one CTA): sum the partials in order, accept / reject, damping schedule, convergence, commit the cameras
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ba_accept(BaState* __restrict__ st, double* __restrict__ cams, const double* __restrict__ dC,
                                                 int nC, const double* __restrict__ cost_part, const double* __restrict__ trial_part,
                                                 const int* __restrict__ bad_part, const double* __restrict__ obs2_part,
                                                 int nparts, double ftol, int max_iter) {
    __shared__ int better_s;
    __shared__ double sh[256 / 32];
    if (st->done) return;
    // ordered sums of the per-block partials: thread t adds partials t, t + 256, ...; then the fixed tree of ba_block_sum
    const bool need_cost = st->have_cost == 0, have_trial = st->accepted > 0;
    double ps = 0.0, ps2 = 0.0, pt = 0.0;
    int pnb = 0;
    for (int i = threadIdx.x; i < nparts; i += blockDim.x) {
        if (need_cost) { ps += cost_part[i]; ps2 += obs2_part[i]; }
        if (have_trial) pt += trial_part[i];
        pnb += bad_part[i];
    }
    const double s = ba_block_sum(ps, sh), s2 = ba_block_sum(ps2, sh), t = ba_block_sum(pt, sh);
    const double nbd = ba_block_sum((double)pnb, sh);
    if (threadIdx.x == 0) {
        if (need_cost) {
            st->cost = 0.5 * s;
            st->floor = 0.5 * s2 * (64.0 * 2.220446049250313e-16) * (64.0 * 2.220446049250313e-16);
            st->have_cost = 1;
        }
        st->n_bad = (int)nbd;
        st->cost_trial = 0.5 * t;
        st->iters += 1;
        const bool better = st->accepted > 0 && st->cost_trial < st->cost;       // NaN / Inf trial cost: not better
        better_s = better ? 1 : 0;
        if (better) {
            const double gain = st->cost - st->cost_trial;
            const bool conv = gain <= ftol * st->cost || st->cost_trial <= st->floor;   // relative decrease, or rounding level
            st->cost = st->cost_trial;
            st->lambda = fmax(st->lambda * 0.1, 1e-15);
            st->accepted = 1;                      // ba_points / ba_finish commit X_trial
            if (conv) st->done = 2;
        } else {
            st->accepted = 0;
            st->lambda *= 10.0;
            if (st->lambda > 1e12) st->done = 3;   // no descent direction any more: the current point is kept
        }
        if (!st->done && st->iters >= max_iter) st->done = 4;
    }
    __syncthreads();
    if (better_s)
        for (int i = threadIdx.x; i < 12 * nC; i += blockDim.x) cams[i] += dC[i];
}

// the cost at the start when no iteration runs (max_iter = 0)
__global__ void ba_cost_only(BaState* __restrict__ st, const double* __restrict__ cost_part, int nparts) {
    if (st->have_cost) return;
    double s = 0.0;
    for (int i = 0; i < nparts; ++i) s += cost_part[i];
    st->cost = 0.5 * s;
    st->have_cost = 1;
}

__global__ void ba_init(BaState* __restrict__ st, double lambda0) {
    st->lambda = lambda0; st->cost = 0.0; st->cost_trial = 0.0;
    st->iters = 0; st->done = 0; st->accepted = 0; st->have_cost = 0; st->n_bad = 0; st->pad = 0; st->floor = 0.0;
}

// after the loop: commit a last accepted trial; points back in the caller's order; scalars
__global__ void __launch_bounds__(256) ba_finish(const BaState* __restrict__ st, double* __restrict__ X,
                                                 const double* __restrict__ Xtrial, int nP, double* __restrict__ cost,
                                                 int* __restrict__ iters, int* __restrict__ status) {
    const bool commit = st->accepted > 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 3 * nP; i += gridDim.x * blockDim.x)
        if (commit) X[i] = Xtrial[i];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (cost) *cost = st->have_cost ? st->cost : __longlong_as_double(0x7ff8000000000000ll);
        if (iters) *iters = st->iters;
        if (status) *status = st->done;
    }
}

// EpsilonBA (tables.py:266-296) for a parameter vector x = [cameras (nC x 12), points (nP x 3)]: interleaved residuals
__global__ void __launch_bounds__(256) ba_residuals(const double* __restrict__ x, int nC, const double* __restrict__ u,
                                                    const double* __restrict__ v, const int* __restrict__ cam_idx,
                                                    const int* __restrict__ pt_idx, int nO, double* __restrict__ out) {
    const double* pts = x + 12 * (size_t)nC;
    for (int o = blockIdx.x * blockDim.x + threadIdx.x; o < nO; o += gridDim.x * blockDim.x) {
        const double* C = x + 12 * (size_t)cam_idx[o];
        const double* X = pts + 3 * (size_t)pt_idx[o];
        const double y0 = C[0] * X[0] + C[1] * X[1] + C[2] * X[2] + C[3];
        const double y1 = C[4] * X[0] + C[5] * X[1] + C[6] * X[2] + C[7];
        const double y2 = C[8] * X[0] + C[9] * X[1] + C[10] * X[2] + C[11];
        out[2 * (size_t)o] = u[o] - y0 / y2;
        out[2 * (size_t)o + 1] = v[o] - y1 / y2;
    }
}

}  // namespace rg
