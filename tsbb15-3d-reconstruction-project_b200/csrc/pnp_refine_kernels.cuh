// Refinement of PnP poses on the device: Levenberg-Marquardt on the reprojection error (DESIGN.md section 4.7).
//
// The reference's live PnP call is OpenCV's cv.solvePnPRansac (tables.py:141), which ends with solvePnP(ITERATIVE,
// useExtrinsicGuess) on the inliers.  This library's RANSAC returns the algebraic DLT pose of pnp.py:132-152; these
// kernels minimise, per view v over its selected correspondences S_v,
//   C_v(R, t) = 1/2 sum_k |W_v (pi(R X_k + t) - y_k)|^2,   pi(p) = (p0 / p2, p1 / p2),   W_v = [[fx, s], [0, fy]] or I
// over R <- exp([dw]_x) R (Rodrigues, FP64) and t <- t + dt.  J_k = W Pi_k [-[R X_k]_x | I]: the row a of W Pi gives the
// row [q x a | a] of J with q = R X_k.  pi is sign-agnostic (synth.pnp_scene has every point at negative depth).
// A robust loss (template parameter kLoss, f_scale = C) replaces |r|^2 by C^2 (rho((r0 / C)^2) + rho((r1 / C)^2)) and
// weights each scalar residual's row of J by rho' in J^T J and J^T r (IRLS, see pr_point).
//
// One pass over the points per iteration: at the trial pose it gives the cost AND the sums of J^T J (21) and J^T r (6);
// an accepted step keeps them as the current system, a rejected one re-solves the saved system with a larger lambda.
// Every sum is in a fixed order (per-thread partials, a fixed shuffle tree, warps / blocks in index order): no
// floating-point atomics, results are bit-reproducible.
//
// Kernels: pnp_refine_init, pnp_refine_fused (a view of <= kPrFusedMaxPts points: the whole loop in one CTA),
//          pnp_refine_pass + pnp_refine_step (larger views: per-block partials, then one CTA per view sums them in block
//          order, solves and accepts / rejects), pnp_refine_export, pnp_refine_consensus (thread per point, FP64).
#pragma once
#include "pnp_kernels.cuh"

namespace rg {

constexpr int kPrSums = 29;             // J^T J upper triangle (21) | J^T r (6) | sum |r|^2 | selected points
constexpr int kPrStride = 32;           // doubles per partial record (256 B)
constexpr int kPrThreads = 256;
constexpr int kPrWarps = kPrThreads / 32;
constexpr int kPrFusedMaxPts = 4096;    // views up to this size: one CTA per view, one launch per round
constexpr double kPrLambda0 = 1e-3;
constexpr double kPrXtol = 1e-14;      // a step below this (radians; relative for t) is rounding: converged

struct PrView {                         // per view, device resident
    double Rt[12];                      // current pose: R row-major, t
    double Rn[12];                      // trial pose (the pose the next pass evaluates)
    double S[kPrSums];                  // sums of the current pose
    double lambda, cost;
    int iters, done, pad0, pad1;        // done: 0 running, 1 pose not finite, 2 converged, 3 lambda > 1e12, 4 max_iter, 5 < 3 points
};

__device__ __forceinline__ constexpr int sym6(int i, int j) {      // packed upper triangle, i <= j
    return i * 6 - i * (i - 1) / 2 + (j - i);
}

// one correspondence: J rows ja, jb (2 x 6) and residual (r0, r1) added to acc.  A robust loss (ic = 1 / C, c2 = C^2)
// weights each scalar residual by w = rho'((r / C)^2) between the two factors of J^T J and J^T r (IRLS, as in
// ba_kernels.cuh) and adds C^2 rho to slot 27 in place of r^2, so that 0.5 * acc[27] is SciPy's robust cost.
template <int kLoss>
__device__ __forceinline__ void pr_point(const double* __restrict__ P, const double w0, const double w1, const double w2,
                                         const double X0, const double X1, const double X2, const double y0, const double y1,
                                         const double ic, const double c2, double (&acc)[kPrSums]) {
    const double q0 = P[0] * X0 + P[1] * X1 + P[2] * X2;
    const double q1 = P[3] * X0 + P[4] * X1 + P[5] * X2;
    const double q2 = P[6] * X0 + P[7] * X1 + P[8] * X2;
    const double iz = 1.0 / (q2 + P[11]);
    const double u = (q0 + P[9]) * iz, v = (q1 + P[10]) * iz;
    const double du = u - y0, dv = v - y1;
    const double r0 = w0 * du + w1 * dv, r1 = w2 * dv;
    // rows of W Pi:  a = (w0, w1, -(w0 u + w1 v)) / z,  b = (0, w2, -w2 v) / z
    const double a0 = w0 * iz, a1 = w1 * iz, a2 = -(w0 * u + w1 * v) * iz;
    const double b1 = w2 * iz, b2 = -w2 * v * iz;
    const double ja[6] = {q1 * a2 - q2 * a1, q2 * a0 - q0 * a2, q0 * a1 - q1 * a0, a0, a1, a2};
    const double jb[6] = {q1 * b2 - q2 * b1, -q0 * b2, q0 * b1, 0.0, b1, b2};
    if constexpr (kLoss == LOSS_LINEAR) {
#pragma unroll
        for (int i = 0; i < 6; ++i) {
#pragma unroll
            for (int j = i; j < 6; ++j) acc[sym6(i, j)] = fma(ja[i], ja[j], fma(jb[i], jb[j], acc[sym6(i, j)]));
            acc[21 + i] = fma(ja[i], r0, fma(jb[i], r1, acc[21 + i]));
        }
        acc[27] = fma(r0, r0, fma(r1, r1, acc[27]));
    } else {
        const double s0 = r0 * ic, s1 = r1 * ic;
        double p0, p1, o0, o1;
        ba_rho<kLoss>(s0 * s0, p0, o0);
        ba_rho<kLoss>(s1 * s1, p1, o1);
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            const double wa = o0 * ja[i], wb = o1 * jb[i];
#pragma unroll
            for (int j = i; j < 6; ++j) acc[sym6(i, j)] = fma(wa, ja[j], fma(wb, jb[j], acc[sym6(i, j)]));
            acc[21 + i] = fma(wa, r0, fma(wb, r1, acc[21 + i]));
        }
        acc[27] = fma(c2, p0 + p1, acc[27]);
    }
    acc[28] += 1.0;
}

// the view's weight W = upper-left 2x2 of K (K validated on the host: K[1][0] == 0, bottom row (0, 0, 1))
__device__ __forceinline__ void pr_weight(const double* __restrict__ W3, int v, double& w0, double& w1, double& w2) {
    if (W3) { w0 = W3[3 * v]; w1 = W3[3 * v + 1]; w2 = W3[3 * v + 2]; }
    else { w0 = 1.0; w1 = 0.0; w2 = 1.0; }
}

// sums of the points [lo, hi) handled by this thread (stride `step` from `first`)
template <int kLoss>
__device__ __forceinline__ void pr_accumulate(const double* __restrict__ X, const double* __restrict__ y,
                                              const unsigned char* __restrict__ mask, const double* P, double w0, double w1,
                                              double w2, int first, int hi, int step, double ic, double c2,
                                              double (&acc)[kPrSums]) {
#pragma unroll
    for (int k = 0; k < kPrSums; ++k) acc[k] = 0.0;
    for (int i = first; i < hi; i += step) {
        if (mask != nullptr && mask[i] == 0) continue;
        pr_point<kLoss>(P, w0, w1, w2, X[3 * (size_t)i], X[3 * (size_t)i + 1], X[3 * (size_t)i + 2], y[2 * (size_t)i],
                        y[2 * (size_t)i + 1], ic, c2, acc);
    }
}

// block sum in a fixed order: shuffle tree per warp, then warps in index order.  out[k] (shared) for k < kPrSums.
__device__ __forceinline__ void pr_block_sum(double (&acc)[kPrSums], double (*red)[kPrStride], double* out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < kPrSums; ++k) {
        double v = acc[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[warp][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < kPrSums) {
        double s = red[0][threadIdx.x];
#pragma unroll
        for (int w = 1; w < kPrWarps; ++w) s += red[w][threadIdx.x];
        out[threadIdx.x] = s;
    }
    __syncthreads();
}

// (A + lambda diag A) dx = -g by a 6x6 Cholesky (one thread); pred = decrease the linear model predicts for dx,
// 1/2 dx^T A dx + lambda dx^T diag(A) dx.  false if the damped system is not positive definite / dx not finite.
__device__ __forceinline__ bool pr_solve(const double* S, const double lambda, double (&dx)[6], double& pred) {
    double L[6][6];
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int j = 0; j < 6; ++j) L[i][j] = (j <= i) ? S[sym6(j, i)] : 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) L[i][i] += lambda * L[i][i];
    bool ok = true;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        double d = L[j][j];
#pragma unroll
        for (int k = 0; k < j; ++k) d -= L[j][k] * L[j][k];
        ok = ok && d > 0.0 && isfinite(d);
        const double ljj = sqrt(d), inv = 1.0 / ljj;
        L[j][j] = ljj;
#pragma unroll
        for (int i = j + 1; i < 6; ++i) {
            double s = L[i][j];
#pragma unroll
            for (int k = 0; k < j; ++k) s -= L[i][k] * L[j][k];
            L[i][j] = s * inv;
        }
    }
    double z[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        double s = -S[21 + i];
#pragma unroll
        for (int k = 0; k < i; ++k) s -= L[i][k] * z[k];
        z[i] = s / L[i][i];
    }
#pragma unroll
    for (int i = 5; i >= 0; --i) {
        double s = z[i];
#pragma unroll
        for (int k = i + 1; k < 6; ++k) s -= L[k][i] * dx[k];
        dx[i] = s / L[i][i];
    }
    double quad = 0.0, damp = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        ok = ok && isfinite(dx[i]);
        double Ai = 0.0;
#pragma unroll
        for (int j = 0; j < 6; ++j) Ai += S[i <= j ? sym6(i, j) : sym6(j, i)] * dx[j];
        quad += dx[i] * Ai;
        damp += S[sym6(i, i)] * dx[i] * dx[i];
    }
    pred = 0.5 * quad + lambda * damp;
    return ok;
}

// out = (exp([dw]_x) R | t + dt); (1 - cos th) / th^2 as 2 sin^2(th/2) / th^2
__device__ __forceinline__ void pr_compose(const double* Rt, const double (&dx)[6], double* out) {
    const double th = sqrt(dx[0] * dx[0] + dx[1] * dx[1] + dx[2] * dx[2]);
    double a = 1.0, b = 0.5;
    if (th > 0.0) {
        a = sin(th) / th;
        const double h = sin(0.5 * th) / (0.5 * th);
        b = 0.5 * h * h;
    }
    const double wx[3][3] = {{0.0, -dx[2], dx[1]}, {dx[2], 0.0, -dx[0]}, {-dx[1], dx[0], 0.0}};
    double E[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const double w2 = wx[i][0] * wx[0][j] + wx[i][1] * wx[1][j] + wx[i][2] * wx[2][j];
            E[i][j] = (i == j ? 1.0 : 0.0) + a * wx[i][j] + b * w2;
        }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) out[3 * i + j] = E[i][0] * Rt[j] + E[i][1] * Rt[3 + j] + E[i][2] * Rt[6 + j];
#pragma unroll
    for (int i = 0; i < 3; ++i) out[9 + i] = Rt[9 + i] + dx[3 + i];
}

// Decision after the pass at the trial pose (sums T), then the next step: the rules of gs_accept (gs_kernels.cuh) —
// lambda / 10 on an accepted step (floor 1e-15), x 10 on a rejected one (NaN trial cost: rejected); status 2 when an
// accepted step decreased the cost by <= ftol * cost, when the model predicts a decrease <= ftol * cost for the next
// step (which is then not taken: its actual decrease would be below the rounding error of the cost) or when that step
// would move the pose by <= kPrXtol (the floor zero-residual data reach), 3 when lambda
// > 1e12, 4 at max_iter.  A damped system that cannot be factorised is a rejected iteration without a pass.
// Returns true when a new trial pose was written to G.Rn.  One thread.
__device__ __forceinline__ bool pr_decide(PrView& G, const double* T, bool have_trial, int max_iter, double ftol) {
    if (have_trial) {
        G.iters += 1;
        const double ct = 0.5 * T[27];
        if (ct < G.cost) {
            const bool conv = G.cost - ct <= ftol * G.cost;
#pragma unroll
            for (int k = 0; k < 12; ++k) G.Rt[k] = G.Rn[k];
#pragma unroll
            for (int k = 0; k < kPrSums; ++k) G.S[k] = T[k];
            G.cost = ct;
            G.lambda = fmax(G.lambda * 0.1, 1e-15);
            if (conv) { G.done = 2; return false; }
        } else {
            G.lambda *= 10.0;
            if (G.lambda > 1e12) { G.done = 3; return false; }
        }
    }
    for (;;) {
        if (G.iters >= max_iter) { G.done = 4; return false; }
        double dx[6], pred;
        if (pr_solve(G.S, G.lambda, dx, pred)) {
            const double nw = sqrt(dx[0] * dx[0] + dx[1] * dx[1] + dx[2] * dx[2]);
            const double nt = sqrt(dx[3] * dx[3] + dx[4] * dx[4] + dx[5] * dx[5]);
            const double t2 = sqrt(G.Rt[9] * G.Rt[9] + G.Rt[10] * G.Rt[10] + G.Rt[11] * G.Rt[11]);
            if (pred <= ftol * G.cost || (nw <= kPrXtol && nt <= kPrXtol * t2)) { G.done = 2; return false; }
            pr_compose(G.Rt, dx, G.Rn);
            return true;
        }
        G.iters += 1;
        G.lambda *= 10.0;
        if (G.lambda > 1e12) { G.done = 3; return false; }
    }
}

// first pass done (sums T at the start pose): cost, fewer-than-3-points check, first step
__device__ __forceinline__ bool pr_start(PrView& G, const double* T, int max_iter, double ftol) {
#pragma unroll
    for (int k = 0; k < kPrSums; ++k) G.S[k] = T[k];
    G.cost = 0.5 * T[27];
    RG_ASSERT(T[28] >= 0.0);
    if (T[28] < 3.0) { G.done = 5; return false; }
    return pr_decide(G, T, false, max_iter, ftol);
}

// state of every view from its start pose (Rt_io, V x 12)
__global__ void __launch_bounds__(64) pnp_refine_init(const double* __restrict__ Rt_io, int V, PrView* __restrict__ st) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= V) return;
    PrView G;
    bool fin = true;
#pragma unroll
    for (int k = 0; k < 12; ++k) { G.Rt[k] = Rt_io[12 * (size_t)v + k]; G.Rn[k] = G.Rt[k]; fin = fin && isfinite(G.Rt[k]); }
#pragma unroll
    for (int k = 0; k < kPrSums; ++k) G.S[k] = 0.0;
    G.lambda = kPrLambda0;
    G.cost = __longlong_as_double(0x7ff8000000000000ll);
    G.iters = 0; G.done = fin ? 0 : 1; G.pad0 = 0; G.pad1 = 0;
    st[v] = G;
}

// The whole loop of ONE view in ONE CTA (views of up to kPrFusedMaxPts points; the Dino views have 37-204).  grid = V.
// kLoss, ic = 1 / C, c2 = C^2: the loss of pr_point.
template <int kLoss>
__global__ void __launch_bounds__(kPrThreads) pnp_refine_fused(const double* __restrict__ X, const double* __restrict__ y,
                                                               const int* __restrict__ off, const double* __restrict__ W3,
                                                               const unsigned char* __restrict__ mask,
                                                               PrView* __restrict__ st, int max_iter, double ftol, double ic,
                                                               double c2) {
    __shared__ PrView G;
    __shared__ double red[kPrWarps][kPrStride];
    __shared__ double T[kPrStride];
    __shared__ int s_go;
    const int v = blockIdx.x;
    if (threadIdx.x == 0) G = st[v];
    __syncthreads();
    if (G.done) return;                                          // uniform
    const int lo = off[v], hi = off[v + 1];
    double w0, w1, w2;
    pr_weight(W3, v, w0, w1, w2);
    double acc[kPrSums];
    pr_accumulate<kLoss>(X, y, mask, G.Rt, w0, w1, w2, lo + threadIdx.x, hi, kPrThreads, ic, c2, acc);
    pr_block_sum(acc, red, T);
    if (threadIdx.x == 0) s_go = pr_start(G, T, max_iter, ftol) ? 1 : 0;
    __syncthreads();
    while (s_go) {
        pr_accumulate<kLoss>(X, y, mask, G.Rn, w0, w1, w2, lo + threadIdx.x, hi, kPrThreads, ic, c2, acc);
        pr_block_sum(acc, red, T);
        if (threadIdx.x == 0) s_go = pr_decide(G, T, true, max_iter, ftol) ? 1 : 0;
        __syncthreads();
    }
    if (threadIdx.x == 0) st[v] = G;
}

// multi-CTA path, pass: per-block partial sums at the pose G.Rn of every running view.  grid = (nb, V).
template <int kLoss>
__global__ void __launch_bounds__(kPrThreads) pnp_refine_pass(const double* __restrict__ X, const double* __restrict__ y,
                                                              const int* __restrict__ off, const double* __restrict__ W3,
                                                              const unsigned char* __restrict__ mask,
                                                              const PrView* __restrict__ st, double* __restrict__ part,
                                                              double ic, double c2) {
    __shared__ double red[kPrWarps][kPrStride];
    __shared__ double P[12];
    const int v = blockIdx.y;
    if (st[v].done) return;
    if (threadIdx.x < 12) P[threadIdx.x] = st[v].Rn[threadIdx.x];
    __syncthreads();
    const int lo = off[v], hi = off[v + 1];
    double w0, w1, w2;
    pr_weight(W3, v, w0, w1, w2);
    double acc[kPrSums];
    pr_accumulate<kLoss>(X, y, mask, P, w0, w1, w2, lo + blockIdx.x * kPrThreads + threadIdx.x, hi, gridDim.x * kPrThreads,
                         ic, c2, acc);
    double* out = part + ((size_t)v * gridDim.x + blockIdx.x) * kPrStride;
    pr_block_sum(acc, red, out);
}

// multi-CTA path, step: the view's partials summed in block order (8 interleaved chains, then the chains in order),
// then the decision of pr_start / pr_decide.  grid = V; n_active (optional): views still running afterwards.
__global__ void __launch_bounds__(kPrThreads) pnp_refine_step(PrView* __restrict__ st, const double* __restrict__ part, int nb,
                                                              int first, int max_iter, double ftol, int* __restrict__ n_active) {
    __shared__ double red[kPrWarps][kPrStride];
    __shared__ double T[kPrStride];
    const int v = blockIdx.x;
    if (st[v].done) return;
    const int k = threadIdx.x & 31, c = threadIdx.x >> 5;
    const double* p = part + (size_t)v * nb * kPrStride;
    double s = 0.0;
    for (int b = c; b < nb; b += kPrWarps) s += p[(size_t)b * kPrStride + k];
    red[c][k] = s;
    __syncthreads();
    if (threadIdx.x < kPrSums) {
        double t = red[0][threadIdx.x];
#pragma unroll
        for (int w = 1; w < kPrWarps; ++w) t += red[w][threadIdx.x];
        T[threadIdx.x] = t;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        PrView& G = st[v];
        const bool go = first ? pr_start(G, T, max_iter, ftol) : pr_decide(G, T, true, max_iter, ftol);
        if (go && n_active != nullptr) atomicAdd(n_active, 1);
    }
}

__global__ void __launch_bounds__(64) pnp_refine_export(const PrView* __restrict__ st, int V, double* __restrict__ Rt_io,
                                                        double* __restrict__ cost, int* __restrict__ iters,
                                                        int* __restrict__ status) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= V) return;
#pragma unroll
    for (int k = 0; k < 12; ++k) Rt_io[12 * (size_t)v + k] = st[v].Rt[k];
    if (cost) cost[v] = st[v].cost;
    if (iters) iters[v] = st[v].iters;
    if (status) status[v] = st[v].done;
}

// consensus at the refined pose over ALL correspondences of the view: thr2 >= e (ransac.py:104-105), FP64.  grid (nbx, V).
__global__ void __launch_bounds__(256) pnp_refine_consensus(const double* __restrict__ X, const double* __restrict__ y,
                                                            const int* __restrict__ off, const PrView* __restrict__ st,
                                                            double thr2, unsigned char* __restrict__ mask) {
    const int v = blockIdx.y;
    double Rt[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) Rt[k] = st[v].Rt[k];
    const int lo = off[v], hi = off[v + 1];
    for (int i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x)
        mask[i] = (unsigned char)pnp_inlier64(Rt, X[3 * (size_t)i], X[3 * (size_t)i + 1], X[3 * (size_t)i + 2],
                                              y[2 * (size_t)i], y[2 * (size_t)i + 1], thr2);
}

}  // namespace rg
