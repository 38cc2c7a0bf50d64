// Gold-standard refinement of a fundamental matrix on the device (SURVEY.md section 8f row N4):
//   minimise  sum_i |pl_i - proj(C1 X_i)|^2 + |pr_i - proj([I|0] X_i)|^2   over C1 (3x4) and the N points X_i
// the cost of lab3.fmatrix_residuals_gs (lab3.py:230-266), which fun.getFFromLabCode hands to SciPy's least_squares
// (fun.py:342-369; 5482 residual evaluations / 267 s for the 257 inliers of the noisy Dino pair (0,1), stopping on
// ftol before the minimum).  Here: Levenberg-Marquardt with Marquardt scaling and the Schur complement of the
// block-diagonal point part, batched over image pairs, no host synchronisation between iterations.
//
// Structure used.  With P2 = d proj / d y at y = C1 Xh (2x3), Q = P2 C1[:, :3], Pr = d proj / d X at X (right camera):
//   J_c^T J_c = (P2^T P2) (x) (Xh Xh^T)          J_c^T J_p = (P2^T Q) (x) Xh          D = Q^T Q + Pr^T Pr
// so the reduced camera system is  S = sum_i (M_i - T_i D_i'^-1 T_i^T) (x) (Xh_i Xh_i^T) + lambda diag(A):
// 60 distinct products per point instead of a 12x12 block, accumulated in registers, reduced per block, atomically added.
// A robust loss (template parameter kLoss, f_scale = C in pixels) replaces every squared residual f^2 by C^2 rho((f / C)^2)
// and weights the products by rho' (IRLS, see gs_blocks_w); the structure above is unchanged.
#pragma once
#include "geom_kernels.cuh"

namespace rg {

constexpr int kGsSums = 60 + 12 + 12 + 1;       // W (x) XX products, rhs (3x4), diag A (3x4), cost
constexpr int kGsThreads = 128;

struct GsPair {                 // per image pair, device resident
    double C1[12];              // current first camera (second is [I | 0])
    double dc[12];              // proposed camera step
    double lambda, cost, cost_trial;
    int iters, done, accepted, have_cost;
    int n_used, pad;
};

// index of (a, b) in the packed upper triangle of a symmetric 3x3 (0..5) / 4x4 (0..9)
__device__ __forceinline__ constexpr int sym3(int a, int b) {
    return (a <= b) ? (a * 3 - a * (a - 1) / 2 + (b - a)) : (b * 3 - b * (b - 1) / 2 + (a - b));
}
__device__ __forceinline__ constexpr int sym4(int a, int b) {
    return (a <= b) ? (a * 4 - a * (a - 1) / 2 + (b - a)) : (b * 4 - b * (b - 1) / 2 + (a - b));
}

// inverse of a symmetric positive definite 3x3 (upper triangle d00 d01 d02 d11 d12 d22) by the adjugate
__device__ __forceinline__ bool inv_sym3(const double (&d)[6], double (&o)[6]) {
    const double c00 = d[3] * d[5] - d[4] * d[4];
    const double c01 = d[2] * d[4] - d[1] * d[5];
    const double c02 = d[1] * d[4] - d[2] * d[3];
    const double det = d[0] * c00 + d[1] * c01 + d[2] * c02;
    if (!(det > 0.0) || !isfinite(det)) return false;
    const double id = 1.0 / det;
    o[0] = c00 * id; o[1] = c01 * id; o[2] = c02 * id;
    o[3] = (d[0] * d[5] - d[2] * d[2]) * id;
    o[4] = (d[1] * d[2] - d[0] * d[4]) * id;
    o[5] = (d[0] * d[3] - d[1] * d[1]) * id;
    return true;
}

// Everything the normal equations need from one correspondence at the current (C1, X).
struct GsPoint {
    double Xh[4];
    double rl[2], rr[2];        // residuals (measured - predicted), left / right
    double P2[2][3], Q[2][3], Pr[2][3];
    bool ok;
};

__device__ __forceinline__ void gs_point(const double* __restrict__ C1, const double4 m, const double X0, const double X1,
                                         const double X2, GsPoint& g) {
    g.Xh[0] = X0; g.Xh[1] = X1; g.Xh[2] = X2; g.Xh[3] = 1.0;
    double y[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) y[a] = C1[4 * a] * X0 + C1[4 * a + 1] * X1 + C1[4 * a + 2] * X2 + C1[4 * a + 3];
    const double iy = 1.0 / y[2], ix = 1.0 / X2;
    const double u0 = y[0] * iy, u1 = y[1] * iy, v0 = X0 * ix, v1 = X1 * ix;
    g.rl[0] = m.x - u0; g.rl[1] = m.y - u1;
    g.rr[0] = m.z - v0; g.rr[1] = m.w - v1;
    g.P2[0][0] = iy; g.P2[0][1] = 0.0; g.P2[0][2] = -u0 * iy;
    g.P2[1][0] = 0.0; g.P2[1][1] = iy; g.P2[1][2] = -u1 * iy;
    g.Pr[0][0] = ix; g.Pr[0][1] = 0.0; g.Pr[0][2] = -v0 * ix;
    g.Pr[1][0] = 0.0; g.Pr[1][1] = ix; g.Pr[1][2] = -v1 * ix;
#pragma unroll
    for (int k = 0; k < 2; ++k)
#pragma unroll
        for (int c = 0; c < 3; ++c) g.Q[k][c] = g.P2[k][0] * C1[c] + g.P2[k][1] * C1[4 + c] + g.P2[k][2] * C1[8 + c];
    g.ok = isfinite(g.rl[0]) && isfinite(g.rl[1]) && isfinite(g.rr[0]) && isfinite(g.rr[1]) && isfinite(iy) && isfinite(ix);
}

// M = P2^T P2 (sym 6), T = P2^T Q (3x3), damped inverse of D = Q^T Q + Pr^T Pr, g_p = -(Q^T rl + Pr^T rr)
__device__ __forceinline__ bool gs_blocks(const GsPoint& g, double lambda, double (&M)[6], double (&T)[3][3], double (&Di)[6],
                                          double (&gp)[3]) {
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = a; b < 3; ++b) M[sym3(a, b)] = g.P2[0][a] * g.P2[0][b] + g.P2[1][a] * g.P2[1][b];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) T[a][c] = g.P2[0][a] * g.Q[0][c] + g.P2[1][a] * g.Q[1][c];
    double D[6];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = a; b < 3; ++b)
            D[sym3(a, b)] = g.Q[0][a] * g.Q[0][b] + g.Q[1][a] * g.Q[1][b] + g.Pr[0][a] * g.Pr[0][b] + g.Pr[1][a] * g.Pr[1][b];
    D[0] += lambda * D[0]; D[3] += lambda * D[3]; D[5] += lambda * D[5];        // Marquardt scaling
#pragma unroll
    for (int c = 0; c < 3; ++c)
        gp[c] = -(g.Q[0][c] * g.rl[0] + g.Q[1][c] * g.rl[1] + g.Pr[0][c] * g.rr[0] + g.Pr[1][c] * g.rr[1]);
    return inv_sym3(D, Di);
}

// Robust loss (ic = 1 / C, c2 = C^2): C^2 (sum of rho((r / C)^2) over the four residuals of g) and the weights
// w = rho'(z) (left x, left y, right x, right y).
template <int kLoss>
__device__ __forceinline__ double gs_rho(const GsPoint& g, const double ic, const double c2, double (&w)[4]) {
    const double s[4] = {g.rl[0] * ic, g.rl[1] * ic, g.rr[0] * ic, g.rr[1] * ic};
    double sum = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        double p;
        ba_rho<kLoss>(s[k] * s[k], p, w[k]);
        sum += p;
    }
    return c2 * sum;
}

// gs_blocks for a loss: the squared loss is gs_blocks itself.  A robust loss puts Wl = diag(w0, w1), Wr = diag(w2, w3)
// between the two factors of every product (IRLS, as in ba_kernels.cuh): M = P2^T Wl P2, T = P2^T Wl Q,
// D = Q^T Wl Q + Pr^T Wr Pr, g_p = -(Q^T Wl rl + Pr^T Wr rr), and the callers' P2^T rl becomes P2^T Wl rl.  It does so by
// scaling each residual of g and its rows of P2, Q, Pr by sqrt(w) in place (w > 0 for every loss), so that the
// unweighted gs_blocks and the callers' code, with their register footprint, stay as they are; take the cost (gs_rho)
// before.
template <int kLoss>
__device__ __forceinline__ bool gs_blocks_w(GsPoint& g, const double (&w)[4], double lambda, double (&M)[6], double (&T)[3][3],
                                            double (&Di)[6], double (&gp)[3]) {
    if constexpr (kLoss != LOSS_LINEAR) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const double sl = sqrt(w[k]), sr = sqrt(w[2 + k]);
            g.rl[k] *= sl; g.rr[k] *= sr;
#pragma unroll
            for (int c = 0; c < 3; ++c) { g.P2[k][c] *= sl; g.Q[k][c] *= sl; g.Pr[k][c] *= sr; }
        }
    }
    return gs_blocks(g, lambda, M, T, Di, gp);
}

// ------------------------------------------------------------------------------------------------
// 12x12 Cholesky of a diagonal block by one warp: lane r holds row r in registers; column j is scaled by rsqrt(d)
// (MUFU.RSQ64H + Newton: no DSQRT / division chain) and broadcast to the other rows through shared memory.
// Ld: row-major lower triangle in shared memory (in: the block, out: its factor), Li[j] = 1 / L[j][j],
// cb: 24 doubles of scratch.  Returns false (uniformly) when a pivot is not positive / finite.
// ------------------------------------------------------------------------------------------------
// (no __restrict__ on these pointers: the lanes communicate through this shared memory, and a restrict-qualified pointer
// lets the compiler move its loads across __syncwarp() — seen as a wrong last pivot in every lane but the writer's)
__device__ __forceinline__ bool ba_chol12(double* Ld, double* Li, double* cb, const int lane) {
    double a[12], dg[12];                                       // own row; every lane's copy of the remaining diagonal
#pragma unroll
    for (int c = 0; c < 12; ++c) {
        a[c] = (lane < 12 && c <= lane) ? Ld[lane * 12 + c] : 0.0;
        dg[c] = Ld[c * 12 + c];
    }
    bool ok = true;
#pragma unroll
    for (int j = 0; j < 12; ++j) {
        const double d = dg[j];                                 // kept up to date below: no shuffle on the critical chain
        ok = ok && d > 0.0 && isfinite(d);                      // no early exit: the loop stays fully unrolled
        const double inv = rsqrt(d);
        if (lane == j) { a[j] = d * inv; Li[j] = inv; }
        else if (lane > j) a[j] *= inv;
        double* col = cb + 12 * (j & 1);
        if (lane > j && lane < 12) col[lane] = a[j];
        __syncwarp();
#pragma unroll
        for (int c = j + 1; c < 12; ++c) {
            const double t = col[c];                            // L[c][j]
            if (lane > c) a[c] = fma(-a[j], t, a[c]);           // L[lane][c] -= L[lane][j] L[c][j]
            dg[c] = fma(-t, t, dg[c]);
            if (lane == c) a[c] = dg[c];                        // the diagonal entry of the own row: same value in every lane
        }
    }
    if (ok && lane < 12) {
#pragma unroll
        for (int c = 0; c < 12; ++c)
            if (c <= lane) Ld[lane * 12 + c] = a[c];
    }
    return ok;
}

// ------------------------------------------------------------------------------------------------
// initial cameras from F (lab3.fmatrix_cameras, lab3.py:353-380): C1 = ([e1]_x F | e1), e1 = left null vector of F
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(64) gs_init(const double* __restrict__ F0, int P, double lambda0, GsPair* __restrict__ gp,
                                              double* __restrict__ C1out, double* __restrict__ C2out) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    double F[9];
    bool fin = true;
#pragma unroll
    for (int k = 0; k < 9; ++k) { F[k] = F0[(size_t)p * 9 + k]; fin = fin && isfinite(F[k]); }
    // right null vector of F^T by one-sided Jacobi: columns of W are the rows of F
    double w[3][3], v[3][3];
#pragma unroll
    for (int j = 0; j < 3; ++j)
#pragma unroll
        for (int i = 0; i < 3; ++i) { w[j][i] = F[3 * j + i]; v[j][i] = (i == j) ? 1.0 : 0.0; }
    jacobi3(w, v);
    int jm = 0;
    double best = INFINITY;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const double n = w[j][0] * w[j][0] + w[j][1] * w[j][1] + w[j][2] * w[j][2];
        if (n < best) { best = n; jm = j; }
    }
    double e[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) e[i] = jm == 0 ? v[0][i] : (jm == 1 ? v[1][i] : v[2][i]);
    const double ne = rsqrt(e[0] * e[0] + e[1] * e[1] + e[2] * e[2]);
#pragma unroll
    for (int i = 0; i < 3; ++i) e[i] *= ne;
    GsPair g;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        g.C1[c]     = -e[2] * F[3 + c] + e[1] * F[6 + c];
        g.C1[4 + c] =  e[2] * F[c]     - e[0] * F[6 + c];
        g.C1[8 + c] = -e[1] * F[c]     + e[0] * F[3 + c];
    }
    g.C1[3] = e[0]; g.C1[7] = e[1]; g.C1[11] = e[2];
#pragma unroll
    for (int k = 0; k < 12; ++k) g.dc[k] = 0.0;
    g.lambda = lambda0; g.cost = 0.0; g.cost_trial = 0.0;
    g.iters = 0; g.done = fin ? 0 : 1; g.accepted = 0; g.have_cost = 0; g.n_used = 0; g.pad = 0;
    gp[p] = g;
#pragma unroll
    for (int k = 0; k < 12; ++k) {
        C1out[(size_t)p * 12 + k] = g.C1[k];
        C2out[(size_t)p * 12 + k] = (k == 0 || k == 5 || k == 10) ? 1.0 : 0.0;
    }
}

// ------------------------------------------------------------------------------------------------
// LM iteration, step 1: commit the previous trial if it was accepted, accumulate the reduced camera system
// grid = (blocks per pair, P); kLoss, ic = 1 / C, c2 = C^2: the loss (gs_rho, gs_blocks_w)
// ------------------------------------------------------------------------------------------------
template <int kLoss>
__global__ void __launch_bounds__(kGsThreads) gs_accumulate(const double4* __restrict__ pts, const unsigned char* __restrict__ mask,
                                                            const int* __restrict__ pair_off, GsPair* __restrict__ gpair,
                                                            double* __restrict__ Xcur, const double* __restrict__ Xtrial,
                                                            double* __restrict__ sums, double ic, double c2) {
    __shared__ double red[kGsSums];
    const int p = blockIdx.y;
    GsPair& G = gpair[p];
    if (G.done) return;
    for (int k = threadIdx.x; k < kGsSums; k += blockDim.x) red[k] = 0.0;
    __syncthreads();
    double C1[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) C1[k] = G.C1[k];
    const double lambda = G.lambda;
    const bool commit = G.accepted != 0;
    const int lo = pair_off[p], hi = pair_off[p + 1];
    double acc[kGsSums];
#pragma unroll
    for (int k = 0; k < kGsSums; ++k) acc[k] = 0.0;
    for (int i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) {
        double X0 = Xcur[3 * (size_t)i], X1 = Xcur[3 * (size_t)i + 1], X2 = Xcur[3 * (size_t)i + 2];
        if (commit) {
            X0 = Xtrial[3 * (size_t)i]; X1 = Xtrial[3 * (size_t)i + 1]; X2 = Xtrial[3 * (size_t)i + 2];
            Xcur[3 * (size_t)i] = X0; Xcur[3 * (size_t)i + 1] = X1; Xcur[3 * (size_t)i + 2] = X2;
        }
        if (mask != nullptr && mask[i] == 0) continue;
        GsPoint g;
        gs_point(C1, pts[i], X0, X1, X2, g);
        if (!g.ok) continue;
        double w[4], rc = 0.0;
        if constexpr (kLoss != LOSS_LINEAR) rc = gs_rho<kLoss>(g, ic, c2, w);
        double M[6], T[3][3], Di[6], gp[3];
        if (!gs_blocks_w<kLoss>(g, w, lambda, M, T, Di, gp)) continue;
        // W = M - T Di T^T  (symmetric 3x3),  z = P2^T rl + T Di gp
        double TD[3][3];
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int c = 0; c < 3; ++c)
                TD[a][c] = T[a][0] * Di[sym3(0, c)] + T[a][1] * Di[sym3(1, c)] + T[a][2] * Di[sym3(2, c)];
        double W[6], z[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int b = a; b < 3; ++b)
                W[sym3(a, b)] = M[sym3(a, b)] - (TD[a][0] * T[b][0] + TD[a][1] * T[b][1] + TD[a][2] * T[b][2]);
            z[a] = g.P2[0][a] * g.rl[0] + g.P2[1][a] * g.rl[1] + TD[a][0] * gp[0] + TD[a][1] * gp[1] + TD[a][2] * gp[2];
        }
        double XX[10];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = a; b < 4; ++b) XX[sym4(a, b)] = g.Xh[a] * g.Xh[b];
#pragma unroll
        for (int wq = 0; wq < 6; ++wq)
#pragma unroll
            for (int x = 0; x < 10; ++x) acc[wq * 10 + x] = fma(W[wq], XX[x], acc[wq * 10 + x]);
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                acc[60 + a * 4 + b] = fma(z[a], g.Xh[b], acc[60 + a * 4 + b]);
                acc[72 + a * 4 + b] = fma(M[sym3(a, a)], XX[sym4(b, b)], acc[72 + a * 4 + b]);
            }
        if constexpr (kLoss == LOSS_LINEAR) acc[84] += g.rl[0] * g.rl[0] + g.rl[1] * g.rl[1] + g.rr[0] * g.rr[0] + g.rr[1] * g.rr[1];
        else acc[84] += rc;
    }
#pragma unroll
    for (int k = 0; k < kGsSums; ++k) {
        double v = acc[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0 && v != 0.0) atomicAdd(&red[k], v);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < kGsSums; k += blockDim.x)
        if (red[k] != 0.0) atomicAdd(&sums[(size_t)p * kGsSums + k], red[k]);
}

// the reduced 12x12 camera system of one pair from its sums s[kGsSums] -> camera step x[12] (one warp; Ld 144, Li 16,
// cb 24, x 12 doubles of shared memory); false if the damped system is not positive definite
__device__ __forceinline__ bool gs_solve_warp(const double* s, const double lambda, double* Ld, double* Li, double* cb,
                                              double* x, const int lane) {
    if (lane < 12) {
        const int a = lane >> 2, b = lane & 3;
        for (int c = 0; c <= lane; ++c) {
            const int a2 = c >> 2, b2 = c & 3;
            Ld[lane * 12 + c] = s[sym3(a, a2) * 10 + sym4(b, b2)];
        }
        for (int c = lane + 1; c < 12; ++c) Ld[lane * 12 + c] = 0.0;
        Ld[lane * 12 + lane] += lambda * s[72 + lane];
        x[lane] = s[60 + lane];
    }
    __syncwarp();
    bool ok = ba_chol12(Ld, Li, cb, lane);
    __syncwarp();
    if (lane == 0 && ok) {                                  // L y = rhs, L^T x = y with the reciprocal diagonal
#pragma unroll
        for (int i = 0; i < 12; ++i) {
            double v = x[i];
#pragma unroll
            for (int k = 0; k < 12; ++k)
                if (k < i) v = fma(-Ld[i * 12 + k], x[k], v);
            x[i] = v * Li[i];
        }
#pragma unroll
        for (int i = 11; i >= 0; --i) {
            double v = x[i];
#pragma unroll
            for (int k = 0; k < 12; ++k)
                if (k > i) v = fma(-Ld[k * 12 + i], x[k], v);
            x[i] = v * Li[i];
            ok = ok && isfinite(x[i]);
        }
    }
    __syncwarp();                                           // x (written by lane 0) is read by the other lanes of the caller
    return __shfl_sync(0xffffffffu, ok ? 1 : 0, 0) != 0;
}

// step 2 (one warp per pair): assemble S, Cholesky (ba_chol12: rows in registers, rsqrt pivots), camera step
constexpr int kGsSolveWarps = 4;
__global__ void __launch_bounds__(32 * kGsSolveWarps) gs_solve(GsPair* __restrict__ gpair, const double* __restrict__ sums, int P) {
    __shared__ double sh[kGsSolveWarps][144 + 16 + 24 + 12];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int p = blockIdx.x * kGsSolveWarps + w;
    if (p >= P) return;                                     // whole warp
    GsPair& G = gpair[p];
    if (G.done) return;
    double* Ld = sh[w];
    double* x = Ld + 144 + 16 + 24;
    const double* s = sums + (size_t)p * kGsSums;
    const double lambda = G.lambda;
    const bool ok = gs_solve_warp(s, lambda, Ld, Ld + 144, Ld + 160, x, lane);
    if (lane == 0) {
        if (!G.have_cost) { G.cost = 0.5 * s[84]; G.have_cost = 1; }
        G.cost_trial = 0.0;
        for (int k = 0; k < 12; ++k) G.dc[k] = ok ? x[k] : 0.0;
        G.accepted = ok ? 1 : -1;          // -1: no step could be computed -> gs_accept raises lambda
    }
}

// step 3: point steps by back-substitution, trial parameters, trial cost
template <int kLoss>
__global__ void __launch_bounds__(kGsThreads) gs_trial(const double4* __restrict__ pts, const unsigned char* __restrict__ mask,
                                                       const int* __restrict__ pair_off, GsPair* __restrict__ gpair,
                                                       const double* __restrict__ Xcur, double* __restrict__ Xtrial, double ic,
                                                       double c2) {
    __shared__ double red;
    const int p = blockIdx.y;
    GsPair& G = gpair[p];
    if (G.done || G.accepted < 0) return;
    if (threadIdx.x == 0) red = 0.0;
    __syncthreads();
    double C1[12], dc[12], Cn[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) { C1[k] = G.C1[k]; dc[k] = G.dc[k]; Cn[k] = C1[k] + dc[k]; }
    const double lambda = G.lambda;
    const int lo = pair_off[p], hi = pair_off[p + 1];
    double cost = 0.0;
    for (int i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) {
        const double X0 = Xcur[3 * (size_t)i], X1 = Xcur[3 * (size_t)i + 1], X2 = Xcur[3 * (size_t)i + 2];
        double n0 = X0, n1 = X1, n2 = X2;
        const bool use = mask == nullptr || mask[i] != 0;
        if (use) {
            const double4 m = pts[i];
            GsPoint g;
            gs_point(C1, m, X0, X1, X2, g);
            double M[6], T[3][3], Di[6], gp[3], w[4];
            if constexpr (kLoss != LOSS_LINEAR) gs_rho<kLoss>(g, ic, c2, w);
            if (g.ok && gs_blocks_w<kLoss>(g, w, lambda, M, T, Di, gp)) {
                // delta_p = D'^-1 (-g_p - B^T dc),  (B^T dc)[c] = sum_a T[a][c] (dc[a, :] . Xh)
                double q[3];
#pragma unroll
                for (int a = 0; a < 3; ++a)
                    q[a] = dc[4 * a] * g.Xh[0] + dc[4 * a + 1] * g.Xh[1] + dc[4 * a + 2] * g.Xh[2] + dc[4 * a + 3];
                double rp[3];
#pragma unroll
                for (int c = 0; c < 3; ++c) rp[c] = -gp[c] - (T[0][c] * q[0] + T[1][c] * q[1] + T[2][c] * q[2]);
                n0 += Di[0] * rp[0] + Di[1] * rp[1] + Di[2] * rp[2];
                n1 += Di[1] * rp[0] + Di[3] * rp[1] + Di[4] * rp[2];
                n2 += Di[2] * rp[0] + Di[4] * rp[1] + Di[5] * rp[2];
                GsPoint t;
                gs_point(Cn, m, n0, n1, n2, t);
                if constexpr (kLoss == LOSS_LINEAR)
                    cost += t.ok ? t.rl[0] * t.rl[0] + t.rl[1] * t.rl[1] + t.rr[0] * t.rr[0] + t.rr[1] * t.rr[1] : INFINITY;
                else
                    cost += t.ok ? gs_rho<kLoss>(t, ic, c2, w) : INFINITY;
            }
        }
        Xtrial[3 * (size_t)i] = n0; Xtrial[3 * (size_t)i + 1] = n1; Xtrial[3 * (size_t)i + 2] = n2;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cost += __shfl_xor_sync(0xffffffffu, cost, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(&red, cost);
    __syncthreads();
    if (threadIdx.x == 0) atomicAdd(&G.cost_trial, 0.5 * red);
}

// step 4 (one thread per pair): accept / reject, damping schedule, convergence, clear the sums
__global__ void __launch_bounds__(32) gs_accept(GsPair* __restrict__ gpair, double* __restrict__ sums, int P, double ftol,
                                                int max_iter, int* __restrict__ n_active) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    GsPair& G = gpair[p];
    if (G.done) return;
    for (int k = 0; k < kGsSums; ++k) sums[(size_t)p * kGsSums + k] = 0.0;
    G.iters += 1;
    const bool better = G.accepted > 0 && G.cost_trial < G.cost;      // NaN / Inf trial cost: not better
    if (better) {
        const double gain = G.cost - G.cost_trial;
        for (int k = 0; k < 12; ++k) G.C1[k] += G.dc[k];
        const bool conv = gain <= ftol * G.cost;
        G.cost = G.cost_trial;
        G.lambda = fmax(G.lambda * 0.1, 1e-15);
        G.accepted = 1;                          // gs_accumulate commits X_trial
        if (conv) G.done = 2;                    // converged: one more commit pass is done by gs_finish
    } else {
        G.accepted = 0;
        G.lambda *= 10.0;
        if (G.lambda > 1e12) G.done = 3;         // no descent direction found any more: current point is kept
    }
    if (!G.done && G.iters >= max_iter) G.done = 4;
    if (n_active != nullptr && !G.done) atomicAdd(n_active, 1);      // host-paced loop: pairs still running after this iteration
}

// after the loop: commit a last accepted trial, export the camera
__global__ void __launch_bounds__(kGsThreads) gs_finish(const int* __restrict__ pair_off, const GsPair* __restrict__ gpair,
                                                        double* __restrict__ Xcur, const double* __restrict__ Xtrial,
                                                        double* __restrict__ C1out) {
    const int p = blockIdx.y;
    const GsPair& G = gpair[p];
    if (blockIdx.x == 0 && threadIdx.x < 12) C1out[(size_t)p * 12 + threadIdx.x] = G.C1[threadIdx.x];
    if (G.accepted <= 0) return;
    const int lo = pair_off[p], hi = pair_off[p + 1];
    for (int i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) {
        Xcur[3 * (size_t)i] = Xtrial[3 * (size_t)i];
        Xcur[3 * (size_t)i + 1] = Xtrial[3 * (size_t)i + 1];
        Xcur[3 * (size_t)i + 2] = Xtrial[3 * (size_t)i + 2];
    }
}

// ------------------------------------------------------------------------------------------------
// The whole Levenberg-Marquardt loop of ONE pair in ONE CTA (pairs of up to a few thousand correspondences: the
// reference's own case has 257): no launch per step, no atomics, every sum in a fixed order.  Per iteration:
//   linearise the points in chunks of kGsFusedThreads into shared-memory records (W = M - T D'^-1 T^T, Xh, z, diag M);
//   3 x 84 entry threads add W (x) Xh Xh^T, z (x) Xh, diag(M) (x) Xh^2 over the chunk; warp 0 solves the 12x12 system;
//   all threads take the point steps and the trial cost; thread 0 accepts / rejects.  Accepted points are swapped in by
//   exchanging the roles of the two point buffers.  grid = P.
// ------------------------------------------------------------------------------------------------
constexpr int kGsFusedThreads = 256;
constexpr int kGsFusedMaxPts = 4096;      // per pair; larger pairs use the multi-kernel path (more than one SM per pair)
constexpr int kGsRec = 15;                // W (6) | X (3) | z (3) | M00, M11, M22

__device__ __forceinline__ double gs_block_sum(double v, double* sh) {      // fixed tree; result in every thread
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sh[w];
    return s;
}

template <int kLoss>
__global__ void __launch_bounds__(kGsFusedThreads) gs_fused(const double4* __restrict__ pts, const unsigned char* __restrict__ mask,
                                                            const int* __restrict__ pair_off, GsPair* __restrict__ gpair,
                                                            double* __restrict__ Xa, double* __restrict__ Xb,
                                                            double* __restrict__ C1out, double ftol, int max_iter, double ic,
                                                            double c2) {
    __shared__ double rec[kGsFusedThreads * kGsRec];
    __shared__ double part[3][84];
    __shared__ double sums[kGsSums];
    __shared__ double solve_ws[144 + 16 + 24 + 12];
    __shared__ double red[kGsFusedThreads / 32];
    __shared__ double sC1[12], sdc[12];
    __shared__ double s_lambda, s_cost;
    __shared__ int s_done, s_ok, s_iters;
    const int p = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    GsPair& G = gpair[p];
    const int lo = pair_off[p], hi = pair_off[p + 1];
    if (tid < 12) sC1[tid] = G.C1[tid];
    if (tid == 0) { s_lambda = G.lambda; s_done = G.done; s_iters = 0; s_cost = 0.0; }
    __syncthreads();
    double* Xc = Xa;                                        // current points / trial points (roles swap on acceptance)
    double* Xt = Xb;
    const int grp = tid / 84, ent = tid - 84 * grp;         // entry threads: 3 groups x 84 sums (tid < 252)
    // static description of the entry owned by this thread
    int e_w = 0, e_a = 0, e_b = 0, e_kind = -1;             // kind 0: W[e_w] Xh[e_a] Xh[e_b]; 1: z[e_w] Xh[e_a]; 2: Md[e_w] Xh[e_a]^2
    if (grp < 3) {
        if (ent < 60) {
            e_kind = 0; e_w = ent / 10;
            const int x = ent - 10 * e_w;
            const int a4[10] = {0, 0, 0, 0, 1, 1, 1, 2, 2, 3}, b4[10] = {0, 1, 2, 3, 1, 2, 3, 2, 3, 3};
            e_a = a4[x]; e_b = b4[x];
        } else if (ent < 72) { e_kind = 1; e_w = (ent - 60) >> 2; e_a = (ent - 60) & 3; }
        else { e_kind = 2; e_w = (ent - 72) >> 2; e_a = (ent - 72) & 3; }
    }
    bool have_cost = false;
    for (int it = 0; it < max_iter && !s_done; ++it) {
        double C1[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) C1[k] = sC1[k];
        const double lambda = s_lambda;
        // ---- accumulate ---------------------------------------------------------------------------------------
        double acc = 0.0, cost = 0.0;
        for (int base = lo; base < hi; base += kGsFusedThreads) {
            const int i = base + tid;
            double* r = rec + tid * kGsRec;
            bool used = false;
            if (i < hi && (mask == nullptr || mask[i] != 0)) {
                GsPoint g;
                gs_point(C1, pts[i], Xc[3 * (size_t)i], Xc[3 * (size_t)i + 1], Xc[3 * (size_t)i + 2], g);
                double M[6], T[3][3], Di[6], gp[3], w[4], rc = 0.0;
                if constexpr (kLoss != LOSS_LINEAR) rc = gs_rho<kLoss>(g, ic, c2, w);
                if (g.ok && gs_blocks_w<kLoss>(g, w, lambda, M, T, Di, gp)) {
                    double TD[3][3];
#pragma unroll
                    for (int a = 0; a < 3; ++a)
#pragma unroll
                        for (int c = 0; c < 3; ++c)
                            TD[a][c] = T[a][0] * Di[sym3(0, c)] + T[a][1] * Di[sym3(1, c)] + T[a][2] * Di[sym3(2, c)];
#pragma unroll
                    for (int a = 0; a < 3; ++a) {
#pragma unroll
                        for (int b = a; b < 3; ++b)
                            r[sym3(a, b)] = M[sym3(a, b)] - (TD[a][0] * T[b][0] + TD[a][1] * T[b][1] + TD[a][2] * T[b][2]);
                        r[9 + a] = g.P2[0][a] * g.rl[0] + g.P2[1][a] * g.rl[1] + TD[a][0] * gp[0] + TD[a][1] * gp[1] + TD[a][2] * gp[2];
                        r[12 + a] = M[sym3(a, a)];
                        r[6 + a] = g.Xh[a];
                    }
                    if constexpr (kLoss == LOSS_LINEAR) cost += g.rl[0] * g.rl[0] + g.rl[1] * g.rl[1] + g.rr[0] * g.rr[0] + g.rr[1] * g.rr[1];
                    else cost += rc;
                    used = true;
                }
            }
            if (!used) {
#pragma unroll
                for (int k = 0; k < kGsRec; ++k) r[k] = 0.0;
            }
            __syncthreads();
            if (e_kind >= 0) {
                const int n = min(kGsFusedThreads, hi - base);
                for (int q = grp; q < n; q += 3) {
                    const double* rq = rec + q * kGsRec;
                    const double xa = e_a < 3 ? rq[6 + e_a] : 1.0;
                    if (e_kind == 0) acc = fma(rq[e_w] * xa, e_b < 3 ? rq[6 + e_b] : 1.0, acc);
                    else if (e_kind == 1) acc = fma(rq[9 + e_w], xa, acc);
                    else acc = fma(rq[12 + e_w] * xa, xa, acc);
                }
            }
            __syncthreads();
        }
        if (e_kind >= 0) part[grp][ent] = acc;
        const double csum = gs_block_sum(cost, red);        // (contains the barriers that publish part[][])
        if (tid < 84) sums[tid] = (part[0][tid] + part[1][tid]) + part[2][tid];
        if (tid == 0 && !have_cost) s_cost = 0.5 * csum;
        have_cost = true;
        __syncthreads();
        // ---- solve --------------------------------------------------------------------------------------------
        if (warp == 0) {
            double* x = solve_ws + 144 + 16 + 24;
            const bool ok = gs_solve_warp(sums, lambda, solve_ws, solve_ws + 144, solve_ws + 160, x, lane);
            if (lane < 12) sdc[lane] = ok ? x[lane] : 0.0;
            if (lane == 0) s_ok = ok ? 1 : 0;
        }
        __syncthreads();
        // ---- trial --------------------------------------------------------------------------------------------
        double tcost = 0.0;
        if (s_ok) {
            double dc[12], Cn[12];
#pragma unroll
            for (int k = 0; k < 12; ++k) { dc[k] = sdc[k]; Cn[k] = C1[k] + dc[k]; }
            for (int i = lo + tid; i < hi; i += kGsFusedThreads) {
                const double X0 = Xc[3 * (size_t)i], X1 = Xc[3 * (size_t)i + 1], X2 = Xc[3 * (size_t)i + 2];
                double n0 = X0, n1 = X1, n2 = X2;
                if (mask == nullptr || mask[i] != 0) {
                    const double4 m = pts[i];
                    GsPoint g;
                    gs_point(C1, m, X0, X1, X2, g);
                    double M[6], T[3][3], Di[6], gp[3], w[4];
                    if constexpr (kLoss != LOSS_LINEAR) gs_rho<kLoss>(g, ic, c2, w);
                    if (g.ok && gs_blocks_w<kLoss>(g, w, lambda, M, T, Di, gp)) {
                        double q[3];
#pragma unroll
                        for (int a = 0; a < 3; ++a)
                            q[a] = dc[4 * a] * g.Xh[0] + dc[4 * a + 1] * g.Xh[1] + dc[4 * a + 2] * g.Xh[2] + dc[4 * a + 3];
                        double rp[3];
#pragma unroll
                        for (int c = 0; c < 3; ++c) rp[c] = -gp[c] - (T[0][c] * q[0] + T[1][c] * q[1] + T[2][c] * q[2]);
                        n0 += Di[0] * rp[0] + Di[1] * rp[1] + Di[2] * rp[2];
                        n1 += Di[1] * rp[0] + Di[3] * rp[1] + Di[4] * rp[2];
                        n2 += Di[2] * rp[0] + Di[4] * rp[1] + Di[5] * rp[2];
                        GsPoint t;
                        gs_point(Cn, m, n0, n1, n2, t);
                        if constexpr (kLoss == LOSS_LINEAR)
                            tcost += t.ok ? t.rl[0] * t.rl[0] + t.rl[1] * t.rl[1] + t.rr[0] * t.rr[0] + t.rr[1] * t.rr[1] : INFINITY;
                        else
                            tcost += t.ok ? gs_rho<kLoss>(t, ic, c2, w) : INFINITY;
                    }
                }
                Xt[3 * (size_t)i] = n0; Xt[3 * (size_t)i + 1] = n1; Xt[3 * (size_t)i + 2] = n2;
            }
        }
        const double ct = 0.5 * gs_block_sum(tcost, red);
        // ---- accept (every thread evaluates the same decision from shared state) --------------------------------
        const double cur = s_cost;
        const bool better = s_ok && ct < cur;                // NaN / Inf trial cost: not better
        __syncthreads();
        if (better) {
            if (tid < 12) sC1[tid] += sdc[tid];
            double* sw = Xc; Xc = Xt; Xt = sw;
        }
        if (tid == 0) {
            s_iters = it + 1;
            if (better) {
                const bool conv = (cur - ct) <= ftol * cur;
                s_cost = ct;
                s_lambda = fmax(lambda * 0.1, 1e-15);
                if (conv) s_done = 2;
            } else {
                s_lambda = lambda * 10.0;
                if (s_lambda > 1e12) s_done = 3;
            }
            if (!s_done && it + 1 >= max_iter) s_done = 4;
        }
        __syncthreads();
    }
    // results: points in Xa, camera, state
    if (Xc != Xa)
        for (int i = 3 * lo + tid; i < 3 * hi; i += kGsFusedThreads) Xa[i] = Xc[i];
    if (tid < 12) { C1out[(size_t)p * 12 + tid] = sC1[tid]; G.C1[tid] = sC1[tid]; }
    if (tid == 0) {
        G.lambda = s_lambda; G.cost = s_cost; G.have_cost = have_cost ? 1 : G.have_cost;
        G.iters = s_iters; G.done = s_done; G.accepted = 0;
    }
}

__global__ void __launch_bounds__(64) gs_export(const GsPair* __restrict__ gpair, int P, double* __restrict__ cost,
                                                int* __restrict__ iters, int* __restrict__ status) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    if (cost) cost[p] = gpair[p].have_cost ? gpair[p].cost : __longlong_as_double(0x7ff8000000000000ll);
    if (iters) iters[p] = gpair[p].iters;
    if (status) status[p] = gpair[p].done;
}

// lab3.fmatrix_residuals_gs (lab3.py:230-266) for one pair: out = [leftx (N), lefty (N), rightx (N), righty (N)]
__global__ void __launch_bounds__(256) gs_residuals(const double* __restrict__ params, const double* __restrict__ pl,
                                                    const double* __restrict__ pr, int N, double* __restrict__ out) {
    double C1[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) C1[k] = params[k];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        const double X0 = params[12 + 3 * (size_t)i], X1 = params[13 + 3 * (size_t)i], X2 = params[14 + 3 * (size_t)i];
        GsPoint g;
        gs_point(C1, make_double4(pl[i], pl[N + i], pr[i], pr[N + i]), X0, X1, X2, g);
        out[i] = g.rl[0]; out[N + i] = g.rl[1]; out[2 * (size_t)N + i] = g.rr[0]; out[3 * (size_t)N + i] = g.rr[1];
    }
}

}  // namespace rg
