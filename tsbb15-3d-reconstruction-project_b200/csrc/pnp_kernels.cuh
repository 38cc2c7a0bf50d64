// Device code of the PnP-RANSAC path (sm_100a).
//
// Reference behaviour being restated (the reference code for this path does not run, SURVEY.md section 8a rows a7/a8):
//   pnp.py:132-152    DLT pose: rows vec(r_l x_k^T), r_l rows of [y_k]_x -> A (3m x 12); c0 = smallest right singular
//                     vector -> C0 = (A|b); tau = sign det A; tau A = U S V^T; R = U V^T; t = (3 tau / tr S) b
//   ransac.py:96-111  y' = R x + t for every correspondence; e = |pnorm(y) - pnorm(y')|^2; member iff thresh >= e;
//                     keep the pose with the largest consensus
//
// Kernels: pnp_bbox_init / pnp_bbox / pnp_frame / pnp_normalise, pnp_solve_rows<n> (default) or pnp_solve_jacobi<n>,
//          score_packed<PnpPolicy>, fixup_list<PnpFix>, pnp_score_fp64, argmax_counts, pnp_finish.
#pragma once
#include "f_kernels.cuh"
#include "jacobi.cuh"

namespace rg {

// FP32 scoring frame of one view:  X' = (X - cX)/sX (|X'| <= 1),  y^ = (y - cy)/sqrt(thr2)  (|y^| <= By)
struct PnpFrame {
    double cX[3], sX;
    double cy[2], sthr;
    double By, thr2;
};

// ------------------------------------------------------------------------------------------------
// exact (FP64) membership test, ransac.py:31-35 + 96-105
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double pnp_err64(const double* __restrict__ Rt /* R row-major (9) then t (3) */, double X0,
                                            double X1, double X2, double y0, double y1) {
    const double p0 = Rt[0] * X0 + Rt[1] * X1 + Rt[2] * X2 + Rt[9];
    const double p1 = Rt[3] * X0 + Rt[4] * X1 + Rt[5] * X2 + Rt[10];
    const double p2 = Rt[6] * X0 + Rt[7] * X1 + Rt[8] * X2 + Rt[11];
    const double a = y0 - p0 / p2;
    const double b = y1 - p1 / p2;
    return a * a + b * b;
}
__device__ __forceinline__ int pnp_inlier64(const double* __restrict__ Rt, double X0, double X1, double X2, double y0,
                                            double y1, double thr2) {
    return thr2 >= pnp_err64(Rt, X0, X1, X2, y0, y1) ? 1 : 0;      // inclusive, NaN -> not a member
}

// FP32 criterion in the view's frame:  q = a^2 + b^2 - w^2  (<= 0  <=>  member); scalar twin of PnpPolicy::eval2
__device__ __forceinline__ float pnp_q32(const float* __restrict__ p, float X0, float X1, float X2, float y0, float y1) {
    const float w  = __fmaf_rn(p[8], X0, __fmaf_rn(p[9], X1, __fmaf_rn(p[10], X2, p[11])));
    const float p0 = __fmaf_rn(p[0], X0, __fmaf_rn(p[1], X1, __fmaf_rn(p[2], X2, p[3])));
    const float p1 = __fmaf_rn(p[4], X0, __fmaf_rn(p[5], X1, __fmaf_rn(p[6], X2, p[7])));
    const float a = __fmaf_rn(y0, w, p0);
    const float b = __fmaf_rn(y1, w, p1);
    const float t2 = __fmaf_rn(b, b, __fmul_rn(a, a));
    return __fmaf_rn(-w, w, t2);
}

// ------------------------------------------------------------------------------------------------
// frame + packed FP32 points:  pair (a,b) = [X0a X0b X1a X1b] [X2a X2b y0a y0b] [y1a y1b 0 0]
// ------------------------------------------------------------------------------------------------
__global__ void pnp_bbox_init(int* __restrict__ bbox, int V) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < V * 10) bbox[i] = ((i % 10) < 5) ? 0x7FFFFFFF : (int)0x80000000;
}

// bounding box of the voting correspondences of every view (grid.y = view)
__global__ void __launch_bounds__(256) pnp_bbox(const double* __restrict__ X, const double* __restrict__ y,
                                                 const PairInfo* __restrict__ pi, int* __restrict__ bbox) {
    const int v = blockIdx.y;
    const PairInfo info = pi[v];
    float mn[5], mx[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) { mn[k] = INFINITY; mx[k] = -INFINITY; }
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < info.n; i += gridDim.x * blockDim.x) {
        const size_t g = (size_t)info.pt_off + i;
        const double c[5] = {X[3 * g], X[3 * g + 1], X[3 * g + 2], y[2 * g], y[2 * g + 1]};
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            if (isfinite(c[k])) {
                mn[k] = fminf(mn[k], __double2float_rd(c[k]));
                mx[k] = fmaxf(mx[k], __double2float_ru(c[k]));
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 5; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mn[k] = fminf(mn[k], __shfl_xor_sync(0xffffffffu, mn[k], o));
            mx[k] = fmaxf(mx[k], __shfl_xor_sync(0xffffffffu, mx[k], o));
        }
    }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            atomicMin(&bbox[v * 10 + k], f2key(mn[k]));
            atomicMax(&bbox[v * 10 + 5 + k], f2key(mx[k]));
        }
    }
}

__global__ void pnp_frame(PnpFrame* __restrict__ fr, const int* __restrict__ bbox, int V, double thr2) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= V) return;
    double c[5], half[5];
    for (int k = 0; k < 5; ++k) {
        float lo = key2f(bbox[v * 10 + k]), hi = key2f(bbox[v * 10 + 5 + k]);
        if (!(lo <= hi)) { lo = 0.f; hi = 0.f; }
        c[k] = 0.5 * ((double)lo + (double)hi);
        half[k] = fmax((double)hi - c[k], c[k] - (double)lo);
    }
    PnpFrame f;
    f.cX[0] = c[0]; f.cX[1] = c[1]; f.cX[2] = c[2];
    f.sX = fmax(fmax(half[0], half[1]), half[2]) * (1.0 + 1e-6) + 1e-300;
    f.cy[0] = c[3]; f.cy[1] = c[4];
    f.sthr = sqrt(thr2);
    f.By = fmax(half[3], half[4]) / f.sthr * (1.0 + 1e-6) + 1e-30;
    f.thr2 = thr2;
    fr[v] = f;
}

__global__ void __launch_bounds__(256) pnp_normalise(const double* __restrict__ X, const double* __restrict__ y,
                                                      const PairInfo* __restrict__ pi, const PnpFrame* __restrict__ frp,
                                                      float4* __restrict__ out) {
    const int v = blockIdx.y;
    const PairInfo info = pi[v];
    const PnpFrame fr = frp[v];
    const float qnan = __int_as_float(0x7FFFFFFF);
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < info.n_pad / 2; j += gridDim.x * blockDim.x) {
        float val[2][5];
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const int i = 2 * j + s;
            if (i < info.n) {
                const size_t g = (size_t)info.pt_off + i;
                val[s][0] = (float)((X[3 * g] - fr.cX[0]) / fr.sX);
                val[s][1] = (float)((X[3 * g + 1] - fr.cX[1]) / fr.sX);
                val[s][2] = (float)((X[3 * g + 2] - fr.cX[2]) / fr.sX);
                val[s][3] = (float)((y[2 * g] - fr.cy[0]) / fr.sthr);
                val[s][4] = (float)((y[2 * g + 1] - fr.cy[1]) / fr.sthr);
            } else {
#pragma unroll
                for (int k = 0; k < 5; ++k) val[s][k] = qnan;
            }
        }
        float4* o = out + ((size_t)info.pt_off32 / 2 + j) * 3;
        o[0] = make_float4(val[0][0], val[1][0], val[0][1], val[1][1]);
        o[1] = make_float4(val[0][2], val[1][2], val[0][3], val[1][3]);
        o[2] = make_float4(val[0][4], val[1][4], 0.f, 0.f);
    }
}

// ------------------------------------------------------------------------------------------------
// pose (FP64) -> Pose32 in the view's frame + rounding band G   (derivation: DESIGN.md "guard band", PnP)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void make_pose32(const double* __restrict__ Rt, const PnpFrame& fr, Pose32* __restrict__ out) {
    // y' = R X + t = (sX R) X' + (R cX + t)
    double row[3][4];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        row[i][0] = Rt[3 * i + 0] * fr.sX;
        row[i][1] = Rt[3 * i + 1] * fr.sX;
        row[i][2] = Rt[3 * i + 2] * fr.sX;
        row[i][3] = Rt[3 * i + 0] * fr.cX[0] + Rt[3 * i + 1] * fr.cX[1] + Rt[3 * i + 2] * fr.cX[2] + Rt[9 + i];
    }
    double q[12];
    const double inv = 1.0 / fr.sthr;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        q[j]     = (fr.cy[0] * row[2][j] - row[0][j]) * inv;      // p0' = (cy0 y'2 - y'0)/sqrt(thr2)
        q[4 + j] = (fr.cy[1] * row[2][j] - row[1][j]) * inv;
        q[8 + j] = row[2][j];
    }
    double rho0 = 0.0, rho1 = 0.0, rho2 = 0.0;
#pragma unroll
    for (int j = 0; j < 4; ++j) { rho0 += fabs(q[j]); rho1 += fabs(q[4 + j]); rho2 += fabs(q[8 + j]); }
    const double phi = fmax(fmax(fr.By * rho2 + rho0, fr.By * rho2 + rho1), rho2);
    Pose32 h;
    if (!(phi > 0.0) || !isfinite(phi)) {
        const float qnan = __int_as_float(0x7FFFFFFF);
#pragma unroll
        for (int k = 0; k < 12; ++k) h.p[k] = qnan;
        h.G = 0.f; h.pad0 = h.pad1 = h.pad2 = 0.f;
        *out = h;
        return;
    }
    const double sc = 1.0 / phi;
#pragma unroll
    for (int k = 0; k < 12; ++k) h.p[k] = (float)(q[k] * sc);
    rho0 *= sc; rho1 *= sc; rho2 *= sc;
    const double eps = 5.9604644775390625e-08;
    const double A0 = fr.By * rho2 + rho0, A1 = fr.By * rho2 + rho1;
    const double G = 1.25 * 14.0 * eps * rho2 * (A0 + A1) +
                     2.0 * (49.0 * eps * eps * (A0 * A0 + A1 * A1) + 16.0 * eps * rho2 * rho2 + 25.0 * eps * eps * rho2 * rho2);
    h.G = __double2float_ru(G);
    if (!(rho2 * rho2 > 1e-28) || !(fr.By < 1e12)) h.G = INFINITY;      // FP32 underflow range: recheck everything in FP64
    h.pad0 = h.pad1 = h.pad2 = 0.f;
    *out = h;
}

__global__ void __launch_bounds__(256) pnp_make_pose32(const double* __restrict__ pose64, const PairInfo* __restrict__ pi,
                                                        int V, int H, const PnpFrame* __restrict__ fr,
                                                        Pose32* __restrict__ pose32) {
    const int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= H) return;
    int lo = 0, hi = V;
    while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (pi[mid].hyp_off <= h) lo = mid; else hi = mid; }
    double Rt[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) Rt[k] = pose64[(size_t)h * 12 + k];
    make_pose32(Rt, fr[lo], pose32 + h);
}

// ------------------------------------------------------------------------------------------------
// constraint enforcement C0 = (A|b) -> (R|t)    pnp.py:147-151
// ------------------------------------------------------------------------------------------------
template <bool FAST = false>
__device__ __forceinline__ void jacobi3(double (&w)[3][3], double (&v)[3][3]) {
    for (int sweep = 0; sweep < 14; ++sweep) {
        bool rotated = false;
#pragma unroll
        for (int pq = 0; pq < 3; ++pq) {
            const int p = (pq == 2) ? 1 : 0;
            const int q = (pq == 0) ? 1 : 2;
            const double a = w[p][0] * w[p][0] + w[p][1] * w[p][1] + w[p][2] * w[p][2];
            const double b = w[q][0] * w[q][0] + w[q][1] * w[q][1] + w[q][2] * w[q][2];
            const double g = w[p][0] * w[q][0] + w[p][1] * w[q][1] + w[p][2] * w[q][2];
            if (FAST ? (g * g > 1e-32 * (a * b)) : (g != 0.0 && fabs(g) > 1e-16 * sqrt(a * b))) {
                double c, s;
                if (FAST) jacobi_rot_fast(a, b, g, c, s); else jacobi_rot(a, b, g, c, s);
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    const double wp = w[p][i], wq = w[q][i];
                    w[p][i] = c * wp - s * wq;
                    w[q][i] = s * wp + c * wq;
                    const double vp = v[p][i], vq = v[q][i];
                    v[p][i] = c * vp - s * vq;
                    v[q][i] = s * vp + c * vq;
                }
                rotated = true;
            }
        }
        if (!rotated) break;
    }
}

__device__ __forceinline__ void cross3(const double* a, const double* b, double* o) {
    o[0] = a[1] * b[2] - a[2] * b[1];
    o[1] = a[2] * b[0] - a[0] * b[2];
    o[2] = a[0] * b[1] - a[1] * b[0];
}

// c0: 12-vector (row-major 3x4).  Rt: R row-major then t.  Returns false if the result is not finite.
template <bool FAST = false>
__device__ __forceinline__ bool enforce_pose(const double* __restrict__ c0, double* __restrict__ Rt) {
    const double A[9] = {c0[0], c0[1], c0[2], c0[4], c0[5], c0[6], c0[8], c0[9], c0[10]};
    const double det = A[0] * (A[4] * A[8] - A[5] * A[7]) - A[1] * (A[3] * A[8] - A[5] * A[6]) +
                       A[2] * (A[3] * A[7] - A[4] * A[6]);
    const double tau = det > 0.0 ? 1.0 : (det < 0.0 ? -1.0 : 0.0);
    double w[3][3], v[3][3];
#pragma unroll
    for (int j = 0; j < 3; ++j)
#pragma unroll
        for (int i = 0; i < 3; ++i) { w[j][i] = tau * A[3 * i + j]; v[j][i] = (i == j) ? 1.0 : 0.0; }
    jacobi3<FAST>(w, v);
    double sg[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) sg[j] = sqrt(w[j][0] * w[j][0] + w[j][1] * w[j][1] + w[j][2] * w[j][2]);
    // the two dominant singular pairs; the third direction follows from orthogonality (det(tau A) > 0 => proper R)
    int i3 = 0;
    if (sg[1] < sg[i3]) i3 = 1;
    if (sg[2] < sg[i3]) i3 = 2;
    double u1[3], u2[3], v1[3], v2[3];
    double s1 = 0.0, s2 = 0.0;
    {
        int cnt = 0;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            if (j == i3) continue;
            double* u = cnt == 0 ? u1 : u2;
            double* vv = cnt == 0 ? v1 : v2;
            const double inv = 1.0 / sg[j];
            u[0] = w[j][0] * inv; u[1] = w[j][1] * inv; u[2] = w[j][2] * inv;
            vv[0] = v[j][0]; vv[1] = v[j][1]; vv[2] = v[j][2];
            if (cnt == 0) s1 = sg[j]; else s2 = sg[j];
            ++cnt;
        }
    }
    double u3[3], v3[3];
    cross3(u1, u2, u3);
    cross3(v1, v2, v3);
    const double lam = 3.0 * tau / (s1 + s2 + sg[i3]);
    bool ok = true;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const double r = u1[i] * v1[j] + u2[i] * v2[j] + u3[i] * v3[j];
            Rt[3 * i + j] = r;
            ok = ok && isfinite(r);
        }
    Rt[9] = lam * c0[3]; Rt[10] = lam * c0[7]; Rt[11] = lam * c0[11];
    ok = ok && isfinite(Rt[9]) && isfinite(Rt[10]) && isfinite(Rt[11]);
    return ok;
}

// ------------------------------------------------------------------------------------------------
// minimal-sample DLT-PnP: one hypothesis per 16-lane group, register-resident one-sided Jacobi on the 3n x 12 matrix
// ------------------------------------------------------------------------------------------------
template <int NPTS>
__global__ void __launch_bounds__(kJacobiThreads) pnp_solve_jacobi(const double* __restrict__ X, const double* __restrict__ y,
                                                                    const int* __restrict__ idx,
                                                                    const PairInfo* __restrict__ pi, int V, int H,
                                                                    const PnpFrame* __restrict__ fr,
                                                                    double* __restrict__ pose64, Pose32* __restrict__ pose32,
                                                                    unsigned char* __restrict__ flags) {
    constexpr int ROWS = 3 * NPTS;
    const int lane = threadIdx.x & 31;
    const int j = lane & 15;
    const int base = lane & 16;
    const int hq = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    const bool live = hq < H;
    const int h = live ? hq : H - 1;
    int view = 0;
    {
        int lo = 0, hi = V;
        while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (pi[mid].hyp_off <= h) lo = mid; else hi = mid; }
        view = lo;
    }
    const int N = pi[view].n_all;
    const size_t pbase = (size_t)pi[view].pt_off;
    const int ca = (j < 12) ? j / 4 : 0;       // which row of C0 this column multiplies
    const int cb = j & 3;                      // which component of the homogeneous world point

    double w[ROWS], v[12];
    bool bad_index = false;
#pragma unroll
    for (int k = 0; k < NPTS; ++k) {
        int q = idx[(size_t)h * NPTS + k];
        bad_index = bad_index || q < 0 || q >= N;                 // reported through flag bit 2 / the call's status
        q = q < 0 ? 0 : (q >= N ? N - 1 : q);
        const size_t gq = pbase + q;
        const double Xh[4] = {X[3 * gq], X[3 * gq + 1], X[3 * gq + 2], 1.0};
        const double y0 = y[2 * gq], y1 = y[2 * gq + 1];
        const double xb = cb == 0 ? Xh[0] : (cb == 1 ? Xh[1] : (cb == 2 ? Xh[2] : 1.0));
        // rows of [y]_x for y = (y0, y1, 1):  r0 = (0,-1,y1)  r1 = (1,0,-y0)  r2 = (-y1,y0,0)
        const double r0 = ca == 0 ? 0.0 : (ca == 1 ? -1.0 : y1);
        const double r1 = ca == 0 ? 1.0 : (ca == 1 ? 0.0 : -y0);
        const double r2 = ca == 0 ? -y1 : (ca == 1 ? y0 : 0.0);
        const bool col = j < 12;
        w[3 * k + 0] = col ? r0 * xb : 0.0;
        w[3 * k + 1] = col ? r1 * xb : 0.0;
        w[3 * k + 2] = col ? r2 * xb : 0.0;
    }
#pragma unroll
    for (int i = 0; i < 12; ++i) v[i] = (i == j) ? 1.0 : 0.0;

    GroupJacobi<ROWS, 12>::run(w, v, j, base);
    double s0, s1, smax;
    const int jm = GroupJacobi<ROWS, 12>::smallest(w, j, s0, s1, smax);
    double c0[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) c0[i] = __shfl_sync(0xffffffffu, v[i], base + jm);
    double Rt[12];
    const bool ok = enforce_pose(c0, Rt);
    if (live && j == 0) {
#pragma unroll
        for (int k = 0; k < 12; ++k) pose64[(size_t)h * 12 + k] = Rt[k];
        unsigned char fl = 0;
        // minimiser not unique: sigma_11 ~ sigma_12 relative to sigma_1
        if (!(sqrt(s1) - sqrt(s0) > 1e-9 * sqrt(smax))) fl |= 1;
        if (!ok) fl |= 2;
        if (bad_index) fl |= 4;                   // a sample index outside [0, N) of the view: clamped, the host call fails
        flags[h] = fl;
        make_pose32(Rt, fr[view], pose32 + h);
    }
}

// ------------------------------------------------------------------------------------------------
// minimal-sample DLT-PnP, default solver (round 2): SIX LANES per hypothesis, matrices in shared memory, no shuffles in
// the rotation loop.
//   1. the 3n x 12 design matrix is written to shared memory (one sample point per lane) and reduced to its triangular
//      factor R by Householder reflections, every lane owning two columns (backward stable; 12 short steps);
//   2. the ROWS of R are orthogonalised by one-sided Jacobi rotations (= Hestenes on R^T): at convergence row i is
//      sigma_i v_i^T — the right singular vectors of A scaled by the singular values — so no V is accumulated and a
//      rotation touches 2 x 12 doubles instead of 2 x (18 + 12).  A sweep is a round-robin tournament of 11 rounds x 6
//      DISJOINT pairs: lane l rotates pair l of the round, all six in parallel, one __syncwarp per round;
//   3. the minimiser c0 = v_12 is the normalised smallest row; when that row is below 1e-4 sigma_1 (exact data: it is pure
//      rounding noise) c0 is instead the unit vector orthogonal to the other eleven rows (projection of the best coordinate
//      vector, applied twice), which has the same eps * sigma_1 / gap accuracy as any SVD.
// Rotations use jacobi_rot_fast: the angle comes from 20-bit reciprocal seeds, c and s are exact functions of it, so the
// transformation stays orthogonal to rounding and only the convergence path changes (the exact formula's two divisions and
// two square roots were two thirds of a rotation's dependent chain).
// History (B200, 8192 hypotheses, config 4): 16-lane group Jacobi on the 18 x 12 matrix with V (round 1, 60 SHFL per
// rotation round) 0.30 ms; one thread per hypothesis with R in shared memory 0.31 ms (exact rotations) -> 0.22 ms (fast
// rotations, three interleaved pairs): pure latency, 256 warps on 592 sub-partitions; this kernel: see DESIGN.md.
// The group Jacobi (pnp_solve_jacobi, the solver BASELINE.json names) stays selectable (rg_set_option(ctx, 7, 1)) and is
// parity-tested against this one.
// ------------------------------------------------------------------------------------------------
constexpr int kRowsLanes = 6;                          // lanes per hypothesis
constexpr int kRowsHypPerWarp = 5;                     // 30 of the 32 lanes carry hypotheses
constexpr int kRowsWarps = 4;
constexpr int kRowsThreads = 32 * kRowsWarps;
constexpr int kRowsHypPerBlock = kRowsHypPerWarp * kRowsWarps;
constexpr int kRS = 14;                                // row stride in doubles: 12 + 2 of padding, so that the 16-byte units of the
                                                       // six rows a hypothesis touches in one round fall into different bank groups
template <int NPTS> __host__ __device__ constexpr int rows_stride() { return 3 * NPTS * kRS + 30; }   // even (16-byte rows), = 5 mod 8 units
template <int NPTS> constexpr size_t rows_smem() { return (size_t)kRowsHypPerBlock * rows_stride<NPTS>() * sizeof(double); }

template <int NPTS>
__global__ void __launch_bounds__(kRowsThreads) pnp_solve_rows(const double* __restrict__ X, const double* __restrict__ y,
                                                                const int* __restrict__ idx, const PairInfo* __restrict__ pi,
                                                                int V, int H, const PnpFrame* __restrict__ fr,
                                                                double* __restrict__ pose64, Pose32* __restrict__ pose32,
                                                                unsigned char* __restrict__ flags) {
    extern __shared__ double rows_sm[];
    constexpr int ROWS = 3 * NPTS;
    constexpr int SH = rows_stride<NPTS>();
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane / kRowsLanes, l = lane - g * kRowsLanes;
    const bool act = g < kRowsHypPerWarp;                              // lanes 30, 31 only take part in the warp-wide votes
    const int hq = (blockIdx.x * kRowsWarps + warp) * kRowsHypPerWarp + g;
    const bool live = act && hq < H;
    const int h = (act && hq < H) ? hq : H - 1;
    double* A = rows_sm + (size_t)(warp * kRowsHypPerWarp + (act ? g : 0)) * SH;      // A[r][c] at A[kRS r + c]
    double* diag = A + ROWS * kRS;                                     // scratch: diag[12], nrm[12], v0, beta, normF2
    double* nrm = diag + 12;
    double* sc = nrm + 12;
    int view = 0;
    {
        int lo = 0, hi = V;
        while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (pi[mid].hyp_off <= h) lo = mid; else hi = mid; }
        view = lo;
    }
    const int N = pi[view].n_all;
    const size_t pbase = (size_t)pi[view].pt_off;

    // ---- 0. design matrix: rows r_l (x) Xh_k, r_l the rows of [y_k]_x -------------------------------------------
    if (act && l == 0) sc[2] = 0.0;
    __syncwarp();
    if (act) {
        for (int k = l; k < NPTS; k += kRowsLanes) {
            int q = idx[(size_t)h * NPTS + k];
            if (q < 0 || q >= N) sc[2] = 1.0;                          // (benign race: every writer stores the same value)
            q = q < 0 ? 0 : (q >= N ? N - 1 : q);
            RG_ASSERT(q >= 0 && q < N && view >= 0 && view < V);
            const size_t gq = pbase + q;
            const double Xh[4] = {X[3 * gq], X[3 * gq + 1], X[3 * gq + 2], 1.0};
            const double y0 = y[2 * gq], y1 = y[2 * gq + 1];
            double* r0 = A + 3 * kRS * k;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                r0[b] = 0.0;                      r0[4 + b] = -Xh[b];               r0[8 + b] = y1 * Xh[b];            // ( 0, -1,  y1)
                r0[kRS + b] = Xh[b];              r0[kRS + 4 + b] = 0.0;            r0[kRS + 8 + b] = -y0 * Xh[b];     // ( 1,  0, -y0)
                r0[2 * kRS + b] = -y1 * Xh[b];    r0[2 * kRS + 4 + b] = y0 * Xh[b]; r0[2 * kRS + 8 + b] = 0.0;         // (-y1, y0,  0)
            }
        }
    }
    __syncwarp();

    // ---- 1. Householder QR, lane l owns columns l and l + 6 --------------------------------------------------------
    for (int k = 0; k < 12; ++k) {
        if (act && l == k % kRowsLanes) {
            double ss = 0.0;
            for (int r = k; r < ROWS; ++r) { const double t = A[kRS * r + k]; ss = fma(t, t, ss); }
            const double x0 = A[kRS * k + k];
            double sigma, beta;
            if (ss > 1e-290 && ss < 1e290) {
                const double ri = rsqrt_nr(ss);
                sigma = ss * ri;
                beta = ri * rcp_nr(sigma + fabs(x0));                  // 1 / (sigma (sigma + |x0|)) = 2 / |v|^2
            } else {
                sigma = sqrt(ss);
                beta = sigma > 0.0 ? 1.0 / (sigma * (sigma + fabs(x0))) : 0.0;
            }
            diag[k] = -copysign(sigma, x0);                            // R[k][k]
            sc[0] = x0 + copysign(sigma, x0);                          // v_k (v_r = A[r][k] for r > k)
            sc[1] = beta;
        }
        __syncwarp();
        if (act) {
            const double v0 = sc[0], beta = sc[1];
            for (int c = l; c < 12; c += kRowsLanes) {
                if (c <= k) continue;
                double d = v0 * A[kRS * k + c];
                for (int r = k + 1; r < ROWS; ++r) d = fma(A[kRS * r + k], A[kRS * r + c], d);
                d *= beta;
                A[kRS * k + c] -= d * v0;
                for (int r = k + 1; r < ROWS; ++r) A[kRS * r + c] = fma(-d, A[kRS * r + k], A[kRS * r + c]);
            }
        }
        __syncwarp();
    }
    if (act) {                                                         // R in rows 0..11: diagonal in place, zeros below it
        for (int c = l; c < 12; c += kRowsLanes) {
            A[kRS * c + c] = diag[c];
            for (int r = c + 1; r < 12; ++r) A[kRS * r + c] = 0.0;
        }
    }
    __syncwarp();

    // ---- 2. one-sided Jacobi on the rows of R, rows in REGISTERS: lane l holds a "top" and a "bottom" row and rotates that
    // pair; between rounds the rows travel round the ring top_1 .. top_5, bottom_5 .. bottom_0 (top_0 fixed) — the circle
    // method: 11 rounds pair every row with every other exactly once.  The exchange is 2 x 12 doubles = 48 SHFL per round
    // for the FIVE hypotheses of the warp (round 1's group Jacobi: 60 SHFL per round for TWO).  A first version kept the
    // rows in shared memory: the loop was bound by shared-memory wavefronts (ncu: 69 % of the LSU peak, 41 % of them bank
    // conflicts, FP64 pipe 27 % busy) at 0.13 ms per 8192 hypotheses.
    double top[12], bot[12];
    double part = 0.0;
    if (act) {
        const double2* At = reinterpret_cast<const double2*>(A + kRS * l);
        const double2* Ab = reinterpret_cast<const double2*>(A + kRS * (11 - l));
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            const double2 u = At[k], w = Ab[k];
            top[2 * k] = u.x; top[2 * k + 1] = u.y; bot[2 * k] = w.x; bot[2 * k + 1] = w.y;
        }
#pragma unroll
        for (int k = 0; k < 12; ++k) part = fma(top[k], top[k], fma(bot[k], bot[k], part));
    } else {
#pragma unroll
        for (int k = 0; k < 12; ++k) { top[k] = 0.0; bot[k] = 0.0; }
    }
    const int gbase = (act ? g : kRowsHypPerWarp - 1) * kRowsLanes;
    double normF2 = 0.0;
#pragma unroll
    for (int t = 0; t < kRowsLanes; ++t) normF2 += __shfl_sync(full, part, gbase + t);
    const double tiny = 7.9e-31 * normF2;
    const int src_left = act ? g * kRowsLanes + (l + kRowsLanes - 1) % kRowsLanes : lane;
    const int src_right = act ? g * kRowsLanes + (l + 1) % kRowsLanes : lane;
    for (int sweep = 0; sweep < kJacobiMaxSweeps; ++sweep) {
        bool rotated = false;
        for (int r = 0; r < 11; ++r) {
            if (act) {
                double a0 = 0.0, a1 = 0.0, b0 = 0.0, b1 = 0.0, g0 = 0.0, g1 = 0.0;
#pragma unroll
                for (int k = 0; k < 12; k += 2) {
                    a0 = fma(top[k], top[k], a0); a1 = fma(top[k + 1], top[k + 1], a1);
                    b0 = fma(bot[k], bot[k], b0); b1 = fma(bot[k + 1], bot[k + 1], b1);
                    g0 = fma(top[k], bot[k], g0); g1 = fma(top[k + 1], bot[k + 1], g1);
                }
                const double a = a0 + a1, b = b0 + b1, gg = g0 + g1;
                const bool conv = !(gg * gg > 1e-30 * (a * b)) || !(fmin(a, b) > tiny);
                if (!conv) {
                    double c, s;
                    jacobi_rot_fast(a, b, gg, c, s);
#pragma unroll
                    for (int k = 0; k < 12; ++k) {
                        const double x = top[k], z = bot[k];
                        top[k] = c * x - s * z;
                        bot[k] = s * x + c * z;
                    }
                    // a rotation by less than 1e-8 leaves an off-diagonal below 1e-16 of the norms (quadratic convergence):
                    // a sweep of only such rotations is the last one, no verification sweep needed
                    rotated = rotated || fabs(s) > 1e-8;
                }
            }
#pragma unroll
            for (int k = 0; k < 12; ++k) {
                const double send = (l == 0) ? bot[k] : top[k];           // lane 0's top never moves: it passes its bottom on
                const double nt = __shfl_sync(full, send, src_left);
                const double nb = __shfl_sync(full, bot[k], src_right);
                const double keep = top[k];
                top[k] = (l == 0) ? keep : nt;
                bot[k] = (l == kRowsLanes - 1) ? keep : nb;
            }
        }
        if (!__any_sync(full, rotated)) break;
    }

    // ---- 3. smallest row -> c0 -> (R | t) ---------------------------------------------------------------------------
    if (act) {                                                         // rows (in whatever order they ended up) back to shared memory
        double2* At = reinterpret_cast<double2*>(A + kRS * (2 * l));
        double2* Ab = reinterpret_cast<double2*>(A + kRS * (2 * l + 1));
        double nt = 0.0, nb = 0.0;
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            At[k] = make_double2(top[2 * k], top[2 * k + 1]);
            Ab[k] = make_double2(bot[2 * k], bot[2 * k + 1]);
        }
#pragma unroll
        for (int k = 0; k < 12; ++k) { nt = fma(top[k], top[k], nt); nb = fma(bot[k], bot[k], nb); }
        nrm[2 * l] = nt;
        nrm[2 * l + 1] = nb;
    }
    __syncwarp();
    if (!(act && l == 0)) return;
    double s0 = INFINITY, s1 = INFINITY, smax = 0.0;
    int jm = 0;
    for (int i = 0; i < 12; ++i) {
        const double t = nrm[i];
        const double key = (t == t) ? t : INFINITY;
        if (key < s0) { s1 = s0; s0 = key; jm = i; }
        else if (key < s1) s1 = key;
        if (t == t) smax = fmax(smax, t);
    }
    double c0[12];
    if (s0 > 1e-8 * smax) {
        const double inv = rsqrt(s0);
#pragma unroll
        for (int k = 0; k < 12; ++k) c0[k] = A[kRS * jm + k] * inv;
    } else {
        // unit vector orthogonal to the eleven other rows; start from the coordinate vector the projector keeps best
        double dg[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) dg[k] = 1.0;
        for (int i = 0; i < 12; ++i) {
            if (i == jm || !(nrm[i] > tiny)) continue;
            const double inv = 1.0 / nrm[i];
#pragma unroll
            for (int k = 0; k < 12; ++k) { const double r = A[kRS * i + k]; dg[k] -= r * r * inv; }
        }
        int e = 0;
#pragma unroll
        for (int k = 1; k < 12; ++k) if (dg[k] > dg[e]) e = k;
#pragma unroll
        for (int k = 0; k < 12; ++k) c0[k] = (k == e) ? 1.0 : 0.0;
        for (int pass = 0; pass < 2; ++pass) {
            for (int i = 0; i < 12; ++i) {
                if (i == jm || !(nrm[i] > tiny)) continue;
                double dot = 0.0;
#pragma unroll
                for (int k = 0; k < 12; ++k) dot = fma(A[kRS * i + k], c0[k], dot);
                dot /= nrm[i];
#pragma unroll
                for (int k = 0; k < 12; ++k) c0[k] -= dot * A[kRS * i + k];
            }
        }
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 12; ++k) t = fma(c0[k], c0[k], t);
        const double inv = rsqrt(t);
#pragma unroll
        for (int k = 0; k < 12; ++k) c0[k] *= inv;
    }
    double Rt[12];
    const bool ok = enforce_pose<true>(c0, Rt);
    if (live) {
#pragma unroll
        for (int k = 0; k < 12; ++k) pose64[(size_t)h * 12 + k] = Rt[k];
        unsigned char fl = 0;
        // minimiser not unique: sigma_11 ~ sigma_12 relative to sigma_1
        if (!(sqrt(s1) - sqrt(s0) > 1e-9 * sqrt(smax))) fl |= 1;
        if (!ok) fl |= 2;
        if (sc[2] != 0.0) fl |= 4;                // a sample index outside [0, N) of the view: clamped, the host call fails
        flags[h] = fl;
        make_pose32(Rt, fr[view], pose32 + h);
    }
}

// ------------------------------------------------------------------------------------------------
// packed FP32 scorer policy for the reprojection criterion
// ------------------------------------------------------------------------------------------------
struct Pose2 { float p[12]; };

struct PnpPolicy {
    typedef Pose32 Rec;
    typedef Pose2 Regs;
    static constexpr bool kBoundOnly = false;
    static constexpr int kVec4PerPair = 3;
    static constexpr int kChunkPts = 512;       // 12 KB of points per stage (two flag words)

    __device__ static __forceinline__ void load(const Pose32* __restrict__ sh, int slot, bool valid, Pose2& out, float& G) {
        if (valid) {
            const float4* p = reinterpret_cast<const float4*>(sh + slot);
            const float4 a = p[0], b = p[1], c = p[2], d = p[3];
            const float f[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
#pragma unroll
            for (int k = 0; k < 12; ++k) out.p[k] = f[k];
            G = d.x;
        } else {
            const float qnan = __int_as_float(0x7FFFFFFF);
#pragma unroll
            for (int k = 0; k < 12; ++k) out.p[k] = qnan;
            G = 0.f;
        }
    }

    template <int K>
    __device__ static __forceinline__ void evalN(const Pose2 (&H)[K], const float4* __restrict__ pr, unsigned (&cnt)[K],
                                                 float (&minabs)[K]) {
        const float4 A = pr[0], B = pr[1];
        const float2 Cc = *reinterpret_cast<const float2*>(pr + 2);
        const float2 X0 = make_float2(A.x, A.y), X1 = make_float2(A.z, A.w), X2 = make_float2(B.x, B.y);
        const float2 y0 = make_float2(B.z, B.w), y1 = Cc;
        float2 w[K], p0[K], p1[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            w[k]  = ffma2_sbs(H[k].p[10], X2, H[k].p[11]);
            p0[k] = ffma2_sbs(H[k].p[2], X2, H[k].p[3]);
            p1[k] = ffma2_sbs(H[k].p[6], X2, H[k].p[7]);
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            w[k]  = ffma2_sbc(H[k].p[9], X1, w[k]);
            p0[k] = ffma2_sbc(H[k].p[1], X1, p0[k]);
            p1[k] = ffma2_sbc(H[k].p[5], X1, p1[k]);
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            w[k]  = ffma2_sbc(H[k].p[8], X0, w[k]);
            p0[k] = ffma2_sbc(H[k].p[0], X0, p0[k]);
            p1[k] = ffma2_sbc(H[k].p[4], X0, p1[k]);
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float2 a = __ffma2_rn(y0, w[k], p0[k]);
            const float2 b = __ffma2_rn(y1, w[k], p1[k]);
            const float2 t2 = __ffma2_rn(b, b, __fmul2_rn(a, a));
            const float2 q = __ffma2_rn(make_float2(-w[k].x, -w[k].y), w[k], t2);
            cnt[k] += __float_as_uint(q.x) >> 31;
            cnt[k] += __float_as_uint(q.y) >> 31;
            minabs[k] = fminf(minabs[k], fminf(fabsf(q.x), fabsf(q.y)));
        }
    }
};

// FP64 re-evaluation of the flagged groups (policy of fixup_scan, score_core.cuh)
struct PnpFix {
    struct Params {
        const float4* pts32; const double* X; const double* y; const Pose32* pose32; const double* pose64;
        const PairInfo* pi; int V; double thr2;
    };
    __device__ static __forceinline__ int pair_of(const Params& p, int h) {
        int lo = 0, hi = p.V;
        while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (p.pi[mid].hyp_off <= h) lo = mid; else hi = mid; }
        return lo;
    }
    __device__ static __forceinline__ int n_points(const Params& p, int view) { return p.pi[view].n; }
    __device__ static __forceinline__ void scan(const Params& p, int h, int flag, int view, unsigned& band, unsigned& sign) {
        const PairInfo& info = p.pi[view];
        const Pose32 ps = p.pose32[h];
        const float4* gp = p.pts32 + ((size_t)info.pt_off32 / 2 + (size_t)flag * (kSub / 2)) * 3;
        float4 v[kSub / 2 * 3];
#pragma unroll
        for (int j = 0; j < kSub / 2 * 3; ++j) v[j] = gp[j];
#pragma unroll
        for (int j = 0; j < kSub / 2; ++j) {
            const float4 A = v[3 * j], B = v[3 * j + 1], Cc = v[3 * j + 2];
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                const int k = 2 * j + s;
                const float q = pnp_q32(ps.p, s ? A.y : A.x, s ? A.w : A.z, s ? B.y : B.x, s ? B.w : B.z, s ? Cc.y : Cc.x);
                const bool valid = flag * kSub + k < info.n;
                band |= (valid && fabsf(q) <= ps.G ? 1u : 0u) << k;
                sign |= (__float_as_uint(q) >> 31) << k;
            }
        }
    }
    __device__ static __forceinline__ int exact(const Params& p, int h, int i, int view) {
        const size_t g = (size_t)p.pi[view].pt_off + i;
        return pnp_inlier64(p.pose64 + (size_t)h * 12, p.X[3 * g], p.X[3 * g + 1], p.X[3 * g + 2], p.y[2 * g], p.y[2 * g + 1],
                            p.thr2);
    }
};

// Plain FP64 scorer (see f_score_fp64): grid (hypothesis blocks, views, N splits)
__global__ void __launch_bounds__(128) pnp_score_fp64(const double* __restrict__ X, const double* __restrict__ y,
                                                       const PairInfo* __restrict__ pi, const double* __restrict__ pose64,
                                                       double thr2, int* __restrict__ counts) {
    __shared__ double sp[256 * 5];
    const PairInfo info = pi[blockIdx.y];
    const int hl = blockIdx.x * blockDim.x + threadIdx.x;
    if (blockIdx.x * blockDim.x >= info.H) return;
    const bool active = hl < info.H;
    double Rt[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) Rt[k] = active ? pose64[(size_t)(info.hyp_off + hl) * 12 + k] : 0.0;
    const int per = (info.n + gridDim.z - 1) / gridDim.z;
    const int n0 = min((int)blockIdx.z * per, info.n), n1 = min(n0 + per, info.n);
    int cnt = 0;
    for (int base = n0; base < n1; base += 256) {
        const int m = min(256, n1 - base);
        __syncthreads();
        for (int i = threadIdx.x; i < m; i += blockDim.x) {
            const size_t g = (size_t)info.pt_off + base + i;
            sp[5 * i + 0] = X[3 * g];
            sp[5 * i + 1] = X[3 * g + 1];
            sp[5 * i + 2] = X[3 * g + 2];
            sp[5 * i + 3] = y[2 * g];
            sp[5 * i + 4] = y[2 * g + 1];
        }
        __syncthreads();
        if (active)
            for (int i = 0; i < m; ++i)
                cnt += pnp_inlier64(Rt, sp[5 * i], sp[5 * i + 1], sp[5 * i + 2], sp[5 * i + 3], sp[5 * i + 4], thr2);
    }
    if (active && cnt) atomicAdd(&counts[info.hyp_off + hl], cnt);
}

// winner's pose + consensus mask over ALL correspondences of every view (FP64); grid (blocks, views)
__global__ void __launch_bounds__(256) pnp_finish(const double* __restrict__ X, const double* __restrict__ y,
                                                   const PairInfo* __restrict__ pi, const double* __restrict__ pose64,
                                                   const int2* __restrict__ best, double thr2,
                                                   unsigned char* __restrict__ mask, double* __restrict__ Rt_out,
                                                   int* __restrict__ best_idx, int* __restrict__ best_count) {
    const int v = blockIdx.y;
    const PairInfo info = pi[v];
    const int2 b = best[v];
    const double* src = pose64 + (size_t)(info.hyp_off + (b.x >= 0 ? b.x : 0)) * 12;
    if (blockIdx.x == 0 && threadIdx.x < 12) Rt_out[v * 12 + threadIdx.x] = b.x >= 0 ? src[threadIdx.x] : nan("");
    if (blockIdx.x == 0 && threadIdx.x == 0) { best_idx[v] = b.x; best_count[v] = b.y; }
    if (mask == nullptr) return;
    double Rt[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) Rt[k] = b.x >= 0 ? src[k] : nan("");
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < info.n_all; i += gridDim.x * blockDim.x) {
        const size_t g = (size_t)info.pt_off + i;
        mask[g] = (unsigned char)pnp_inlier64(Rt, X[3 * g], X[3 * g + 1], X[3 * g + 2], y[2 * g], y[2 * g + 1], thr2);
    }
}

}  // namespace rg
