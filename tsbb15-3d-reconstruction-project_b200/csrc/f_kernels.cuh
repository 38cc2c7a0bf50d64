// Device code of the F-matrix RANSAC path (sm_100a).
//
// Reference behaviour being reproduced (paths relative to the reference root):
//   fun.py:303-328   RANSAC loop: sample 8 -> fmatrix_stls -> fmatrix_residuals on all N -> max|d| < thr -> best
//   lab3.py:269-329  fmatrix_stls (Hartley scaling, A = [Xx Xy X Yx Yy Y x y 1], null vector, rank 2, denormalise)
//   lab3.py:188-227  fmatrix_residuals (signed point-to-epipolar-line distances in both images)
//
// Kernels (launch order of one batched call):
//   f_bbox / f_normalise                           per-pair FP32 scoring frame + NaN-padded packed FP32 points
//                                                  (bounding-box keys start at 0: cleared by the pass's one memset)
//   f8_solve_qr (or f8_solve_jacobi)               one hypothesis per thread (or 16-lane group), FP64
//   score_packed<EpiPolicy>                        FP32 fma.rn.f32x2 scorer, 2 hypotheses x 2 points per thread-step
//   fixup_list<EpiFix>                             FP64 re-evaluation of the flagged guard-band groups -> exact counts
//   argmax_counts / f_tie_stats / f_tie_resolve / f_mask   selection + winner's inlier mask (FP64)
#pragma once
#include "common.cuh"
#include "score_core.cuh"
#include "philox.cuh"

namespace rg {


// ------------------------------------------------------------------------------------------------
// exact (FP64) criterion, same formula as lab3.py:213-227 + fun.py:316-317
// ------------------------------------------------------------------------------------------------
// returns d = max(|res1|, |res2|) (EPI_MAX) or the Sampson distance; NaN propagates like numpy.
__device__ __forceinline__ double epi_dist64(const double* __restrict__ F, double x0, double x1, double y0, double y1,
                                             int mode) {
    const double l1x = F[0] * y0 + F[1] * y1 + F[2];
    const double l1y = F[3] * y0 + F[4] * y1 + F[5];
    const double l1z = F[6] * y0 + F[7] * y1 + F[8];
    const double l2x = F[0] * x0 + F[3] * x1 + F[6];
    const double l2y = F[1] * x0 + F[4] * x1 + F[7];
    const double l2z = F[2] * x0 + F[5] * x1 + F[8];
    const double s1 = l1x * l1x + l1y * l1y;
    const double s2 = l2x * l2x + l2y * l2y;
    const double r1 = l1x * x0 + l1y * x1 + l1z;
    if (mode == MODE_SAMPSON) return sqrt(r1 * r1 / (s1 + s2));
    const double r2 = l2x * y0 + l2y * y1 + l2z;
    const double d1 = fabs(r1 / sqrt(s1));
    const double d2 = fabs(r2 / sqrt(s2));
    // np.max propagates NaN (fmax would drop it)
    if (d1 != d1) return d1;
    if (d2 != d2) return d2;
    return d1 > d2 ? d1 : d2;
}

__device__ __forceinline__ int epi_inlier64(const double* __restrict__ F, double x0, double x1, double y0, double y1,
                                            double thr, int mode) {
    return epi_dist64(F, x0, x1, y0, y1, mode) < thr ? 1 : 0;   // strict <, NaN -> outlier (fun.py:317)
}

// ------------------------------------------------------------------------------------------------
// FP32 criterion in the pair's normalised frame (threshold == 1):  q = r^2 - min(s1, s2)  (< 0 <=> inlier)
// Scalar form; op-for-op the same IEEE sequence as the packed form used by the hot kernel.
// ------------------------------------------------------------------------------------------------
template <int MODE>
__device__ __forceinline__ float epi_q32(const float* __restrict__ f, const float* __restrict__ g, float x0, float x1, float y0,
                                         float y1) {
    const float l1x = __fmaf_rn(f[0], y0, __fmaf_rn(f[1], y1, f[2]));
    const float l1y = __fmaf_rn(f[3], y0, __fmaf_rn(f[4], y1, f[5]));
    const float l1z = __fmaf_rn(f[6], y0, __fmaf_rn(f[7], y1, f[8]));
    const float r   = __fmaf_rn(l1x, x0, __fmaf_rn(l1y, x1, l1z));
    const float l2x = __fmaf_rn(g[0], x0, __fmaf_rn(g[1], x1, g[2]));      // rotated image-2 normal: 3 FMA instead of 4
    const float l2y = __fmaf_rn(g[3], x1, g[4]);
    const float s1  = __fmaf_rn(l1x, l1x, __fmul_rn(l1y, l1y));
    const float s2  = __fmaf_rn(l2x, l2x, __fmul_rn(l2y, l2y));
    const float m   = (MODE == MODE_SAMPSON) ? __fadd_rn(s1, s2) : fminf(s1, s2);
    return __fmaf_rn(r, r, -m);
}

// ------------------------------------------------------------------------------------------------
// bounding boxes (FP32, rounded outwards) via ordered-key atomics
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int f2key(float f) {
    int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7FFFFFFF;
}
__device__ __forceinline__ float key2f(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7FFFFFFF); }

// unsigned monotone key, > 0 for every float except the NaN with all mantissa bits set: a zeroed array is the
// identity of atomicMax, so the bounding boxes need no initialisation kernel (the pass's memset clears them)
__device__ __forceinline__ unsigned f2ukey(float f) {
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ukey2f(unsigned k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k); }

// bbox[p*8 + k] = key(max of -coordinate k) for k < 4, key(max of coordinate k-4) for k >= 4; 0 = no finite point seen
__global__ void __launch_bounds__(256) f_bbox(const double4* __restrict__ pts, const PairInfo* __restrict__ pi,
                                               unsigned* __restrict__ bbox) {
    const int p = blockIdx.y;
    const PairInfo info = pi[p];
    float mn[4] = {INFINITY, INFINITY, INFINITY, INFINITY};
    float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < info.n; i += gridDim.x * blockDim.x) {
        const double4 v = pts[info.pt_off + i];
        const double c[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (isfinite(c[k])) {      // non-finite input can never be an inlier; keep it out of the frame
                mn[k] = fminf(mn[k], __double2float_rd(c[k]));
                mx[k] = fmaxf(mx[k], __double2float_ru(c[k]));
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mn[k] = fminf(mn[k], __shfl_xor_sync(0xffffffffu, mn[k], o));
            mx[k] = fmaxf(mx[k], __shfl_xor_sync(0xffffffffu, mx[k], o));
        }
    }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (mn[k] <= mx[k]) {       // this warp saw at least one finite value of coordinate k
                atomicMax(&bbox[p * 8 + k], f2ukey(-mn[k]));
                atomicMax(&bbox[p * 8 + 4 + k], f2ukey(mx[k]));
            }
        }
    }
}

__device__ __forceinline__ PairFrame frame_from_bbox(const unsigned* __restrict__ bb, double thr, double band_scale) {
    double c[4], half = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        float lo = 0.f, hi = 0.f;
        if (bb[k] != 0u && bb[4 + k] != 0u) { lo = -ukey2f(bb[k]); hi = ukey2f(bb[4 + k]); }
        if (!(lo <= hi)) { lo = 0.f; hi = 0.f; }          // empty pair or all points non-finite
        c[k] = 0.5 * ((double)lo + (double)hi);
        half = fmax(half, fmax((double)hi - c[k], c[k] - (double)lo));
    }
    PairFrame o;
    o.c1x = c[0]; o.c1y = c[1]; o.c2x = c[2]; o.c2y = c[3];
    o.thr = thr;
    // bound on |normalised coordinate| with head-room for the FP64 division and FP32 rounding
    o.B = (half / thr) * (1.0 + 1e-6) + 1e-30;
    o.band_scale = band_scale;
    o.pad = 0.0;
    return o;
}

// FP32 copy in the scoring frame, laid out for the packed scorer: point pair (a, b) occupies 32 bytes
//   [x0a x0b x1a x1b] [y0a y0b y1a y1b]
// Points beyond n (padding up to a multiple of kSub) are NaN: they can never count and never flag.
// Every block derives the pair's frame from the bounding box; block x == 0 also stores it for the later kernels.
__global__ void __launch_bounds__(256) f_normalise(const double4* __restrict__ pts, const PairInfo* __restrict__ pi,
                                                    const unsigned* __restrict__ bbox, double thr, double band_scale,
                                                    PairFrame* __restrict__ frames, float4* __restrict__ pts32) {
    const int p = blockIdx.y;
    const PairInfo info = pi[p];
    const PairFrame fr = frame_from_bbox(bbox + p * 8, thr, band_scale);
    if (blockIdx.x == 0 && threadIdx.x == 0) frames[p] = fr;
    const float qnan = __int_as_float(0x7FFFFFFF);
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < info.n_pad / 2; j += gridDim.x * blockDim.x) {
        float a[4], b[4];
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const int i = 2 * j + s;
            float* dst = s ? b : a;
            if (i < info.n) {
                const double4 v = pts[info.pt_off + i];
                dst[0] = (float)((v.x - fr.c1x) / fr.thr);
                dst[1] = (float)((v.y - fr.c1y) / fr.thr);
                dst[2] = (float)((v.z - fr.c2x) / fr.thr);
                dst[3] = (float)((v.w - fr.c2y) / fr.thr);
            } else {
                dst[0] = dst[1] = dst[2] = dst[3] = qnan;
            }
        }
        float4* out = pts32 + (size_t)(info.pt_off32 / 2 + j) * 2;
        out[0] = make_float4(a[0], b[0], a[1], b[1]);
        out[1] = make_float4(a[2], b[2], a[3], b[3]);
    }
}

// ------------------------------------------------------------------------------------------------
// F (pixel frame, FP64) -> Hyp32 (normalised frame, FP32) + rigorous rounding band G
// ------------------------------------------------------------------------------------------------
// Derivation in DESIGN.md ("guard band").  eps = 2^-24.  With F~ scaled so that
//   sum_ij |f_ij| w_i w_j = 1,  w = (B, B, 1)
// every partial sum of r = x~^T F~ y~ is bounded by 1, |l1x|<=rho0, |l1y|<=rho1, |l2x|<=kap0, |l2y|<=kap1 and
//   |q^ - q| <= 2 sqrt(Mb) 8eps + 64 eps^2 + 10 eps Smax + 2 eps Mb      whenever the decision could flip,
// where S1 = rho0^2+rho1^2, S2 = kap0^2+kap1^2, Mb = min(S1,S2) (EPI) or S1+S2 (Sampson), Smax likewise.
template <int MODE>
__device__ __forceinline__ void make_hyp32(const double* __restrict__ F, const PairFrame& fr, Hyp32* __restrict__ out) {
    const double t = fr.thr, B = fr.B;
    double g[9], ft[9];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        g[3 * i + 0] = F[3 * i + 0] * t;
        g[3 * i + 1] = F[3 * i + 1] * t;
        g[3 * i + 2] = F[3 * i + 0] * fr.c2x + F[3 * i + 1] * fr.c2y + F[3 * i + 2];
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        ft[0 + j] = t * g[0 + j];
        ft[3 + j] = t * g[3 + j];
        ft[6 + j] = fr.c1x * g[0 + j] + fr.c1y * g[3 + j] + g[6 + j];
    }
    const double w[3] = {B, B, 1.0};
    double phi = 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) phi += fabs(ft[3 * i + j]) * w[i] * w[j];
    Hyp32 h;
    if (!(phi > 0.0) || !isfinite(phi)) {          // zero / NaN / inf hypothesis: never an inlier anywhere
        const float qnan = __int_as_float(0x7FFFFFFF);
#pragma unroll
        for (int k = 0; k < 9; ++k) h.f[k] = qnan;
#pragma unroll
        for (int k = 0; k < 5; ++k) h.g[k] = qnan;
        h.G = 0.f; h.T = 0.f;
        *out = h;
        return;
    }
    const double inv = 1.0 / phi;
    double a[9], fd[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) { fd[k] = ft[k] * inv; a[k] = fabs(fd[k]); h.f[k] = (float)fd[k]; }
    // l2 = (f0 x0 + f3 x1 + f6, f1 x0 + f4 x1 + f7) rotated by (cos, sin) = (f0, f1) / hypot(f0, f1): the second component
    // loses its x0 term; |l2'| = |l2| exactly, so s2 and every bound on it carry over with the rotated coefficients
    double gd[5];
    {
        const double hh = sqrt(fd[0] * fd[0] + fd[1] * fd[1]);
        if (hh > 0.0) {
            const double ih = 1.0 / hh;
            gd[0] = hh;
            gd[1] = (fd[0] * fd[3] + fd[1] * fd[4]) * ih;
            gd[2] = (fd[0] * fd[6] + fd[1] * fd[7]) * ih;
            gd[3] = (fd[0] * fd[4] - fd[1] * fd[3]) * ih;
            gd[4] = (fd[0] * fd[7] - fd[1] * fd[6]) * ih;
        } else {
            gd[0] = 0.0; gd[1] = fd[3]; gd[2] = fd[6]; gd[3] = fd[4]; gd[4] = fd[7];
        }
    }
#pragma unroll
    for (int k = 0; k < 5; ++k) h.g[k] = (float)gd[k];
    const double rho0 = a[0] * B + a[1] * B + a[2];
    const double rho1 = a[3] * B + a[4] * B + a[5];
    const double kap0 = fabs(gd[0]) * B + fabs(gd[1]) * B + fabs(gd[2]);       // bounds on |l2x'|, |l2y'| over the frame
    const double kap1 = fabs(gd[3]) * B + fabs(gd[4]);
    const double S1 = rho0 * rho0 + rho1 * rho1;
    const double S2 = kap0 * kap0 + kap1 * kap1;
    const double eps = 5.9604644775390625e-08;   // 2^-24
    double Mb, Smax;
    if (MODE == MODE_SAMPSON) { Mb = S1 + S2; Smax = 1.1 * (S1 + S2); }
    else                      { Mb = fmin(S1, S2); Smax = fmax(S1, S2); }
    const double G = 1.25 * 16.0 * eps * sqrt(Mb) + 2.0 * (100.0 * eps * eps + 10.0 * eps * Smax + 2.0 * eps * Mb);
    h.G = __double2float_ru(G * fr.band_scale);
    // the bound assumes no FP32 underflow: with an extreme threshold / point spread (s1, s2 ~ 1/B^2 near the denormal
    // range) every evaluation of this hypothesis is sent to the FP64 recheck instead
    if (!(Mb > 1e-28) || !(B < 1e12)) h.G = INFINITY;
    // bound-only prefix scorer (EpiBoundPolicy): a reference inlier has q^ <= G (the band above) and m^ <= Mb (1 + eps)^14
    // + 2^-146 (coefficients rounded, |x~|, |y~| <= B, subnormal results included), so r^2 < T (DESIGN.md section 4.2).
    // G = inf gives T = inf: every evaluation counts and the pair falls back to the full sweep.
    h.T = __double2float_ru((1.0 + 0x1p-16) * Mb + (1.0 + 0x1p-20) * (double)h.G + 0x1p-126);
    *out = h;
}

template <int MODE>
__global__ void __launch_bounds__(256) f_make_hyp32(const double* __restrict__ F64, const PairInfo* __restrict__ pi,
                                                     const PairFrame* __restrict__ frames, int P, int Htot,
                                                     Hyp32* __restrict__ hyp32) {
    const int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= Htot) return;
    int lo = 0, hi = P;
    while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (pi[mid].hyp_off <= h) lo = mid; else hi = mid; }
    double F[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) F[k] = F64[(size_t)h * 9 + k];
    make_hyp32<MODE>(F, frames[lo], hyp32 + h);
}

// ------------------------------------------------------------------------------------------------
// fast reciprocal / reciprocal square root / rotation helpers of the one-thread-per-hypothesis solvers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double rcp_approx(double x) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    return y;
}
// 1/sqrt(x) to full double precision from the 20-bit hardware seed (MUFU.RSQ64H) + two Newton steps: ~10 dependent
// instructions instead of the ~60 of sqrt() followed by a division.  x > 0, normal range.
__device__ __forceinline__ double rsqrt_nr(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double hx = 0.5 * x;
    y = y * fma(-hx * y, y, 1.5);
    y = y * fma(-hx * y, y, 1.5);
    return y;
}
// 1/x to full double precision: 20-bit seed (MUFU.RCP64H) + two Newton steps.  x finite, normal, non-zero.
__device__ __forceinline__ double rcp_nr(double x) {
    double y = rcp_approx(x);
    y = y * fma(-x, y, 2.0);
    y = y * fma(-x, y, 2.0);
    return y;
}
// Jacobi rotation for the thread-per-hypothesis solvers.  Any rotation with c^2 + s^2 = 1 (to rounding) keeps the
// iteration an orthogonal transformation, so only c and s = c t have to be exact functions of t; the ANGLE itself only
// steers convergence and is computed from 20-bit reciprocal / reciprocal-square-root seeds (a 1e-6 relative error in t
// leaves an off-diagonal of 1e-6 of the old one instead of zero: at most one extra sweep, measured none).  The exact
// formula (jacobi_rot: two divisions, two square roots) was ~750 dependent cycles of the ~1100 per rotation.
__device__ __forceinline__ void jacobi_rot_fast(double a, double b, double g, double& c, double& s) {
    const double zeta = (b - a) * 0.5 * rcp_approx(g);
    const double w = fma(zeta, zeta, 1.0);
    double rs;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(rs) : "d"(w));
    const double root = w * rs;                                   // ~ sqrt(1 + zeta^2)
    double t = copysign(rcp_approx(fabs(zeta) + root), zeta);
    if (!(fabs(t) <= 1.0)) t = 0.0;       // zeta^2 overflowed (needs a column ratio > 1e278, excluded by the `tiny` test): no rotation
    c = rsqrt_nr(fma(t, t, 1.0));
    s = c * t;
}


// ------------------------------------------------------------------------------------------------
// 3x3: right singular vector of the smallest singular value by one-sided Jacobi, then rank-2 projection
//      Fs <- Fs - (Fs v3) v3^T      (== U diag(s1,s2,0) V^T, lab3.py:321-324)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void jacobi_rot(double a, double b, double g, double& c, double& s) {
    // rotation that orthogonalises two columns with squared norms a, b and inner product g
    const double zeta = (b - a) / (2.0 * g);
    const double t = copysign(1.0, zeta) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
    c = rsqrt(1.0 + t * t);
    s = c * t;
}

__device__ __forceinline__ void rank2_project(double* __restrict__ Fs /* row-major 3x3, in/out */) {
    // columns of W = Fs*V and of V
    double w[3][3], v[3][3];
#pragma unroll
    for (int j = 0; j < 3; ++j)
#pragma unroll
        for (int i = 0; i < 3; ++i) { w[j][i] = Fs[3 * i + j]; v[j][i] = (i == j) ? 1.0 : 0.0; }
    for (int sweep = 0; sweep < 12; ++sweep) {
        bool rotated = false;
#pragma unroll
        for (int pq = 0; pq < 3; ++pq) {
            const int p = (pq == 2) ? 1 : 0;
            const int q = (pq == 0) ? 1 : 2;
            const double a = w[p][0] * w[p][0] + w[p][1] * w[p][1] + w[p][2] * w[p][2];
            const double b = w[q][0] * w[q][0] + w[q][1] * w[q][1] + w[q][2] * w[q][2];
            const double g = w[p][0] * w[q][0] + w[p][1] * w[q][1] + w[p][2] * w[q][2];
            if (g != 0.0 && fabs(g) > 1e-16 * sqrt(a * b)) {
                double c, s;
                jacobi_rot(a, b, g, c, s);
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
    double n0 = w[0][0] * w[0][0] + w[0][1] * w[0][1] + w[0][2] * w[0][2];
    double n1 = w[1][0] * w[1][0] + w[1][1] * w[1][1] + w[1][2] * w[1][2];
    double n2 = w[2][0] * w[2][0] + w[2][1] * w[2][1] + w[2][2] * w[2][2];
    int jm = 0;
    if (n1 < n0) { jm = 1; n0 = n1; }
    if (n2 < n0) { jm = 2; }
    double v3[3], fv[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) v3[i] = (jm == 0) ? v[0][i] : (jm == 1 ? v[1][i] : v[2][i]);
    // re-normalise v3 (rotations keep it unit up to rounding)
    const double nv = rsqrt(v3[0] * v3[0] + v3[1] * v3[1] + v3[2] * v3[2]);
#pragma unroll
    for (int i = 0; i < 3; ++i) v3[i] *= nv;
#pragma unroll
    for (int i = 0; i < 3; ++i) fv[i] = Fs[3 * i] * v3[0] + Fs[3 * i + 1] * v3[1] + Fs[3 * i + 2] * v3[2];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) Fs[3 * i + j] -= fv[i] * v3[j];
}

// rank-2 projection for the thread-per-hypothesis solver: same iteration with approximate-angle rotations (the rotation
// stays orthogonal to rounding, see jacobi_rot_fast) and a square-root-free convergence test — the exact version's
// divisions and square roots were a third of f8_solve_qr's dependent chain
__device__ __forceinline__ void rank2_project_fast(double* __restrict__ Fs /* row-major 3x3, in/out */) {
    double w[3][3], v[3][3];
#pragma unroll
    for (int j = 0; j < 3; ++j)
#pragma unroll
        for (int i = 0; i < 3; ++i) { w[j][i] = Fs[3 * i + j]; v[j][i] = (i == j) ? 1.0 : 0.0; }
    for (int sweep = 0; sweep < 14; ++sweep) {
        bool rotated = false;
#pragma unroll
        for (int pq = 0; pq < 3; ++pq) {
            const int p = (pq == 2) ? 1 : 0;
            const int q = (pq == 0) ? 1 : 2;
            const double a = w[p][0] * w[p][0] + w[p][1] * w[p][1] + w[p][2] * w[p][2];
            const double b = w[q][0] * w[q][0] + w[q][1] * w[q][1] + w[q][2] * w[q][2];
            const double g = w[p][0] * w[q][0] + w[p][1] * w[q][1] + w[p][2] * w[q][2];
            if (g * g > 1e-32 * (a * b)) {
                double c, s;
                jacobi_rot_fast(a, b, g, c, s);
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
    double n0 = w[0][0] * w[0][0] + w[0][1] * w[0][1] + w[0][2] * w[0][2];
    double n1 = w[1][0] * w[1][0] + w[1][1] * w[1][1] + w[1][2] * w[1][2];
    double n2 = w[2][0] * w[2][0] + w[2][1] * w[2][1] + w[2][2] * w[2][2];
    int jm = 0;
    if (n1 < n0) { jm = 1; n0 = n1; }
    if (n2 < n0) { jm = 2; }
    double v3[3], fv[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) v3[i] = (jm == 0) ? v[0][i] : (jm == 1 ? v[1][i] : v[2][i]);
    const double nv = rsqrt_nr(v3[0] * v3[0] + v3[1] * v3[1] + v3[2] * v3[2]);
#pragma unroll
    for (int i = 0; i < 3; ++i) v3[i] *= nv;
#pragma unroll
    for (int i = 0; i < 3; ++i) fv[i] = Fs[3 * i] * v3[0] + Fs[3 * i + 1] * v3[1] + Fs[3 * i + 2] * v3[2];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) Fs[3 * i + j] -= fv[i] * v3[j];
}

// Hartley scaling with one reciprocal square root instead of a square root and three divisions (a = 1/L to full precision)
__device__ __forceinline__ void hartley8_fast(const double* __restrict__ px, const double* __restrict__ py, double& a, double& b,
                                              double& c) {
    double mx = 0.0, my = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { mx += px[k]; my += py[k]; }
    mx *= 0.125; my *= 0.125;
    double ss = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { const double dx = px[k] - mx, dy = py[k] - my; ss += dx * dx + dy * dy; }
    const double q = ss * 0.0625;
    if (q > 1e-290 && q < 1e290) {
        a = rsqrt_nr(q);
    } else {                                  // coincident / non-finite samples: the exact formula's inf / NaN behaviour
        a = 1.0 / sqrt(q);
    }
    b = -mx * a;
    c = -my * a;
}

// Hartley scaling of 8 points (lab3.py:288-295): returns a = 1/L, b = -mx/L, c = -my/L
__device__ __forceinline__ void hartley8(const double* __restrict__ px, const double* __restrict__ py, double& a, double& b,
                                         double& c) {
    double mx = 0.0, my = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { mx += px[k]; my += py[k]; }
    mx *= 0.125; my *= 0.125;
    double ss = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { const double dx = px[k] - mx, dy = py[k] - my; ss += dx * dx + dy * dy; }
    const double L = sqrt(ss / 16.0);      // sqrt(1/2/N * sum), N = 8
    a = 1.0 / L;
    b = -mx / L;
    c = -my / L;
}

// F = S^T Fs T with S = [[a1,0,b1],[0,a1,c1],[0,0,1]], T = [[a2,0,b2],[0,a2,c2],[0,0,1]]   (lab3.py:327)
__device__ __forceinline__ void denormalise(const double* __restrict__ Fs, double a1, double b1, double c1, double a2,
                                            double b2, double c2, double* __restrict__ F) {
    double g[9];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        g[3 * i + 0] = Fs[3 * i + 0] * a2;
        g[3 * i + 1] = Fs[3 * i + 1] * a2;
        g[3 * i + 2] = Fs[3 * i + 0] * b2 + Fs[3 * i + 1] * c2 + Fs[3 * i + 2];
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        F[0 + j] = a1 * g[0 + j];
        F[3 + j] = a1 * g[3 + j];
        F[6 + j] = b1 * g[0 + j] + c1 * g[3 + j] + g[6 + j];
    }
}

// ------------------------------------------------------------------------------------------------
// 8-point solve, QR form: one hypothesis per thread.
// The null vector of the 8x9 design matrix A is the last column of Q in A^T = Q R (Householder, backward
// stable: it is the exact null vector of A + E, |E| <= c u |A| — the same guarantee LAPACK's SVD gives).
// ------------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(128) f8_solve_qr(const double4* __restrict__ pts, const int* __restrict__ idx,
                                                    unsigned long long seed, unsigned first_pair,
                                                    const PairInfo* __restrict__ pi, const PairFrame* __restrict__ frames,
                                                    int P, int Htot, double* __restrict__ F64, Hyp32* __restrict__ hyp32,
                                                    unsigned char* __restrict__ flags) {
    const int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= Htot) return;
    int lo = 0, hi = P;
    while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (pi[mid].hyp_off <= h) lo = mid; else hi = mid; }
    const PairInfo& info = pi[lo];

    double X[8], Y[8], x[8], y[8];
    bool bad_index = false;
    {
        int id[8];
        if (idx != nullptr) {
            const int4 i0 = reinterpret_cast<const int4*>(idx)[(size_t)h * 2];
            const int4 i1 = reinterpret_cast<const int4*>(idx)[(size_t)h * 2 + 1];
            id[0] = i0.x; id[1] = i0.y; id[2] = i0.z; id[3] = i0.w; id[4] = i1.x; id[5] = i1.y; id[6] = i1.z; id[7] = i1.w;
        } else {      // seeded call: the sample is a pure function of (seed, global pair id, hypothesis index) — philox.cuh
            sample_distinct<8>(seed, first_pair + (unsigned)lo, (unsigned)(info.hyp_first + (h - info.hyp_off)),
                               (unsigned)max(info.n, 8), id);
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            int j = id[k];
            bad_index = bad_index || j < 0 || j >= info.n;       // reported through flag bit 2 / the call's status
            j = j < 0 ? 0 : (j >= info.n ? info.n - 1 : j);     // never read out of the pair
            RG_ASSERT(j >= 0 && j < info.n && h >= info.hyp_off && h < info.hyp_off + info.H);
            const double4 v = pts[info.pt_off + j];
            X[k] = v.x; Y[k] = v.y; x[k] = v.z; y[k] = v.w;
        }
    }
    double a1, b1, c1, a2, b2, c2;
    hartley8_fast(X, Y, a1, b1, c1);
    hartley8_fast(x, y, a2, b2, c2);

    // rows of A (== columns of A^T)
    double A[8][9];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const double Xh = X[k] * a1 + b1, Yh = Y[k] * a1 + c1;
        const double xh = x[k] * a2 + b2, yh = y[k] * a2 + c2;
        A[k][0] = Xh * xh; A[k][1] = Xh * yh; A[k][2] = Xh;
        A[k][3] = Yh * xh; A[k][4] = Yh * yh; A[k][5] = Yh;
        A[k][6] = xh;      A[k][7] = yh;      A[k][8] = 1.0;
    }
    double beta[8];
    double rmin = INFINITY, rmax = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        double ss = 0.0;
#pragma unroll
        for (int i = k; i < 9; ++i) ss += A[k][i] * A[k][i];
        const double x0 = A[k][k];
        double sigma, bk;
        if (ss > 1e-290 && ss < 1e290) {                        // reciprocal square root + reciprocal, Newton-refined to full
            const double r = rsqrt_nr(ss);                      // precision: no sqrt / division chain on the critical path
            sigma = ss * r;
            bk = r * rcp_nr(sigma + fabs(x0));                  // 1 / (sigma (sigma + |x0|)) = 2 / |v|^2
        } else {
            sigma = sqrt(ss);
            bk = sigma > 0.0 ? 1.0 / (sigma * (sigma + fabs(x0))) : 0.0;
        }
        rmin = fmin(rmin, sigma);
        rmax = fmax(rmax, sigma);
        if (sigma > 0.0) A[k][k] = x0 + copysign(sigma, x0);    // v0 = x0 - alpha, alpha = -sign(x0) sigma
        beta[k] = bk;
#pragma unroll
        for (int j = k + 1; j < 8; ++j) {
            double d = 0.0;
#pragma unroll
            for (int i = k; i < 9; ++i) d += A[k][i] * A[j][i];
            d *= beta[k];
#pragma unroll
            for (int i = k; i < 9; ++i) A[j][i] -= d * A[k][i];
        }
    }
    double nv[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) nv[i] = (i == 8) ? 1.0 : 0.0;
#pragma unroll
    for (int k = 7; k >= 0; --k) {
        double d = 0.0;
#pragma unroll
        for (int i = k; i < 9; ++i) d += A[k][i] * nv[i];
        d *= beta[k];
#pragma unroll
        for (int i = k; i < 9; ++i) nv[i] -= d * A[k][i];
    }
    // unit norm (Q is orthogonal up to rounding; LAPACK's V[-1] is unit norm too)
    {
        double ss = 0.0;
#pragma unroll
        for (int i = 0; i < 9; ++i) ss += nv[i] * nv[i];
        const double inv = rsqrt(ss);
#pragma unroll
        for (int i = 0; i < 9; ++i) nv[i] *= inv;
    }
    rank2_project_fast(nv);
    double F[9];
    denormalise(nv, a1, b1, c1, a2, b2, c2, F);
    bool finite = true;
#pragma unroll
    for (int k = 0; k < 9; ++k) { F64[(size_t)h * 9 + k] = F[k]; finite = finite && isfinite(F[k]); }
    unsigned char fl = 0;
    if (!(rmin > 1e-9 * rmax)) fl |= 1;       // (nearly) rank-deficient sample: null direction not unique
    if (!finite) fl |= 2;
    if (bad_index) fl |= 4;                   // a sample index outside [0, n): clamped, and the host call fails
    flags[h] = fl;
    make_hyp32<MODE>(F, frames[lo], hyp32 + h);
}

// ------------------------------------------------------------------------------------------------
// FP32 packed scorer policy for the epipolar criterion
// ------------------------------------------------------------------------------------------------
struct Hyp2 {            // one hypothesis: 9 + 5 scalar coefficients, broadcast inside FFMA2 (.F32 operand form)
    float f[9];
    float g[5];
};

template <int MODE>
struct EpiPolicy {
    typedef Hyp32 Rec;
    typedef Hyp2 Regs;
    static constexpr bool kBoundOnly = false;
    static constexpr int kVec4PerPair = 2;      // [x0a x0b x1a x1b] [y0a y0b y1a y1b]
    static constexpr int kChunkPts = RG_EPI_CHUNK;   // 16 KB of points per stage by default

    // hypothesis record from the item's shared-memory stage (or an all-NaN hypothesis past the end of the pair)
    __device__ static __forceinline__ void load(const Hyp32* __restrict__ sh, int slot, bool valid, Hyp2& out, float& G) {
        if (valid) {
            const float4* p = reinterpret_cast<const float4*>(sh + slot);
            const float4 a = p[0], b = p[1], c = p[2], d = p[3];
            const float f[9] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x};
            const float g[5] = {c.y, c.z, c.w, d.x, d.y};
#pragma unroll
            for (int k = 0; k < 9; ++k) out.f[k] = f[k];
#pragma unroll
            for (int k = 0; k < 5; ++k) out.g[k] = g[k];
            G = d.z;
        } else {
            const float qnan = __int_as_float(0x7FFFFFFF);
#pragma unroll
            for (int k = 0; k < 9; ++k) out.f[k] = qnan;
#pragma unroll
            for (int k = 0; k < 5; ++k) out.g[k] = qnan;
            G = 0.f;
        }
    }

    // two correspondences (a,b) against K hypotheses, written step-major across the hypotheses so that consecutive
    // FFMA2 share their point operand (operand-reuse cache: the scorer is register-file-port bound, DESIGN.md);
    // per lane the IEEE op sequence is identical to epi_q32
    template <int K>
    __device__ static __forceinline__ void evalN(const Hyp2 (&H)[K], const float4* __restrict__ pr, unsigned (&cnt)[K],
                                                 float (&minabs)[K]) {
        const float4 X = pr[0], Y = pr[1];
        const float2 x0 = make_float2(X.x, X.y), x1 = make_float2(X.z, X.w);
        const float2 y0 = make_float2(Y.x, Y.y), y1 = make_float2(Y.z, Y.w);
        float2 l1x[K], l1y[K], l1z[K], l2x[K], l2y[K], r[K], s1[K], s2[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            l1x[k] = ffma2_sbs(H[k].f[1], y1, H[k].f[2]);
            l1y[k] = ffma2_sbs(H[k].f[4], y1, H[k].f[5]);
            l1z[k] = ffma2_sbs(H[k].f[7], y1, H[k].f[8]);
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            l1x[k] = ffma2_sbc(H[k].f[0], y0, l1x[k]);
            l1y[k] = ffma2_sbc(H[k].f[3], y0, l1y[k]);
            l1z[k] = ffma2_sbc(H[k].f[6], y0, l1z[k]);
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            l2x[k] = ffma2_sbs(H[k].g[1], x1, H[k].g[2]);
            l2y[k] = ffma2_sbs(H[k].g[3], x1, H[k].g[4]);      // rotated normal: no x0 term
            r[k]   = __ffma2_rn(l1y[k], x1, l1z[k]);
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            l2x[k] = ffma2_sbc(H[k].g[0], x0, l2x[k]);
            r[k]   = __ffma2_rn(l1x[k], x0, r[k]);
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            s1[k] = __ffma2_rn(l1x[k], l1x[k], __fmul2_rn(l1y[k], l1y[k]));
            s2[k] = __ffma2_rn(l2x[k], l2x[k], __fmul2_rn(l2y[k], l2y[k]));
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            float2 nm;
            if (MODE == MODE_SAMPSON) {
                const float2 m = __fadd2_rn(s1[k], s2[k]);
                nm = make_float2(-m.x, -m.y);
            } else {
                nm = make_float2(-fminf(s1[k].x, s2[k].x), -fminf(s1[k].y, s2[k].y));
            }
            const float2 q = __ffma2_rn(r[k], r[k], nm);
            cnt[k] += __float_as_uint(q.x) >> 31;
            cnt[k] += __float_as_uint(q.y) >> 31;
            minabs[k] = fminf(minabs[k], fminf(fabsf(q.x), fabsf(q.y)));
        }
    }
};

// Bound-only policy of the bounded sweep's prefix stage: counts r^2 < T (Hyp32::T), an upper bound on the exact count
// (every reference inlier passes, DESIGN.md section 4.2).  r is computed with EpiPolicy's op sequence, so it is bit-identical
// to the guarded scorer's; no image-2 normal, no norms, no guard band, no fix-up.  MODE only selects T (make_hyp32).
struct HypBound {
    float f[9];
    float nT;            // -T
};

struct EpiBoundPolicy {
    typedef Hyp32 Rec;
    typedef HypBound Regs;
    static constexpr bool kBoundOnly = true;
    static constexpr int kVec4PerPair = 2;
    static constexpr int kChunkPts = RG_EPI_CHUNK;

    __device__ static __forceinline__ void load(const Hyp32* __restrict__ sh, int slot, bool valid, HypBound& out, float& G) {
        G = 0.f;
        if (valid) {
            const float4* p = reinterpret_cast<const float4*>(sh + slot);
            const float4 a = p[0], b = p[1], c = p[2], d = p[3];
            const float f[9] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x};
#pragma unroll
            for (int k = 0; k < 9; ++k) out.f[k] = f[k];
            out.nT = -d.w;
        } else {                          // NaN r: q is a positive NaN and never counts
            const float qnan = __int_as_float(0x7FFFFFFF);
#pragma unroll
            for (int k = 0; k < 9; ++k) out.f[k] = qnan;
            out.nT = 0.f;
        }
    }

    template <int K>
    __device__ static __forceinline__ void evalN(const HypBound (&H)[K], const float4* __restrict__ pr, unsigned (&cnt)[K]) {
        const float4 X = pr[0], Y = pr[1];
        const float2 x0 = make_float2(X.x, X.y), x1 = make_float2(X.z, X.w);
        const float2 y0 = make_float2(Y.x, Y.y), y1 = make_float2(Y.z, Y.w);
        float2 l1x[K], l1y[K], l1z[K], r[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            l1x[k] = ffma2_sbs(H[k].f[1], y1, H[k].f[2]);
            l1y[k] = ffma2_sbs(H[k].f[4], y1, H[k].f[5]);
            l1z[k] = ffma2_sbs(H[k].f[7], y1, H[k].f[8]);
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            l1x[k] = ffma2_sbc(H[k].f[0], y0, l1x[k]);
            l1y[k] = ffma2_sbc(H[k].f[3], y0, l1y[k]);
            l1z[k] = ffma2_sbc(H[k].f[6], y0, l1z[k]);
        }
#pragma unroll
        for (int k = 0; k < K; ++k) r[k] = __ffma2_rn(l1y[k], x1, l1z[k]);
#pragma unroll
        for (int k = 0; k < K; ++k) r[k] = __ffma2_rn(l1x[k], x0, r[k]);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float2 q = __ffma2_rn(r[k], r[k], make_float2(H[k].nT, H[k].nT));     // sign bit set <=> r^2 < T
            cnt[k] += __float_as_uint(q.x) >> 31;
            cnt[k] += __float_as_uint(q.y) >> 31;
        }
    }
};

// FP64 re-evaluation of the flagged groups (policy of fixup_scan, score_core.cuh)
template <int MODE>
struct EpiFix {
    struct Params {
        const float4* pts32; const double4* pts64; const Hyp32* hyp32; const double* F64; const PairInfo* pi;
        const PairFrame* fr; int P;
        const int* map = nullptr;      // bounded sweep, candidate stage: compact hypothesis index -> index into F64
    };
    __device__ static __forceinline__ int pair_of(const Params& p, int h) {
        int lo = 0, hi = p.P;
        while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (p.pi[mid].hyp_off <= h) lo = mid; else hi = mid; }
        return lo;
    }
    __device__ static __forceinline__ int n_points(const Params& p, int pair) { return p.pi[pair].n; }
    // FP32 pass over one flagged group (kSub consecutive correspondences of one hypothesis)
    __device__ static __forceinline__ void scan(const Params& p, int h, int flag, int pair, unsigned& band, unsigned& sign) {
        const PairInfo& info = p.pi[pair];
        const Hyp32 hy = p.hyp32[h];
        const float4* gp = p.pts32 + (size_t)info.pt_off32 + (size_t)flag * kSub;      // kSub/2 point pairs, 2 float4 each
        float4 v[kSub];
#pragma unroll
        for (int j = 0; j < kSub; ++j) v[j] = gp[j];
#pragma unroll
        for (int j = 0; j < kSub / 2; ++j) {
            const float4 X = v[2 * j], Y = v[2 * j + 1];
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                const int k = 2 * j + s;
                const float q = epi_q32<MODE>(hy.f, hy.g, s ? X.y : X.x, s ? X.w : X.z, s ? Y.y : Y.x, s ? Y.w : Y.z);
                const bool valid = flag * kSub + k < info.n;
                band |= (valid && fabsf(q) <= hy.G ? 1u : 0u) << k;
                sign |= (__float_as_uint(q) >> 31) << k;
            }
        }
    }
    __device__ static __forceinline__ int exact(const Params& p, int h, int i, int pair) {
        const PairInfo& info = p.pi[pair];
        const double4 v = p.pts64[info.pt_off + i];
        const size_t g = p.map != nullptr ? (size_t)p.map[h] : (size_t)h;
        return epi_inlier64(p.F64 + g * 9, v.x, v.y, v.z, v.w, p.fr[pair].thr, MODE);
    }
};

// Plain FP64 scorer (reference formula for every evaluation): the SCORE_FP64 path and the on-device exact answer in
// tests.  One hypothesis per thread, points broadcast from shared memory; N may be split over gridDim.z (counts must be
// zeroed beforehand, partial sums are added atomically).
__global__ void __launch_bounds__(128) f_score_fp64(const double4* __restrict__ pts64, const double* __restrict__ F64,
                                                     const PairInfo* __restrict__ pi, double thr, int mode,
                                                     int* __restrict__ counts) {
    __shared__ double4 sp[256];
    const int p = blockIdx.y;
    const PairInfo info = pi[p];
    const int hl = blockIdx.x * blockDim.x + threadIdx.x;           // hypothesis inside the pair
    if (blockIdx.x * blockDim.x >= info.H) return;
    const bool active = hl < info.H;
    double F[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) F[k] = active ? F64[(size_t)(info.hyp_off + hl) * 9 + k] : 0.0;
    const int per = (info.n + gridDim.z - 1) / gridDim.z;
    const int n0 = min((int)blockIdx.z * per, info.n), n1 = min(n0 + per, info.n);
    int cnt = 0;
    for (int base = n0; base < n1; base += 256) {
        const int m = min(256, n1 - base);
        __syncthreads();
        for (int i = threadIdx.x; i < m; i += blockDim.x) sp[i] = pts64[info.pt_off + base + i];
        __syncthreads();
        if (active) {
            for (int i = 0; i < m; ++i) {
                const double4 v = sp[i];
                cnt += epi_inlier64(F, v.x, v.y, v.z, v.w, thr, mode);
            }
        }
    }
    if (active && cnt) atomicAdd(&counts[info.hyp_off + hl], cnt);
}

// ------------------------------------------------------------------------------------------------
// selection
// ------------------------------------------------------------------------------------------------
// tie_stats[h] = {std(d), ||d||_2} over all N points (FP64), only for hypotheses whose count equals the pair maximum
// (the only ones the reference's tie rule fun.py:324-328 can ever look at once the maximum has appeared).
__global__ void __launch_bounds__(256) f_tie_stats(const double4* __restrict__ pts64, const double* __restrict__ F64,
                                                    const int* __restrict__ counts, const PairInfo* __restrict__ pi, int P,
                                                    int Htot, const int2* __restrict__ best, int mode,
                                                    double2* __restrict__ tie_stats) {
    __shared__ double red[3][8];
    for (int h = blockIdx.x; h < Htot; h += gridDim.x) {
        int lo = 0, hi = P;
        while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (pi[mid].hyp_off <= h) lo = mid; else hi = mid; }
        const PairInfo& info = pi[lo];
        if (counts[h] != best[lo].y || best[lo].x < 0) continue;          // uniform per block
        const double* F = F64 + (size_t)h * 9;
        // two-pass like np.std: mean first, then mean of squared deviations
        double s = 0.0, s2 = 0.0;
        for (int i = threadIdx.x; i < info.n; i += blockDim.x) {
            const double4 v = pts64[info.pt_off + i];
            const double d = epi_dist64(F, v.x, v.y, v.z, v.w, mode);
            s += d; s2 += d * d;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
        __syncthreads();
        if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s; red[1][threadIdx.x >> 5] = s2; }
        __syncthreads();
        double S = 0.0, S2 = 0.0;
        for (int w = 0; w < 8; ++w) { S += red[0][w]; S2 += red[1][w]; }
        const double mean = S / (double)info.n;
        double dv = 0.0;
        for (int i = threadIdx.x; i < info.n; i += blockDim.x) {
            const double4 v = pts64[info.pt_off + i];
            const double d = epi_dist64(F, v.x, v.y, v.z, v.w, mode) - mean;
            dv += d * d;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) dv += __shfl_xor_sync(0xffffffffu, dv, o);
        if ((threadIdx.x & 31) == 0) red[2][threadIdx.x >> 5] = dv;
        __syncthreads();
        if (threadIdx.x == 0) {
            double DV = 0.0;
            for (int w = 0; w < 8; ++w) DV += red[2][w];
            tie_stats[h] = make_double2(sqrt(DV / (double)info.n), sqrt(S2));
        }
        __syncthreads();
    }
}

// sequential replay of fun.py:320-328 over the maximal-count hypotheses, in hypothesis order (one warp per pair)
__global__ void __launch_bounds__(32) f_tie_resolve(const int* __restrict__ counts, const PairInfo* __restrict__ pi,
                                                     const double2* __restrict__ tie_stats, int2* __restrict__ best,
                                                     unsigned long long* __restrict__ keys) {
    const int p = blockIdx.x;
    const PairInfo info = pi[p];
    const int2 b = best[p];
    if (b.x < 0) {
        if (keys != nullptr && threadIdx.x == 0) keys[p] = 0ull;
        return;
    }
    const int lane = threadIdx.x;
    int cur = -1;
    double cur_std = 0.0;
    for (int base = 0; base < info.H; base += 32) {
        const int h = base + lane;
        const bool cand = h < info.H && counts[info.hyp_off + h] == b.y;
        double2 st = make_double2(0.0, 0.0);
        if (cand) st = tie_stats[info.hyp_off + h];
        unsigned m = __ballot_sync(0xffffffffu, cand);
        while (m) {
            const int src = __ffs(m) - 1;
            m &= m - 1;
            const double sd = __shfl_sync(0xffffffffu, st.x, src);
            const double nr = __shfl_sync(0xffffffffu, st.y, src);
            if (cur < 0) { cur = base + src; cur_std = sd; }                 // first arrival at the max: strict >
            else if (fabs(cur_std) > nr) { cur = base + src; cur_std = sd; } // norm(std_best) > norm(d_new)
        }
    }
    if (lane == 0) {
        best[p] = make_int2(cur, b.y);
        if (keys != nullptr)
            keys[p] = ((unsigned long long)(unsigned)b.y << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)(info.hyp_first + cur));
    }
}

// inlier mask of the winner (FP64 reference formula) + copy of its F
__global__ void __launch_bounds__(256) f_mask(const double4* __restrict__ pts64, const double* __restrict__ F64,
                                               const PairInfo* __restrict__ pi, const int2* __restrict__ best, double thr,
                                               int mode, unsigned char* __restrict__ mask, double* __restrict__ best_F,
                                               int* __restrict__ best_idx, int* __restrict__ best_count) {
    const int p = blockIdx.y;
    const PairInfo info = pi[p];
    const int2 b = best[p];
    if (blockIdx.x == 0 && threadIdx.x < 9) {
        best_F[p * 9 + threadIdx.x] = b.x >= 0 ? F64[(size_t)(info.hyp_off + b.x) * 9 + threadIdx.x] : nan("");
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { best_idx[p] = b.x; best_count[p] = b.y; }
    if (mask == nullptr) return;
    double F[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) F[k] = b.x >= 0 ? F64[(size_t)(info.hyp_off + b.x) * 9 + k] : nan("");
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < info.n; i += gridDim.x * blockDim.x) {
        const double4 v = pts64[info.pt_off + i];
        mask[info.pt_off + i] = (unsigned char)epi_inlier64(F, v.x, v.y, v.z, v.w, thr, mode);
    }
}

// inlier masks of caller-supplied F matrices (FP64 reference formula), up to 64 pairs per launch: the hypothesis-split mode
// computes the winner's mask on every rank from the F that came out of the exchange
struct MaskPairs { int off[65]; };
__global__ void __launch_bounds__(256) f_mask_given(const double4* __restrict__ pts64, MaskPairs mp,
                                                     const double* __restrict__ F_in, double thr, int mode,
                                                     unsigned char* __restrict__ mask) {
    const int p = blockIdx.y;
    double F[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) F[k] = F_in[p * 9 + k];
    for (int i = mp.off[p] + blockIdx.x * blockDim.x + threadIdx.x; i < mp.off[p + 1]; i += gridDim.x * blockDim.x) {
        const double4 v = pts64[i];
        mask[i] = (unsigned char)epi_inlier64(F, v.x, v.y, v.z, v.w, thr, mode);
    }
}

// signed residuals of one F over N points (lab3.fmatrix_residuals drop-in): out[0..N) = res1, out[N..2N) = res2
__global__ void __launch_bounds__(256) f_residuals(const double* __restrict__ F9, const double* __restrict__ x,
                                                    const double* __restrict__ y, int N, double* __restrict__ out) {
    double F[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) F[k] = F9[k];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        const double x0 = x[i], x1 = x[N + i], y0 = y[i], y1 = y[N + i];
        const double l1x = F[0] * y0 + F[1] * y1 + F[2];
        const double l1y = F[3] * y0 + F[4] * y1 + F[5];
        const double l1z = F[6] * y0 + F[7] * y1 + F[8];
        const double l2x = F[0] * x0 + F[3] * x1 + F[6];
        const double l2y = F[1] * x0 + F[4] * x1 + F[7];
        const double l2z = F[2] * x0 + F[5] * x1 + F[8];
        out[i]     = (l1x * x0 + l1y * x1 + l1z) / sqrt(l1x * l1x + l1y * l1y);
        out[N + i] = (l2x * y0 + l2y * y1 + l2z) / sqrt(l2x * l2x + l2y * l2y);
    }
}

}  // namespace rg
