// K3 + K4: seeded RANSAC homography and Levenberg-Marquardt refit, one CTA per frame pair.
// Replaces cv2.findHomography(a, b, cv2.RANSAC, thresh) (reference matching.py:156-157,
// utils.py:356-358) and the 70 % gate of compute_homography (utils.py:359-360).
//
// ransac_score_kernel (256 threads, one CTA per pair, 4 CTAs per SM)
//   staging  the pair's point list (float4 ax,ay,bx,by; contiguous, 16-byte aligned) arrives in shared memory by one bulk
//            copy (cp.async.bulk + mbarrier); with a pre-transform (pre_H) a load loop maps the points on the way;
//   pass 0   every hypothesis: counter-based PCG sample of 4 distinct matches, closed-form 4-point solve in f64 registers
//            (projective basis), orientation / collinearity test, ordered compaction of the valid ones; the f32 model of
//            a valid hypothesis goes to a per-pair model cache in global memory (hyp_model) so that later stages load
//            32 bytes instead of solving again;
//   scoring  all matches are scored against the thread's hypotheses (broadcast LDS.128, counts in registers).  The inlier
//            test is OpenCV's f32 computeError <= thresh^2 with individually rounded operations.  To avoid paying ~35
//            instructions for every evaluation, a fused (FFMA + rcp.approx, ~11 instructions) value is classified
//            against per-hypothesis thresholds tlo / thi derived from a rounding-error bound, which gives count bounds
//            [lo, hi]; only hypotheses whose bounds still matter are rescored with the exact formula (one warp per
//            hypothesis, ballot / popc).  Level 1 runs in stages over matches partitioned by the leading hypothesis and
//            drops hypotheses that can no longer win; level 2 searches for the first hypothesis that counts every point.
//            Counts and the (count desc, hypothesis asc) arg-max are identical to evaluating the exact formula for every
//            hypothesis (EVZ_OPT_RANSAC_EXACT / EVZ_OPT_RANSAC_NO_PRUNE force that, for the tests).
// ransac_refit_kernel (64 threads, one CTA per pair that found a model)
//   phase 3  inlier mask of the winner (exact formula, pixel coordinates) and the bounding boxes of its inliers, then an
//            LM refit on the 8 free parameters in f64 with OpenCV's damping schedule, started undamped from the winning
//            model and run in coordinates normalised by those boxes (see LmNorm);
//   phase 4  final mask = f32 error of the refined H <= thresh^2, inlier count, 70 % gate.
//
// This file is compiled with --fmad=false: the f64 solver must round exactly like the NumPy
// oracle (oracle/ransac.py) so that identical seeds give bit-identical inlier masks.
#include "evz_common.cuh"
#include "evz_ptx.cuh"
#include <cfloat>

namespace evz {

constexpr int kRsThreads = 256;   // scoring kernel
constexpr int kRfThreads = 64;    // refit kernel
constexpr int kHpt = 4;           // hypotheses scored concurrently per thread
constexpr int kGrp = 32;          // hypotheses per group of the level-2 search (first_perfect_search)
constexpr int kStagesMax = 6;     // stages of the level-1 staged scoring
constexpr int kLmMaxIters = 20;   // OpenCV uses 10 from a DLT start; we start from the 4-point model
constexpr double kPxTol = 1e-6;   // LM stops when a step moves every point by less than this many pixels
constexpr double kPxApply = 1e-3; // an undamped step smaller than this is applied without a confirming pass (see the LM loop)
constexpr int kNSums = 32;        // 21 JtJ + 8 Jtr + S + max|r| (+1 pad)

__device__ __forceinline__ uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16; return x;
}
__device__ __forceinline__ uint32_t pcg_next(uint32_t& s) {
    s = s * 747796405u + 2891336453u;
    const uint32_t w = ((s >> ((s >> 28) + 4u)) ^ s) * 277803737u;
    return (w >> 22) ^ w;
}
// 4 distinct indices in [0, m), m >= 4 (oracle/ransac.py hyp_indices)
__device__ __forceinline__ void sample4(uint32_t seed, uint32_t pair_level, uint32_t hyp, int m, int (&idx)[4]) {
    uint32_t s = mix32(seed ^ mix32(pair_level + 0x9E3779B9u));
    s = mix32(s + hyp * 0x9E3779B9u);
    int sorted[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t r = pcg_next(s);
        int c = static_cast<int>(__umulhi(r, static_cast<uint32_t>(m - k)));
#pragma unroll
        for (int j = 0; j < k; ++j) c += (c >= sorted[j]);
        idx[k] = c;
        // insert into the sorted prefix
        int v = c;
#pragma unroll
        for (int j = 0; j < k; ++j) { if (v < sorted[j]) { const int t = sorted[j]; sorted[j] = v; v = t; } }
        sorted[k] = v;
    }
}

__device__ __forceinline__ double area2(double ax, double ay, double bx, double by, double cx, double cy) {
    return (bx - ax) * (cy - ay) - (by - ay) * (cx - ax);
}

// closed-form homography through 4 correspondences (oracle/ransac.py solve4, same operation order)
__device__ __forceinline__ bool solve4(const float4 (&p)[4], double (&H)[9]) {
    const double x0 = p[0].x, y0 = p[0].y, u0 = p[0].z, v0 = p[0].w;
    const double x1 = p[1].x, y1 = p[1].y, u1 = p[1].z, v1 = p[1].w;
    const double x2 = p[2].x, y2 = p[2].y, u2 = p[2].z, v2 = p[2].w;
    const double x3 = p[3].x, y3 = p[3].y, u3 = p[3].z, v3 = p[3].w;
    const double l0 = area2(x3, y3, x1, y1, x2, y2);
    const double l1 = area2(x0, y0, x3, y3, x2, y2);
    const double l2 = area2(x0, y0, x1, y1, x3, y3);
    const double lt = area2(x0, y0, x1, y1, x2, y2);
    const double m0 = area2(u3, v3, u1, v1, u2, v2);
    const double m1 = area2(u0, v0, u3, v3, u2, v2);
    const double m2 = area2(u0, v0, u1, v1, u3, v3);
    const double mt = area2(u0, v0, u1, v1, u2, v2);
    const double eps = 1e-6;
    const int neg = (lt * mt < 0) + (l0 * m0 < 0) + (l1 * m1 < 0) + (l2 * m2 < 0);
    const bool big = fabs(lt) > eps && fabs(l0) > eps && fabs(l1) > eps && fabs(l2) > eps &&
                     fabs(mt) > eps && fabs(m0) > eps && fabs(m1) > eps && fabs(m2) > eps;
    bool ok = big && (neg == 0 || neg == 4);
    const double w0 = m0 * (l1 * l2);
    const double w1 = m1 * (l0 * l2);
    const double w2 = m2 * (l0 * l1);
    const double c0[3] = {y1 - y2, x2 - x1, x1 * y2 - y1 * x2};
    const double c1[3] = {y2 - y0, x0 - x2, x2 * y0 - y2 * x0};
    const double c2[3] = {y0 - y1, x1 - x0, x0 * y1 - y0 * x1};
    const double q0[3] = {u0, v0, 1.0}, q1[3] = {u1, v1, 1.0}, q2[3] = {u2, v2, 1.0};
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const double a0 = w0 * q0[r], a1 = w1 * q1[r], a2 = w2 * q2[r];
#pragma unroll
        for (int j = 0; j < 3; ++j) H[3 * r + j] = (a0 * c0[j] + a1 * c1[j]) + a2 * c2[j];
    }
    const double inv = 1.0 / H[8];
    ok = ok && isfinite(inv);
#pragma unroll
    for (int i = 0; i < 8; ++i) H[i] = H[i] * inv;
    H[8] = 1.0;
    return ok;
}

// OpenCV HomographyEstimatorCallback::computeError, f32, no contraction
__device__ __forceinline__ float reproj_err32(const float (&h)[8], const float4 p) {
    const float den = __fadd_rn(__fadd_rn(__fmul_rn(h[6], p.x), __fmul_rn(h[7], p.y)), 1.f);
    const float ww = __frcp_rn(den);
    const float dx = __fsub_rn(__fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(h[0], p.x), __fmul_rn(h[1], p.y)), h[2]), ww), p.z);
    const float dy = __fsub_rn(__fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(h[3], p.x), __fmul_rn(h[4], p.y)), h[5]), ww), p.w);
    return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
}

// matrix_H_prev pre-transform of compute_homography (utils.py:351-355): f64 map, f32 result
__device__ __forceinline__ float2 pre_map(const double* T, float x, float y) {
    const double X = (T[0] * x + T[1] * y) + T[2];
    const double Y = (T[3] * x + T[4] * y) + T[5];
    const double W = (T[6] * x + T[7] * y) + T[8];
    return make_float2(static_cast<float>(X / W), static_cast<float>(Y / W));
}

struct FhArgs {
    const float* pts; const int32_t* off; const int32_t* cnt;
    const double* pre_H;
    int n_hyp; uint32_t seed; int64_t pair_id_base; int level;
    float thresh2; double min_inlier_frac; int fail_status;
    int32_t* status; double* H; uint8_t* mask; int32_t* inl_cnt;
    int32_t* best_hyp; int32_t* best_cnt; uint8_t* mask_best; double* H_best;
    int max_cnt;
    int exact_only;
    int no_prune;
    float4* hcache;     // [n_pairs][n_hyp][2] f32 models of the hypotheses that passed pass 0 (null: solved again where needed)
    const int64_t* pair_ids;   // [n_pairs] sampler id of every pair (null: pair_id_base + p)
};

// 8x8 symmetric positive-definite system through an LDL^T factorisation held in registers
// (all loops unrolled -> static indexing).  A: full symmetric 8x8 (shared memory), diag_add added to
// the diagonal.  Returns false when a pivot is not positive / finite.
struct Ldl8 { double L[8][8]; double d[8]; double inv[8]; bool ok; };
__device__ __forceinline__ void ldl8_factor(const double* A, const double* diag_add, double lam, Ldl8& f) {
    f.ok = true;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        double dj = A[j * 8 + j] + (diag_add ? lam * diag_add[j] : 0.0);
#pragma unroll
        for (int k = 0; k < j; ++k) dj -= f.L[j][k] * f.L[j][k] * f.d[k];
        f.ok = f.ok && (dj > 0.0) && isfinite(dj);
        f.d[j] = dj;
        const double inv = 1.0 / dj;
        f.inv[j] = inv;
#pragma unroll
        for (int i = j + 1; i < 8; ++i) {
            double v = A[i * 8 + j];
#pragma unroll
            for (int k = 0; k < j; ++k) v -= f.L[i][k] * f.L[j][k] * f.d[k];
            f.L[i][j] = v * inv;
        }
    }
}
__device__ __forceinline__ void ldl8_solve(const Ldl8& f, const double (&b)[8], double (&x)[8]) {
    double y[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        double v = b[i];
#pragma unroll
        for (int k = 0; k < i; ++k) v -= f.L[i][k] * y[k];
        y[i] = v;
    }
#pragma unroll
    for (int i = 7; i >= 0; --i) {
        double v = y[i] * f.inv[i];      // the pivot reciprocals of the factorisation: no second set of divisions
#pragma unroll
        for (int k = i + 1; k < 8; ++k) v -= f.L[k][i] * x[k];
        x[i] = v;
    }
}

// index of (i, j), i <= j, in the packed accumulators described in lm_accumulate
//   sums[0..5]   P  = sum p p^T            (p = (Mx ww, My ww, ww)) : 00 01 02 11 12 22
//   sums[6..11]  Px = sum -xi p p2^T       (3 x 2)                   : 00 01 10 11 20 21
//   sums[12..17] Py = sum -yi p p2^T       (3 x 2)
//   sums[18..20] Q  = sum (xi^2+yi^2) p2 p2^T                         : 00 01 11
//   sums[21..23] sum p rx, [24..26] sum p ry, [27..28] sum -(xi rx + yi ry) p2
//   sums[29] S = sum r^2, sums[30] = max |r|
// (explicit fma(): this file is compiled with --fmad=false for the bit-exact kernels, but the refit only has
// to reach the same optimum -- shared products and fused accumulation halve its f64 instruction count)
// 1 / x for the refit: single-precision seed + two Newton steps in double (full double accuracy for |x| in the
// float range; the denominator of a homography over image coordinates is ~1).  The IEEE division it replaces is
// ~15 instructions per point; the refit only has to reach the same optimum, not the same bits.
__device__ __forceinline__ double refit_rcp(double x) {
    float rf;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rf) : "f"(static_cast<float>(x)));
    double r = static_cast<double>(rf);
    r = fma(fma(-x, r, 1.0), r, r);
    r = fma(fma(-x, r, 1.0), r, r);
    return r;
}
// The LM runs in normalised coordinates: a' = (a - ca) / sa, b' = (b - cb) / sb with ca, cb the centres of the bounding
// boxes of the winner's inliers and sa, sb powers of two that bound their half-extents, so |a'|, |b'| <= 1 over the
// inliers and both maps are exact in f64.  In pixel coordinates far from the origin J^T J is close to singular in f64
// (a 96 x 54 px patch at (1500, 800): the LM stalled up to 1.66 px from the optimum); in these it stays well
// conditioned.  The residuals are those
// in pixels of b divided by sb, so the minimiser is the same.
struct LmNorm { double cax, cay, ia, cbx, cby, ib; };
__device__ __forceinline__ void lm_point(const double* h, const LmNorm& nm, const float4 pt, double* s) {
    const double Mx = (pt.x - nm.cax) * nm.ia, My = (pt.y - nm.cay) * nm.ia;
    const double bx = (pt.z - nm.cbx) * nm.ib, by = (pt.w - nm.cby) * nm.ib;
    double ww = fma(h[6], Mx, fma(h[7], My, 1.0));
    ww = fabs(ww) > DBL_EPSILON ? refit_rcp(ww) : 0.0;
    const double xi = fma(h[0], Mx, fma(h[1], My, h[2])) * ww;
    const double yi = fma(h[3], Mx, fma(h[4], My, h[5])) * ww;
    const double rx = xi - bx, ry = yi - by;
    const double p0 = Mx * ww, p1 = My * ww, p2 = ww;
    const double p00 = p0 * p0, p01 = p0 * p1, p02 = p0 * p2, p11 = p1 * p1, p12 = p1 * p2, p22 = p2 * p2;
    s[0] += p00; s[1] += p01; s[2] += p02; s[3] += p11; s[4] += p12; s[5] += p22;
    s[6] = fma(-xi, p00, s[6]); s[7] = fma(-xi, p01, s[7]); s[8] = fma(-xi, p01, s[8]); s[9] = fma(-xi, p11, s[9]);
    s[10] = fma(-xi, p02, s[10]); s[11] = fma(-xi, p12, s[11]);
    s[12] = fma(-yi, p00, s[12]); s[13] = fma(-yi, p01, s[13]); s[14] = fma(-yi, p01, s[14]); s[15] = fma(-yi, p11, s[15]);
    s[16] = fma(-yi, p02, s[16]); s[17] = fma(-yi, p12, s[17]);
    const double e = fma(xi, xi, yi * yi);
    s[18] = fma(e, p00, s[18]); s[19] = fma(e, p01, s[19]); s[20] = fma(e, p11, s[20]);
    s[21] = fma(p0, rx, s[21]); s[22] = fma(p1, rx, s[22]); s[23] = fma(p2, rx, s[23]);
    s[24] = fma(p0, ry, s[24]); s[25] = fma(p1, ry, s[25]); s[26] = fma(p2, ry, s[26]);
    const double g = fma(xi, rx, yi * ry);
    s[27] = fma(-g, p0, s[27]); s[28] = fma(-g, p1, s[28]);
    s[29] = fma(rx, rx, fma(ry, ry, s[29]));
    s[30] = fmax(s[30], fmax(fabs(rx), fabs(ry)));
}
// expand packed sums to the full symmetric 8x8 JtJ and Jtr
__device__ void lm_expand(const double* s, double* A, double* v) {
    for (int i = 0; i < 64; ++i) A[i] = 0.0;
    const int tri[3][3] = {{0, 1, 2}, {1, 3, 4}, {2, 4, 5}};
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) {
        A[i * 8 + j] = s[tri[i][j]];
        A[(3 + i) * 8 + 3 + j] = s[tri[i][j]];
    }
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 2; ++j) {
        A[i * 8 + 6 + j] = s[6 + 2 * i + j];        A[(6 + j) * 8 + i] = s[6 + 2 * i + j];
        A[(3 + i) * 8 + 6 + j] = s[12 + 2 * i + j]; A[(6 + j) * 8 + 3 + i] = s[12 + 2 * i + j];
    }
    A[6 * 8 + 6] = s[18]; A[6 * 8 + 7] = s[19]; A[7 * 8 + 6] = s[19]; A[7 * 8 + 7] = s[20];
    for (int i = 0; i < 3; ++i) { v[i] = s[21 + i]; v[3 + i] = s[24 + i]; }
    v[6] = s[27]; v[7] = s[28];
}

// G = T_b H T_a^-1 with T(p) = (p - c) / s, scaled to g22 = 1; x receives the 8 free entries
__device__ void lm_to_normalised(const double* H, const LmNorm& nm, double sa, double* x) {
    double M[9];                                              // H T_a^-1
    for (int r = 0; r < 3; ++r) {
        M[3 * r] = H[3 * r] * sa;
        M[3 * r + 1] = H[3 * r + 1] * sa;
        M[3 * r + 2] = (H[3 * r] * nm.cax + H[3 * r + 1] * nm.cay) + H[3 * r + 2];
    }
    double G[9];
    for (int j = 0; j < 3; ++j) {
        G[j] = (M[j] - nm.cbx * M[6 + j]) * nm.ib;
        G[3 + j] = (M[3 + j] - nm.cby * M[6 + j]) * nm.ib;
        G[6 + j] = M[6 + j];
    }
    const double inv = 1.0 / G[8];
    for (int i = 0; i < 8; ++i) x[i] = G[i] * inv;
}
// H = T_b^-1 G T_a, scaled to h22 = 1 (all 9 entries written)
__device__ void lm_from_normalised(const double* x, const LmNorm& nm, double sb, double* H) {
    double N[9];                                              // G T_a
    for (int r = 0; r < 3; ++r) {
        const double g0 = x[3 * r], g1 = x[3 * r + 1], g2 = r == 2 ? 1.0 : x[3 * r + 2];
        N[3 * r] = g0 * nm.ia;
        N[3 * r + 1] = g1 * nm.ia;
        N[3 * r + 2] = g2 - (g0 * nm.cax + g1 * nm.cay) * nm.ia;
    }
    double K[9];
    for (int j = 0; j < 3; ++j) {
        K[j] = N[j] * sb + nm.cbx * N[6 + j];
        K[3 + j] = N[3 + j] * sb + nm.cby * N[6 + j];
        K[6 + j] = N[6 + j];
    }
    const double inv = 1.0 / K[8];
    for (int i = 0; i < 8; ++i) H[i] = K[i] * inv;
    H[8] = 1.0;
}

struct LmShared {
    double x[8], A[64], v[8], D[8];     // x: parameters in normalised coordinates (g22 = 1)
    double H[9];                        // the model in pixel coordinates (h22 = 1)
    double S, lam, lc;
    double px_prev;                     // pixels moved by the last evaluated step if it was undamped and accepted, else inf
    double sums[kNSums];
    double wsum[kRfThreads / 32][kNSums];
    float box_w[kRfThreads / 32][8];    // per warp: min and -max of ax, ay, bx, by
    LmNorm nm;
    int iter, go;
};

// all threads: accumulate the packed sums at parameters h over the inliers flagged in msk
__device__ void lm_accumulate(const double* h, const float4* pts, const uint8_t* msk, int m, LmShared& L) {
    double s[kNSums];
#pragma unroll
    for (int i = 0; i < kNSums; ++i) s[i] = 0.0;
    const LmNorm nm = L.nm;
    for (int i = threadIdx.x; i < m; i += blockDim.x) if (msk[i]) lm_point(h, nm, pts[i], s);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // warp reduction of the 30 sums as a transposing butterfly: at every step a lane keeps one half of its values
    // and trades the other half, so that lane i ends up with the warp total of sum i (31 exchanges instead of
    // 30 x 5); the maximum (s[30]) is reduced on its own
    double mx = s[30];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffff, mx, o));
    double v[32];
#pragma unroll
    for (int i = 0; i < 30; ++i) v[i] = s[i];
    v[30] = 0.0; v[31] = 0.0;
#pragma unroll
    for (int n = 16; n > 0; n >>= 1) {
        const bool up = (lane & n) != 0;
#pragma unroll
        for (int i = 0; i < n; ++i) {
            const double keep = up ? v[i + n] : v[i];
            const double send = up ? v[i] : v[i + n];
            v[i] = keep + __shfl_xor_sync(0xffffffff, send, n);
        }
    }
    __syncthreads();
    if (lane < 31) L.wsum[warp][lane] = lane == 30 ? mx : v[0];
    __syncthreads();
    if (threadIdx.x < 31) {
        double t = L.wsum[0][threadIdx.x];
        for (int w = 1; w < kRfThreads / 32; ++w)
            t = (threadIdx.x == 30) ? fmax(t, L.wsum[w][threadIdx.x]) : t + L.wsum[w][threadIdx.x];
        L.sums[threadIdx.x] = t;
    }
    __syncthreads();
}

// fused (FFMA + approximate reciprocal) evaluation of the same quantity as reproj_err32
__device__ __forceinline__ float reproj_err_fused(const float (&h)[8], const float4 p) {
    const float den = __fmaf_rn(h[6], p.x, __fmaf_rn(h[7], p.y, 1.f));
    float ww;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(ww) : "f"(den));
    const float X = __fmaf_rn(h[0], p.x, __fmaf_rn(h[1], p.y, h[2]));
    const float Y = __fmaf_rn(h[3], p.x, __fmaf_rn(h[4], p.y, h[5]));
    const float dx = __fmaf_rn(X, ww, -p.z);
    const float dy = __fmaf_rn(Y, ww, -p.w);
    return __fmaf_rn(dx, dx, __fmul_rn(dy, dy));
}

// Thresholds outside of which the fused value decides the exact test  err_exact <= t.
// u = 2^-24; |coords| <= cmax; Bd >= |h6 x| + |h7 y| + 1; Bx >= |h0 x| + |h1 y| + |h2|.  Over the
// data range den >= 1 - (|h6|+|h7|) cmax; in addition an evaluation is only classified when
// |den_fused| >= kDenMin.  With the 8 u Bd rounding slack both give |den| >= dm on both paths
//   dm = max(0.9 kDenMin, 1 - (|h6|+|h7|) cmax - 8 u Bd)        (requires 8 u Bd <= 0.1 kDenMin).
// Then, for either path,
//   rel. error of ww            <= rho = 4u Bd/dm + 2u                     (rcp.approx: 2^-23)
//   abs. error of X ww - u_i    <= (Bx/dm)(6u + rho) + u cmax
// so the paths differ by at most dX (dY) below (x1.25 safety) and, with D = dX + dY,
//   |err_exact - err_fused| <= 2 D sqrt(max err) + 6u max err.
// Solving the two one-sided implications for the fused value gives
//   err_fused >= t + 2D^2 + 2D sqrt(D^2 + t)  =>  err_exact >  t      (thi, margin x1.25 + 1e-4)
//   err_fused <= t - 6D            (D < 2)    =>  err_exact <= t      (tlo, margin x1.25 + 1e-4)
// Everything else (inside the band, |den| small, NaN) is "unsure" and counted in hi only.
constexpr float kDenMin = 0.0625f;
// true when |den| >= kDenMin is guaranteed on both the fused and the exact path for every point with
// |x|, |y| <= cmax: den >= 1 - (|h6|+|h7|) cmax - 8 u Bd (same bound as dm in fused_thresholds)
__device__ __forceinline__ bool den_safe(float h6, float h7, float cmax) {
    const float u = 5.9604645e-8f;
    const float a6 = fabsf(h6) + fabsf(h7);
    const float Bd = a6 * cmax + 1.f;
    return (8.f * u * Bd <= 0.1f * kDenMin) && ((1.f - a6 * cmax - 8.f * u * Bd) * 0.999999f >= kDenMin);
}
__device__ __forceinline__ void fused_thresholds(const float (&h)[8], float cmax, float t, bool exact_only,
                                                 float& tlo, float& thi) {
    const float u = 5.9604645e-8f;
    const float a6 = fabsf(h[6]) + fabsf(h[7]);
    const float Bd = a6 * cmax + 1.f;
    const float Bx = (fabsf(h[0]) + fabsf(h[1])) * cmax + fabsf(h[2]);
    const float By = (fabsf(h[3]) + fabsf(h[4])) * cmax + fabsf(h[5]);
    const float dm = fmaxf(0.9f * kDenMin, (1.f - a6 * cmax - 8.f * u * Bd) * 0.999999f);
    const float rho = 4.f * u * Bd / dm + 2.f * u;
    const float dX = 2.5f * ((Bx / dm) * (6.f * u + rho) + u * cmax);
    const float dY = 2.5f * ((By / dm) * (6.f * u + rho) + u * cmax);
    const float D = dX + dY;
    tlo = -INFINITY;
    thi = INFINITY;
    if (exact_only || !(8.f * u * Bd <= 0.1f * kDenMin) || !(D < 1e6f)) return;      // no usable bound: all unsure
    thi = t + 1.25f * (2.f * D * D + 2.f * D * sqrtf(D * D + t)) + 1e-4f;
    if (D < 2.f) tlo = t - 1.25f * 6.f * D - 1e-4f;
}

// Fused scoring of NJ hypotheses per thread (slots s0 + j*kRsThreads + tid) against all matches;
// writes the count bounds of every live slot and returns the thread's best lower bound.
// kCheckDen = false is used for hypotheses whose denominator provably stays >= kDenMin over the data range
// (den_safe below), for which the per-evaluation |den| test can never fire.
// Range of matches a scoring call covers.  FULL: all matches, final bounds.  PREFIX: matches [0, i1), the raw
// partial counts (sure-in, sure-out) are parked in lo_s / hi_s.  SUFFIX: matches [i0, m) on top of the parked
// partial counts, final bounds.  (Two-phase scoring, see ransac_score_kernel.)
struct PtRange { int i0, i1, mode; };
// kMid: a middle stage of the staged scoring -- starts from the parked partial counts and parks them again
constexpr int kFull = 0, kPrefix = 1, kSuffix = 2, kMid = 3;
constexpr int kLead = 32;                    // hypotheses of the fully scored leading batch of the two-phase scoring

// the four sampled correspondences of a hypothesis: sample indices refer to the caller's order, pos[] maps them to
// where the point lives in shared memory (identity until the level-1 partition by the leader's residuals)
__device__ __forceinline__ void load_sample(const float4* pts, const uint16_t* pos, const int (&idx)[4], float4 (&q)[4]) {
#pragma unroll
    for (int k = 0; k < 4; ++k) q[k] = pts[pos[idx[k]]];
}

// f32 model of hypothesis `hyp`: pass 0 solved it once (f64, cast to f32) and left it in the per-pair model cache in
// global memory (32 bytes, an L2 hit a few microseconds later); without a cache the sample is drawn and solved again.
// A staged level-1 scoring looks at a surviving hypothesis once per stage and a sliced row once per slice: the
// closed-form solve (~150 f64 instructions) is several times the price of the two loads.
__device__ __forceinline__ void hyp_model(const FhArgs& a, const float4* pts, const uint16_t* pos, int hyp, int m,
                                          uint32_t pair_level, float (&hf)[8]) {
    if (a.hcache) {
        const float4* hc = a.hcache + (static_cast<size_t>(blockIdx.x) * a.n_hyp + hyp) * 2;
        const float4 u = __ldcg(hc), v = __ldcg(hc + 1);
        hf[0] = u.x; hf[1] = u.y; hf[2] = u.z; hf[3] = u.w; hf[4] = v.x; hf[5] = v.y; hf[6] = v.z; hf[7] = v.w;
    } else {
        int idx[4];
        sample4(a.seed, pair_level, static_cast<uint32_t>(hyp), m, idx);
        float4 q[4];
        load_sample(pts, pos, idx, q);
        double H[9];
        solve4(q, H);
#pragma unroll
        for (int i = 0; i < 8; ++i) hf[i] = static_cast<float>(H[i]);
    }
}

template <int NJ, bool kCheckDen>
__device__ __forceinline__ int score_batch(const FhArgs& a, const float4* pts, const uint16_t* pos, const uint16_t* vlist,
                                           uint16_t* lo_s, uint16_t* hi_s, int s0, int n_valid, int m, float cmax,
                                           uint32_t pair_level, int* cut, const PtRange rg) {
    const int tid = threadIdx.x;
    float hf[NJ][8];
    float tlo[NJ], thi[NJ];
    int lo[NJ], out[NJ];
    bool any_live = false;                                 // (a live slot is recognisable by thi > -inf)
    const int cutv = *cut;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const int slot = s0 + j * kRsThreads + tid;
        lo[j] = 0; out[j] = 0;
        tlo[j] = -INFINITY; thi[j] = -INFINITY;            // idle slot: everything "sure out"
#pragma unroll
        for (int i = 0; i < 8; ++i) hf[j][i] = 0.f;
        // hypotheses behind the cut (see the pruning note in ransac_score_kernel) stay idle: lo = hi = 0
        if (slot < n_valid && static_cast<int>(vlist[slot]) < cutv) {
            hyp_model(a, pts, pos, vlist[slot], m, pair_level, hf[j]);
            fused_thresholds(hf[j], cmax, a.thresh2, a.exact_only != 0, tlo[j], thi[j]);
            any_live = true;
            if (rg.mode == kSuffix || rg.mode == kMid) { lo[j] = lo_s[slot]; out[j] = hi_s[slot]; }
        }
    }
    const int i_end = __any_sync(0xffffffff, any_live) ? rg.i1 : 0;   // a warp without live hypotheses skips the matches
    for (int i = rg.i0; i < i_end; ++i) {
        const float4 pt = pts[i];
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const float den = __fmaf_rn(hf[j][6], pt.x, __fmaf_rn(hf[j][7], pt.y, 1.f));
            float ww;
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(ww) : "f"(den));
            const float X = __fmaf_rn(hf[j][0], pt.x, __fmaf_rn(hf[j][1], pt.y, hf[j][2]));
            const float Y = __fmaf_rn(hf[j][3], pt.x, __fmaf_rn(hf[j][4], pt.y, hf[j][5]));
            const float dx = __fmaf_rn(X, ww, -pt.z);
            const float dy = __fmaf_rn(Y, ww, -pt.w);
            const float e = __fmaf_rn(dx, dx, __fmul_rn(dy, dy));
            // |den| too small: not classifiable -> NaN fails both tests below (counted as unsure)
            const float e2 = (!kCheckDen || fabsf(den) >= kDenMin) ? e : __int_as_float(0x7fc00000);
            asm("{\n\t.reg .pred p;\n\tsetp.le.f32 p, %1, %2;\n\t@p add.s32 %0, %0, 1;\n\t}" : "+r"(lo[j]) : "f"(e2), "f"(tlo[j]));
            asm("{\n\t.reg .pred p;\n\tsetp.ge.f32 p, %1, %2;\n\t@p add.s32 %0, %0, 1;\n\t}" : "+r"(out[j]) : "f"(e2), "f"(thi[j]));
        }
    }
    int my_lo = 0;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const int slot = s0 + j * kRsThreads + tid;
        if (thi[j] > -INFINITY) {
            if (rg.mode == kPrefix || rg.mode == kMid) {
                lo_s[slot] = static_cast<uint16_t>(lo[j]); hi_s[slot] = static_cast<uint16_t>(out[j]);
            } else {
                lo_s[slot] = static_cast<uint16_t>(lo[j]); hi_s[slot] = static_cast<uint16_t>(m - out[j]);
                // every match is a sure inlier: no hypothesis with a larger index can win any more
                if (lo[j] == m) atomicMin(cut, static_cast<int>(vlist[slot]));
                my_lo = max(my_lo, lo[j]);
            }
        }
    }
    return my_lo;
}

// The last, partially filled row of hypotheses (L < kRsThreads live slots starting at r0): instead of
// letting most threads idle through all m matches, the threads are regrouped as (hypothesis, slice): Lp =
// L rounded up to a power of two >= 32, slice = tid / Lp of kRsThreads / Lp slices, and every slice scores
// a strided share of the matches; partial counts meet in shared memory.  Same classification per
// evaluation as score_batch<.., true>, so the bounds are identical.
__device__ __forceinline__ void score_partial_row(const FhArgs& a, const float4* pts, const uint16_t* pos, const uint16_t* vlist,
                                                  uint16_t* lo_s, uint16_t* hi_s, int* part, int* lbest, int* cut, int r0, int L, int m,
                                                  float cmax, uint32_t pair_level, const PtRange rg) {
    const int tid = threadIdx.x;
    int Lp = 16;
    while (Lp < L) Lp <<= 1;
    const int slices = kRsThreads / Lp;
    const int k = tid & (Lp - 1), slice = tid / Lp;
    const bool live = k < L && static_cast<int>(vlist[r0 + k]) < *cut;     // behind the cut: idle, lo = hi = 0
    float hf[8];
    float tlo = -INFINITY, thi = -INFINITY;                  // idle lane: everything "sure out"
#pragma unroll
    for (int i = 0; i < 8; ++i) hf[i] = 0.f;
    if (live) {
        hyp_model(a, pts, pos, vlist[r0 + k], m, pair_level, hf);
        fused_thresholds(hf, cmax, a.thresh2, a.exact_only != 0, tlo, thi);
    }
    part[tid] = 0; part[kRsThreads + tid] = 0;
    __syncthreads();
    int lo = 0, out = 0;
    const int i_end = __any_sync(0xffffffff, live) ? rg.i1 : 0;      // a warp without live hypotheses skips the matches
    auto eval = [&](const float4 pt) {
        const float den = __fmaf_rn(hf[6], pt.x, __fmaf_rn(hf[7], pt.y, 1.f));
        float ww;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(ww) : "f"(den));
        const float X = __fmaf_rn(hf[0], pt.x, __fmaf_rn(hf[1], pt.y, hf[2]));
        const float Y = __fmaf_rn(hf[3], pt.x, __fmaf_rn(hf[4], pt.y, hf[5]));
        const float dx = __fmaf_rn(X, ww, -pt.z);
        const float dy = __fmaf_rn(Y, ww, -pt.w);
        const float e = __fmaf_rn(dx, dx, __fmul_rn(dy, dy));
        const float e2 = fabsf(den) >= kDenMin ? e : __int_as_float(0x7fc00000);
        asm("{\n\t.reg .pred p;\n\tsetp.le.f32 p, %1, %2;\n\t@p add.s32 %0, %0, 1;\n\t}" : "+r"(lo) : "f"(e2), "f"(tlo));
        asm("{\n\t.reg .pred p;\n\tsetp.ge.f32 p, %1, %2;\n\t@p add.s32 %0, %0, 1;\n\t}" : "+r"(out) : "f"(e2), "f"(thi));
    };
    {   // four points per trip: the loads are issued together and the loop overhead is shared
        int i = rg.i0 + slice;
        for (; i + 3 * slices < i_end; i += 4 * slices) {
            const float4 p0 = pts[i], p1 = pts[i + slices], p2 = pts[i + 2 * slices], p3 = pts[i + 3 * slices];
            eval(p0); eval(p1); eval(p2); eval(p3);
        }
        for (; i < i_end; i += slices) eval(pts[i]);
    }
    if (live) { atomicAdd(&part[k], lo); atomicAdd(&part[kRsThreads + k], out); }
    __syncthreads();
    if (live && slice == 0) {
        int l = part[k], o = part[kRsThreads + k];
        if (rg.mode == kSuffix || rg.mode == kMid) { l += lo_s[r0 + k]; o += hi_s[r0 + k]; }
        lo_s[r0 + k] = static_cast<uint16_t>(l);
        if (rg.mode == kPrefix || rg.mode == kMid) {
            hi_s[r0 + k] = static_cast<uint16_t>(o);
        } else {
            hi_s[r0 + k] = static_cast<uint16_t>(m - o);
            atomicMax(lbest, l);
            if (l == m) atomicMin(cut, static_cast<int>(vlist[r0 + k]));
        }
    }
    __syncthreads();                                         // part[] may be reused by a later call
}

// Scores the slots [s_begin, s_end) of vlist over the match range rg: whole rows of kRsThreads slots in
// batches of up to kHpt rows (rows that lie entirely below n_safe run without the denominator test; the
// remaining safe slots share their rows with the unsafe ones, never more thread-rows than a single region
// would need), then the last partial row sliced over the matches.  With `prune`, batches and rows whose
// hypotheses all lie behind the cut are skipped.
__device__ __forceinline__ void score_slots(const FhArgs& a, const float4* pts, const uint16_t* pos, const uint16_t* vlist, uint16_t* lo_s,
                                            uint16_t* hi_s, int* part_s, int* s_lbest, int* s_cut, int s_begin, int s_end,
                                            int n_safe, int m, float cmax, uint32_t pair_level, bool prune,
                                            bool first_row_alone, const PtRange rg) {
    const int tid = threadIdx.x;
    if (s_end <= s_begin) return;
    const int n_nochk = s_begin + max(0, min(n_safe, s_end) - s_begin) / kRsThreads * kRsThreads;
    int n_full = n_nochk + (s_end - n_nochk) / kRsThreads * kRsThreads;           // end of the last full row
    // a tail of at least half a row joins the batched rows (its idle slots cost less than a one-hypothesis-per-thread
    // pass over the matches); shorter tails are sliced over the matches below
    if (s_end - n_full >= kRsThreads / 2) n_full = s_end;
#pragma unroll 1
    for (int region = 0; region < 2; ++region) {
        const int r_begin = region ? n_nochk : s_begin, r_end = region ? n_full : n_nochk;
        for (int s0 = r_begin; s0 < r_end; ) {
            // live hypotheses per thread in this batch (1..kHpt): idle slots are not evaluated
            const int nj = (first_row_alone && s0 == s_begin) ? 1 : min(kHpt, (r_end - s0 + kRsThreads - 1) / kRsThreads);
            if (prune) {
                __syncthreads();                                   // s_cut of the previous batch is visible
                const int cutv = *s_cut;
                int alive = 0;
#pragma unroll
                for (int j = 0; j < kHpt; ++j) {
                    const int slot = s0 + j * kRsThreads + tid;
                    if (j < nj && slot < r_end && static_cast<int>(vlist[slot]) < cutv) alive = 1;
                }
                if (!__syncthreads_or(alive)) { s0 += nj * kRsThreads; continue; }
            }
            int my_lo;
            if (region == 0) {
                switch (nj) {
                    case 1:  my_lo = score_batch<1, false>(a, pts, pos, vlist, lo_s, hi_s, s0, r_end, m, cmax, pair_level, s_cut, rg); break;
                    case 2:  my_lo = score_batch<2, false>(a, pts, pos, vlist, lo_s, hi_s, s0, r_end, m, cmax, pair_level, s_cut, rg); break;
                    case 3:  my_lo = score_batch<3, false>(a, pts, pos, vlist, lo_s, hi_s, s0, r_end, m, cmax, pair_level, s_cut, rg); break;
                    default: my_lo = score_batch<4, false>(a, pts, pos, vlist, lo_s, hi_s, s0, r_end, m, cmax, pair_level, s_cut, rg); break;
                }
            } else {
                switch (nj) {
                    case 1:  my_lo = score_batch<1, true>(a, pts, pos, vlist, lo_s, hi_s, s0, r_end, m, cmax, pair_level, s_cut, rg); break;
                    case 2:  my_lo = score_batch<2, true>(a, pts, pos, vlist, lo_s, hi_s, s0, r_end, m, cmax, pair_level, s_cut, rg); break;
                    case 3:  my_lo = score_batch<3, true>(a, pts, pos, vlist, lo_s, hi_s, s0, r_end, m, cmax, pair_level, s_cut, rg); break;
                    default: my_lo = score_batch<4, true>(a, pts, pos, vlist, lo_s, hi_s, s0, r_end, m, cmax, pair_level, s_cut, rg); break;
                }
            }
            atomicMax(s_lbest, my_lo);
            s0 += nj * kRsThreads;
        }
        if (region == 1 && n_full < s_end) {
            int alive = 1;
            if (prune) {
                __syncthreads();
                const int slot = n_full + tid;
                alive = __syncthreads_or(slot < s_end && static_cast<int>(vlist[slot]) < *s_cut);
            }
            if (alive)
                score_partial_row(a, pts, pos, vlist, lo_s, hi_s, part_s, s_lbest, s_cut, n_full, s_end - n_full, m, cmax, pair_level, rg);
        }
    }
}

// Level >= 2 (static points: nearly every point is an inlier of nearly every hypothesis).  The arg-max is
// (count desc, index asc), and no count exceeds m: the winner is the LOWEST-INDEX hypothesis that counts every point,
// if there is one.  Hypotheses are therefore examined in index order, kGrp at a time (thread = hypothesis x slice of
// the points, the model solved once per hypothesis and shared through shared memory), and a hypothesis is dropped at
// its first SURE outlier -- it cannot reach m.  The search stops at the first group that holds a hypothesis with m sure
// inliers (its index goes to *cut).  Candidates = that hypothesis and every earlier one without a sure outlier
// (unsure evaluations only): they are appended to slist and counted exactly by the rescoring pass.  Returns false
// when no hypothesis counts every point as a sure inlier: the caller then scores everything the general way.
__device__ __forceinline__ bool first_perfect_search(const FhArgs& a, const float4* pts, const uint16_t* pos, uint16_t* slist, int* part,
                                                     float* grp, int* dead, int* n_surv, int* cut, int m, float cmax,
                                                     uint32_t pair_level) {
    const int tid = threadIdx.x;
    constexpr int kSlices = kRsThreads / kGrp;
    const int k = tid & (kGrp - 1), slice = tid / kGrp;
    for (int g0 = 0; g0 < a.n_hyp; g0 += kGrp) {
        if (tid < kGrp) {
            const int hyp = g0 + tid;
            int ok = 0;
            if (hyp < a.n_hyp) {
                int idx[4];
                sample4(a.seed, pair_level, static_cast<uint32_t>(hyp), m, idx);
                float4 q[4];
                load_sample(pts, pos, idx, q);
                double H[9];
                ok = solve4(q, H) ? 1 : 0;
                float hf[8], tlo, thi;
#pragma unroll
                for (int i = 0; i < 8; ++i) { hf[i] = static_cast<float>(H[i]); grp[tid * 10 + i] = hf[i]; }
                fused_thresholds(hf, cmax, a.thresh2, false, tlo, thi);
                grp[tid * 10 + 8] = tlo; grp[tid * 10 + 9] = thi;
            }
            dead[tid] = ok ? 0 : 1;
            part[tid] = 0;
        }
        __syncthreads();
        float hf[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) hf[i] = grp[k * 10 + i];
        const float tlo = grp[k * 10 + 8], thi = grp[k * 10 + 9];
        volatile int* vdead = dead;
        int lo = 0;
        for (int i = slice; i < m && !vdead[k]; i += 4 * kSlices) {
            int outl = 0;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int ii = i + u * kSlices;
                if (ii < m) {
                    const float4 pt = pts[ii];
                    const float den = __fmaf_rn(hf[6], pt.x, __fmaf_rn(hf[7], pt.y, 1.f));
                    const float e = reproj_err_fused(hf, pt);
                    const bool cls = fabsf(den) >= kDenMin;
                    lo += (cls && e <= tlo) ? 1 : 0;
                    outl |= (cls && e >= thi) ? 1 : 0;
                }
            }
            if (outl) vdead[k] = 1;
        }
        if (lo) atomicAdd(&part[k], lo);
        __syncthreads();
        if (tid < kGrp && g0 + tid < a.n_hyp && !dead[tid]) {
            if (part[tid] == m) atomicMin(cut, g0 + tid);
            slist[atomicAdd(n_surv, 1)] = static_cast<uint16_t>(g0 + tid);
        }
        __syncthreads();
        if (*cut != 0x7FFFFFFF) return true;
    }
    __syncthreads();
    if (tid == 0) *n_surv = 0;               // no perfect hypothesis: the general path starts from scratch
    __syncthreads();
    return false;
}


// dynamic shared memory of the scoring kernel: float4 pts[max_cnt] | u16 pos[max_cnt (rounded up to 8)] |
// u16 vlist, slist, lo_s, hi_s [n_hyp] each.  kGlobalLists: the four hypothesis lists are the pair's slice
// glists + 4 n_hyp p of handle scratch instead (chosen by the host when they do not fit in shared memory next to the
// points: 12 288 points leave room for 944 hypotheses).  Only the block's own threads touch its slice, and every
// cross-thread hand-over in this kernel already passes a __syncthreads, which orders global memory as well.
template <bool kGlobalLists>
__global__ void __launch_bounds__(kRsThreads, 4)
ransac_score_kernel(const FhArgs a, double* __restrict__ Hbest_out, int32_t* __restrict__ phase, uint16_t* glists) {
    extern __shared__ __align__(16) uint8_t fh_smem[];
    float4* pts = reinterpret_cast<float4*>(fh_smem);
    uint16_t* pos = reinterpret_cast<uint16_t*>(fh_smem + static_cast<size_t>(a.max_cnt) * 16);      // sample index -> position in pts
    uint16_t* vlist = kGlobalLists ? glists + static_cast<size_t>(blockIdx.x) * 4 * a.n_hyp           // valid hypotheses
                                   : pos + ((a.max_cnt + 7) & ~7);
    uint16_t* slist = vlist + a.n_hyp;                                                                // survivors to rescore
    uint16_t* lo_s = slist + a.n_hyp;                                                                 // count bounds per valid slot
    uint16_t* hi_s = lo_s + a.n_hyp;
    __shared__ unsigned long long red[kRsThreads / 32];
    __shared__ float cmax_s[kRsThreads / 32];
    __shared__ int warp_sums[2 * (kRsThreads / 32)];
    __shared__ int part_s[2 * kRsThreads];
    __shared__ float lead_s[10];
    __shared__ float grp_s[kGrp * 10];
    __shared__ int grp_dead[kGrp];
    __shared__ int s_flag, s_nvalid, s_nsafe, s_nsurv, s_lbest, s_cut, s_leader;
    __shared__ __align__(8) uint64_t stage_bar;

    const int p = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) phase[p] = 0;
    // the three per-pair scalars are loaded together (one round trip to L2 instead of three dependent ones)
    const int st_p = a.status[p];
    const int m = a.cnt[p];
    const int64_t o = a.off[p];
    if (st_p != EVZ_ST_OK) return;
    if (m < 4) { if (tid == 0) a.status[p] = EVZ_ST_FEW_POINTS; return; }
    // max_cnt sizes the shared-memory tables: a pair that exceeds it (the caller's bound was wrong) is reported as
    // failed, not truncated and not staged past the end of the tables
    if (m > a.max_cnt) { if (tid == 0) a.status[p] = a.fail_status; return; }

    // stage the point pairs (optionally through matrix_H_prev); track max |coordinate|
    const double* T = a.pre_H ? a.pre_H + static_cast<size_t>(p) * 9 : nullptr;
    float cmax = 0.f;
    if (T) {
        for (int i = tid; i < m; i += blockDim.x) {
            float4 v = reinterpret_cast<const float4*>(a.pts)[o + i];
            const float2 pa = pre_map(T, v.x, v.y), pb = pre_map(T, v.z, v.w);
            v = make_float4(pa.x, pa.y, pb.x, pb.y);
            pts[i] = v;
            pos[i] = static_cast<uint16_t>(i);
            cmax = fmaxf(cmax, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
        }
    } else {
        // one bulk copy (TMA) of the pair's contiguous, 16-byte aligned point list
        if (tid == 0) { mbar_init(&stage_bar, 1); fence_mbar_init(); }
        __syncthreads();
        if (tid == 0) {
            mbar_arrive_expect_tx(&stage_bar, static_cast<uint32_t>(m) * 16u);
            bulk_load_1d(pts, reinterpret_cast<const float4*>(a.pts) + o, static_cast<uint32_t>(m) * 16u, &stage_bar);
        }
        for (int i = tid; i < m; i += blockDim.x) pos[i] = static_cast<uint16_t>(i);
        mbar_wait(&stage_bar, 0);
        for (int i = tid; i < m; i += blockDim.x) {
            const float4 v = pts[i];
            cmax = fmaxf(cmax, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
        }
    }
#pragma unroll
    for (int of = 16; of > 0; of >>= 1) cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffff, cmax, of));
    if (lane == 0) cmax_s[warp] = cmax;
    if (tid == 0) { s_nvalid = 0; s_nsurv = 0; s_lbest = 0; s_cut = 0x7FFFFFFF; s_leader = 0x7FFFFFFF; }
    __syncthreads();
#pragma unroll
    for (int w = 0; w < kRsThreads / 32; ++w) cmax = fmaxf(cmax, cmax_s[w]);

    const uint32_t pair_level = static_cast<uint32_t>((a.pair_ids ? a.pair_ids[p] : a.pair_id_base + p) * 2 + a.level);
    if (m == 4) {
        // findHomography: npoints == 4 -> exact model through the 4 points, mask = ones, no LM
        if (tid == 0) {
            const float4 q[4] = {pts[0], pts[1], pts[2], pts[3]};
            double H[9];
            solve4(q, H);
            bool fin = true;
            for (int i = 0; i < 9; ++i) fin = fin && isfinite(H[i]);
            if (!fin) a.status[p] = a.fail_status;
            else {
                for (int i = 0; i < 9; ++i) { a.H[static_cast<size_t>(p) * 9 + i] = H[i]; Hbest_out[static_cast<size_t>(p) * 9 + i] = H[i]; }
                if (a.best_hyp) a.best_hyp[p] = -1;
                if (a.best_cnt) a.best_cnt[p] = 4;
                if (a.inl_cnt) a.inl_cnt[p] = 4;
            }
            s_flag = fin;
        }
        __syncthreads();
        if (s_flag && tid < 4) { if (a.mask_best) a.mask_best[o + tid] = 1; if (a.mask) a.mask[o + tid] = 1; }
        return;
    }

    // ---------------- pass 0: which hypotheses pass the orientation / collinearity test (ordered compaction);
    // those with a provably safe denominator go first (vlist[0, n_safe)), the others after them
    const bool prune = a.exact_only == 0 && a.no_prune == 0;
    bool found = false;
    if (prune && a.level >= 2)
        found = first_perfect_search(a, pts, pos, slist, part_s, grp_s, grp_dead, &s_nsurv, &s_cut, m, cmax, pair_level);
    if (!found) {
        int base = 0, base_u = 0;
        for (int h0 = 0; h0 < a.n_hyp; h0 += kRsThreads) {
            const int hyp = h0 + tid;
            int ok = 0, safe = 0;
            if (hyp < a.n_hyp) {
                int idx[4];
                sample4(a.seed, pair_level, static_cast<uint32_t>(hyp), m, idx);
                float4 q[4];
                load_sample(pts, pos, idx, q);
                double H[9];
                ok = solve4(q, H) ? 1 : 0;
                safe = ok && den_safe(static_cast<float>(H[6]), static_cast<float>(H[7]), cmax);
                if (ok && a.hcache) {
                    float4* hc = a.hcache + (static_cast<size_t>(p) * a.n_hyp + hyp) * 2;
                    __stcg(hc, make_float4(static_cast<float>(H[0]), static_cast<float>(H[1]), static_cast<float>(H[2]), static_cast<float>(H[3])));
                    __stcg(hc + 1, make_float4(static_cast<float>(H[4]), static_cast<float>(H[5]), static_cast<float>(H[6]), static_cast<float>(H[7])));
                }
            }
            const unsigned bal_s = __ballot_sync(0xffffffff, safe);
            const unsigned bal_u = __ballot_sync(0xffffffff, ok && !safe);
            if (lane == 0) { warp_sums[warp] = __popc(bal_s); warp_sums[kRsThreads / 32 + warp] = __popc(bal_u); }
            __syncthreads();
            int before = 0, total = 0, before_u = 0, total_u = 0;
#pragma unroll
            for (int w = 0; w < kRsThreads / 32; ++w) {
                const int c = warp_sums[w], cu = warp_sums[kRsThreads / 32 + w];
                before += w < warp ? c : 0; total += c;
                before_u += w < warp ? cu : 0; total_u += cu;
            }
            const unsigned below = (1u << lane) - 1u;
            if (safe) vlist[base + before + __popc(bal_s & below)] = static_cast<uint16_t>(hyp);
            else if (ok) slist[base_u + before_u + __popc(bal_u & below)] = static_cast<uint16_t>(hyp);
            base += total; base_u += total_u;
            __syncthreads();
        }
        for (int k = tid; k < base_u; k += kRsThreads) vlist[base + k] = slist[k];
        if (tid == 0) { s_nvalid = base + base_u; s_nsafe = base; }
    }
    __syncthreads();
    int n_valid = found ? 0 : s_nvalid, n_safe = found ? 0 : s_nsafe;

    // ---------------- pass 1: fused scoring of the valid hypotheses with count bounds [lo, hi]
    unsigned long long best_key = 0;      // (exact count << 32) | ~hyp   of hypotheses whose count is already exact
    const int start = 0;
    for (int slot = start + tid; slot < n_valid; slot += kRsThreads) { lo_s[slot] = 0; hi_s[slot] = 0; }   // skipped slots: hi = 0
    __syncthreads();
    // Staged scoring at level 1 (exact).  A leading batch of kLead hypotheses is scored against every match (sliced
    // over the matches like a partial row); its best sure-inlier count lb is a true lower bound on the winning
    // count, so a hypothesis that has collected more than m - lb sure outliers can no longer win.  To make the
    // others collect their outliers EARLY, the matches are partitioned in place by the leader (the leading
    // hypothesis that reached lb): the m - lb matches it does not count as sure inliers first -- true outliers are
    // outliers for every good hypothesis -- then the rest (pos[] keeps the sample indices valid).  The other
    // hypotheses then run in stages over the matches; after every stage those with more than m - lb sure outliers,
    // or behind the cut, are removed by an ordered compaction.  Outlier-contaminated hypotheses retire after the
    // first stage (m - lb + 32 matches), good-but-worse ones a few stages later; only hypotheses as good as the
    // leader see every match.  Counts do not depend on the order of the matches: results are identical to scoring
    // everything (EVZ_OPT_RANSAC_NO_PRUNE).
    // (At level >= 2 the first row goes alone instead: the rows after it are usually pruned by the cut it finds.)
    const bool lead = prune && a.level == 1;
    const int s1 = start + (lead ? kLead : kRsThreads);
    const bool staged = lead && n_valid > s1;
    if (found) {
        // level >= 2: the candidates are already in slist
    } else if (!staged) {
        score_slots(a, pts, pos, vlist, lo_s, hi_s, part_s, &s_lbest, &s_cut, start, n_valid, n_safe, m, cmax, pair_level, prune,
                    prune && a.level >= 2, PtRange{0, m, kFull});
    } else {
        score_slots(a, pts, pos, vlist, lo_s, hi_s, part_s, &s_lbest, &s_cut, start, s1, n_safe, m, cmax, pair_level, prune, false,
                    PtRange{0, m, kFull});
        __syncthreads();
        const int lb = s_lbest;
        int b1 = m;                                    // end of the first stage
        int leader_hyp = 0x7FFFFFFF;
        if (lb >= 4) {
            // leader = lowest slot of the leading batch that reached lb; its model goes to shared memory
            if (start + tid < s1 && lo_s[start + tid] == lb) atomicMin(&s_leader, start + tid);
            __syncthreads();
            if (tid == 0) {
                int idx[4];
                sample4(a.seed, pair_level, static_cast<uint32_t>(vlist[s_leader]), m, idx);
                float4 q[4];
                load_sample(pts, pos, idx, q);
                double H[9];
                solve4(q, H);
                float hf[8], tlo, thi;
                for (int i = 0; i < 8; ++i) { hf[i] = static_cast<float>(H[i]); lead_s[i] = hf[i]; }
                fused_thresholds(hf, cmax, a.thresh2, a.exact_only != 0, tlo, thi);
                lead_s[8] = tlo;
            }
            __syncthreads();
            leader_hyp = vlist[s_leader];
            float hl[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) hl[i] = lead_s[i];
            const float tlo_l = lead_s[8];
            // class of a point: 1 = not a sure inlier of the leader (goes first).  Unordered in-place partition: the
            // k-th misplaced "rest" point of the front region trades places with the k-th misplaced "first" point
            // of the back region (lists of positions in slist / part_s).
            int n_first = 0;
            for (int c0 = 0; c0 < m; c0 += kRsThreads) {               // count the class-1 points
                const int i = c0 + tid;
                int f = 0;
                if (i < m) {
                    const float4 pt = pts[i];
                    const float den = __fmaf_rn(hl[6], pt.x, __fmaf_rn(hl[7], pt.y, 1.f));
                    const float e = reproj_err_fused(hl, pt);
                    f = !(fabsf(den) >= kDenMin && e <= tlo_l);
                }
                n_first += __syncthreads_count(f);
            }
            uint16_t* list_a = slist;                                      // misplaced class-0 points in [0, n_first)
            uint16_t* list_b = reinterpret_cast<uint16_t*>(part_s);        // misplaced class-1 points in [n_first, m); <= 1024 entries
            const int cap_b = static_cast<int>(sizeof(part_s) / sizeof(uint16_t));
            int na = 0, nb = 0;
            bool fits = true;
            for (int c0 = 0; c0 < m; c0 += kRsThreads) {
                const int i = c0 + tid;
                int f = -1;
                if (i < m) {
                    const float4 pt = pts[i];
                    const float den = __fmaf_rn(hl[6], pt.x, __fmaf_rn(hl[7], pt.y, 1.f));
                    const float e = reproj_err_fused(hl, pt);
                    f = !(fabsf(den) >= kDenMin && e <= tlo_l);
                }
                const int mis_a = i < m && i < n_first && f == 0, mis_b = i < m && i >= n_first && f == 1;
                const unsigned bal_a = __ballot_sync(0xffffffff, mis_a), bal_b = __ballot_sync(0xffffffff, mis_b);
                if (lane == 0) { warp_sums[warp] = __popc(bal_a); warp_sums[kRsThreads / 32 + warp] = __popc(bal_b); }
                __syncthreads();
                int before_a = 0, total_a = 0, before_b = 0, total_b = 0;
#pragma unroll
                for (int w = 0; w < kRsThreads / 32; ++w) {
                    const int ca = warp_sums[w], cb = warp_sums[kRsThreads / 32 + w];
                    before_a += w < warp ? ca : 0; total_a += ca;
                    before_b += w < warp ? cb : 0; total_b += cb;
                }
                const unsigned below = (1u << lane) - 1u;
                if (mis_a && na + before_a + __popc(bal_a & below) < a.n_hyp) list_a[na + before_a + __popc(bal_a & below)] = static_cast<uint16_t>(i);
                if (mis_b && nb + before_b + __popc(bal_b & below) < cap_b) list_b[nb + before_b + __popc(bal_b & below)] = static_cast<uint16_t>(i);
                na += total_a; nb += total_b;
                __syncthreads();
            }
            fits = na <= a.n_hyp && nb <= cap_b;            // (na == nb always; the lists live in borrowed buffers)
            if (fits) {
                for (int k = tid; k < na; k += kRsThreads) {
                    const int ia = list_a[k], ib = list_b[k];
                    const float4 va = pts[ia], vb = pts[ib];
                    pts[ia] = vb; pts[ib] = va;
                    pos[ia] = static_cast<uint16_t>(ib); pos[ib] = static_cast<uint16_t>(ia);
                }
                b1 = min(m, (n_first + 32 + 31) & ~31);
            }
            __syncthreads();
        }
        // stages over the matches: [0, b1), then up to kStages - 1 equal parts of at least 128 matches
        int n_rest_stages = b1 < m ? max(1, min(kStagesMax - 1, (m - b1) / 128)) : 0;
        if (!(lb >= 4 && b1 * 5 <= m * 4)) { b1 = m; n_rest_stages = 0; }      // nothing to gain: one pass over everything
        const int step = n_rest_stages ? ((m - b1 + n_rest_stages - 1) / n_rest_stages + 31) & ~31 : 0;
        int i0 = 0, i1 = b1;
        for (int stage = 0; ; ++stage) {
            const bool last = i1 >= m;
            const int mode = stage == 0 ? (last ? kFull : kPrefix) : (last ? kSuffix : kMid);
            score_slots(a, pts, pos, vlist, lo_s, hi_s, part_s, &s_lbest, &s_cut, s1, n_valid, n_safe, m, cmax, pair_level, prune, false,
                        PtRange{i0, min(i1, m), mode});
            if (last) break;
            __syncthreads();
            // ordered in-place compaction of the hypotheses that can still reach lb (new position <= old position;
            // every chunk is read, then written)
            const int cutv = s_cut;
            int base = s1, safe_alive = 0;
            for (int c0 = s1; c0 < n_valid; c0 += kRsThreads) {
                const int slot = c0 + tid;
                int hyp = 0, l = 0, ot = 0, alive = 0;
                if (slot < n_valid) {
                    hyp = vlist[slot]; l = lo_s[slot]; ot = hi_s[slot];
                    // (count desc, index asc): behind the leader a hypothesis needs strictly more than lb inliers
                    alive = (ot <= m - lb - (hyp > leader_hyp ? 1 : 0) && hyp < cutv) ? 1 : 0;
                }
                const unsigned bal = __ballot_sync(0xffffffff, alive);
                const unsigned bal_sf = __ballot_sync(0xffffffff, alive && slot < n_safe);
                if (lane == 0) { warp_sums[warp] = __popc(bal); warp_sums[kRsThreads / 32 + warp] = __popc(bal_sf); }
                __syncthreads();
                int before = 0, total = 0;
#pragma unroll
                for (int w = 0; w < kRsThreads / 32; ++w) {
                    const int c = warp_sums[w];
                    before += w < warp ? c : 0; total += c; safe_alive += warp_sums[kRsThreads / 32 + w];
                }
                if (alive) {
                    const int d = base + before + __popc(bal & ((1u << lane) - 1u));
                    vlist[d] = static_cast<uint16_t>(hyp); lo_s[d] = static_cast<uint16_t>(l); hi_s[d] = static_cast<uint16_t>(ot);
                }
                base += total;
                __syncthreads();
            }
            n_safe = min(n_safe, s1) + safe_alive;
            n_valid = base;
            i0 = i1; i1 = min(m, i1 + step);
            if (n_valid <= s1) break;                     // nobody left: the leading batch holds the winner
        }
    }
    __syncthreads();
    const int lbest = s_lbest;
    // hypotheses that can still be the arg-max: hi >= lbest.  Exact already if hi == lo, else rescore.
    for (int slot = tid; slot < n_valid; slot += kRsThreads) {
        const int lo = lo_s[slot], hi = hi_s[slot];
        if (hi >= lbest && hi > 0) {
            if (hi == lo) {
                const unsigned long long key = (static_cast<unsigned long long>(static_cast<uint32_t>(lo)) << 32) |
                                               (0xFFFFFFFFu - static_cast<uint32_t>(vlist[slot]));
                best_key = key > best_key ? key : best_key;
            } else {
                slist[atomicAdd(&s_nsurv, 1)] = vlist[slot];
            }
        }
    }
    __syncthreads();

    // ---------------- pass 2: exact rescoring of the survivors, one warp per hypothesis, ballot / popc counts
    const int n_surv = s_nsurv;
    for (int k = warp; k < n_surv; k += kRsThreads / 32) {
        const int hyp = slist[k];
        int idx[4];
        sample4(a.seed, pair_level, static_cast<uint32_t>(hyp), m, idx);
        float4 q[4];
        load_sample(pts, pos, idx, q);
        double H[9];
        solve4(q, H);
        float hf[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) hf[i] = static_cast<float>(H[i]);
        int c = 0;
        for (int i0 = 0; i0 < m; i0 += 32) {
            const int i = i0 + lane;
            const bool in = i < m && reproj_err32(hf, pts[i]) <= a.thresh2;
            c += __popc(__ballot_sync(0xffffffff, in));
        }
        const unsigned long long key = (static_cast<unsigned long long>(static_cast<uint32_t>(c)) << 32) |
                                       (0xFFFFFFFFu - static_cast<uint32_t>(hyp));
        if (c > 0) best_key = key > best_key ? key : best_key;
    }
    // block arg-max on (count desc, hypothesis asc)
    unsigned long long key = best_key;
#pragma unroll
    for (int of = 16; of > 0; of >>= 1) { const unsigned long long u = __shfl_xor_sync(0xffffffff, key, of); key = u > key ? u : key; }
    if (lane == 0) red[warp] = key;
    __syncthreads();
    if (tid == 0) {
        unsigned long long k = red[0];
        for (int w = 1; w < kRsThreads / 32; ++w) k = red[w] > k ? red[w] : k;
        const int bc = static_cast<int>(k >> 32);
        const int bh = k ? static_cast<int>(0xFFFFFFFFu - static_cast<uint32_t>(k & 0xFFFFFFFFu)) : -1;
        if (a.best_hyp) a.best_hyp[p] = bh;
        if (a.best_cnt) a.best_cnt[p] = bc;
        if (bc >= 4) {
            int idx[4];
            sample4(a.seed, pair_level, static_cast<uint32_t>(bh), m, idx);
            float4 q[4];
            load_sample(pts, pos, idx, q);
            double H[9];
            solve4(q, H);
            for (int i = 0; i < 9; ++i) Hbest_out[static_cast<size_t>(p) * 9 + i] = H[i];
            phase[p] = 1;
        } else {
            a.status[p] = a.fail_status;
        }
    }
}

__global__ void __launch_bounds__(kRfThreads, 6)
ransac_refit_kernel(const FhArgs a, const double* __restrict__ Hbest_in, const int32_t* __restrict__ phase) {
    extern __shared__ __align__(16) uint8_t fh_smem[];
    float4* pts = reinterpret_cast<float4*>(fh_smem);
    uint8_t* msk = fh_smem + static_cast<size_t>(a.max_cnt) * 16;
    __shared__ LmShared L;
    __shared__ int red[kRfThreads / 32];
    __shared__ __align__(8) uint64_t stage_bar;

    const int p = blockIdx.x;
    if (phase[p] != 1) return;
    const int m = a.cnt[p];
    const int64_t o = a.off[p];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double* T = a.pre_H ? a.pre_H + static_cast<size_t>(p) * 9 : nullptr;
    if (T) {
        for (int i = tid; i < m; i += blockDim.x) {
            float4 v = reinterpret_cast<const float4*>(a.pts)[o + i];
            const float2 pa = pre_map(T, v.x, v.y), pb = pre_map(T, v.z, v.w);
            pts[i] = make_float4(pa.x, pa.y, pb.x, pb.y);
        }
        if (tid < 9) L.H[tid] = Hbest_in[static_cast<size_t>(p) * 9 + tid];
    } else {
        // one bulk copy (TMA, 16 bytes per point) instead of a latency-bound loop of 64-thread loads: the point list of a
        // pair is contiguous and 16-byte aligned
        if (tid == 0) { mbar_init(&stage_bar, 1); fence_mbar_init(); }
        __syncthreads();
        if (tid == 0) {
            mbar_arrive_expect_tx(&stage_bar, static_cast<uint32_t>(m) * 16u);
            bulk_load_1d(pts, reinterpret_cast<const float4*>(a.pts) + o, static_cast<uint32_t>(m) * 16u, &stage_bar);
        }
        if (tid < 9) L.H[tid] = Hbest_in[static_cast<size_t>(p) * 9 + tid];
        mbar_wait(&stage_bar, 0);
    }
    __syncthreads();

    // ---------------- phase 3: winner's inlier mask (pixel coordinates, f32 formula) and the bounding boxes of its
    // inliers in a and b, as (min, -max) so that one fminf reduction serves both.  The boxes of the inliers, not of all
    // points: outliers spread over the frame would leave inliers clustered in a corner ill-conditioned again.
    float box[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) box[k] = INFINITY;
    {
        float hb[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) hb[i] = static_cast<float>(L.H[i]);
        uint8_t* mask_out = a.mask_best ? a.mask_best + o : nullptr;
        for (int i = tid; i < m; i += blockDim.x) {
            const float4 v = pts[i];
            const uint8_t in = reproj_err32(hb, v) <= a.thresh2 ? 1 : 0;
            msk[i] = in;
            if (mask_out) mask_out[i] = in;
            if (in) {
                box[0] = fminf(box[0], v.x); box[1] = fminf(box[1], v.y); box[2] = fminf(box[2], v.z); box[3] = fminf(box[3], v.w);
                box[4] = fminf(box[4], -v.x); box[5] = fminf(box[5], -v.y); box[6] = fminf(box[6], -v.z); box[7] = fminf(box[7], -v.w);
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
#pragma unroll
        for (int of = 16; of > 0; of >>= 1) box[k] = fminf(box[k], __shfl_xor_sync(0xffffffff, box[k], of));
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) L.box_w[warp][k] = box[k];
    }
    __syncthreads();
    if (tid == 0) {
        // (the winner counts at least 4 inliers, so the boxes are finite)
        for (int w = 1; w < kRfThreads / 32; ++w)
            for (int k = 0; k < 8; ++k) box[k] = fminf(box[k], L.box_w[w][k]);
        // centre: an f32 value, so that x - c is exact in f64; scale: a power of two >= the half-extent (at least 1 px)
        LmNorm nm;
        double sc[2];
        for (int q = 0; q < 2; ++q) {
            const float lx = box[2 * q], ly = box[2 * q + 1], hx = -box[4 + 2 * q], hy = -box[5 + 2 * q];
            const float cx = 0.5f * lx + 0.5f * hx, cy = 0.5f * ly + 0.5f * hy;
            const double ext = fmax(1.0, fmax(fmax(static_cast<double>(hx) - cx, static_cast<double>(cx) - lx),
                                              fmax(static_cast<double>(hy) - cy, static_cast<double>(cy) - ly)));
            int e;
            frexp(ext, &e);
            sc[q] = ldexp(1.0, e);
            if (q == 0) { nm.cax = cx; nm.cay = cy; } else { nm.cbx = cx; nm.cby = cy; }
        }
        nm.ia = 1.0 / sc[0]; nm.ib = 1.0 / sc[1];
        L.nm = nm;
        lm_to_normalised(L.H, nm, sc[0], L.x);
    }
    __syncthreads();
    const double sb = 1.0 / L.nm.ib;                       // pixels of b per normalised unit
    const double s_eps = DBL_EPSILON * L.nm.ib * L.nm.ib;  // OpenCV's DBL_EPSILON guards, in px^2, in units of S
    // first LM pass over the inliers
    lm_accumulate(L.x, pts, msk, m, L);
    if (tid == 0) {
        lm_expand(L.sums, L.A, L.v);
        for (int i = 0; i < 8; ++i) L.D[i] = L.A[i * 8 + i];
        L.S = L.sums[29];
        // (OpenCV starts at lambda = 1 from a DLT estimate; from the winning 4-point model an undamped first step saves
        // one pass over the inliers -- a step that does not reduce S is damped as usual)
        L.lam = 0.0; L.lc = 0.75; L.iter = 0; L.px_prev = INFINITY;
        L.go = L.sums[30] * sb >= static_cast<double>(FLT_EPSILON);
    }
    __syncthreads();
    while (L.go) {
        // every thread solves (A + lambda diag(D)) d = v redundantly in registers: no serial section
        double d[8], xd[8], px;
        {
            Ldl8 f;
            ldl8_factor(L.A, L.D, L.lam, f);
            double vv[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) vv[i] = L.v[i];
            ldl8_solve(f, vv, d);
#pragma unroll
            for (int i = 0; i < 8; ++i) { if (!f.ok) d[i] = 0.0; xd[i] = L.x[i] - d[i]; }
            // a step that moves no inlier by more than kPxTol pixels of b is not worth a pass over the inliers: converged
            // (every thread holds the same d, so the exit is uniform).  px estimates that movement from the entries of d:
            // |a'|, |b'| <= 1 over the inliers and den ~ 1, so a point moves by about |d0| x' + |d1| y' + |d2| +
            // (|d6| x' + |d7| y') |xi'| normalised units; the largest entries stand in for the sums (within a factor of
            // ~2 either way), and sb converts to pixels.
            px = f.ok ? (fmax(fmax(fabs(d[0]), fabs(d[1])), fmax(fabs(d[3]), fabs(d[4]))) + fmax(fabs(d[2]), fabs(d[5])) +
                         fmax(fabs(d[6]), fabs(d[7]))) * sb : 0.0;
            if (f.ok && px < kPxTol) break;
            // an undamped step below kPxApply pixels is taken without the pass that would only confirm it when the step
            // after it, px times the contraction px / px_prev of the last two Gauss-Newton steps, is below kPxTol: x - d
            // is then the point the full iteration stops at as well.  Without a previous undamped step the contraction
            // is taken to be small (the first step from the 4-point model).  The contraction is ~1e-3 on full-frame sets
            // but 1e-2 and more on small noisy patches, where a fixed assumption left the result 1e-5 px short.
            if (f.ok && px < kPxApply && L.lam == 0.0 && px * px < kPxTol * L.px_prev) {
                __syncthreads();
                if (tid < 8) L.x[tid] = xd[tid];
                __syncthreads();
                break;
            }
        }
        lm_accumulate(xd, pts, msk, m, L);
        if (tid == 0) {
            const double Sd = L.sums[29];
            const double lam_step = L.lam;
            double dS = 0.0, tdv = 0.0;
            for (int i = 0; i < 8; ++i) {
                double Ad = 0.0;
                for (int j = 0; j < 8; ++j) Ad += L.A[i * 8 + j] * d[j];
                dS += d[i] * (2.0 * L.v[i] - Ad);
                tdv += d[i] * L.v[i];
            }
            const double R = (L.S - Sd) / (fabs(dS) > s_eps ? dS : 1.0);
            if (R > 0.75) {
                L.lam *= 0.5;
                if (L.lam < L.lc) L.lam = 0.0;
            } else if (R < 0.25) {
                double nu = (Sd - L.S) / (fabs(tdv) > s_eps ? tdv : 1.0) + 2.0;
                nu = fmin(fmax(nu, 2.0), 10.0);
                if (L.lam == 0.0) {
                    // lambda = lc = 1 / max |diag(A^-1)|
                    double maxval = DBL_EPSILON;
                    Ldl8 f;
                    ldl8_factor(L.A, nullptr, 0.0, f);
                    if (f.ok) {
                        for (int c = 0; c < 8; ++c) {
                            double e[8], col[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) e[i] = i == c ? 1.0 : 0.0;
                            ldl8_solve(f, e, col);
                            double cc = 0.0;
#pragma unroll
                            for (int i = 0; i < 8; ++i) cc = i == c ? col[i] : cc;
                            maxval = fmax(maxval, fabs(cc));
                        }
                    }
                    L.lam = L.lc = 1.0 / maxval;
                    nu *= 0.5;
                }
                L.lam *= nu;
            }
            double rmax = 0.0;
            L.px_prev = INFINITY;
            if (Sd < L.S) {
                if (lam_step == 0.0) L.px_prev = px;
                L.S = Sd;
                for (int i = 0; i < 8; ++i) L.x[i] = xd[i];
                lm_expand(L.sums, L.A, L.v);
                rmax = L.sums[30];
            } else {
                rmax = 1.0;     // residual at the kept x is unchanged and was >= eps
            }
            L.iter++;
            // OpenCV also stops on a step below FLT_EPSILON in parameter units; here every step that reaches this point
            // moves some point by kPxTol or more, except the zero step of a failed factorisation, which ends the loop
            L.go = L.iter < kLmMaxIters && px > 0.0 && rmax * sb >= static_cast<double>(FLT_EPSILON);
        }
        __syncthreads();
    }

    // ---------------- phase 4: final mask under the refined H (pixel coordinates), count, gate
    if (tid == 0) lm_from_normalised(L.x, L.nm, sb, L.H);
    __syncthreads();
    float hfin[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) hfin[i] = static_cast<float>(L.H[i]);
    int c = 0;
    for (int i = tid; i < m; i += blockDim.x) {
        const int in = reproj_err32(hfin, pts[i]) <= a.thresh2 ? 1 : 0;
        if (a.mask) a.mask[o + i] = static_cast<uint8_t>(in);
        c += in;
    }
#pragma unroll
    for (int of = 16; of > 0; of >>= 1) c += __shfl_xor_sync(0xffffffff, c, of);
    if (lane == 0) red[warp] = c;
    __syncthreads();
    if (tid == 0) {
        int tot = 0;
        for (int w = 0; w < kRfThreads / 32; ++w) tot += red[w];
        if (a.inl_cnt) a.inl_cnt[p] = tot;
        for (int i = 0; i < 9; ++i) a.H[static_cast<size_t>(p) * 9 + i] = L.H[i];
        if (a.min_inlier_frac > 0.0 && static_cast<double>(tot) < a.min_inlier_frac * static_cast<double>(m))
            a.status[p] = EVZ_ST_FEW_INLIERS;
    }
}

}  // namespace evz

// evz_find_homography (pair_ids = null) and evz_find_homography_ids (pair_ids set): the kernels are shared, the only
// difference is the sampler id of pair p (FhArgs::pair_ids).  `fn` names the entry point in the error text.
#define FH_REQUIRE(cond, msg) do { if (!(cond)) { EVZ_SET_ERR(h, "%s: %s", fn, msg); return EVZ_E_ARG; } } while (0)
static int find_homography(const char* fn, evz_handle* h, const float* pts, const int32_t* off, const int32_t* cnt, int n_pairs,
                           int max_cnt, const double* pre_H, int n_hyp, uint32_t seed, int64_t pair_id_base,
                           const int64_t* pair_ids, int level, double thresh, double min_inlier_frac, int fail_status,
                           int32_t* status, double* H, uint8_t* mask, int32_t* inl_cnt,
                           int32_t* best_hyp, int32_t* best_cnt, uint8_t* mask_best, double* H_best,
                           void* stream) {
    FH_REQUIRE(pts && off && cnt && status && H, "null pointer");
    FH_REQUIRE(n_hyp > 0, "n_hyp must be positive");
    FH_REQUIRE(n_hyp <= 65535, "n_hyp must be below 65536");
    FH_REQUIRE((reinterpret_cast<uintptr_t>(pts) & 15) == 0, "pts must be 16-byte aligned");
    if (max_cnt > EVZ_MAX_KP) {
        EVZ_SET_ERR(h, "%s: max_cnt %d exceeds the supported %d points per pair", fn, max_cnt, EVZ_MAX_KP);
        return EVZ_E_UNSUPPORTED;
    }
    if (n_pairs <= 0) return EVZ_OK;
    if (max_cnt < 4) max_cnt = 4;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // the scoring kernel keeps its four u16 hypothesis lists (8 B per hypothesis) in shared memory when they fit next to
    // the points, else in handle scratch; the room is the device's per-block opt-in limit less the kernel's static part
    if (h->score_smem_room < 0) {
        int optin = 0;
        cudaFuncAttributes fa;
        EVZ_CUDA_CHECK(h, cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
        EVZ_CUDA_CHECK(h, cudaFuncGetAttributes(&fa, evz::ransac_score_kernel<false>));
        h->score_smem_room = optin - static_cast<int>(fa.sharedSizeBytes);
    }
    const int smem_pts = max_cnt * 16 + ((max_cnt + 7) & ~7) * 2 + 16;
    const bool glists = smem_pts + 8 * n_hyp > h->score_smem_room;
    const int smem_score = glists ? smem_pts : smem_pts + 8 * n_hyp;
    // scratch: phase[P] | H_best[P][9] when the caller does not want it | hypothesis lists | model cache
    void* scr = nullptr;
    const size_t ph_bytes = evz_align_up(static_cast<size_t>(n_pairs) * 4, 256);
    const size_t hb_bytes = evz_align_up(H_best ? 0 : static_cast<size_t>(n_pairs) * 72, 256);
    const size_t hl_bytes = glists ? evz_align_up(static_cast<size_t>(n_pairs) * static_cast<size_t>(n_hyp) * 8, 256) : 0;
    // model cache of the scoring kernel (hyp_model): 32 bytes per hypothesis, written and read by the pair's own CTA
    size_t hc_bytes = static_cast<size_t>(n_pairs) * static_cast<size_t>(n_hyp) * 32;
    if (hc_bytes > (size_t(4) << 30) || h->opt_ransac_exact) hc_bytes = 0;
    int rc = evz_scratch(h, ph_bytes + hb_bytes + hl_bytes + hc_bytes + 256, &scr);
    if (rc) return rc;
    uint8_t* scr8 = static_cast<uint8_t*>(scr);
    int32_t* phase = static_cast<int32_t*>(scr);
    double* hb = H_best ? H_best : reinterpret_cast<double*>(scr8 + ph_bytes);
    uint16_t* hlists = glists ? reinterpret_cast<uint16_t*>(scr8 + ph_bytes + hb_bytes) : nullptr;
    float4* hcache = hc_bytes ? reinterpret_cast<float4*>(scr8 + ph_bytes + hb_bytes + hl_bytes) : nullptr;
    const int smem_refit = max_cnt * 17 + 16;
    int& attr_score = glists ? h->attr_score_g : h->attr_score;
    if (smem_score > attr_score) {
        EVZ_CUDA_CHECK(h, cudaFuncSetAttribute(glists ? evz::ransac_score_kernel<true> : evz::ransac_score_kernel<false>,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, smem_score));
        attr_score = smem_score;
    }
    if (smem_refit > h->attr_refit) {
        EVZ_CUDA_CHECK(h, cudaFuncSetAttribute(evz::ransac_refit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_refit));
        h->attr_refit = smem_refit;
    }
    const float t = static_cast<float>(thresh * thresh);
    evz::FhArgs a{pts, off, cnt, pre_H, n_hyp, seed, pair_id_base, level, t, min_inlier_frac, fail_status,
                  status, H, mask, inl_cnt, best_hyp, best_cnt, mask_best, H_best, max_cnt, h->opt_ransac_exact, h->opt_ransac_no_prune, hcache,
                  pair_ids};
    if (glists) evz::ransac_score_kernel<true><<<n_pairs, evz::kRsThreads, smem_score, st>>>(a, hb, phase, hlists);
    else evz::ransac_score_kernel<false><<<n_pairs, evz::kRsThreads, smem_score, st>>>(a, hb, phase, nullptr);
    EVZ_LAUNCH_CHECK(h);
    evz::ransac_refit_kernel<<<n_pairs, evz::kRfThreads, smem_refit, st>>>(a, hb, phase);
    EVZ_LAUNCH_CHECK(h);
    return EVZ_OK;
}
#undef FH_REQUIRE

extern "C" int evz_find_homography(evz_handle* h, const float* pts, const int32_t* off, const int32_t* cnt, int n_pairs,
                                   int max_cnt, const double* pre_H, int n_hyp, uint32_t seed, int64_t pair_id_base, int level,
                                   double thresh, double min_inlier_frac, int fail_status,
                                   int32_t* status, double* H, uint8_t* mask, int32_t* inl_cnt,
                                   int32_t* best_hyp, int32_t* best_cnt, uint8_t* mask_best, double* H_best,
                                   void* stream) {
    if (!h) return EVZ_E_ARG;
    EVZ_ENTER(h);
    return find_homography(__func__, h, pts, off, cnt, n_pairs, max_cnt, pre_H, n_hyp, seed, pair_id_base, nullptr, level, thresh,
                           min_inlier_frac, fail_status, status, H, mask, inl_cnt, best_hyp, best_cnt, mask_best, H_best, stream);
}

extern "C" int evz_find_homography_ids(evz_handle* h, const float* pts, const int32_t* off, const int32_t* cnt, int n_pairs,
                                       int max_cnt, const double* pre_H, int n_hyp, uint32_t seed, const int64_t* pair_id,
                                       int level, double thresh, double min_inlier_frac, int fail_status,
                                       int32_t* status, double* H, uint8_t* mask, int32_t* inl_cnt,
                                       int32_t* best_hyp, int32_t* best_cnt, uint8_t* mask_best, double* H_best,
                                       void* stream) {
    if (!h) return EVZ_E_ARG;
    EVZ_ENTER(h);
    EVZ_REQUIRE(h, pair_id, "null pointer");
    return find_homography(__func__, h, pts, off, cnt, n_pairs, max_cnt, pre_H, n_hyp, seed, 0, pair_id, level, thresh,
                           min_inlier_frac, fail_status, status, H, mask, inl_cnt, best_hyp, best_cnt, mask_best, H_best, stream);
}
