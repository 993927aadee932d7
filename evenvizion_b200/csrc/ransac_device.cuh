// Device helpers of the RANSAC scoring kernels: sampler, 4-point solve, f32 error formulas, fused count bounds, staged
// scoring of hypothesis slots and the level-2 first-perfect search.  Shared by ransac_kernels.cu (fixed hypothesis count,
// refit) and ransac_adaptive.cu (confidence-bounded stop); both are compiled with --fmad=false.
#pragma once
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
    // the threshold's share of the fused_thresholds cuts, the same for every hypothesis (set_fused_cut)
    float thresh_sqrt, cut_k, cut_rnd;
};

__host__ __device__ inline void set_fused_cut(FhArgs& a) {
    a.thresh_sqrt = sqrtf(a.thresh2);                                    // correctly rounded on host and device
    a.cut_k = 2.5f * a.thresh_sqrt;
    a.cut_rnd = fmaxf(1e-4f, 8.f * 5.9604645e-8f * a.thresh2);          // max(1e-4, 8u t)
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
// so the paths differ by at most dX (dY) below (twice that, x1.25 safety) and, with D = dX + dY, the residual vectors r = (dx, dy)
// of the two paths satisfy  | |r_exact| - |r_fused| | <= D  (triangle inequality).  The two f32 squares and the sum
// round with at most 2u relative error on either path: err = |r|^2 (1 +- 2.0001u).  With s = sqrt(t):
//   err_fused <= (s - D)^2 (1 - 4u) = t - 2 s D + D^2 - ..  =>  err_exact <= t      (needs D < s)
//   err_fused >= (s + D)^2 (1 + 4u) = t + 2 s D + D^2 + ..  =>  err_exact >  t
// The cuts below take the D terms x1.25 (which also absorbs the rounding of these few f32 operations on them) and a
// rounding term 8u t >= the 4u t above plus the two roundings of t +- ..; it never falls below 1e-4, which keeps the
// cuts of small thresholds at their earlier values:
//   thi = t + 1.25 (2D^2 + 2D sqrt(D^2 + t)) + max(1e-4, 8u t)          (2D sqrt(D^2 + t) >= 2 s D)
//   tlo = t - 2.5 s D - max(1e-4, 8u t)                  (D < s; tlo < 0 never fires, err_fused >= 0)
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
// t, s = sqrt(t), 2.5 s and the rounding term come from a (set_fused_cut)
__device__ __forceinline__ void fused_thresholds(const float (&h)[8], float cmax, const FhArgs& a, bool exact_only,
                                                 float& tlo, float& thi) {
    const float t = a.thresh2, s = a.thresh_sqrt, rnd = a.cut_rnd;
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
    thi = t + 1.25f * (2.f * D * D + 2.f * D * sqrtf(D * D + t)) + rnd;
    if (D < s) tlo = t - a.cut_k * D - rnd;
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
            fused_thresholds(hf[j], cmax, a, a.exact_only != 0, tlo[j], thi[j]);
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
        fused_thresholds(hf, cmax, a, a.exact_only != 0, tlo, thi);
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
                fused_thresholds(hf, cmax, a, false, tlo, thi);
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

}  // namespace evz

// host: launches the scoring kernel of evz_find_homography_adaptive (ransac_adaptive.cu) with `smem` bytes of dynamic
// shared memory (the points and their positions, as for ransac_score_kernel)
int evz_launch_adaptive_score(evz_handle* h, const evz::FhArgs& a, double confidence, int32_t* n_used, double* Hbest,
                              int32_t* phase, int n_pairs, int smem, cudaStream_t st);
