// Confidence-bounded RANSAC stop of evz_find_homography_adaptive: the scoring stage for OpenCV's iteration bound.  The
// refit is ransac_refit_kernel's (ransac_kernels.cu), fed through the same Hbest / phase hand-over.
//
// Compiled with --fmad=false like ransac_kernels.cu: the sampler, the 4-point solve and the count formulas are the shared
// helpers of ransac_device.cuh and must round exactly as there.
#include "ransac_device.cuh"

namespace evz {

// OpenCV's RANSACUpdateNumIters(p, ep, 4, max_iters) (ptsetreg.cpp), literally: the number of iterations after which a
// model with inlier ratio 1 - ep would have been drawn from an all-inlier sample with probability p
__device__ __forceinline__ int ransac_update_num_iters(double p, double ep, int max_iters) {
    p = fmin(fmax(p, 0.0), 1.0);
    ep = fmin(fmax(ep, 0.0), 1.0);
    double num = fmax(1.0 - p, DBL_MIN);
    double denom = 1.0 - pow(1.0 - ep, 4);
    if (denom < DBL_MIN) return 0;
    num = log(num);
    denom = log(denom);
    return denom >= 0 || -num >= max_iters * (-denom) ? max_iters : __double2int_rn(num / denom);
}

constexpr int kAdGrp0 = 32;       // hypotheses of the first group: at >= 80 % inliers the bound is ~10
constexpr int kAdGrpMax = 512;    // groups grow x4 up to this size
constexpr uint16_t kAdInvalid = 0xFFFF;

// Stages the point pairs of pair p in shared memory and returns the block's maximum |coordinate|: the staging of
// ransac_score_kernel (whose inline copy is kept as it is so that its code does not change).
__device__ __forceinline__ float ad_stage_points(const FhArgs& a, int p, int m, int64_t o, float4* pts, uint16_t* pos,
                                                 uint64_t* stage_bar, float* cmax_s) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
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
        if (tid == 0) { mbar_init(stage_bar, 1); fence_mbar_init(); }
        __syncthreads();
        if (tid == 0) {
            mbar_arrive_expect_tx(stage_bar, static_cast<uint32_t>(m) * 16u);
            bulk_load_1d(pts, reinterpret_cast<const float4*>(a.pts) + o, static_cast<uint32_t>(m) * 16u, stage_bar);
        }
        for (int i = tid; i < m; i += blockDim.x) pos[i] = static_cast<uint16_t>(i);
        mbar_wait(stage_bar, 0);
        for (int i = tid; i < m; i += blockDim.x) {
            const float4 v = pts[i];
            cmax = fmaxf(cmax, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
        }
    }
#pragma unroll
    for (int of = 16; of > 0; of >>= 1) cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffff, cmax, of));
    if (lane == 0) cmax_s[warp] = cmax;
    __syncthreads();
#pragma unroll
    for (int w = 0; w < kRsThreads / 32; ++w) cmax = fmaxf(cmax, cmax_s[w]);
    return cmax;
}

// The scoring stage of evz_find_homography_adaptive: one CTA per pair walks the hypothesis stream 0, 1, .. n_hyp - 1 in
// index-ordered groups (kAdGrp0, then x4 up to kAdGrpMax) and stops where OpenCV's RANSAC loop would.  Per group:
//   pass 0   sample + solve + validity test of every hypothesis of the group, ordered compaction (safe denominators
//            first, as in ransac_score_kernel); the f32 models go to the model cache;
//   scoring  score_slots over all matches (fused bounds [lo, hi]);  a hypothesis whose count can be neither the new best
//            nor, while no model has more than 3 inliers, the fallback arg-max (hi <= best at group start, best >= 4) is
//            settled without its exact count; lo == hi is exact; the rest are rescored exactly, one warp each;
//   walk     warp 0 applies the update / stop rule in index order, 32 hypotheses per step: it counts the valid ones,
//            finds the first that beats max(best, 3) and the first at which it >= niters, and recomputes niters at
//            every new best (rare: the walk costs a few ballots per 32 hypotheses).
// The (count desc, index asc) arg-max over the consumed prefix goes to the refit kernel through Hbest / phase exactly as
// from ransac_score_kernel, so every output equals evz_find_homography's with n_hyp = n_used[p].  Only group-sized lists
// live in shared memory.
__global__ void __launch_bounds__(kRsThreads, 2)
ransac_adaptive_kernel(const FhArgs a, double confidence, int32_t* __restrict__ n_used, double* __restrict__ Hbest_out,
                       int32_t* __restrict__ phase) {
    extern __shared__ __align__(16) uint8_t fh_smem[];
    float4* pts = reinterpret_cast<float4*>(fh_smem);
    uint16_t* pos = reinterpret_cast<uint16_t*>(fh_smem + static_cast<size_t>(a.max_cnt) * 16);
    __shared__ uint16_t vlist[kAdGrpMax], slist[kAdGrpMax], lo_s[kAdGrpMax], hi_s[kAdGrpMax];
    __shared__ uint16_t gcnt[kAdGrpMax];         // per hypothesis of the group: exact count, 0 if settled, kAdInvalid
    __shared__ float cmax_s[kRsThreads / 32];
    __shared__ int warp_sums[2 * (kRsThreads / 32)];
    __shared__ int part_s[2 * kRsThreads];
    __shared__ int s_nsurv, s_lbest, s_cut, s_best, s_stop, s_flag;
    __shared__ unsigned long long s_key;
    __shared__ __align__(8) uint64_t stage_bar;

    const int p = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) { phase[p] = 0; if (n_used) n_used[p] = 0; }
    const int st_p = a.status[p];
    const int m = a.cnt[p];
    const int64_t o = a.off[p];
    if (st_p != EVZ_ST_OK) return;
    if (m < 4) { if (tid == 0) a.status[p] = EVZ_ST_FEW_POINTS; return; }
    if (m > a.max_cnt) { if (tid == 0) a.status[p] = a.fail_status; return; }
    const float cmax = ad_stage_points(a, p, m, o, pts, pos, &stage_bar, cmax_s);
    const uint32_t pair_level = static_cast<uint32_t>((a.pair_ids ? a.pair_ids[p] : a.pair_id_base + p) * 2 + a.level);
    if (m == 4) {
        // the m == 4 path of ransac_score_kernel: exact model through the 4 points, mask = ones, no LM
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
    if (tid == 0) { s_lbest = 0; s_cut = 0x7FFFFFFF; s_best = 0; s_stop = 0; s_key = 0; }
    // walk state, held by warp 0 (uniform across its lanes)
    int best = 0, niters = a.n_hyp, it = 0, used = a.n_hyp;
    bool stop = false;
    unsigned long long key = 0;        // (count << 32) | ~hyp over the consumed prefix, counts > 0 only
    const bool settle = a.no_prune == 0;
    for (int g0 = 0, G = kAdGrp0; g0 < a.n_hyp; g0 += G, G = min(G * 4, kAdGrpMax)) {
        const int gn = min(G, a.n_hyp - g0);
        // ---- pass 0 of the group
        int base = 0, base_u = 0;
        for (int r0 = 0; r0 < gn; r0 += kRsThreads) {
            const int j = r0 + tid, hyp = g0 + j;
            int ok = 0, safe = 0;
            if (j < gn) {
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
                gcnt[j] = ok ? 0 : kAdInvalid;
                lo_s[j] = 0; hi_s[j] = 0;
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
        if (tid == 0) s_nsurv = 0;
        __syncthreads();
        const int n_valid = base + base_u;
        // ---- fused count bounds of the valid hypotheses of the group over all matches
        score_slots(a, pts, pos, vlist, lo_s, hi_s, part_s, &s_lbest, &s_cut, 0, n_valid, base, m, cmax, pair_level, false,
                    false, PtRange{0, m, kFull});
        __syncthreads();
        // a count <= the best at group start (>= 4) can change neither the winner nor niters
        const int thr = settle && s_best >= 4 ? s_best : 0;
        for (int slot = tid; slot < n_valid; slot += kRsThreads) {
            const int hyp = vlist[slot], lo = lo_s[slot], hi = hi_s[slot];
            if (hi <= thr) gcnt[hyp - g0] = 0;
            else if (lo == hi) gcnt[hyp - g0] = static_cast<uint16_t>(lo);
            else slist[atomicAdd(&s_nsurv, 1)] = static_cast<uint16_t>(hyp);
        }
        __syncthreads();
        const int n_surv = s_nsurv;
        for (int k = warp; k < n_surv; k += kRsThreads / 32) {
            const int hyp = slist[k];
            float hf[8];
            hyp_model(a, pts, pos, hyp, m, pair_level, hf);
            int c = 0;
            for (int i0 = 0; i0 < m; i0 += 32) {
                const int i = i0 + lane;
                const bool in = i < m && reproj_err32(hf, pts[i]) <= a.thresh2;
                c += __popc(__ballot_sync(0xffffffff, in));
            }
            if (lane == 0) gcnt[hyp - g0] = static_cast<uint16_t>(c);
        }
        __syncthreads();
        // ---- the update / stop rule in index order
        if (warp == 0) {
            for (int c0 = 0; c0 < gn && !stop; c0 += 32) {
                const int j = c0 + lane;
                const int g = j < gn ? gcnt[j] : kAdInvalid;
                const bool valid = g != kAdInvalid;
                const int c = valid ? g : 0;
                const unsigned vb = __ballot_sync(0xffffffff, valid);
                const int itl = it + __popc(vb & (lane == 31 ? 0xffffffffu : (2u << lane) - 1u));
                int end = 32, from = 0;
                while (true) {
                    const unsigned um = __ballot_sync(0xffffffff, valid && lane >= from && c > max(best, 3));
                    const unsigned sm = __ballot_sync(0xffffffff, valid && lane >= from && itl >= niters);
                    const int u = um ? __ffs(um) - 1 : 32, s = sm ? __ffs(sm) - 1 : 32;
                    if (s < u) { end = s + 1; stop = true; break; }
                    if (u == 32) break;
                    best = __shfl_sync(0xffffffff, c, u);
                    niters = ransac_update_num_iters(confidence, static_cast<double>(m - best) / m, niters);
                    if (__shfl_sync(0xffffffff, itl, u) >= niters) { end = u + 1; stop = true; break; }
                    from = u + 1;
                }
                unsigned long long k = valid && lane < end && c > 0
                    ? (static_cast<unsigned long long>(static_cast<uint32_t>(c)) << 32) | (0xFFFFFFFFu - static_cast<uint32_t>(g0 + j))
                    : 0ull;
#pragma unroll
                for (int of = 16; of > 0; of >>= 1) { const unsigned long long v = __shfl_xor_sync(0xffffffff, k, of); k = v > k ? v : k; }
                key = k > key ? k : key;
                it += __popc(vb);
                if (stop) used = g0 + c0 + end;
            }
            if (lane == 0) { s_best = best; s_stop = stop; s_key = key; }
        }
        __syncthreads();
        if (s_stop) break;
    }
    if (tid == 0) {
        const unsigned long long k = s_key;
        const int bc = static_cast<int>(k >> 32);
        const int bh = k ? static_cast<int>(0xFFFFFFFFu - static_cast<uint32_t>(k & 0xFFFFFFFFu)) : -1;
        if (n_used) n_used[p] = used;
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

}  // namespace evz

int evz_launch_adaptive_score(evz_handle* h, const evz::FhArgs& a, double confidence, int32_t* n_used, double* Hbest,
                              int32_t* phase, int n_pairs, int smem, cudaStream_t st) {
    if (smem > h->attr_score_a) {
        EVZ_CUDA_CHECK(h, cudaFuncSetAttribute(evz::ransac_adaptive_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        h->attr_score_a = smem;
    }
    evz::ransac_adaptive_kernel<<<n_pairs, evz::kRsThreads, smem, st>>>(a, confidence, n_used, Hbest, phase);
    EVZ_LAUNCH_CHECK(h);
    return EVZ_OK;
}
