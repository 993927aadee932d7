// K5 static-point filter, K6 None-H fallback + cumulative superposition (parallel prefix product
// of 3x3 f64 matrices), K7 object-coordinate remap, dense max-movement metric.
// All HBM-bound f64 work; compiled with --fmad=false so that the rounded displacement bins of K5
// are computed with the same individually rounded operations as the oracle.
#include "evz_common.cuh"
#include <climits>

namespace evz {

// ------------------------------------------------------------------------------------ K5
// one CTA per pair; histogram of rounded displacements in shared memory:
//   hist  uint32 [(R_MAX+2)/2]  two 16-bit counters per word,  first int32 [R_MAX+2] first index per bin
constexpr int kBins = EVZ_R_MAX + 2;      // bin R_MAX+1 collects overflow / non-finite

__device__ __forceinline__ int disp_bin(const double* H, const float4 p) {
    const double ax = p.x, ay = p.y, bx = p.z, by = p.w;
    const double X = (H[0] * ax + H[1] * ay) + H[2];
    const double Y = (H[3] * ax + H[4] * ay) + H[5];
    const double W = (H[6] * ax + H[7] * ay) + H[8];
    const double dx = X / W - bx, dy = Y / W - by;
    const double dist = sqrt(dx * dx + dy * dy);
    if (!(dist <= static_cast<double>(EVZ_R_MAX))) return EVZ_R_MAX + 1;     // also catches NaN
    return static_cast<int>(rint(dist));                                      // half-to-even, like Python round()
}

constexpr int kSfWindow = 2048;            // displacement bins histogrammed at a time (the used range is usually < 100 wide)

// One CTA per pair.  Pass A computes every point's rounded displacement once (f64) into shared memory and
// the used range [rmin, rmax]; the histogram / first-occurrence tables only cover windows of that range
// (typically a single window), instead of zeroing and scanning all EVZ_R_MAX + 2 bins; the compaction
// compares the cached bins.  Shared memory: u16 r[EVZ_MAX_KP] | u32 hist[kSfWindow] | i32 first[kSfWindow].
__global__ void __launch_bounds__(256)
static_filter_kernel(const float* __restrict__ pts, const int32_t* __restrict__ off, const int32_t* __restrict__ cnt,
                     const double* __restrict__ Hs, const int32_t* __restrict__ status,
                     float* __restrict__ out_pts, int32_t* __restrict__ out_cnt, int32_t* __restrict__ best_r,
                     int32_t* __restrict__ flags, int32_t* __restrict__ r_out) {
    extern __shared__ __align__(16) uint8_t sf_smem[];
    uint16_t* r_s = reinterpret_cast<uint16_t*>(sf_smem);
    uint32_t* hist = reinterpret_cast<uint32_t*>(sf_smem + EVZ_MAX_KP * 2);
    int32_t* first = reinterpret_cast<int32_t*>(hist + kSfWindow);
    __shared__ unsigned long long red[8];
    __shared__ int warp_sums[32];
    __shared__ int s_best, s_rmin, s_rmax;
    const int p = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (status[p] != EVZ_ST_OK) { if (tid == 0) { out_cnt[p] = 0; best_r[p] = -1; flags[p] = 0; } return; }
    // the host entry point refuses max_cnt > EVZ_MAX_KP; a pair that exceeds it anyway (the caller's bound was wrong)
    // is reported, not truncated
    if (cnt[p] > EVZ_MAX_KP) { if (tid == 0) { out_cnt[p] = 0; best_r[p] = -1; flags[p] = EVZ_FLAG_TOO_MANY_POINTS; } return; }
    const int m = cnt[p];
    const int64_t o = off[p];
    double H[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) H[i] = Hs[static_cast<size_t>(p) * 9 + i];
    if (tid == 0) { s_rmin = INT_MAX; s_rmax = -1; }
    __syncthreads();
    const float4* P = reinterpret_cast<const float4*>(pts) + o;
    int rmin = INT_MAX, rmax = -1;
    for (int i = tid; i < m; i += blockDim.x) {
        const int r = disp_bin(H, P[i]);
        if (r_out) r_out[o + i] = r;
        r_s[i] = static_cast<uint16_t>(r);
        rmin = min(rmin, r); rmax = max(rmax, r);
    }
#pragma unroll
    for (int of = 16; of > 0; of >>= 1) {
        rmin = min(rmin, __shfl_xor_sync(0xffffffff, rmin, of));
        rmax = max(rmax, __shfl_xor_sync(0xffffffff, rmax, of));
    }
    if (lane == 0 && rmax >= 0) { atomicMin(&s_rmin, rmin); atomicMax(&s_rmax, rmax); }
    __syncthreads();
    rmin = s_rmin; rmax = s_rmax;
    // arg-max over bins: (count desc, first-inserted asc)  == reference's strict '>' over dict order
    unsigned long long key = 0;
    for (int w0 = rmin; w0 <= rmax; w0 += kSfWindow) {
        for (int i = tid; i < kSfWindow; i += blockDim.x) { hist[i] = 0; first[i] = INT_MAX; }
        __syncthreads();
        for (int i = tid; i < m; i += blockDim.x) {
            const int b = static_cast<int>(r_s[i]) - w0;
            if (b >= 0 && b < kSfWindow) { atomicAdd(&hist[b], 1u); atomicMin(&first[b], i); }
        }
        __syncthreads();
        for (int b = tid; b < kSfWindow; b += blockDim.x) {
            const unsigned int c = hist[b];
            if (c) {
                const unsigned long long k = (static_cast<unsigned long long>(c) << 48) |
                                             (static_cast<unsigned long long>(0xFFFFFFu - static_cast<unsigned int>(first[b])) << 24) |
                                             static_cast<unsigned long long>(b + w0);
                key = k > key ? k : key;
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int of = 16; of > 0; of >>= 1) { const unsigned long long u = __shfl_xor_sync(0xffffffff, key, of); key = u > key ? u : key; }
    if (lane == 0) red[warp] = key;
    __syncthreads();
    if (tid == 0) {
        unsigned long long k = red[0];
        for (int w = 1; w < 8; ++w) k = red[w] > k ? red[w] : k;
        s_best = m > 0 ? static_cast<int>(k & 0xFFFFFFu) : -1;
    }
    __syncthreads();
    const int best = s_best;
    int base = 0;
    for (int ib = 0; ib < m; ib += blockDim.x) {
        const int i = ib + tid;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        int keep = 0;
        if (i < m) { v = P[i]; keep = static_cast<int>(r_s[i]) == best; }
        // block exclusive scan of keep
        int incl = keep;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffff, incl, d); if (lane >= d) incl += t; }
        if (lane == 31) warp_sums[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int w = lane < 8 ? warp_sums[lane] : 0;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffff, w, d); if (lane >= d) w += t; }
            warp_sums[lane] = w;
        }
        __syncthreads();
        const int pos = base + incl - keep + (warp > 0 ? warp_sums[warp - 1] : 0);
        if (keep) reinterpret_cast<float4*>(out_pts)[o + pos] = v;
        base += warp_sums[7];
        __syncthreads();
    }
    if (tid == 0) { out_cnt[p] = base; best_r[p] = best; flags[p] = rmax > EVZ_R_MAX ? EVZ_FLAG_DISP_OVERFLOW : 0; }
}

// ------------------------------------------------------------------------------------ K6
struct M3 { double m[9]; };

__device__ __forceinline__ M3 m3_identity() { M3 r; for (int i = 0; i < 9; ++i) r.m[i] = (i % 4 == 0) ? 1.0 : 0.0; return r; }
__device__ __forceinline__ M3 m3_load(const double* p) { M3 r; for (int i = 0; i < 9; ++i) r.m[i] = p[i]; return r; }
__device__ __forceinline__ void m3_store(double* p, const M3& a) { for (int i = 0; i < 9; ++i) p[i] = a.m[i]; }
// a . b inside the scan.  The reference divides the running product by its [2][2] at every step (utils.py:139-145);
// a homography is defined up to scale, so only the matrices that are STORED need that normalisation.  Inside the
// tree the partial products (G3 . G4, block totals: products the reference never forms) are kept in range by an
// exact power-of-two scale instead -- a partial product whose [2][2] happens to be ~0 must not poison its prefix.
__device__ __forceinline__ M3 m3_mul_scaled(const M3& a, const M3& b) {
    M3 r;
    double mx = 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            r.m[3 * i + j] = (a.m[3 * i] * b.m[j] + a.m[3 * i + 1] * b.m[3 + j]) + a.m[3 * i + 2] * b.m[6 + j];
            mx = fmax(mx, fabs(r.m[3 * i + j]));
        }
    if (mx > 0.0 && mx < 1.0 / 0.0) {
        const int e = -ilogb(mx);
#pragma unroll
        for (int i = 0; i < 9; ++i) r.m[i] = scalbn(r.m[i], e);
    }
    return r;
}
__device__ __forceinline__ M3 m3_norm22(const M3& a) {
    M3 r;
    const double s = a.m[8];
#pragma unroll
    for (int i = 0; i < 9; ++i) r.m[i] = a.m[i] / s;
    return r;
}
// normalise(a . b), for the few products that are stored directly
__device__ __forceinline__ M3 m3_mul_norm(const M3& a, const M3& b) { return m3_norm22(m3_mul_scaled(a, b)); }
__device__ __forceinline__ M3 m3_inverse(const M3& a) {
    const double* m = a.m;
    M3 r;
    r.m[0] = m[4] * m[8] - m[5] * m[7]; r.m[1] = m[2] * m[7] - m[1] * m[8]; r.m[2] = m[1] * m[5] - m[2] * m[4];
    r.m[3] = m[5] * m[6] - m[3] * m[8]; r.m[4] = m[0] * m[8] - m[2] * m[6]; r.m[5] = m[2] * m[3] - m[0] * m[5];
    r.m[6] = m[3] * m[7] - m[4] * m[6]; r.m[7] = m[1] * m[6] - m[0] * m[7]; r.m[8] = m[0] * m[4] - m[1] * m[3];
    const double det = m[0] * r.m[0] + m[1] * r.m[3] + m[2] * r.m[6];
    const double inv = 1.0 / det;
#pragma unroll
    for (int i = 0; i < 9; ++i) r.m[i] *= inv;
    return r;
}
__device__ __forceinline__ M3 m3_shfl_up(const M3& a, int d) {
    M3 r;
#pragma unroll
    for (int i = 0; i < 9; ++i) r.m[i] = __shfl_up_sync(0xffffffff, a.m[i], d);
    return r;
}

constexpr int kScanBlock = 256;

// The scan kernels run over one chain (seg_blk = null: block b covers pairs [256 b, 256 b + 256) of n) or over several
// independent chains (evz_chain_scan_segments): segment s holds pairs [seg_off[s], seg_off[s+1]) and owns the block slots
// [seg_blk[s], seg_blk[s+1]), one per 256 pairs counted from the segment's own start, so that every block of a segment
// computes exactly what the one-chain scan of that segment alone computes in the same block.  Indices inside a segment
// (k, src[]) are segment-relative; `base` turns them into rows of G / S / H_fixed.
struct ScanBlock { int base, n, blk, slot; };
// false: a surplus block of the segmented grid (the grid is sized by a host-known bound)
__device__ __forceinline__ bool scan_block(const int32_t* seg_off, const int32_t* seg_blk, int n_segs, int n, ScanBlock& sb) {
    const int g = blockIdx.x;
    if (!seg_blk) { sb.base = 0; sb.n = n; sb.blk = g; sb.slot = g; return true; }
    if (g >= seg_blk[n_segs]) return false;
    int lo = 0, hi = n_segs - 1;                                  // last s with seg_blk[s] <= g (a non-empty segment)
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (seg_blk[mid] <= g) lo = mid; else hi = mid - 1; }
    sb.base = seg_off[lo]; sb.n = seg_off[lo + 1] - seg_off[lo]; sb.blk = g - seg_blk[lo]; sb.slot = g;
    return true;
}
// segmented scan set-up (single CTA): seg_blk[s] = sum over s' < s of ceil(len(s') / 256)
__global__ void __launch_bounds__(kScanBlock)
seg_blocks_kernel(const int32_t* __restrict__ seg_off, int n_segs, int32_t* __restrict__ seg_blk) {
    __shared__ int ws[kScanBlock / 32];
    __shared__ int carry_s;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int carry = 0;
    for (int s0 = 0; s0 < n_segs; s0 += kScanBlock) {
        const int s = s0 + threadIdx.x;
        const int nb = s < n_segs ? (seg_off[s + 1] - seg_off[s] + kScanBlock - 1) / kScanBlock : 0;
        int v = nb;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffff, v, d); if (lane >= d) v += t; }
        if (lane == 31) ws[warp] = v;
        __syncthreads();
        int c = carry;
        for (int w = 0; w < warp; ++w) c += ws[w];
        if (s < n_segs) seg_blk[s] = c + v - nb;
        if (threadIdx.x == kScanBlock - 1) carry_s = c + v;
        __syncthreads();
        carry = carry_s;
        __syncthreads();
    }
    if (threadIdx.x == 0) seg_blk[n_segs] = carry;
}

// phase A1: src[k] = index of the last valid pair at or before k within the block (or -1);
// block_last[b] = last valid index of block b (or -1)
__global__ void __launch_bounds__(kScanBlock)
fill_local_kernel(const int32_t* __restrict__ status, int n, int32_t* __restrict__ src, int32_t* __restrict__ block_last,
                  const int32_t* __restrict__ seg_off, const int32_t* __restrict__ seg_blk, int n_segs) {
    __shared__ int ws[kScanBlock / 32];
    ScanBlock sb;
    if (!scan_block(seg_off, seg_blk, n_segs, n, sb)) return;
    const int k = sb.blk * kScanBlock + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int v = (k < sb.n && status[sb.base + k] == EVZ_ST_OK) ? k : -1;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffff, v, d); if (lane >= d) v = max(v, t); }
    if (lane == 31) ws[warp] = v;
    __syncthreads();
    int carry = -1;
    for (int w = 0; w < warp; ++w) carry = max(carry, ws[w]);
    v = max(v, carry);
    if (k < sb.n) src[sb.base + k] = v;
    if (threadIdx.x == kScanBlock - 1) block_last[sb.slot] = v;
}
// phase A2 (one CTA per segment): running max over block_last -> block_carry[b] = last valid before block b
__global__ void fill_carry_kernel(const int32_t* __restrict__ block_last, int nb, int32_t* __restrict__ block_carry,
                                  const int32_t* __restrict__ seg_blk) {
    if (threadIdx.x == 0) {
        const int b0 = seg_blk ? seg_blk[blockIdx.x] : 0, b1 = seg_blk ? seg_blk[blockIdx.x + 1] : nb;
        int c = -1;
        for (int b = b0; b < b1; ++b) { block_carry[b] = c; c = max(c, block_last[b]); }
    }
}
// phase A3: fold the cross-block carry into src
__global__ void __launch_bounds__(kScanBlock)
fill_apply_kernel(int32_t* __restrict__ src, const int32_t* __restrict__ block_carry, int n,
                  const int32_t* __restrict__ seg_off, const int32_t* __restrict__ seg_blk, int n_segs) {
    ScanBlock sb;
    if (!scan_block(seg_off, seg_blk, n_segs, n, sb)) return;
    const int k = sb.blk * kScanBlock + threadIdx.x;
    if (k < sb.n) src[sb.base + k] = max(src[sb.base + k], block_carry[sb.slot]);
}
// phase B1: Gf[k] = filled step matrix; local inclusive product scan; block totals.  Only block 0 of an unseeded scan holds
// true prefixes, which are normalised here; every other block stores its block-local prefix (a partial product, whose
// [2][2] may be 0) with its power-of-two scale, and prod_apply_kernel normalises it once the carry is applied.
__global__ void __launch_bounds__(kScanBlock)
prod_local_kernel(const double* __restrict__ G, const int32_t* __restrict__ src,
                  int n, int policy, const double* __restrict__ seed_G, int has_seed,
                  double* __restrict__ S, double* __restrict__ block_tot,
                  const int32_t* __restrict__ seg_off, const int32_t* __restrict__ seg_blk, int n_segs) {
    __shared__ double wt[kScanBlock / 32][9];
    ScanBlock sb;
    if (!scan_block(seg_off, seg_blk, n_segs, n, sb)) return;
    const int k = sb.blk * kScanBlock + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    M3 v = m3_identity();
    if (k < sb.n) {
        int s = src[sb.base + k];
        if (policy == 0 && s != k) s = -2;                       // identity step for an invalid pair
        if (s >= 0) v = m3_load(G + static_cast<size_t>(sb.base + s) * 9);
        else if (s == -1 && policy != 0 && seed_G) v = m3_load(seed_G);
    }
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const M3 t = m3_shfl_up(v, d);
        if (lane >= d) v = m3_mul_scaled(t, v);
    }
    if (lane == 31) m3_store(wt[warp], v);
    __syncthreads();
    if (warp > 0) {
        M3 c = m3_load(wt[0]);
        for (int w = 1; w < warp; ++w) c = m3_mul_scaled(c, m3_load(wt[w]));
        v = m3_mul_scaled(c, v);
    }
    if (k < sb.n) m3_store(S + static_cast<size_t>(sb.base + k) * 9, (sb.blk == 0 && !has_seed) ? m3_norm22(v) : v);
    if (threadIdx.x == kScanBlock - 1) m3_store(block_tot + static_cast<size_t>(sb.slot) * 9, v);
}
// phase B2 (one CTA per segment): exclusive prefix of the block totals, seeded.  Block-wide shuffle scan over
// chunks of kScanBlock totals (a serial loop over blocks costs ~1 us per block: L2 latency + f64 divides)
__global__ void __launch_bounds__(kScanBlock)
prod_carry_kernel(const double* __restrict__ block_tot, int nb, const double* __restrict__ seed_S,
                  double* __restrict__ block_pre, const int32_t* __restrict__ seg_blk) {
    __shared__ double wt[kScanBlock / 32][9];
    __shared__ double carry_s[9];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (seg_blk) {
        const int b0 = seg_blk[blockIdx.x];
        nb = seg_blk[blockIdx.x + 1] - b0;
        block_tot += static_cast<size_t>(b0) * 9;
        block_pre += static_cast<size_t>(b0) * 9;
    }
    M3 carry = seed_S ? m3_load(seed_S) : m3_identity();
    for (int b0 = 0; b0 < nb; b0 += kScanBlock) {
        const int b = b0 + threadIdx.x;
        M3 v = b < nb ? m3_load(block_tot + static_cast<size_t>(b) * 9) : m3_identity();
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const M3 t = m3_shfl_up(v, d);
            if (lane >= d) v = m3_mul_scaled(t, v);
        }
        if (lane == 31) m3_store(wt[warp], v);
        __syncthreads();
        M3 c = carry;
        for (int w = 0; w < warp; ++w) c = m3_mul_scaled(c, m3_load(wt[w]));
        const M3 incl = m3_mul_scaled(c, v);                       // inclusive prefix through block b
        // exclusive prefix = inclusive prefix of the previous block
        M3 excl = m3_shfl_up(incl, 1);
        if (lane == 0) excl = c;
        if (b < nb) m3_store(block_pre + static_cast<size_t>(b) * 9, excl);
        if (threadIdx.x == kScanBlock - 1) m3_store(carry_s, incl);
        __syncthreads();
        carry = m3_load(carry_s);
        __syncthreads();
    }
}
// phase B3: S[k] = block_pre[b] . S_local[k]
__global__ void __launch_bounds__(kScanBlock)
prod_apply_kernel(double* __restrict__ S, const double* __restrict__ block_pre, int n, int has_seed,
                  const int32_t* __restrict__ seg_off, const int32_t* __restrict__ seg_blk, int n_segs) {
    ScanBlock sb;
    if (!scan_block(seg_off, seg_blk, n_segs, n, sb)) return;
    const int k = sb.blk * kScanBlock + threadIdx.x;
    if (k >= sb.n || (sb.blk == 0 && !has_seed)) return;
    double* Sk = S + static_cast<size_t>(sb.base + k) * 9;
    m3_store(Sk, m3_mul_norm(m3_load(block_pre + static_cast<size_t>(sb.slot) * 9), m3_load(Sk)));
}
// H_fixed[k] = normalise(S[k] . S[k-1]^-1)
__global__ void __launch_bounds__(kScanBlock)
fixed_plane_kernel(const double* __restrict__ S, const double* __restrict__ seed_S, int n, double* __restrict__ Hf,
                   const int32_t* __restrict__ seg_off, const int32_t* __restrict__ seg_blk, int n_segs) {
    ScanBlock sb;
    if (!scan_block(seg_off, seg_blk, n_segs, n, sb)) return;
    const int k = sb.blk * kScanBlock + threadIdx.x;
    if (k >= sb.n) return;
    const double* Sk = S + static_cast<size_t>(sb.base + k) * 9;
    const M3 prev = k > 0 ? m3_load(Sk - 9) : (seed_S ? m3_load(seed_S) : m3_identity());
    m3_store(Hf + static_cast<size_t>(sb.base + k) * 9, m3_mul_norm(m3_load(Sk), m3_inverse(prev)));
}

// Reference-exact chain step (video_processing.py:119-149 on the device), one thread per chain c:
//   H = H2[c] if status[c] == EVZ_ST_OK, else H_prev[c] if policy and not first, else the identity;  H_out[c] = H;
//   S_state[c] = H if first, else C / C[2][2] with C = H . S_state[c].
// The product uses one fixed operation order, fma(H[i][2], S[2][j], fma(H[i][1], S[1][j], H[i][0] * S[0][j])), followed by
// an IEEE division: the order in which NumPy's np.dot (OpenBLAS dgemm) forms a 3x3 f64 product, so the device chain
// follows the host loop bit for bit wherever the host's BLAS does the same.  H_prev may alias H_out (each thread reads
// its own row before it writes it).
__global__ void __launch_bounds__(kScanBlock)
chain_ref_step_kernel(const double* __restrict__ H2, const int32_t* __restrict__ status, int n, int first, int policy,
                      double* __restrict__ S_state, const double* H_prev, double* H_out) {
    const int c = blockIdx.x * kScanBlock + threadIdx.x;
    if (c >= n) return;
    M3 H;
    if (status[c] == EVZ_ST_OK) H = m3_load(H2 + static_cast<size_t>(c) * 9);
    else if (policy && !first) H = m3_load(H_prev + static_cast<size_t>(c) * 9);
    else H = m3_identity();
    m3_store(H_out + static_cast<size_t>(c) * 9, H);
    double* Sc = S_state + static_cast<size_t>(c) * 9;
    if (first) { m3_store(Sc, H); return; }
    const M3 S = m3_load(Sc);
    M3 R;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j)
            R.m[3 * i + j] = __fma_rn(H.m[3 * i + 2], S.m[6 + j], __fma_rn(H.m[3 * i + 1], S.m[3 + j], __dmul_rn(H.m[3 * i], S.m[j])));
    const double d = R.m[8];
#pragma unroll
    for (int i = 0; i < 9; ++i) Sc[i] = __ddiv_rn(R.m[i], d);
}
// shard summary for the cross-GPU all-gather (see evz.h)
__global__ void summary_kernel(const double* __restrict__ G, const int32_t* __restrict__ src, const double* __restrict__ S_noseed_tot,
                               int n, double* __restrict__ summary) {
    if (threadIdx.x != 0) return;
    const int last = src[n - 1];
    for (int i = 0; i < 9; ++i) summary[i] = S_noseed_tot[i];
    for (int i = 0; i < 9; ++i) summary[9 + i] = last >= 0 ? G[static_cast<size_t>(last) * 9 + i] : ((i % 4 == 0) ? 1.0 : 0.0);
    int lead = 0;
    if (last < 0) lead = n;
    else { int lo = 0, hi = n - 1; while (lo < hi) { const int mid = (lo + hi) / 2; if (src[mid] >= 0) hi = mid; else lo = mid + 1; } lead = lo; }
    summary[18] = static_cast<double>(lead);
    summary[19] = last >= 0 ? 1.0 : 0.0;
}

// ---- cross-GPU seeding on the device (port of evenvizion_b200/distributed.py::seeds_from_summaries).
// summaries: [world][20] as written by summary_kernel on every rank and all-gathered.  Single thread:
//   seed_S  superposition before this rank's first pair, seed_G last valid step before it (identity when there is none,
//           which is what an absent seed means to the fill), A = seed_S . seed_G^lead = the factor that turns this rank's
//           UNSEEDED local scan into the global one from its first valid pair on (lead = its number of leading
//           invalid pairs); the first `lead` rows of S (S_k = seed_S . seed_G^(k+1)) are written here, serially.
// seeds_out: [27] = seed_S | seed_G | A
__global__ void seed_kernel(const double* __restrict__ summaries, int world, int rank, int policy, int n,
                            double* __restrict__ S, double* __restrict__ seeds_out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    M3 Sm = m3_identity(), lastG = m3_identity();
    bool have = false;
    for (int r = 0; r < rank; ++r) {
        const double* s = summaries + static_cast<size_t>(r) * 20;
        const int lead = static_cast<int>(s[18] + 0.5);
        if (policy != 0 && have)
            for (int i = 0; i < lead; ++i) Sm = m3_mul_norm(Sm, lastG);       // leading failures of shard r repeat the carried step
        if (s[19] > 0.5) { Sm = m3_mul_norm(Sm, m3_load(s)); lastG = m3_load(s + 9); have = true; }
    }
    const M3 G = (policy != 0 && have) ? lastG : m3_identity();
    m3_store(seeds_out, Sm);
    m3_store(seeds_out + 9, G);
    const int lead = min(n, static_cast<int>(summaries[static_cast<size_t>(rank) * 20 + 18] + 0.5));
    M3 A = Sm;
    for (int k = 0; k < lead; ++k) { A = m3_mul_norm(A, G); m3_store(S + static_cast<size_t>(k) * 9, A); }
    m3_store(seeds_out + 18, A);
}
// S[k] = normalise(A . S_local[k]) for the pairs from the first valid one on
__global__ void __launch_bounds__(kScanBlock)
seed_apply_kernel(double* __restrict__ S, const double* __restrict__ summaries, int rank, const double* __restrict__ seeds, int n) {
    const int k = blockIdx.x * kScanBlock + threadIdx.x;
    const int lead = static_cast<int>(summaries[static_cast<size_t>(rank) * 20 + 18] + 0.5);
    if (k >= n || k < lead) return;
    m3_store(S + static_cast<size_t>(k) * 9, m3_mul_norm(m3_load(seeds + 18), m3_load(S + static_cast<size_t>(k) * 9)));
}

// ------------------------------------------------------------------------------------ K7
__global__ void __launch_bounds__(256)
remap_kernel(const double* __restrict__ pin, const int32_t* __restrict__ frame_idx, int64_t n,
             const double* __restrict__ S, double sx, double sy, int inverse, double* __restrict__ pout) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double2 p = reinterpret_cast<const double2*>(pin)[i];
    M3 T = m3_load(S + static_cast<size_t>(frame_idx[i]) * 9);
    if (inverse) T = m3_inverse(T);
    const double x = sx * p.x, y = sy * p.y;
    const double X = (T.m[0] * x + T.m[1] * y) + T.m[2];
    const double Y = (T.m[3] * x + T.m[4] * y) + T.m[5];
    const double W = (T.m[6] * x + T.m[7] * y) + T.m[8];
    double2 r;
    r.x = rint((X / W) * 100.0) / 100.0;        // np.around(v, 2)
    r.y = rint((Y / W) * 100.0) / 100.0;
    reinterpret_cast<double2*>(pout)[i] = r;
}

// dense max-movement: max over frames and pixels of max(x', y').  gridDim.y is at most 65 535, so y-block b covers
// frames b, b + gridDim.y, ...; one partial per (y-block, x-block).
__global__ void __launch_bounds__(256)
max_movement_kernel(const double* __restrict__ S, int n_frames, int height, int width, double* __restrict__ partial) {
    __shared__ double ws[8];
    double best = -1.0 / 0.0;
    const int npix = height * width;
    for (int f = blockIdx.y; f < n_frames; f += gridDim.y) {
        const M3 T = m3_load(S + static_cast<size_t>(f) * 9);
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += gridDim.x * blockDim.x) {
            const double x = static_cast<double>(i % width), y = static_cast<double>(i / width);
            const double X = (T.m[0] * x + T.m[1] * y) + T.m[2];
            const double Y = (T.m[3] * x + T.m[4] * y) + T.m[5];
            const double W = (T.m[6] * x + T.m[7] * y) + T.m[8];
            best = fmax(best, fmax(X / W, Y / W));
        }
    }
#pragma unroll
    for (int of = 16; of > 0; of >>= 1) best = fmax(best, __shfl_xor_sync(0xffffffff, best, of));
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) best = fmax(best, ws[w]);
        partial[static_cast<size_t>(blockIdx.y) * gridDim.x + blockIdx.x] = best;
    }
}
__global__ void max_reduce_kernel(const double* __restrict__ partial, int n, double* __restrict__ out) {
    __shared__ double ws[32];
    double best = -1.0 / 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) best = fmax(best, partial[i]);
#pragma unroll
    for (int of = 16; of > 0; of >>= 1) best = fmax(best, __shfl_xor_sync(0xffffffff, best, of));
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < static_cast<int>(blockDim.x >> 5); ++w) best = fmax(best, ws[w]);
        *out = best;
    }
}

}  // namespace evz

extern "C" int evz_static_filter(evz_handle* h, const float* pts, const int32_t* off, const int32_t* cnt, int n_pairs,
                                 int max_cnt, const double* H, const int32_t* status,
                                 float* out_pts, int32_t* out_cnt, int32_t* best_r, int32_t* flags, int32_t* r_out,
                                 void* stream) {
    if (!h) return EVZ_E_ARG;
    EVZ_ENTER(h);
    EVZ_REQUIRE(h, pts && off && cnt && H && status && out_pts && out_cnt && best_r && flags, "null pointer");
    if (max_cnt > EVZ_MAX_KP) {
        EVZ_SET_ERR(h, "evz_static_filter: max_cnt %d exceeds the supported %d points per pair", max_cnt, EVZ_MAX_KP);
        return EVZ_E_UNSUPPORTED;
    }
    if (n_pairs <= 0) return EVZ_OK;
    const int smem = EVZ_MAX_KP * 2 + evz::kSfWindow * 8;
    if (!h->attr_static) {
        EVZ_CUDA_CHECK(h, cudaFuncSetAttribute(evz::static_filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        h->attr_static = true;
    }
    evz::static_filter_kernel<<<n_pairs, 256, smem, static_cast<cudaStream_t>(stream)>>>(pts, off, cnt, H, status, out_pts, out_cnt, best_r, flags, r_out);
    EVZ_LAUNCH_CHECK(h);
    return EVZ_OK;
}

extern "C" int evz_chain_scan(evz_handle* h, const double* G, const int32_t* status, int n_pairs, int policy,
                              const double* seed_S, const double* seed_G,
                              double* S, double* H_fixed, double* summary, void* stream) {
    if (!h) return EVZ_E_ARG;
    EVZ_ENTER(h);
    EVZ_REQUIRE(h, G && status, "null pointer");
    EVZ_REQUIRE(h, S || summary, "nothing to compute");
    if (n_pairs <= 0) return EVZ_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int nb = (n_pairs + evz::kScanBlock - 1) / evz::kScanBlock;
    // scratch: src[n] | block_last[nb] | block_carry[nb] | block_tot[nb*9] | block_pre[nb*9] | S_tmp[n*9] (summary-only mode)
    const size_t need = evz_align_up(static_cast<size_t>(n_pairs) * 4, 256) + 2 * evz_align_up(static_cast<size_t>(nb) * 4, 256) +
                        2 * evz_align_up(static_cast<size_t>(nb) * 72, 256) + (S ? 0 : static_cast<size_t>(n_pairs) * 72) + 256;
    void* scr = nullptr;
    int rc = evz_scratch(h, need, &scr);
    if (rc) return rc;
    uint8_t* b = static_cast<uint8_t*>(scr);
    int32_t* src = reinterpret_cast<int32_t*>(b); b += evz_align_up(static_cast<size_t>(n_pairs) * 4, 256);
    int32_t* block_last = reinterpret_cast<int32_t*>(b); b += evz_align_up(static_cast<size_t>(nb) * 4, 256);
    int32_t* block_carry = reinterpret_cast<int32_t*>(b); b += evz_align_up(static_cast<size_t>(nb) * 4, 256);
    double* block_tot = reinterpret_cast<double*>(b); b += evz_align_up(static_cast<size_t>(nb) * 72, 256);
    double* block_pre = reinterpret_cast<double*>(b); b += evz_align_up(static_cast<size_t>(nb) * 72, 256);
    double* S_work = S ? S : reinterpret_cast<double*>(b);

    evz::fill_local_kernel<<<nb, evz::kScanBlock, 0, st>>>(status, n_pairs, src, block_last, nullptr, nullptr, 0);
    EVZ_LAUNCH_CHECK(h);
    evz::fill_carry_kernel<<<1, 32, 0, st>>>(block_last, nb, block_carry, nullptr);
    EVZ_LAUNCH_CHECK(h);
    evz::fill_apply_kernel<<<nb, evz::kScanBlock, 0, st>>>(src, block_carry, n_pairs, nullptr, nullptr, 0);
    EVZ_LAUNCH_CHECK(h);
    const bool seeded = seed_S != nullptr || seed_G != nullptr;
    if (summary || (S && !seeded)) {
        // unseeded pass: leading invalid pairs are identity steps, so the total is R
        evz::prod_local_kernel<<<nb, evz::kScanBlock, 0, st>>>(G, src, n_pairs, policy, nullptr, 0, S_work, block_tot, nullptr, nullptr, 0);
        EVZ_LAUNCH_CHECK(h);
        evz::prod_carry_kernel<<<1, evz::kScanBlock, 0, st>>>(block_tot, nb, nullptr, block_pre, nullptr);
        EVZ_LAUNCH_CHECK(h);
        evz::prod_apply_kernel<<<nb, evz::kScanBlock, 0, st>>>(S_work, block_pre, n_pairs, 0, nullptr, nullptr, 0);
        EVZ_LAUNCH_CHECK(h);
        if (summary) {
            evz::summary_kernel<<<1, 32, 0, st>>>(G, src, S_work + static_cast<size_t>(n_pairs - 1) * 9, n_pairs, summary);
            EVZ_LAUNCH_CHECK(h);
        }
    }
    if (S && seeded) {
        evz::prod_local_kernel<<<nb, evz::kScanBlock, 0, st>>>(G, src, n_pairs, policy, seed_G, seed_S ? 1 : 0, S, block_tot, nullptr, nullptr, 0);
        EVZ_LAUNCH_CHECK(h);
        evz::prod_carry_kernel<<<1, evz::kScanBlock, 0, st>>>(block_tot, nb, seed_S, block_pre, nullptr);
        EVZ_LAUNCH_CHECK(h);
        evz::prod_apply_kernel<<<nb, evz::kScanBlock, 0, st>>>(S, block_pre, n_pairs, seed_S ? 1 : 0, nullptr, nullptr, 0);
        EVZ_LAUNCH_CHECK(h);
    }
    if (S && H_fixed) {
        evz::fixed_plane_kernel<<<nb, evz::kScanBlock, 0, st>>>(S, seed_S, n_pairs, H_fixed, nullptr, nullptr, 0);
        EVZ_LAUNCH_CHECK(h);
    }
    return EVZ_OK;
}

extern "C" int evz_chain_scan_segments(evz_handle* h, const double* G, const int32_t* status, int n_pairs,
                                       const int32_t* seg_off, int n_segs, int policy, double* S, double* H_fixed, void* stream) {
    if (!h) return EVZ_E_ARG;
    EVZ_ENTER(h);
    EVZ_REQUIRE(h, G && status && seg_off && S, "null pointer");
    EVZ_REQUIRE(h, n_segs >= 0, "n_segs must not be negative");
    if (n_pairs <= 0 || n_segs == 0) return EVZ_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // host-known bound of the block slots: sum over s of ceil(len(s) / 256) <= ceil(n_pairs / 256) + n_segs
    const int nb = (n_pairs + evz::kScanBlock - 1) / evz::kScanBlock + n_segs;
    // scratch: src[n] | block_last[nb] | block_carry[nb] | block_tot[nb*9] | block_pre[nb*9] | seg_blk[n_segs+1]
    const size_t need = evz_align_up(static_cast<size_t>(n_pairs) * 4, 256) + 2 * evz_align_up(static_cast<size_t>(nb) * 4, 256) +
                        2 * evz_align_up(static_cast<size_t>(nb) * 72, 256) + evz_align_up(static_cast<size_t>(n_segs + 1) * 4, 256) + 256;
    void* scr = nullptr;
    int rc = evz_scratch(h, need, &scr);
    if (rc) return rc;
    uint8_t* b = static_cast<uint8_t*>(scr);
    int32_t* src = reinterpret_cast<int32_t*>(b); b += evz_align_up(static_cast<size_t>(n_pairs) * 4, 256);
    int32_t* block_last = reinterpret_cast<int32_t*>(b); b += evz_align_up(static_cast<size_t>(nb) * 4, 256);
    int32_t* block_carry = reinterpret_cast<int32_t*>(b); b += evz_align_up(static_cast<size_t>(nb) * 4, 256);
    double* block_tot = reinterpret_cast<double*>(b); b += evz_align_up(static_cast<size_t>(nb) * 72, 256);
    double* block_pre = reinterpret_cast<double*>(b); b += evz_align_up(static_cast<size_t>(nb) * 72, 256);
    int32_t* seg_blk = reinterpret_cast<int32_t*>(b);

    evz::seg_blocks_kernel<<<1, evz::kScanBlock, 0, st>>>(seg_off, n_segs, seg_blk);
    EVZ_LAUNCH_CHECK(h);
    evz::fill_local_kernel<<<nb, evz::kScanBlock, 0, st>>>(status, n_pairs, src, block_last, seg_off, seg_blk, n_segs);
    EVZ_LAUNCH_CHECK(h);
    evz::fill_carry_kernel<<<n_segs, 32, 0, st>>>(block_last, nb, block_carry, seg_blk);
    EVZ_LAUNCH_CHECK(h);
    evz::fill_apply_kernel<<<nb, evz::kScanBlock, 0, st>>>(src, block_carry, n_pairs, seg_off, seg_blk, n_segs);
    EVZ_LAUNCH_CHECK(h);
    evz::prod_local_kernel<<<nb, evz::kScanBlock, 0, st>>>(G, src, n_pairs, policy, nullptr, 0, S, block_tot, seg_off, seg_blk, n_segs);
    EVZ_LAUNCH_CHECK(h);
    evz::prod_carry_kernel<<<n_segs, evz::kScanBlock, 0, st>>>(block_tot, nb, nullptr, block_pre, seg_blk);
    EVZ_LAUNCH_CHECK(h);
    evz::prod_apply_kernel<<<nb, evz::kScanBlock, 0, st>>>(S, block_pre, n_pairs, 0, seg_off, seg_blk, n_segs);
    EVZ_LAUNCH_CHECK(h);
    if (H_fixed) {
        evz::fixed_plane_kernel<<<nb, evz::kScanBlock, 0, st>>>(S, nullptr, n_pairs, H_fixed, seg_off, seg_blk, n_segs);
        EVZ_LAUNCH_CHECK(h);
    }
    return EVZ_OK;
}

extern "C" int evz_chain_ref_step(evz_handle* h, const double* H2, const int32_t* status, int n_chains, int first, int policy,
                                  double* S_state, const double* H_prev, double* H_out, void* stream) {
    if (!h) return EVZ_E_ARG;
    EVZ_ENTER(h);
    EVZ_REQUIRE(h, H2 && status && S_state && H_out, "null pointer");
    EVZ_REQUIRE(h, first || !policy || H_prev, "null pointer (H_prev is required after the first step when policy = 1)");
    if (n_chains <= 0) return EVZ_OK;
    const int nb = (n_chains + evz::kScanBlock - 1) / evz::kScanBlock;
    evz::chain_ref_step_kernel<<<nb, evz::kScanBlock, 0, static_cast<cudaStream_t>(stream)>>>(H2, status, n_chains, first ? 1 : 0,
                                                                                             policy ? 1 : 0, S_state, H_prev, H_out);
    EVZ_LAUNCH_CHECK(h);
    return EVZ_OK;
}

extern "C" int evz_chain_seed_apply(evz_handle* h, const double* summaries, int world, int rank, int policy, int n_pairs,
                                    double* S, double* H_fixed, double* seeds_out, void* stream) {
    if (!h) return EVZ_E_ARG;
    EVZ_ENTER(h);
    EVZ_REQUIRE(h, summaries && S && seeds_out, "null pointer");
    EVZ_REQUIRE(h, world >= 1 && rank >= 0 && rank < world, "rank must be in [0, world)");
    if (n_pairs <= 0) return EVZ_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int nb = (n_pairs + evz::kScanBlock - 1) / evz::kScanBlock;
    evz::seed_kernel<<<1, 32, 0, st>>>(summaries, world, rank, policy, n_pairs, S, seeds_out);
    EVZ_LAUNCH_CHECK(h);
    evz::seed_apply_kernel<<<nb, evz::kScanBlock, 0, st>>>(S, summaries, rank, seeds_out, n_pairs);
    EVZ_LAUNCH_CHECK(h);
    if (H_fixed) {
        evz::fixed_plane_kernel<<<nb, evz::kScanBlock, 0, st>>>(S, seeds_out, n_pairs, H_fixed, nullptr, nullptr, 0);
        EVZ_LAUNCH_CHECK(h);
    }
    return EVZ_OK;
}

extern "C" int evz_remap(evz_handle* h, const double* pts_in, const int32_t* frame_idx, int64_t n,
                         const double* S, int n_frames, double sx, double sy, int inverse,
                         double* pts_out, void* stream) {
    if (!h) return EVZ_E_ARG;
    EVZ_ENTER(h);
    EVZ_REQUIRE(h, pts_in && frame_idx && S && pts_out && n_frames > 0, "null pointer");
    if (n <= 0) return EVZ_OK;
    const int64_t nb = (n + 255) / 256;
    evz::remap_kernel<<<static_cast<unsigned int>(nb), 256, 0, static_cast<cudaStream_t>(stream)>>>(pts_in, frame_idx, n, S, sx, sy, inverse, pts_out);
    EVZ_LAUNCH_CHECK(h);
    return EVZ_OK;
}

extern "C" int evz_max_movement(evz_handle* h, const double* S, int n_frames, int height, int width,
                                double* out_max, void* stream) {
    if (!h) return EVZ_E_ARG;
    EVZ_ENTER(h);
    EVZ_REQUIRE(h, S && out_max && n_frames > 0 && height > 0 && width > 0, "bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int bx = (height * width + 256 * 8 - 1) / (256 * 8);
    if (bx < 1) bx = 1;
    if (bx > 64) bx = 64;
    const int by = n_frames < 65535 ? n_frames : 65535;         // the limit of gridDim.y; the kernel loops over the rest
    void* scr = nullptr;
    int rc = evz_scratch(h, static_cast<size_t>(by) * bx * 8 + 256, &scr);
    if (rc) return rc;
    dim3 grid(bx, by);
    evz::max_movement_kernel<<<grid, 256, 0, st>>>(S, n_frames, height, width, static_cast<double*>(scr));
    EVZ_LAUNCH_CHECK(h);
    evz::max_reduce_kernel<<<1, 1024, 0, st>>>(static_cast<const double*>(scr), by * bx, out_max);
    EVZ_LAUNCH_CHECK(h);
    return EVZ_OK;
}
