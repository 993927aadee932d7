// K1: exact brute-force 2-NN of u8 descriptors as a batched u8 x u8 -> s32 tcgen05 contraction
// with a fused distance / top-2 epilogue.  Replaces cv2 BFMatcher.knnMatch(q, t, 2)
// (reference evenvizion/processing/matching.py:102-108).
//
// Two kernels share the TMA / tcgen05 front end (work item = (pair, block of 256 query rows); per 256-row
// train tile one 128 x 256 accumulator per 128-row query sub-tile, K = 128 bytes = 4 x tcgen05.mma.kind::i8):
//
//  * match_top2_vkernel ("V-space", default; second half of this file): the train norm enters the accumulator
//    through a fifth K block, so the epilogue is a max tree over raw accumulator values -- about half the
//    instructions per output of the key-space epilogue.  Rows it cannot certify are recomputed by
//    match_fixup_kernel; match_prepare_kernel writes its fifth K block.
//  * match_top2_kernel ("key-space", this half): the fallback for pairs whose train frame has a norm range the
//    fifth K block cannot encode, and every pair with EVZ_OPT_MATCH_VARIANT = 5.
// The other epilogues tried for both kernels, and why they lost, are in DESIGN.md K1; their source is in the
// history of this file.
//
// Key-space epilogue, per accumulator element (row r = query, column c = train):
//   key = ckey[c] - 512 * acc = ((||t_c||^2 - 2 q.t_c) << 8) | c      (one IMAD on the FMA pipe; the
//   multiplier is a kernel argument so that ptxas cannot strength-reduce it onto the ALU pipe)
// ckey[c] = (||t_c||^2 << 8) | (c & 255) comes from the frame store, INT32_MAX for padding rows;
// it is staged by 1 KB bulk copies into its own ring.  ||t||^2 - 2 q.t >= -||q||^2 >= -8323200,
// so the key fits in int32, and a signed min over keys is the lexicographic (distance, index)
// minimum: ties go to the lowest train index exactly as OpenCV's batchDistance does.  ||q||^2 is
// added once per row after the reduction.
//
// The K dimension is only 128, so the kernel is bound by the epilogue's instruction issue, not by
// the tensor pipe: an exact running top-2 costs 2.5 min/max per element on the ALU pipe.  This
// epilogue spends ~1 ALU op per element instead:
//   * every aligned chunk of 8 columns is reduced to its minimum key with 3-input mins, and a
//     running top-2 of CHUNK minima is kept per thread;
//   * whenever a chunk minimum beats the thread's running best, the chunk's raw keys are saved to
//     a per-thread shared-memory slot by two predicated 128-bit stores, so at the end of the
//     item the slot holds the keys of the chunk that contains the nearest neighbour;
//   * the second neighbour is the smaller of the second-best chunk minimum and the best of the
//     other keys in that slot -- both exact, no recomputation.
// The running best crosses tile boundaries as a sentinel key (V1 << 8, made distinct from every
// real key of the thread's column range), so a later tile only wins with a strictly smaller distance.
//
// Warp roles (128 + 256 threads, 1 CTA / SM, persistent over items):
//   warp 0 : TMA producer (query block, train tiles, item descriptor ring)   warp 1 : MMA issuer
//   warp 2 : TMEM allocator        warp 3 : ckey producer
//   warps 4-11 : epilogue; warp w reads TMEM lanes 32*(w%4).. and the column half (w-4)/4
#include "evz_common.cuh"
#include "evz_ptx.cuh"
#include <climits>

namespace evz {

constexpr int kBlockQ      = 256;   // query rows per item (two 128-row MMA sub-tiles)
constexpr int kBlockT      = 256;   // train rows per tile (MMA N)
constexpr int kRowBytes    = 128;   // descriptor bytes = one SWIZZLE_128B row
constexpr int kStages      = 3;     // train-tile ring depth (released by the MMA commit alone)
constexpr int kCkStages    = 8;     // ckey-tile ring depth (released by the epilogue)
constexpr int kTileBytes   = kBlockT * kRowBytes;   // 32 KB
constexpr int kQBytes      = kBlockQ * kRowBytes;   // 32 KB
constexpr int kCkeyBytes   = kBlockT * 4;           // 1 KB
constexpr int kAbsent      = 0x7FFFFF;              // INT32_MAX >> 8: "no neighbour"

struct Item {
    int q_row0, nq_left, t_row0, nt, n_tiles, n_sub, out_row0, pad;
};

// Key-space kernel.  Every epilogue thread drains two query rows (one per sub-tile); the two accumulators
// alternate between the sub-tiles.
struct MatchCfg {
    static constexpr int epi_warps   = 8;                         // two column halves x four TMEM lane quarters
    static constexpr int epi_threads = epi_warps * 32;
    static constexpr int threads     = 128 + epi_threads;
    static constexpr int groups      = 2;                         // column groups of the accumulator
    static constexpr int cols        = kBlockT / groups;          // accumulator columns per epilogue thread and tile
    static constexpr int rows_per_thread = 2;                     // query rows (sub-tiles) per epilogue thread
    static constexpr int acc_readers = epi_warps;                 // epilogue warps that drain one accumulator
    static constexpr int chunk       = 8;                         // keys per save slot
    static constexpr int part_stride = epi_threads * 16;          // save slots are laid out [sub][part][thread] x 16 B
    static constexpr int parts       = chunk / 4;
    // offsets into dynamic shared memory (base aligned to 1024)
    static constexpr int q_off     = 0;                               // 2 x 32 KB
    static constexpr int t_off     = q_off + 2 * kQBytes;             // kStages x 32 KB
    static constexpr int ckey_off  = t_off + kStages * kTileBytes;    // kCkStages x 1 KB
    static constexpr int merge_rows = 256;                            // one merge buffer: 256 query rows x int4
    static constexpr int merge_off = ckey_off + kCkStages * kCkeyBytes; // two buffers, alternating per item
    static constexpr int slot_off  = merge_off + 2 * merge_rows * 16;
    static constexpr int item_off  = slot_off + rows_per_thread * parts * part_stride;
    static constexpr int bar_off   = item_off + 2 * static_cast<int>(sizeof(Item));
    static constexpr int n_bars    = 2 * kStages + 2 * kCkStages + 2 + 2 + 2 + 2;
    static constexpr int tmem_off  = bar_off + n_bars * 8;
    static constexpr int total     = tmem_off + 16;
    static constexpr int smem_bytes = total + 1024;               // + alignment slack
    static_assert(smem_bytes <= 227 * 1024, "match kernel shared memory exceeds 227 KB");
};

struct MatchArgs {
    const int32_t* ckey;
    const int32_t* row_off;
    const int32_t* n_kp;
    const int32_t* pair_q;
    const int32_t* pair_t;
    const int32_t* out_off;
    const int32_t* items;      // [n_items][2] = (pair, query block)
    const int32_t* n_items;    // device scalar
    int32_t* top2_idx;
    int32_t* top2_d2;
    int neg512;                // -512, passed at run time (see header)
    // V-space kernel only (match_top2_vkernel)
    const int32_t* pair_hmax;  // [n_pairs] max over the train frame of ||t||^2 >> 1
    const uint8_t* ecode;      // [total_rows / 256][8 KB] fifth K block of the train operand
    const uint32_t* pbits;     // [total_rows / 256][8] parity of ||t||^2, one bit per train row
    uint32_t mul256;           // 256, passed at run time (keeps the chunk-key IMAD on the FMA pipe)
    int32_t* fix_count;        // number of rows left to match_fixup_kernel (reset by match_prepare_kernel)
    int32_t* fix_list;         // [fix_capacity] item * 256 + row
    int fix_capacity;
    int pair_mode;             // always 0.  1 decoded items of 512 query rows for the CTA-pair kernel removed after round 2;
                               //    the decode stays in load_item because without it the V-space kernel measured 0.2 %
                               //    slower at ORB width (B200 at 1000 W, same-run A/B: 1.030 vs 1.028 ms per 2 000 pairs;
                               //    removing only this field did not change that), an effect of code placement
    int n_kb;                  // data K blocks of 32 bytes that hold descriptor bytes: 4 for SIFT (128 B), 1 for ORB (32 B);
                               //    the rest of the 128-byte row is zero padding and is not multiplied (match_top2_vkernel)
};

__device__ __forceinline__ Item load_item(const MatchArgs& a, int it) {
    Item r;
    const int li = a.pair_mode ? it >> 1 : it;
    const int p = a.items[2 * li];
    int blk = a.items[2 * li + 1];
    const int qf = a.pair_q[p], tf = a.pair_t[p];
    const int nq = a.n_kp[qf];
    int sub_left = nq - blk * kBlockQ;
    if (a.pair_mode) {                              // never taken (see MatchArgs::pair_mode)
        sub_left = nq - 2 * blk * kBlockQ;
        blk = 2 * blk + (it & 1);
    }
    r.q_row0 = a.row_off[qf] + blk * kBlockQ;
    r.nq_left = nq - blk * kBlockQ;                 // valid query rows in this block (may exceed 256)
    r.n_sub = sub_left > 128 ? 2 : 1;
    r.t_row0 = a.row_off[tf];
    r.nt = a.n_kp[tf];
    r.n_tiles = (r.nt + kBlockT - 1) / kBlockT;
    r.out_row0 = a.out_off[p] + blk * kBlockQ;
    r.pad = a.pair_hmax ? a.pair_hmax[p] : 0;      // V-space kernel: hmax of the train frame
    return r;
}

// lexicographic (value, index) insertion into a running top-2
__device__ __forceinline__ void top2_insert(int v, int i, int& V1, int& I1, int& V2, int& I2) {
    const bool lt1 = (v < V1) || (v == V1 && i < I1);
    const bool lt2 = (v < V2) || (v == V2 && i < I2);
    if (lt1)      { V2 = V1; I2 = I1; V1 = v; I1 = i; }
    else if (lt2) { V2 = v;  I2 = i; }
}

// 128-bit shared-memory load through a 32-bit shared address (the dynamic smem base is realigned by
// integer arithmetic, which hides the address space from nvcc: plain loads would become generic LD)
__device__ __forceinline__ int4 lds128(uint32_t addr) {
    int4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ int mad_key(uint32_t acc, int mul, int ck) {
    int r;
    asm("mad.lo.s32 %0, %1, %2, %3;" : "=r"(r) : "r"(static_cast<int>(acc)), "r"(mul), "r"(ck));
    return r;
}

// exact running top-2 of packed keys, two elements at a time (5 ALU ops / 2 elements)
__device__ __forceinline__ void top2_pair(int k0, int k1, int& m1, int& m2) {
    const int lo = min(k0, k1), hi = max(k0, k1);
    m2 = __vimin3_s32(m2, hi, max(m1, lo));
    m1 = min(m1, lo);
}

// chunk minimum + predicated save of the best chunk's keys: returns min(cm, m1); when cm < m1 the
// chunk's keys go to the slot (setp + selp fuse into one VIMNMX with a predicate output)
__device__ __forceinline__ int save_if_less8(int cm, int m1, uint32_t slot, const int* k) {
    int mn;
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "setp.lt.s32 p, %1, %2;\n\t"
                 "selp.s32 %0, %1, %2, p;\n\t"
                 "@p st.shared.v4.b32 [%3], {%4, %5, %6, %7};\n\t"
                 "@p st.shared.v4.b32 [%3+%12], {%8, %9, %10, %11};\n\t}"
                 : "=r"(mn) : "r"(cm), "r"(m1), "r"(slot), "r"(k[0]), "r"(k[1]), "r"(k[2]), "r"(k[3]),
                    "r"(k[4]), "r"(k[5]), "r"(k[6]), "r"(k[7]), "n"(MatchCfg::part_stride));
    return mn;
}

// 32 accumulator columns (r) against their ckey values (ck): update the thread's running (m1, m2)
__device__ __forceinline__ void pass32(const uint32_t (&r)[32], const int4 (&ck)[8], int mul, int& m1, int& m2,
                                       uint32_t slot) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        int k[8];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int4 c = ck[q * 2 + j];
            k[4 * j + 0] = mad_key(r[q * 8 + 4 * j + 0], mul, c.x);
            k[4 * j + 1] = mad_key(r[q * 8 + 4 * j + 1], mul, c.y);
            k[4 * j + 2] = mad_key(r[q * 8 + 4 * j + 2], mul, c.z);
            k[4 * j + 3] = mad_key(r[q * 8 + 4 * j + 3], mul, c.w);
        }
        const int cm = __vimin3_s32(__vimin3_s32(k[0], k[1], k[2]), __vimin3_s32(k[3], k[4], k[5]), min(k[6], k[7]));
        const int mn = save_if_less8(cm, m1, slot, k);
        m2 = min(m2, max(m1, cm));
        m1 = mn;
    }
}

// Drain this thread's columns of one accumulator in batches.  The accumulator is handed back to the MMA
// warp as soon as its last column is in registers.
// Software pipeline over batches of 32 columns: the TMEM load and the eight broadcast ckey loads of batch
// b+1 are issued before batch b is processed, so only the first load of an accumulator is exposed (the two
// epilogue warps of a scheduler drain the same accumulator in lockstep and cannot hide each other's load
// latency).
__device__ __forceinline__ void drain_acc(uint32_t taddr, uint32_t ck, int mul, int& m1, int& m2, uint32_t slot,
                                          uint64_t* acc_empty, int lane) {
    constexpr int kBatches = MatchCfg::cols / 32;
    constexpr int kBuf = 2;
    uint32_t r[kBuf][32];
    int4 ckv[kBuf][8];
    auto issue = [&](int b) {
        tmem_ld_32x32b_x32(taddr + b * 32, r[b % kBuf]);
#pragma unroll
        for (int j = 0; j < 8; ++j) ckv[b % kBuf][j] = lds128(ck + b * 128 + j * 16);
    };
    issue(0);
#pragma unroll
    for (int b = 0; b < kBatches; ++b) {
        tmem_ld_wait_dep(r[b % kBuf]);
        if (b + 1 < kBatches) issue(b + 1);
        if (b == kBatches - 1) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty);
        }
        pass32(r[b % kBuf], ckv[b % kBuf], mul, m1, m2, slot);
    }
}

__global__ void __launch_bounds__(MatchCfg::threads, 1)
match_top2_kernel(const __grid_constant__ CUtensorMap tmap, const MatchArgs args) {
    using Cfg = MatchCfg;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* q_s = smem + Cfg::q_off;
    uint8_t* t_s = smem + Cfg::t_off;
    int32_t* ckey_s = reinterpret_cast<int32_t*>(smem + Cfg::ckey_off);
    int4* merge_s = reinterpret_cast<int4*>(smem + Cfg::merge_off);
    Item* item_s = reinterpret_cast<Item*>(smem + Cfg::item_off);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::bar_off);
    uint64_t* full = bars;                       // [kStages] train tile landed (TMA tx)
    uint64_t* empty = full + kStages;            // [kStages] MMA commit
    uint64_t* ck_full = empty + kStages;         // [kCkStages] ckey tile landed
    uint64_t* ck_empty = ck_full + kCkStages;    // [kCkStages] epilogue warp arrivals
    uint64_t* q_full = ck_empty + kCkStages;     // [2] query block landed + item descriptor published
    uint64_t* q_empty = q_full + 2;              // [2] MMA commit + epilogue warp arrivals
    uint64_t* acc_full = q_empty + 2;            // [2] accumulator ready (MMA commit)
    uint64_t* acc_empty = acc_full + 2;          // [2] accumulator drained (epilogue warp arrivals)
    uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(smem + Cfg::tmem_off);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmap);
        for (int i = 0; i < kStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < kCkStages; ++i) { mbar_init(&ck_full[i], 1); mbar_init(&ck_empty[i], Cfg::epi_warps); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&q_full[i], 1); mbar_init(&q_empty[i], 1 + Cfg::epi_warps);
            mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], Cfg::acc_readers);
        }
        fence_mbar_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_ptr_s, 512);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_s;
    const int n_items = *args.n_items;

    if (warp == 0) {
        // ------------------------------------------------------------- TMA producer
        if (lane == 0) {
            uint32_t stage = 0, sphase = 0, qi = 0;
            for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
                const Item im = load_item(args, it);
                const uint32_t qb = qi & 1, qph = (qi >> 1) & 1;
                ++qi;
                mbar_wait(&q_empty[qb], qph ^ 1);
                item_s[qb] = im;                           // published by the arrive below (release)
                if (im.n_tiles == 0) { mbar_arrive(&q_full[qb]); continue; }   // empty train frame: nothing to multiply
                mbar_arrive_expect_tx(&q_full[qb], kQBytes);
                tma_load_2d(q_s + qb * kQBytes, &tmap, 0, im.q_row0, &q_full[qb]);
                for (int n = 0; n < im.n_tiles; ++n) {
                    mbar_wait(&empty[stage], sphase ^ 1);
                    mbar_arrive_expect_tx(&full[stage], kTileBytes);
                    tma_load_2d(t_s + stage * kTileBytes, &tmap, 0, im.t_row0 + n * kBlockT, &full[stage]);
                    if (++stage == kStages) { stage = 0; sphase ^= 1; }
                }
            }
        }
    } else if (warp == 3) {
        // ------------------------------------------------------------- ckey producer
        if (lane == 0) {
            uint32_t cs = 0, cph = 0;
            for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
                const Item im = load_item(args, it);
                for (int n = 0; n < im.n_tiles; ++n) {
                    mbar_wait(&ck_empty[cs], cph ^ 1);
                    mbar_arrive_expect_tx(&ck_full[cs], kCkeyBytes);
                    bulk_load_1d(ckey_s + cs * kBlockT, args.ckey + im.t_row0 + n * kBlockT, kCkeyBytes, &ck_full[cs]);
                    if (++cs == kCkStages) { cs = 0; cph ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------- MMA issuer
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_u8(128, kBlockT);
            uint32_t stage = 0, sphase = 0, qi = 0, g = 0;
            for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
                const uint32_t qb = qi & 1, qph = (qi >> 1) & 1;
                ++qi;
                mbar_wait(&q_full[qb], qph);
                const int n_tiles = item_s[qb].n_tiles, n_sub = item_s[qb].n_sub;
                const uint32_t q_addr = smem_u32(q_s + qb * kQBytes);
                for (int n = 0; n < n_tiles; ++n) {
                    mbar_wait(&full[stage], sphase);
                    const uint32_t t_addr = smem_u32(t_s + stage * kTileBytes);
                    for (int sub = 0; sub < n_sub; ++sub, ++g) {
                        const uint32_t acc = g & 1, aph = (g >> 1) & 1;
                        mbar_wait(&acc_empty[acc], aph ^ 1);
                        tc_fence_after();
#pragma unroll
                        for (int k = 0; k < kRowBytes / 32; ++k) {
                            const uint64_t da = umma_desc_sw128(q_addr + sub * (128 * kRowBytes) + k * 32);
                            const uint64_t db = umma_desc_sw128(t_addr + k * 32);
                            umma_i8(tmem_base + acc * kBlockT, da, db, idesc, k > 0 ? 1u : 0u);
                        }
                        umma_commit(&acc_full[acc]);
                    }
                    umma_commit(&empty[stage]);
                    if (++stage == kStages) { stage = 0; sphase ^= 1; }
                }
                umma_commit(&q_empty[qb]);
            }
        }
    } else if (warp >= 4) {
        // ------------------------------------------------------------- epilogue
        constexpr int kR = Cfg::rows_per_thread;
        const int quarter = warp & 3;                          // TMEM lane quarter this warp may read
        const int cgrp = (warp - 4) >> 2;                      // column group of the accumulator
        const int colbase = cgrp * Cfg::cols;
        const int row_in_sub = quarter * 32 + lane;
        const int sent_adj = colbase == 0 ? 1 : 0;   // sentinel distinct from every key of this column range
        const uint32_t slot0 = smem_u32(smem + Cfg::slot_off) + (threadIdx.x - 128) * 16;
        const uint32_t ckey_base = smem_u32(ckey_s);
        constexpr int bar_id = 1, bar_threads = Cfg::epi_threads;
        uint32_t cs = 0, cph = 0, g = 0, qi = 0;
        for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
            const uint32_t qb = qi & 1, qph = (qi >> 1) & 1;
            ++qi;
            mbar_wait(&q_full[qb], qph);
            const Item im = item_s[qb];
            // ||q||^2 of this thread's query rows: loaded now, needed when the item is written out
            int qkey[kR];
#pragma unroll
            for (int s = 0; s < kR; ++s)
                qkey[s] = cgrp == 0 ? __ldg(args.ckey + im.q_row0 + s * 128 + row_in_sub) : 0;
            // running best / second best of this thread's column range as packed keys (distance << 8 | column
            // within the tile) plus the tile they came from; decoded once per item
            int B1[kR], T1[kR], B2[kR], T2[kR];
#pragma unroll
            for (int s = 0; s < kR; ++s) { B1[s] = kAbsent * 256; T1[s] = -1; B2[s] = INT_MAX; T2[s] = -1; }
            for (int n = 0; n < im.n_tiles; ++n) {
                mbar_wait(&ck_full[cs], cph);
                const uint32_t ck = ckey_base + (cs * kBlockT + colbase) * 4;
#pragma unroll
                for (int s = 0; s < kR; ++s) {
                    const int sub = s;
                    if (sub < im.n_sub) {
                        const uint32_t acc = g & 1, aph = (g >> 1) & 1;
                        mbar_wait(&acc_full[acc], aph);
                        tc_fence_after();
                        const uint32_t taddr = tmem_base + acc * kBlockT + colbase + (static_cast<uint32_t>(quarter * 32) << 16);
                        // the running best enters the tile as a sentinel: a chunk only wins (and is saved)
                        // with a strictly smaller distance
                        const int sentinel = (B1[s] & ~255) - sent_adj;
                        int m1 = sentinel, m2 = INT_MAX;
                        drain_acc(taddr, ck, args.neg512, m1, m2, slot0 + s * (Cfg::parts * Cfg::part_stride), &acc_empty[acc], lane);
                        if (m1 != sentinel) {
                            const bool demote = m2 == sentinel;      // the old best is the new second best
                            B2[s] = demote ? B1[s] : m2; T2[s] = demote ? T1[s] : n;
                            B1[s] = m1; T1[s] = n;
                        } else if (m2 < (B2[s] & ~255)) {
                            B2[s] = m2; T2[s] = n;
                        }
                        ++g;
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&ck_empty[cs]);
                if (++cs == kCkStages) { cs = 0; cph ^= 1; }
            }
            int V1[kR], I1[kR], V2[kR], I2[kR];
#pragma unroll
            for (int s = 0; s < kR; ++s) {
                V1[s] = T1[s] >= 0 ? B1[s] >> 8 : kAbsent; I1[s] = T1[s] >= 0 ? T1[s] * kBlockT + (B1[s] & 255) : -1;
                V2[s] = T2[s] >= 0 ? B2[s] >> 8 : kAbsent; I2[s] = T2[s] >= 0 ? T2[s] * kBlockT + (B2[s] & 255) : -1;
            }
            // exact second neighbour: the other keys of the chunk that holds the nearest one
#pragma unroll
            for (int s = 0; s < kR; ++s) {
                if (I1[s] >= 0) {
                    const int wkey = B1[s];
                    int cand = INT_MAX;
#pragma unroll
                    for (int part = 0; part < Cfg::parts; ++part) {
                        const int4 k = lds128(slot0 + s * (Cfg::parts * Cfg::part_stride) + part * Cfg::part_stride);
                        cand = min(cand, k.x == wkey ? INT_MAX : k.x);
                        cand = min(cand, k.y == wkey ? INT_MAX : k.y);
                        cand = min(cand, k.z == wkey ? INT_MAX : k.z);
                        cand = min(cand, k.w == wkey ? INT_MAX : k.w);
                    }
                    const int v = cand >> 8, i = (I1[s] & ~255) + (cand & 255);
                    if (v < V2[s] || (v == V2[s] && i < I2[s])) { V2[s] = v; I2[s] = i; }
                }
            }
            // merge the two column groups through shared memory: group 1 hands its candidates to group 0 and
            // moves on (bar.arrive); the merge buffer alternates per item, and a writer can be at most two
            // accumulators ahead of group 0, so a buffer is never rewritten before it has been read.
            int4* mbuf = merge_s + (qi & 1) * Cfg::merge_rows;
            if (cgrp > 0) {
#pragma unroll
                for (int s = 0; s < kR; ++s)
                    mbuf[s * 128 + row_in_sub] = make_int4(V1[s], I1[s], V2[s], I2[s]);
                named_bar_arrive(bar_id, bar_threads);
            } else {
                named_bar_sync(bar_id, bar_threads);
#pragma unroll
                for (int s = 0; s < kR; ++s) {
                    const int sub = s;
                    const int4 o = mbuf[sub * 128 + row_in_sub];
                    if (o.y >= 0) top2_insert(o.x, o.y, V1[s], I1[s], V2[s], I2[s]);
                    if (o.w >= 0) top2_insert(o.z, o.w, V1[s], I1[s], V2[s], I2[s]);
                    const int r = sub * 128 + row_in_sub;
                    if (r < im.nq_left) {
                        const int qn = qkey[s] >> 8;
                        const int64_t o_row = static_cast<int64_t>(im.out_row0) + r;
                        int2 oi, od;
                        oi.x = I1[s]; od.x = I1[s] >= 0 ? V1[s] + qn : -1;
                        oi.y = I2[s]; od.y = I2[s] >= 0 ? V2[s] + qn : -1;
                        reinterpret_cast<int2*>(args.top2_idx)[o_row] = oi;
                        reinterpret_cast<int2*>(args.top2_d2)[o_row] = od;
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&q_empty[qb]);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, 512);
}

// items[i] = (pair, query block): one entry per block of kBlockQ rows of every pair's query frame.
// Single CTA; pairs are scanned in chunks of blockDim.x.
__global__ void build_items_kernel(const int32_t* n_kp, const int32_t* pair_q, int n_pairs,
                                   int32_t* items, int32_t* n_items, int capacity,
                                   const int32_t* pair_flag, int want) {
    __shared__ int warp_sums[32];
    __shared__ int base_s;
    if (threadIdx.x == 0) base_s = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (int p0 = 0; p0 < n_pairs; p0 += blockDim.x) {
        const int p = p0 + threadIdx.x;
        // pair_flag selects the pairs of this list (V-space kernel: 0, key-space fallback: 1)
        const bool take = p < n_pairs && (pair_flag == nullptr || pair_flag[p] == want);
        const int nb = take ? (n_kp[pair_q[p]] + kBlockQ - 1) / kBlockQ : 0;
        int incl = nb;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffff, incl, d); if (lane >= d) incl += t; }
        if (lane == 31) warp_sums[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int w = lane < nwarps ? warp_sums[lane] : 0;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffff, w, d); if (lane >= d) w += t; }
            warp_sums[lane] = w;
        }
        __syncthreads();
        const int base = base_s;
        int start = base + incl - nb + (warp > 0 ? warp_sums[warp - 1] : 0);
        for (int b = 0; b < nb; ++b) {
            if (start + b < capacity) { items[2 * (start + b)] = p; items[2 * (start + b) + 1] = b; }
        }
        __syncthreads();
        if (threadIdx.x == 0) base_s = base + warp_sums[nwarps - 1];
        __syncthreads();
    }
    if (threadIdx.x == 0) *n_items = min(base_s, capacity);
}


// =====================================================================================================
// V-space kernel: the train norm enters the accumulator through a fifth K block, so the epilogue needs
// no per-element arithmetic at all -- only a max tree over the raw accumulator.
//
//   V[r][c] = q_r . t_c + E_c,   E_c = hmax + 1 - (||t_c||^2 >> 1)  (real columns),  E_c = 0 (padding)
//   =>  ||t_c||^2 - 2 q_r . t_c = 2 (hmax + 1 - V[r][c]) + (||t_c||^2 & 1)
// hmax = max over the train frame of ||t||^2 >> 1.  A larger V is a strictly smaller distance; equal V
// differ by the norm parity only.  E_c is a u8 x u8 dot product of the constant query-side vector
// a = (255 x 30, 1, 0) with 32 code bytes per train row (match_prepare_kernel writes them, in the no-swizzle
// core-matrix layout the MMA reads, plus one norm-parity bit per row), good for hmax - hmin < kEMax;
// pairs with a wider norm range or more than EVZ_MAX_KP train rows go through the key-space kernel.
//
// Epilogue (8 warps; warps 4-7 drain accumulator 0 = query sub-tile 0, warps 8-11 accumulator 1; one query
// row and all 256 columns of a tile per thread): every aligned chunk of 16 columns is reduced to its
// maximum (8 three-input max), packed with its position ((V << 8) | (254 - chunk), earlier = larger), and a
// sorted top-3 of chunk keys is kept (5 min/max).  A chunk that beats the second-best key is saved raw
// into the slot that holds the second-best chunk (4 predicated 128-bit stores); when it also beats the
// best key the two slots swap roles.  At the end of the item the two slots hold the two best chunks:
// their 32 columns are evaluated exactly (norm parity from the shared-memory bitmap, index), and the result
// is exact whenever the second-best distance found is strictly below the bound 2 (hmax + 1 - V3) of every
// other column (V3 = third chunk maximum).  Rows that cannot be certified (a value tie between the second
// and third chunk: ~1e-3 of the rows on descriptor-like data, every row on degenerate data) are flagged
// and recomputed by match_fixup_kernel (dp4a brute force, one CTA per row).
//
// Measured (B200, 2048 keypoints/frame, profiles/r01e_*, r01f): 1.8 warp instructions per 32 outputs against 3.3
// in the key-space kernel; tensor pipe active 56 % (45 % algorithmic + the fifth K block), issue slots 45 %,
// ALU pipe 57 %.  The TMA / tcgen05 front end alone (accumulators released undrained) runs at 2.75 POP/s (2048
// keypoints) to 3.2 POP/s (8192), the rate of the cuBLASLt int8 GEMM; the kernel runs at 1.9-2.0 / 2.3, so the
// epilogue is the bound, and in it the four predicated STS.128 of a chunk: they cost 22 % of the kernel whether
// or not any lane stores (see vchunk).  Neither the shared-memory data pipe nor the accumulator hand-off is the
// bound: CTA pairs (cta_group::2), eight or sixteen drain warps per accumulator, a two-pass drain and 16-column
// TMEM loads all measured equal or slower (DESIGN.md K1), as did chunks of 32 columns, N = 128 MMAs and polling
// barriers from all threads (r01e).  Chunks of 8 columns halve the saved bytes but add instructions: faster at
// 1024 keypoints, slower at 8192.
// The kernel is plain, non-templated code on purpose: a template instance of the same source compiled to a 4 %
// slower kernel (same-run A/B, r01g), and a run-time option test in the tile loop cost another 1.4 %.
constexpr int kECodeBytes = kBlockT * 32;                 // fifth K block of one train tile
constexpr int kEMax       = 255 * (30 * 255) + 254;       // largest representable E_c
constexpr int kFlagged    = -2;                           // top2_idx[row][0] of a row left to the fix-up kernel

constexpr int kVC    = 16;               // columns per chunk of the V-space epilogue
constexpr int kVCps  = kBlockT / kVC;    // chunks per tile
constexpr int kVClog = 4;                // log2(kVCps)
struct VCfg {
    static constexpr int threads   = 384;
    static constexpr int q_off     = 0;                                // 2 x 32 KB
    static constexpr int t_off     = q_off + 2 * kQBytes;              // kStages x 32 KB
    static constexpr int e_off     = t_off + kStages * kTileBytes;     // kStages x 8 KB
    static constexpr int a_off     = e_off + kStages * kECodeBytes;    // 4 KB: query-side fifth K block
    static constexpr int slot_off  = a_off + 128 * 32;                 // [slot 2][part 4][row 256] x 16 B
    static constexpr int part_stride = 256 * 16;
    static constexpr int slot_stride = (kVC / 4) * part_stride;
    static constexpr int pb_bytes  = (EVZ_MAX_KP / kBlockT) * 32;      // norm parity bitmap of one train frame
    static constexpr int pb_off    = slot_off + 2 * slot_stride;       // 2 x pb_bytes, alternating per item
    static constexpr int item_off  = pb_off + 2 * pb_bytes;
    static constexpr int bar_off   = item_off + 2 * static_cast<int>(sizeof(Item));
    static constexpr int n_bars    = 2 * kStages + 2 + 2 + 2 + 2;
    static constexpr int tmem_off  = bar_off + n_bars * 8;
    static constexpr int total     = tmem_off + 16;
    static constexpr int smem_bytes = total + 1024;
    static_assert(smem_bytes <= 227 * 1024, "V-space match kernel shared memory exceeds 227 KB");
};

// one chunk of kVC raw accumulator values: chunk key, sorted top-3 update, predicated save
__device__ __forceinline__ void vchunk(const uint32_t* r, uint32_t tagc, uint32_t mul, uint32_t& M1, uint32_t& M2,
                                       uint32_t& M3, uint32_t& sec, uint32_t sum) {
    static_assert(kVC == 16, "four 128-bit stores per chunk");
    const uint32_t a = __vimax3_u32(r[0], r[1], r[2]), b = __vimax3_u32(r[3], r[4], r[5]), c = __vimax3_u32(r[6], r[7], r[8]);
    const uint32_t d = __vimax3_u32(r[9], r[10], r[11]), e = __vimax3_u32(r[12], r[13], r[14]);
    const uint32_t cm = max(__vimax3_u32(a, b, c), __vimax3_u32(d, e, r[15]));
    uint32_t cmk;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(cmk) : "r"(cm), "r"(mul), "r"(tagc));
    // the next store address goes to a different register (early clobber): overwriting `sec` in place would wait
    // for the stores to have read it (write-after-read on the short scoreboard, ~35 clk per chunk)
    const uint32_t alt = sum - sec;
    uint32_t nsec;
    // (a predicated-off STS.128 still costs its LSU issue slot: all-false predicates measured no faster, removing the
    // four stores +28 %; skipping them with a warp-uniform vote + branch when no lane saves measured 18 % SLOWER)
    asm volatile("{\n\t.reg .pred p1, p2;\n\t"
                 "setp.gt.u32 p2, %2, %4;\n\t"
                 "setp.gt.u32 p1, %2, %3;\n\t"
                 "@p2 st.shared.v4.b32 [%1], {%6, %7, %8, %9};\n\t"
                 "@p2 st.shared.v4.b32 [%1+%22], {%10, %11, %12, %13};\n\t"
                 "@p2 st.shared.v4.b32 [%1+2*%22], {%14, %15, %16, %17};\n\t"
                 "@p2 st.shared.v4.b32 [%1+3*%22], {%18, %19, %20, %21};\n\t"
                 "selp.u32 %0, %5, %1, p1;\n\t}"
                 : "=&r"(nsec) : "r"(sec), "r"(cmk), "r"(M1), "r"(M2), "r"(alt),
                   "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
                   "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]),
                   "r"(r[14]), "r"(r[15]), "n"(VCfg::part_stride) : "memory");
    sec = nsec;
    const uint32_t t = min(M1, cmk), u = __vimin3_u32(M1, M2, cmk);
    M1 = max(M1, cmk);
    M3 = max(M3, u);
    M2 = max(M2, t);
}

// K-major operand tile without swizzle: 8-row x 16-byte core matrices (128 contiguous bytes); lbo = byte
// distance between the two core matrices along K, sbo = byte distance between 8-row groups.
__device__ __forceinline__ uint64_t umma_desc_nosw(uint32_t smem_addr_bytes, uint32_t lbo, uint32_t sbo) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr_bytes & 0x3FFFF) >> 4);
    d |= static_cast<uint64_t>(lbo >> 4) << 16;
    d |= static_cast<uint64_t>(sbo >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;                                 // version = 1 (sm_100), layout = none
    return d;
}

// keeps 16 registers allocated up to this point: the predicated stores of a chunk read them late, and a
// temporary that the allocator placed on one of them would wait for those reads (write-after-read stall)
__device__ __forceinline__ void keep_alive16(const uint32_t* r) {
    asm volatile("" :: "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
                       "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]));
}

// one accumulator row (256 columns): 8 batches of 32 columns, TMEM loads one batch ahead; the accumulator is
// handed back to the MMA warp as soon as its last column is in registers
__device__ __forceinline__ void drain_v(uint32_t taddr, uint32_t mul, uint32_t& M1, uint32_t& M2, uint32_t& M3,
                                        uint32_t& sec, uint32_t sum, uint64_t* acc_empty, int lane) {
    uint32_t r[2][32];
    tmem_ld_32x32b_x32(taddr, r[0]);
#pragma unroll
    for (int b = 0; b < 8; ++b) {
        tmem_ld_wait_dep(r[b & 1]);
        if (b + 1 < 8) {
            tmem_ld_32x32b_x32(taddr + (b + 1) * 32, r[(b + 1) & 1]);
        } else {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty);
        }
#pragma unroll
        for (int c = 0; c < 32 / kVC; ++c) vchunk(&r[b & 1][kVC * c], 254 - (32 / kVC) * b - c, mul, M1, M2, M3, sec, sum);
        keep_alive16(&r[b & 1][0]);
        keep_alive16(&r[b & 1][16]);
    }
}

__global__ void __launch_bounds__(VCfg::threads, 1)
match_top2_vkernel(const __grid_constant__ CUtensorMap tmap, const MatchArgs args) {
    using Cfg = VCfg;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* q_s = smem + Cfg::q_off;
    uint8_t* t_s = smem + Cfg::t_off;
    uint8_t* e_s = smem + Cfg::e_off;
    uint8_t* a_s = smem + Cfg::a_off;
    Item* item_s = reinterpret_cast<Item*>(smem + Cfg::item_off);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::bar_off);
    uint64_t* full = bars;                       // [kStages] train tile + its fifth K block landed (TMA tx)
    uint64_t* empty = full + kStages;            // [kStages] MMA commit
    uint64_t* q_full = empty + kStages;          // [2] query block landed + item descriptor published
    uint64_t* q_empty = q_full + 2;              // [2] MMA commit + 8 epilogue warps
    uint64_t* acc_full = q_empty + 2;            // [2] accumulator (= query sub-tile) ready (MMA commit)
    uint64_t* acc_empty = acc_full + 2;          // [2] accumulator drained (4 epilogue warps each)
    uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(smem + Cfg::tmem_off);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmap);
        for (int i = 0; i < kStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&q_full[i], 1); mbar_init(&q_empty[i], 1 + 8);
            mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 4);
        }
        fence_mbar_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_ptr_s, 512);
        tmem_relinquish();
    }
    if (warp == 3) {
        // query-side fifth K block: every row = (255 x 30, 1, 0), no-swizzle core-matrix layout
        for (int i = lane; i < 256; i += 32) {
            const bool second = (i >> 3) & 1;          // [group 16][k half 2][row 8] x 16 B
            reinterpret_cast<uint4*>(a_s)[i] = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, second ? 0x0001FFFFu : 0xFFFFFFFFu);
        }
        fence_proxy_async();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_s;
    const int n_items = *args.n_items;

    if (warp == 0) {
        // ------------------------------------------------------------- TMA producer (polling waits, single thread)
        if (lane == 0) {
            uint32_t stage = 0, sphase = 0, qi = 0;
            for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
                const Item im = load_item(args, it);
                const uint32_t qb = qi & 1, qph = (qi >> 1) & 1;
                ++qi;
                mbar_wait_spin(&q_empty[qb], qph ^ 1);
                item_s[qb] = im;
                if (im.n_tiles == 0) { mbar_arrive(&q_full[qb]); continue; }
                mbar_arrive_expect_tx(&q_full[qb], kQBytes + im.n_tiles * 32);
                tma_load_2d(q_s + qb * kQBytes, &tmap, 0, im.q_row0, &q_full[qb]);
                bulk_load_1d(smem + Cfg::pb_off + qb * Cfg::pb_bytes, args.pbits + static_cast<size_t>(im.t_row0 >> 8) * 8,
                             im.n_tiles * 32, &q_full[qb]);
                const uint8_t* ecode = args.ecode + static_cast<size_t>(im.t_row0 >> 8) * kECodeBytes;
                for (int n = 0; n < im.n_tiles; ++n) {
                    // the ring is only kStages deep: pull the tile that will be loaded kStages iterations from now
                    // into L2 already, so that its TMA load is an L2 hit
                    if (n + kStages < im.n_tiles) {
                        tma_prefetch_2d(&tmap, 0, im.t_row0 + (n + kStages) * kBlockT);
                        bulk_prefetch_1d(ecode + static_cast<size_t>(n + kStages) * kECodeBytes, kECodeBytes);
                    }
                    mbar_wait_spin(&empty[stage], sphase ^ 1);
                    mbar_arrive_expect_tx(&full[stage], kTileBytes + kECodeBytes);
                    tma_load_2d(t_s + stage * kTileBytes, &tmap, 0, im.t_row0 + n * kBlockT, &full[stage]);
                    bulk_load_1d(e_s + stage * kECodeBytes, ecode + static_cast<size_t>(n) * kECodeBytes, kECodeBytes, &full[stage]);
                    if (++stage == kStages) { stage = 0; sphase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------- MMA issuer
        if (lane == 0) {
            // accumulator = query sub-tile.  The waits of this single thread poll: a tcgen05.mma issue blocks
            // until the tensor pipe accepts it, so the pipe only stays fed while this thread is never late,
            // and a suspended try_wait wakes up late.
            constexpr uint32_t idesc = umma_idesc_u8(128, kBlockT);
            const uint64_t da_e = umma_desc_nosw(smem_u32(a_s), 128, 256);
            const int n_kb = args.n_kb;
            uint32_t stage = 0, sphase = 0, qi = 0, gs[2] = {0, 0};
            for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
                const uint32_t qb = qi & 1, qph = (qi >> 1) & 1;
                ++qi;
                mbar_wait_spin(&q_full[qb], qph);
                const int n_tiles = item_s[qb].n_tiles, n_sub = item_s[qb].n_sub;
                const uint32_t q_addr = smem_u32(q_s + qb * kQBytes);
                for (int n = 0; n < n_tiles; ++n) {
                    mbar_wait_spin(&full[stage], sphase);
                    const uint32_t t_addr = smem_u32(t_s + stage * kTileBytes);
                    const uint64_t db_e = umma_desc_nosw(smem_u32(e_s + stage * kECodeBytes), 128, 256);
                    for (int sub = 0; sub < n_sub; ++sub) {
                        const uint32_t aph = gs[sub]++ & 1;
                        mbar_wait_spin(&acc_empty[sub], aph ^ 1);
                        tc_fence_after();
                        if (n_kb == kRowBytes / 32) {
#pragma unroll
                            for (int k = 0; k < kRowBytes / 32; ++k) {
                                const uint64_t da = umma_desc_sw128(q_addr + sub * (128 * kRowBytes) + k * 32);
                                const uint64_t db = umma_desc_sw128(t_addr + k * 32);
                                umma_i8(tmem_base + sub * kBlockT, da, db, idesc, k > 0 ? 1u : 0u);
                            }
                        } else {
                            // short descriptors (ORB: one 32-byte K block): the zero padding is not multiplied
                            for (int k = 0; k < n_kb; ++k) {
                                const uint64_t da = umma_desc_sw128(q_addr + sub * (128 * kRowBytes) + k * 32);
                                const uint64_t db = umma_desc_sw128(t_addr + k * 32);
                                umma_i8(tmem_base + sub * kBlockT, da, db, idesc, k > 0 ? 1u : 0u);
                            }
                        }
                        umma_i8(tmem_base + sub * kBlockT, da_e, db_e, idesc, 1u);
                        umma_commit(&acc_full[sub]);
                    }
                    umma_commit(&empty[stage]);
                    if (++stage == kStages) { stage = 0; sphase ^= 1; }
                }
                umma_commit(&q_empty[qb]);
            }
        }
    } else if (warp >= 4) {
        // ------------------------------------------------------------- epilogue
        const int grp = (warp - 4) >> 2;                       // query sub-tile = accumulator
        const int quarter = warp & 3;                          // TMEM lane quarter this warp may read
        const int row = grp * 128 + quarter * 32 + lane;       // query row within the block
        const uint32_t slot_a = smem_u32(smem + Cfg::slot_off) + row * 16, slot_b = slot_a + Cfg::slot_stride;
        const uint32_t sum = slot_a + slot_b;
        const uint32_t taddr = tmem_base + grp * kBlockT + (static_cast<uint32_t>(quarter * 32) << 16);
        uint32_t g = 0, qi = 0;
        for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
            const uint32_t qb = qi & 1, qph = (qi >> 1) & 1;
            ++qi;
            mbar_wait(&q_full[qb], qph);
            const Item im = item_s[qb];
            if (grp < im.n_sub) {
                const int qkey = __ldg(args.ckey + im.q_row0 + row);
                // sorted top-3 of chunk keys, the slot that holds the second-best chunk, and the position
                // (tile * 16 + chunk) of the chunks in the best / second-best slot
                uint32_t M1 = 0, M2 = 0, M3 = 0, sec = slot_b;
                int Tb = -1, Ts = -1;
                for (int n = 0; n < im.n_tiles; ++n) {
                    // keys of earlier tiles beat every key of this tile with the same V (lowest index wins)
                    M1 |= 255u; M2 |= 255u; M3 |= 255u;
                    const uint32_t o1 = M1, o2 = M2;
                    mbar_wait(&acc_full[grp], g & 1);
                    tc_fence_after();
                    drain_v(taddr, args.mul256, M1, M2, M3, sec, sum, &acc_empty[grp], lane);
                    ++g;
                    const int nTb = M1 == o1 ? Tb : n * kVCps + 254 - static_cast<int>(M1 & 255u);
                    Ts = (M1 != o1 && M2 == o1) ? Tb : (M2 == o2 ? Ts : n * kVCps + 254 - static_cast<int>(M2 & 255u));
                    Tb = nTb;
                }
                // exact evaluation of the two saved chunks: ||t||^2 - 2 q.t = 2 (hmax + 1 - V) + parity, packed
                // with the ordinal of the column among the 32 candidates (the slot with the lower position
                // first), so that a signed min is the lexicographic (distance, index) minimum.  Padding
                // columns have V = 0, i.e. a distance above every real column: they sort last by themselves.
                const int hm1 = im.pad + 1;
                const bool best_first = Ts < 0 || Tb < Ts;
                int k[2 * kVC];
#pragma unroll
                for (int s = 0; s < 2; ++s) {
                    const int T = s == 0 ? Tb : Ts;
                    const uint32_t sa = s == 0 ? sum - sec : sec;
                    if (T >= 0) {
                        const int base = (T >> kVClog) * kBlockT + (T & (kVCps - 1)) * kVC;
                        const int cs = (2 * hm1) * 256 + ((s == 0) == best_first ? 0 : kVC);
                        uint32_t ps;                       // norm parity of the chunk's columns, moved to bits 8..
                        asm volatile("ld.shared.u16 %0, [%1];" : "=r"(ps) : "r"(smem_u32(smem + Cfg::pb_off) + qb * Cfg::pb_bytes + (base >> 3)));
                        ps <<= 8;
#pragma unroll
                        for (int part = 0; part < kVC / 4; ++part) {
                            const int4 v = lds128(sa + part * Cfg::part_stride);
                            k[s * kVC + part * 4 + 0] = mad_key(v.x, args.neg512, cs) + (((ps >> (part * 4 + 0)) & 256) + part * 4 + 0);
                            k[s * kVC + part * 4 + 1] = mad_key(v.y, args.neg512, cs) + (((ps >> (part * 4 + 1)) & 256) + part * 4 + 1);
                            k[s * kVC + part * 4 + 2] = mad_key(v.z, args.neg512, cs) + (((ps >> (part * 4 + 2)) & 256) + part * 4 + 2);
                            k[s * kVC + part * 4 + 3] = mad_key(v.w, args.neg512, cs) + (((ps >> (part * 4 + 3)) & 256) + part * 4 + 3);
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < kVC; ++i) k[s * kVC + i] = INT_MAX;
                    }
                }
                int m1 = INT_MAX, m2 = INT_MAX;
#pragma unroll
                for (int i = 0; i < kVC; ++i) top2_pair(k[2 * i], k[2 * i + 1], m1, m2);
                const int base_b = Tb >= 0 ? (Tb >> kVClog) * kBlockT + (Tb & (kVCps - 1)) * kVC : 0;
                const int base_s = Ts >= 0 ? (Ts >> kVClog) * kBlockT + (Ts & (kVCps - 1)) * kVC : 0;
                const int base_lo = best_first ? base_b : base_s, base_hi = best_first ? base_s : base_b;
                const int c1 = ((m1 & kVC) ? base_hi : base_lo) + (m1 & (kVC - 1)), c2 = ((m2 & kVC) ? base_hi : base_lo) + (m2 & (kVC - 1));
                const int I1 = (m1 != INT_MAX && c1 < im.nt) ? c1 : -1, I2 = (m2 != INT_MAX && c2 < im.nt) ? c2 : -1;
                const int V1 = m1 >> 8, V2 = m2 >> 8;
                // every column outside the two slots has V <= V3, i.e. ||t||^2 - 2 q.t >= 2 (hmax + 1 - V3)
                const bool third = M3 > 255u;
                const int bound = 2 * (hm1 - static_cast<int>(M3 >> 8));
                const bool flagged = third && (I2 < 0 || V2 >= bound);
                if (row < im.nq_left) {
                    const int qn = qkey >> 8;
                    const int64_t o_row = static_cast<int64_t>(im.out_row0) + row;
                    int2 oi, od;
                    oi.x = flagged ? kFlagged : I1; od.x = I1 >= 0 ? V1 + qn : -1;
                    oi.y = I2;                      od.y = I2 >= 0 ? V2 + qn : -1;
                    reinterpret_cast<int2*>(args.top2_idx)[o_row] = oi;
                    reinterpret_cast<int2*>(args.top2_d2)[o_row] = od;
                    if (flagged) {
                        const int pos = atomicAdd(args.fix_count, 1);
                        if (pos < args.fix_capacity) args.fix_list[pos] = it * 256 + row;
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&q_empty[qb]);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, 512);
}

// Per pair: hmax / range test of the train frame, then the 32 code bytes of every train row in the
// no-swizzle core-matrix layout the fifth MMA reads ([tile][group of 8 rows][k half][row][16 B]).
// One CTA of 256 threads per pair; pairs that share a train frame write identical bytes.
__global__ void __launch_bounds__(256)
match_prepare_kernel(const int32_t* ckey, const int32_t* row_off, const int32_t* n_kp, const int32_t* pair_t,
                     int32_t* pair_hmax, int32_t* pair_flag, uint8_t* ecode, uint32_t* pbits, int32_t* fix_count) {
    __shared__ int s_max[8], s_min[8];
    const int p = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (p == 0 && tid == 0) *fix_count = 0;
    const int tf = pair_t[p], nt = n_kp[tf], base = row_off[tf];
    int hmax = 0, hmin = INT_MAX;
    for (int c = tid; c < nt; c += 256) {
        const int h = ckey[base + c] >> 9;
        hmax = max(hmax, h); hmin = min(hmin, h);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        hmax = max(hmax, __shfl_xor_sync(0xffffffff, hmax, d));
        hmin = min(hmin, __shfl_xor_sync(0xffffffff, hmin, d));
    }
    if (lane == 0) { s_max[warp] = hmax; s_min[warp] = hmin; }
    __syncthreads();
    hmax = s_max[0]; hmin = s_min[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) { hmax = max(hmax, s_max[w]); hmin = min(hmin, s_min[w]); }
    // (frames above EVZ_MAX_KP would overflow the kernel's parity bitmap buffers: key-space kernel as well)
    const bool wide = nt > 0 && (hmax - hmin + 1 > kEMax || nt > EVZ_MAX_KP);
    if (tid == 0) { pair_hmax[p] = hmax; pair_flag[p] = wide ? 1 : 0; }
    if (wide) return;
    const int n_tiles = (nt + kBlockT - 1) / kBlockT;
    for (int n = 0; n < n_tiles; ++n) {
        const int c = n * kBlockT + tid;
        uint32_t w[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        const int ckv = c < nt ? ckey[base + c] : 0;
        const unsigned par = __ballot_sync(0xffffffff, (ckv >> 8) & 1);
        if (lane == 0) pbits[(static_cast<size_t>(base >> 8) + n) * 8 + warp] = par;
        if (c < nt) {
            const int E = hmax + 1 - (ckv >> 9);
            const int m = E / 255, r = E - 255 * m;
#pragma unroll
            for (int k = 0; k < 30; ++k) {
                const uint32_t b = static_cast<uint32_t>(min(max(m - 255 * k, 0), 255));
                w[k >> 2] |= b << (8 * (k & 3));
            }
            w[7] |= static_cast<uint32_t>(r) << 16;
        }
        uint8_t* tile = ecode + (static_cast<size_t>(base >> 8) + n) * kECodeBytes + (tid >> 3) * 256 + (tid & 7) * 16;
        *reinterpret_cast<uint4*>(tile) = make_uint4(w[0], w[1], w[2], w[3]);
        *reinterpret_cast<uint4*>(tile + 128) = make_uint4(w[4], w[5], w[6], w[7]);
    }
}

// Rows the V-space kernel could not certify (listed in fix_list, top2_idx[row][0] == kFlagged): exact
// brute-force 2-NN with dp4a, one CTA of 128 threads per row.
__global__ void __launch_bounds__(128)
match_fixup_kernel(const uint8_t* desc, const MatchArgs args) {
    __shared__ int4 s_part[4];
    const int n_fix = min(*args.fix_count, args.fix_capacity);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int e = blockIdx.x; e < n_fix; e += gridDim.x) {
        const int code = args.fix_list[e];
        const Item im = load_item(args, code >> 8);
        const int r = code & 255;
        const uint4* qp = reinterpret_cast<const uint4*>(desc + static_cast<size_t>(im.q_row0 + r) * kRowBytes);
        uint4 q[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) q[j] = __ldg(qp + j);
        int V1 = kAbsent, I1 = -1, V2 = kAbsent, I2 = -1;
        for (int c = tid; c < im.nt; c += 128) {
            const uint4* tp = reinterpret_cast<const uint4*>(desc + static_cast<size_t>(im.t_row0 + c) * kRowBytes);
            uint4 t[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) t[j] = __ldg(tp + j);
            unsigned dot = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                dot = __dp4a(q[j].x, t[j].x, dot); dot = __dp4a(q[j].y, t[j].y, dot);
                dot = __dp4a(q[j].z, t[j].z, dot); dot = __dp4a(q[j].w, t[j].w, dot);
            }
            top2_insert((__ldg(args.ckey + im.t_row0 + c) >> 8) - 2 * static_cast<int>(dot), c, V1, I1, V2, I2);
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const int oV1 = __shfl_xor_sync(0xffffffff, V1, d), oI1 = __shfl_xor_sync(0xffffffff, I1, d);
            const int oV2 = __shfl_xor_sync(0xffffffff, V2, d), oI2 = __shfl_xor_sync(0xffffffff, I2, d);
            if (oI1 >= 0) top2_insert(oV1, oI1, V1, I1, V2, I2);
            if (oI2 >= 0) top2_insert(oV2, oI2, V1, I1, V2, I2);
        }
        if (lane == 0) s_part[warp] = make_int4(V1, I1, V2, I2);
        __syncthreads();
        if (tid == 0) {
#pragma unroll
            for (int w = 1; w < 4; ++w) {
                const int4 o = s_part[w];
                if (o.y >= 0) top2_insert(o.x, o.y, V1, I1, V2, I2);
                if (o.w >= 0) top2_insert(o.z, o.w, V1, I1, V2, I2);
            }
            const int qn = __ldg(args.ckey + im.q_row0 + r) >> 8;
            const int64_t o = static_cast<int64_t>(im.out_row0) + r;
            reinterpret_cast<int2*>(args.top2_idx)[o] = make_int2(I1, I2);
            reinterpret_cast<int2*>(args.top2_d2)[o] = make_int2(I1 >= 0 ? V1 + qn : -1, I2 >= 0 ? V2 + qn : -1);
        }
        __syncthreads();
    }
}

}  // namespace evz

static int ensure_tmap(evz_handle* h, const uint8_t* desc, int64_t total_rows) {
    if (h->tmap_ptr == desc && h->tmap_rows == total_rows) return EVZ_OK;
    if (!h->encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        EVZ_CUDA_CHECK(h, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (!fn || qres != cudaDriverEntryPointSuccess) {
            EVZ_SET_ERR(h, "cuTensorMapEncodeTiled not available from the driver");
            return EVZ_E_CUDA;
        }
        h->encode = reinterpret_cast<evz_encode_tiled_fn>(fn);
    }
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(evz::kRowBytes), static_cast<cuuint64_t>(total_rows)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(evz::kRowBytes)};
    const cuuint32_t box[2] = {static_cast<cuuint32_t>(evz::kRowBytes), 256u};
    const cuuint32_t estr[2] = {1u, 1u};
    const CUresult r = h->encode(&h->tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t*>(desc), dims, strides, box, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                 CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        EVZ_SET_ERR(h, "cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld)", static_cast<int>(r), static_cast<long long>(total_rows));
        return EVZ_E_CUDA;
    }
    h->tmap_ptr = desc;
    h->tmap_rows = total_rows;
    return EVZ_OK;
}

extern "C" int evz_match_top2(evz_handle* h, const uint8_t* desc, const int32_t* ckey, int64_t total_rows,
                              const int32_t* row_off, const int32_t* n_kp,
                              const int32_t* pair_q, const int32_t* pair_t, const int32_t* out_off, int n_pairs,
                              int32_t* top2_idx, int32_t* top2_d2, void* stream) {
    return evz_match_top2_d(h, desc, EVZ_DESC_BYTES, ckey, total_rows, row_off, n_kp, pair_q, pair_t, out_off, n_pairs, top2_idx, top2_d2, stream);
}

extern "C" int evz_match_top2_d(evz_handle* h, const uint8_t* desc, int desc_bytes, const int32_t* ckey, int64_t total_rows,
                                const int32_t* row_off, const int32_t* n_kp,
                                const int32_t* pair_q, const int32_t* pair_t, const int32_t* out_off, int n_pairs,
                                int32_t* top2_idx, int32_t* top2_d2, void* stream) {
    if (!h) return EVZ_E_ARG;
    EVZ_ENTER(h);
    EVZ_REQUIRE(h, desc_bytes > 0 && desc_bytes <= EVZ_DESC_BYTES, "desc_bytes must be in [1, 128]");
    EVZ_REQUIRE(h, desc && ckey && row_off && n_kp && pair_q && pair_t && out_off && top2_idx && top2_d2, "null pointer");
    EVZ_REQUIRE(h, total_rows > 0 && total_rows % EVZ_ROW_ALIGN == 0 && total_rows < (int64_t(1) << 31), "total_rows must be a positive multiple of 256 below 2^31");
    EVZ_REQUIRE(h, (reinterpret_cast<uintptr_t>(desc) & 127) == 0 && (reinterpret_cast<uintptr_t>(ckey) & 15) == 0, "desc must be 128-byte and ckey 16-byte aligned");
    if (n_pairs <= 0) return EVZ_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = ensure_tmap(h, desc, total_rows);
    if (rc) return rc;
    // every pair owns at most ceil(n_kp/256) <= rows/256 + 1 items
    const size_t capacity = static_cast<size_t>(total_rows / evz::kBlockQ) + static_cast<size_t>(n_pairs);
    EVZ_REQUIRE(h, capacity < (size_t(1) << 30), "too many work items");
    // EVZ_OPT_MATCH_VARIANT: 0 = V-space kernel for the pairs it can encode, key-space kernel for the rest (default);
    // 5 = key-space kernel for every pair (evz_set_option accepts no other value)
    const bool vspace = h->opt_match_variant == 0;
    // scratch: [counters 256 B][items A][items B][pair_hmax][pair_flag][ecode]
    const size_t items_bytes = evz_align_up(capacity * 8, 256), pair_bytes = evz_align_up(static_cast<size_t>(n_pairs) * 4, 256);
    const size_t fix_bytes = evz_align_up(capacity * 256 * 4, 256);          // every row of every item, at worst
    const size_t pbits_bytes = evz_align_up(static_cast<size_t>(total_rows) / 8, 256);     // one bit per store row
    const size_t ecode_off = evz_align_up(256 + 2 * items_bytes + 2 * pair_bytes + fix_bytes + pbits_bytes, 1024);
    EVZ_REQUIRE(h, !vspace || capacity < (size_t(1) << 22), "too many work items for the V-space kernel (set EVZ_OPT_MATCH_VARIANT=5)");
    void* scr = nullptr;
    rc = evz_scratch(h, vspace ? ecode_off + static_cast<size_t>(total_rows) * 32 : 256 + items_bytes, &scr);
    if (rc) return rc;
    uint8_t* sb = static_cast<uint8_t*>(scr);
    int32_t* n_items = reinterpret_cast<int32_t*>(sb);
    int32_t* items = reinterpret_cast<int32_t*>(sb + 256);
    evz::MatchArgs a{ckey, row_off, n_kp, pair_q, pair_t, out_off, items, n_items, top2_idx, top2_d2, -512, nullptr, nullptr, nullptr, 256u,
                     nullptr, nullptr, 0, 0, (desc_bytes + 31) / 32};
    if (vspace) {
        int32_t* n_items_slow = n_items + 16;
        int32_t* items_slow = reinterpret_cast<int32_t*>(sb + 256 + items_bytes);
        int32_t* pair_hmax = reinterpret_cast<int32_t*>(sb + 256 + 2 * items_bytes);
        int32_t* pair_flag = reinterpret_cast<int32_t*>(sb + 256 + 2 * items_bytes + pair_bytes);
        uint8_t* ecode = sb + ecode_off;
        a.fix_count = n_items + 32;
        a.fix_list = reinterpret_cast<int32_t*>(sb + 256 + 2 * items_bytes + 2 * pair_bytes);
        a.fix_capacity = static_cast<int>(capacity * 256);
        uint32_t* pbits = reinterpret_cast<uint32_t*>(sb + 256 + 2 * items_bytes + 2 * pair_bytes + fix_bytes);
        a.pbits = pbits;
        evz::match_prepare_kernel<<<n_pairs, 256, 0, st>>>(ckey, row_off, n_kp, pair_t, pair_hmax, pair_flag, ecode, pbits, a.fix_count);
        EVZ_LAUNCH_CHECK(h);
        evz::build_items_kernel<<<1, 1024, 0, st>>>(n_kp, pair_q, n_pairs, items, n_items, static_cast<int>(capacity), pair_flag, 0);
        evz::build_items_kernel<<<1, 1024, 0, st>>>(n_kp, pair_q, n_pairs, items_slow, n_items_slow, static_cast<int>(capacity), pair_flag, 1);
        EVZ_LAUNCH_CHECK(h);
        a.pair_hmax = pair_hmax;
        a.ecode = ecode;
        if (!(h->attr_match & 2u)) {
            EVZ_CUDA_CHECK(h, cudaFuncSetAttribute(evz::match_top2_vkernel, cudaFuncAttributeMaxDynamicSharedMemorySize, evz::VCfg::smem_bytes));
            h->attr_match |= 2u;
        }
        cudaEvent_t* tev = nullptr;
        if (h->opt_time_match) {
            if (!h->match_ev_made) {
                for (auto& pr : h->match_ev) { EVZ_CUDA_CHECK(h, cudaEventCreate(&pr[0])); EVZ_CUDA_CHECK(h, cudaEventCreate(&pr[1])); }
                h->match_ev_made = true;
            }
            tev = h->match_ev[h->match_calls++ & 15];
            EVZ_CUDA_CHECK(h, cudaEventRecord(tev[0], st));
        }
        evz::match_top2_vkernel<<<h->sm_count, evz::VCfg::threads, evz::VCfg::smem_bytes, st>>>(h->tmap, a);
        EVZ_LAUNCH_CHECK(h);
        if (tev) EVZ_CUDA_CHECK(h, cudaEventRecord(tev[1], st));
        evz::match_fixup_kernel<<<h->sm_count * 16, 128, 0, st>>>(desc, a);      // latency-bound (one row per CTA at a time): fill the SMs
        EVZ_LAUNCH_CHECK(h);
        // pairs whose train frame has a norm range the fifth K block cannot encode go to the key-space kernel
        // below (normally no items)
        a.items = items_slow;
        a.n_items = n_items_slow;
        a.pair_hmax = nullptr;
    } else {
        evz::build_items_kernel<<<1, 1024, 0, st>>>(n_kp, pair_q, n_pairs, items, n_items, static_cast<int>(capacity), nullptr, 0);
        EVZ_LAUNCH_CHECK(h);
    }
    if (!(h->attr_match & 1u)) {
        EVZ_CUDA_CHECK(h, cudaFuncSetAttribute(evz::match_top2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, evz::MatchCfg::smem_bytes));
        h->attr_match |= 1u;
    }
    evz::match_top2_kernel<<<h->sm_count, evz::MatchCfg::threads, evz::MatchCfg::smem_bytes, st>>>(h->tmap, a);
    EVZ_LAUNCH_CHECK(h);
    return EVZ_OK;
}
