/*
 * evz.h -- C ABI of libevz.so: the B200 (sm_100a) implementation of EvenVizion's
 * frame-to-frame geometry hot path.
 *
 * The reference (gridl/EvenVizion) is pure Python and has no FFI of its own; the heavy
 * arithmetic of this path lives behind two OpenCV call sites.  Each entry point below
 * names the reference code it replaces (paths relative to the reference repo root).
 * The Python shim in evenvizion_b200/ binds these with ctypes (see INTEGRATION.md for
 * the stub a maintainer of the reference would add).
 *
 * Conventions
 *   - every pointer marked DEV is a CUDA device pointer owned by the caller; the
 *     library owns only scratch inside the handle;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), performs
 *     no host synchronisation except when scratch has to grow, and returns 0 on
 *     success or a negative EVZ_E_* code (evz_last_error() has the text);
 *   - per-pair outcomes are status codes in an output array (EVZ_ST_*), mirroring the
 *     reference's NoMatchesException / HomographyException control flow;
 *   - one handle per device, not thread-safe;
 *   - there is no CPU fallback: without a CUDA device evz_create() fails.
 *
 * Frame store layout (built by evz_ingest)
 *   A video is F frames; frame f has n_kp[f] keypoints stored in rows
 *   [row_off[f], row_off[f] + n_kp[f]) of four parallel arrays.  row_off[f] is a
 *   multiple of EVZ_ROW_ALIGN (256) and row_off[F] is the total row count, so every
 *   256-row tensor-core tile belongs to exactly one frame; padding rows hold zero
 *   descriptors and ckey = INT32_MAX.
 *     desc   uint8  [rows][128]   descriptors, zero-padded to 128 bytes (ORB: 32 used)
 *     ckey   int32  [rows]        (||d||^2 << 8) | (row & 255)
 *     coords float  [rows][2]     keypoint (x, y)
 *     canon  int32  [rows]        frame-local index of the first keypoint of the frame
 *                                 with bit-identical (x, y)   (for remove_double_matching)
 *   A frame pair p is (query frame pair_q[p] = the NEW frame = `self` in the reference,
 *   train frame pair_t[p] = the PREVIOUS frame = `acceding`).  Per-pair variable-length
 *   results start at row out_off[p] of the per-row output arrays and have capacity
 *   n_kp[pair_q[p]]; for a video chain out_off[p] = row_off[pair_q[p]].
 */
#ifndef EVZ_H
#define EVZ_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EVZ_VERSION       100
#define EVZ_ROW_ALIGN     256
#define EVZ_DESC_BYTES    128
#define EVZ_R_MAX         16383   /* largest displacement bin resolved exactly by evz_static_filter */
#define EVZ_MAX_KP        12288   /* keypoints per frame supported by the shared-memory per-pair tables */

/* error codes */
#define EVZ_OK             0
#define EVZ_E_CUDA        -1
#define EVZ_E_ARG         -2
#define EVZ_E_NOMEM       -3
#define EVZ_E_NODEVICE    -4
#define EVZ_E_UNSUPPORTED -5

/* per-pair status (reference exception it mirrors) */
#define EVZ_ST_OK           0
#define EVZ_ST_FEW_MATCHES  1  /* NoMatchesException "len(matches) < min_matching_pts"   matching.py:113-116 */
#define EVZ_ST_FEW_POINTS   3  /* < 4 points reach findHomography: cv2.error, uncaught in the reference     */
#define EVZ_ST_NO_MODEL_1   4  /* NoMatchesException "can't find homography matrix"       matching.py:158-159 */
#define EVZ_ST_NO_MODEL_2   5  /* HomographyException()                                    utils.py:361-362   */
#define EVZ_ST_FEW_INLIERS  6  /* HomographyException "not enough points ..."              utils.py:359-360   */

/* flags written by evz_static_filter into flags[p] */
#define EVZ_FLAG_DISP_OVERFLOW 1 /* a displacement was non-finite or > EVZ_R_MAX (reference round() raises) */
#define EVZ_FLAG_TOO_MANY_POINTS 2 /* cnt[p] > EVZ_MAX_KP although max_cnt promised otherwise: nothing was written */

/* A handle belongs to ONE device and ONE host thread / stream at a time: its grow-only scratch block is shared by all
 * entry points, so two calls that overlap in time on different streams (or threads) would race on it.  Every entry point
 * makes the handle's device current (cudaSetDevice) before it launches.  Growing the scratch block synchronises the
 * device once (cudaDeviceSynchronize + cudaFree + cudaMalloc); steady-state calls do not synchronise. */
typedef struct evz_handle evz_handle;

int         evz_version(void);
int         evz_create(int device, evz_handle** out);
void        evz_destroy(evz_handle* h);
const char* evz_last_error(const evz_handle* h);     /* h may be NULL: last creation error */
int         evz_sm_count(const evz_handle* h);

/* debugging / A-B options; results are identical for every setting, only the route differs */
#define EVZ_OPT_RANSAC_EXACT   1  /* 1: score every hypothesis x match with the exactly-rounded formula (no fused fast path) */
#define EVZ_OPT_MATCH_VARIANT  2  /* match route: 0 (default) = the "V-space" kernel (the train norm enters the accumulator
                                     through a fifth K block, max-tree epilogue, exact resolution from two saved chunks +
                                     fix-up) for every pair whose train frame it can encode, the key-space kernel for the rest;
                                     5 = the key-space kernel (distance/index keys formed per element, chunk-8 minima + saved
                                     best chunk) for every pair.  Any other value returns EVZ_E_ARG */
#define EVZ_OPT_RANSAC_NO_PRUNE 3  /* 1: score every valid hypothesis even after one of them counted all matches as inliers
                                     (default 0: hypotheses that can no longer win the (count desc, index asc) arg-max are skipped) */
#define EVZ_OPT_TIME_MATCH     4  /* 1: evz_match_top2 brackets its main kernel with CUDA events on the caller's stream (a ring of
                                     16 pairs, one per call); read them with evz_match_kernel_ms after synchronising */
int         evz_set_option(evz_handle* h, int option, int value);
/* elapsed time of the main match kernel of the k-th most recent evz_match_top2 call (k = 0: the last one), for the
 * roofline line of bench.py.  The stream must have been synchronised; returns EVZ_E_ARG when no such record exists. */
int         evz_match_kernel_ms(evz_handle* h, int k, float* ms);

/* ---- ingest: the step before the path (SURVEY 8f-1).  Replaces the implicit
 * np.float32 -> cv::Mat conversion inside knnMatch (matching.py:108) and prepares
 * remove_double_matching's key comparison (utils.py:63-64).
 *   raw_desc   DEV  [sum n_kp][d] of uint8 (raw_is_f32 = 0) or float (raw_is_f32 = 1),
 *                   frames concatenated without padding; d <= 128
 *   raw_coords DEV  float [sum n_kp][2]
 *   raw_off    DEV  int64 [F+1]  first raw row of every frame
 *   row_off    DEV  int32 [F+1]  first padded row of every frame (multiples of 256)
 *   bad_count  DEV  int32 [1]    incremented for every descriptor value that is not an
 *                                integer in [0,255] (float input; SURF cannot use this path)
 */
int evz_ingest(evz_handle* h, const void* raw_desc, int raw_is_f32, int d,
               const float* raw_coords, const int64_t* raw_off, const int32_t* row_off, int n_frames,
               uint8_t* desc, int32_t* ckey, float* coords, int32_t* canon, int32_t* bad_count,
               void* stream);

/* ---- K1: exact brute-force 2-NN.  Replaces
 * cv2.DescriptorMatcher_create("BruteForce").knnMatch(q, t, 2) at matching.py:102-108.
 * u8 x u8 -> s32 tcgen05.mma (kind::i8), TMA-staged tiles, TMEM accumulators, fused
 * ||a||^2 + ||b||^2 - 2ab / top-2 epilogue.  Ties resolve to the lowest train index.
 * Uses handle scratch of about 33 bytes per store row + 1 KB per 256-row query block
 * (fifth-K-block codes, norm parity bitmap, work items, fix-up list).
 *   top2_idx DEV int32 [rows][2]  train keypoint index (frame-local), -1 when absent
 *   top2_d2  DEV int32 [rows][2]  exact squared L2 distance,          -1 when absent
 * (knnMatch's DMatch.distance is sqrtf((float)d2), bit for bit.)
 */
int evz_match_top2(evz_handle* h, const uint8_t* desc, const int32_t* ckey, int64_t total_rows,
                   const int32_t* row_off, const int32_t* n_kp,
                   const int32_t* pair_q, const int32_t* pair_t, const int32_t* out_off, int n_pairs,
                   int32_t* top2_idx, int32_t* top2_d2, void* stream);
/* The same with the number of descriptor bytes that are in use (the rest of every 128-byte row is zero padding):
 * 32 for ORB (frame_processing.py:59-61) -- one 32-byte K block is multiplied instead of four.  Results are those of
 * evz_match_top2 (which is this call with desc_bytes = 128). */
int evz_match_top2_d(evz_handle* h, const uint8_t* desc, int desc_bytes, const int32_t* ckey, int64_t total_rows,
                     const int32_t* row_off, const int32_t* n_kp,
                     const int32_t* pair_q, const int32_t* pair_t, const int32_t* out_off, int n_pairs,
                     int32_t* top2_idx, int32_t* top2_d2, void* stream);


/* ---- K1b/K2: Lowe ratio test + many-to-one filter + coordinate de-dup + gather.  Replaces
 * lowes_ratio_test / filter_corresponding_points (matching.py:166-239), the point gather
 * (matching.py:117-118) and remove_double_matching (utils.py:41-68).
 *   max_kp   upper bound of n_kp over the frames involved (sizes shared memory; <= EVZ_MAX_KP)
 *   surv     DEV uint8  [rows]     1 where the query passes the ratio test (may be NULL)
 *   m_idx    DEV int32  [rows][2]  (query, train) of the de-duplicated matches, in order
 *   m_pts    DEV float  [rows][4]  (ax, ay, bx, by): a = query/self, b = train/acceding
 *   m_cnt    DEV int32  [P]        number of matches after de-dup
 *   n_filtered DEV int32 [P]       len(matches) before de-dup (what min_matching_pts tests)
 *   status   DEV int32  [P]        EVZ_ST_OK or EVZ_ST_FEW_MATCHES
 */
int evz_filter_matches(evz_handle* h, const int32_t* top2_idx, const int32_t* top2_d2,
                       const float* coords, const int32_t* canon,
                       const int32_t* row_off, const int32_t* n_kp,
                       const int32_t* pair_q, const int32_t* pair_t, const int32_t* out_off, int n_pairs,
                       int max_kp, double ratio, int min_matching_pts,
                       uint8_t* surv, int32_t* m_idx, float* m_pts, int32_t* m_cnt,
                       int32_t* n_filtered, int32_t* status, void* stream);

/* ---- K3 + K4: seeded RANSAC homography + refit.  Replaces
 * cv2.findHomography(a, b, cv2.RANSAC, thresh) at matching.py:156-157 (level 1) and
 * utils.py:356-358 (level 2), including the 70 % inlier gate of utils.py:359-360 when
 * min_inlier_frac > 0.  Pairs whose status is non-zero on entry are skipped.
 *   pts        DEV float [rows][4]  point pairs of pair p at rows [off[p], off[p]+cnt[p])
 *   max_cnt    upper bound of cnt[p] (sizes shared memory; <= EVZ_MAX_KP, else EVZ_E_UNSUPPORTED); a pair with
 *              cnt[p] > max_cnt gets fail_status
 *   pre_H      DEV double [P][9] or NULL: both point sets are first mapped through this
 *              matrix in f64 and rounded to f32 (utils.py:351-355, matrix_H_prev)
 *   n_hyp      hypotheses per pair, 1 .. 65535 (else EVZ_E_ARG) (counter-based sampler: seed, pair_id_base + p, level)
 *   fail_status value written to status[p] when no model is found (EVZ_ST_NO_MODEL_1/2)
 * outputs (any may be NULL except H and status)
 *   H          DEV double [P][9]  refined homography, h22 = 1: Levenberg-Marquardt on the 8 free parameters over the
 *                                 winner's inlier set (OpenCV's damping schedule and stop rule), started from the winning
 *                                 4-point model -- not from a normalised DLT as cv2 does; same optimum (<= 1e-3 px),
 *                                 first step undamped, stop when a step moves no point by more than 1e-6 px (an undamped
 *                                 step below 1e-3 px is applied without a confirming pass), <= 20 steps
 *   mask       DEV uint8 [rows]   final inlier mask: f32 reprojection error of the REFINED H <= thresh^2.  This is what
 *                                 cv2 >= 4.x returns (the oracle is pinned to cv2 4.13); the opencv-contrib 3.4.2 pinned by
 *                                 the reference's requirements.txt returns the RANSAC consensus mask (= mask_best) instead,
 *                                 so the 70 % gate can differ for pairs that sit on the boundary
 *   inl_cnt    DEV int32 [P]      sum(mask): the count the min_inlier_frac gate (utils.py:359) is applied to
 *   best_hyp   DEV int32 [P]      winning hypothesis (max inliers, ties -> lowest index)
 *   best_cnt   DEV int32 [P]      its inlier count
 *   mask_best  DEV uint8 [rows]   its inlier mask (the refit set)
 *   H_best     DEV double [P][9]  its 4-point model
 * Every max_cnt <= EVZ_MAX_KP and 1 <= n_hyp <= 65535 runs, with the same results whichever memory holds the tables.
 * Handle scratch used by this call: 4 B + 72 B per pair, plus a model cache of 32 B per (pair, hypothesis) when that stays
 * below 4 GB (without it every scoring stage solves its hypotheses again; the results are the same).  The scoring kernel
 * keeps 8 B per hypothesis of lists in shared memory next to 18 B per point of max_cnt; when both do not fit in the
 * device's per-block shared memory (on a B200: n_hyp > 944 at max_cnt = EVZ_MAX_KP, n_hyp > 28 582 at any max_cnt) the
 * lists take 8 B per (pair, hypothesis) of handle scratch instead, e.g. 8 MB for 1 000 pairs x 1 024 hypotheses or
 * 5.2 GB for 10 000 pairs x 65 535; EVZ_E_NOMEM when that cannot be allocated.
 */
int evz_find_homography(evz_handle* h, const float* pts, const int32_t* off, const int32_t* cnt, int n_pairs,
                        int max_cnt, const double* pre_H, int n_hyp, uint32_t seed, int64_t pair_id_base, int level,
                        double thresh, double min_inlier_frac, int fail_status,
                        int32_t* status, double* H, uint8_t* mask, int32_t* inl_cnt,
                        int32_t* best_hyp, int32_t* best_cnt, uint8_t* mask_best, double* H_best,
                        void* stream);
/* The same with a sampler id per pair instead of pair_id_base + p: pair p is seeded with pair_id[p].  Replaces the same
 * call sites; used to run the pairs of several videos in one launch while pair k of every video keeps id k, so that each
 * pair gets the result of a call on its video alone (video_processing.py:67-105 runs one video per call).
 *   pair_id    DEV int64 [P] (required)
 * Every other argument and result is that of evz_find_homography; with pair_id[p] = pair_id_base + p the results are
 * identical to it.
 */
int evz_find_homography_ids(evz_handle* h, const float* pts, const int32_t* off, const int32_t* cnt, int n_pairs,
                            int max_cnt, const double* pre_H, int n_hyp, uint32_t seed, const int64_t* pair_id, int level,
                            double thresh, double min_inlier_frac, int fail_status,
                            int32_t* status, double* H, uint8_t* mask, int32_t* inl_cnt,
                            int32_t* best_hyp, int32_t* best_cnt, uint8_t* mask_best, double* H_best,
                            void* stream);

/* ---- K5: displacement-mode static-point filter.  Replaces find_point_displacement
 * (utils.py:289-325) + get_largest_group_points (utils.py:258-286).
 *   out_pts DEV float [rows][4] kept point pairs (order preserved), out_cnt DEV int32 [P],
 *   best_r  DEV int32 [P] the winning rounded displacement, flags DEV int32 [P] (EVZ_FLAG_*)
 *   r_out   DEV int32 [rows] or NULL: round(||H a - b||) of every point (find_point_displacement's key)
 *   max_cnt upper bound of cnt[] known to the host; > EVZ_MAX_KP -> EVZ_E_UNSUPPORTED (like evz_find_homography)
 */
int evz_static_filter(evz_handle* h, const float* pts, const int32_t* off, const int32_t* cnt, int n_pairs,
                      int max_cnt, const double* H, const int32_t* status,
                      float* out_pts, int32_t* out_cnt, int32_t* best_r, int32_t* flags, int32_t* r_out,
                      void* stream);

/* ---- K5b: static points of several feature types, concatenated and de-duplicated per pair.  Replaces the tail of
 * FrameProcessing.concatenate_all_features_types (frame_processing.py:91-104: extend over the feature types, then
 * remove_double_matching, utils.py:41-68): the a-points of pair p are the keys in first-occurrence order over
 * type 0, type 1, ...; the b-point kept for a key is that of its LAST occurrence.
 *   n_types <= EVZ_MAX_TYPES; pts[t] DEV float [rows_t][4], off[t] / cnt[t] DEV int32 [P] (HOST arrays of device pointers)
 *   status  DEV int32 [P] non-zero: the pair produces no points
 *   out_off DEV int32 [P] first output row of pair p (capacity >= sum over t of cnt[t][p]); max_total: host-known upper
 *           bound of that sum, > EVZ_MAX_KP -> EVZ_E_UNSUPPORTED
 *   out_pts DEV float [out rows][4], out_cnt DEV int32 [P]
 */
#define EVZ_MAX_TYPES 4
int evz_concat_dedup(evz_handle* h, int n_types, const float* const* pts, const int32_t* const* off, const int32_t* const* cnt,
                     int n_pairs, const int32_t* status, int max_total, const int32_t* out_off,
                     float* out_pts, int32_t* out_cnt, void* stream);

/* ---- K6: None-H fallback + cumulative superposition as a parallel prefix product.
 * Replaces video_processing.py:94-103 and matrix_superposition / superposition_dict
 * (utils.py:118-145, 184-211).
 *   G       DEV double [P][9]  frame-plane step matrices (new frame -> previous frame)
 *   status  DEV int32  [P]     non-zero = "H is None"
 *   policy  1 = none_H_processing=True (reuse the previous pair's matrix), 0 = identity step
 *   seed_S  DEV double [9] or NULL  superposition before the first pair (identity if NULL)
 *   seed_G  DEV double [9] or NULL  last valid step matrix before the first pair
 * outputs
 *   S       DEV double [P][9]  S_k = normalise(S_{k-1} . Gfilled_k): frame k+1 -> fixed plane
 *   H_fixed DEV double [P][9]  S_k . S_{k-1}^-1 normalised: what the reference stores in
 *                              dict_with_homography_matrix.json (may be NULL)
 *   summary DEV double [20]    shard summary for the cross-GPU all-gather (may be NULL):
 *             [0..8]  R = product of the steps from the first valid pair on (filled)
 *             [9..17] last valid G of the shard, [18] number of leading invalid pairs,
 *             [19] 1 if the shard has a valid pair
 */
int evz_chain_scan(evz_handle* h, const double* G, const int32_t* status, int n_pairs, int policy,
                   const double* seed_S, const double* seed_G,
                   double* S, double* H_fixed, double* summary, void* stream);

/* ---- K6, many chains in one call: evz_chain_scan (no seeds, no summary) over every segment of the pair list.
 * Replaces video_processing.py:94-103 and superposition_dict (utils.py:184-211) for several videos at once: segment s is
 * one video's chain, pairs [seg_off[s], seg_off[s+1]); the None-H fill and the product restart at its first pair.
 *   seg_off DEV int32 [n_segs+1], non-decreasing, seg_off[0] = 0, seg_off[n_segs] = n_pairs; empty segments are allowed
 *   S       DEV double [P][9] (required), H_fixed DEV double [P][9] or NULL
 * The rows of every segment are bit-identical to what evz_chain_scan writes for that segment alone (same policy): the
 * segment is cut into 256-pair blocks counted from its own start and scanned by the same kernels.  A fixed number of
 * launches, whatever n_segs; handle scratch of about 4 B per pair + 160 B per (256 pairs + 1 segment).
 */
int evz_chain_scan_segments(evz_handle* h, const double* G, const int32_t* status, int n_pairs,
                            const int32_t* seg_off, int n_segs, int policy, double* S, double* H_fixed, void* stream);

/* ---- K6c: one step of the reference-exact chain for n_chains independent chains.  Replaces the host loop body of
 * video_processing.py:94-105 (None-H policy, matrix_superposition utils.py:118-145) so that a chain advances without a
 * host round trip; the next step's RANSAC #2 reads S_state as its pre_H.  Chain c:
 *   H = H2[c]        if status[c] == EVZ_ST_OK
 *     = H_prev[c]    elif policy and not first              (video_processing.py:95-96)
 *     = identity     otherwise                              (the reference crashes here; DESIGN.md deviation 4)
 *   H_out[c] = H;  S_state[c] = H if first (un-normalised, as the reference), else C / C[2][2] with C = H . S_state[c]
 *   C[i][j] = fma(H[i][2], S[2][j], fma(H[i][1], S[1][j], H[i][0] * S[0][j])), each operation rounded once (the order of
 *   NumPy's np.dot on 3x3 f64 through OpenBLAS), then an IEEE division of every element by C[2][2].
 *   H2, H_out DEV double [n_chains][9]; status DEV int32 [n_chains]; S_state DEV double [n_chains][9] (in/out)
 *   H_prev DEV double [n_chains][9]: the previous step's H_out (may alias H_out); NULL allowed when first or policy = 0
 * n_chains = 0 is a no-op.  Chains that end early are dropped from the end: order chains by length, longest first.
 */
int evz_chain_ref_step(evz_handle* h, const double* H2, const int32_t* status, int n_chains, int first, int policy,
                       double* S_state, const double* H_prev, double* H_out, void* stream);

/* ---- K6b: cross-GPU seeding of the scan, on the device (no host round trip).  Every rank calls evz_chain_scan with
 * S and summary (no seeds: an UNSEEDED local scan), all-gathers the 20-double summaries into `summaries`
 * (ncclAllGather / torch.distributed.all_gather_into_tensor), then calls this: S becomes the rank's slice of the global
 * scan (identical to evz_chain_scan over the whole video up to the rounding of a different association order).
 *   summaries DEV double [world][20]; S DEV double [P][9] in: unseeded local scan, out: global scan
 *   H_fixed   DEV double [P][9] or NULL;  seeds_out DEV double [27]: seed_S | seed_G | seed_S . seed_G^lead
 */
int evz_chain_seed_apply(evz_handle* h, const double* summaries, int world, int rank, int policy, int n_pairs,
                         double* S, double* H_fixed, double* seeds_out, void* stream);

/* ---- K7: object-coordinate remap.  Replaces from_original_to_fix / from_fix_to_original
 * (fixed_coordinate_system.py:19-122): (x', y') = around(T . (sx*x, sy*y, 1), 2) with
 * T = S[frame] (inverse = 0) or S[frame]^-1 (inverse = 1).
 *   pts_in DEV double [n][2], frame_idx DEV int32 [n] (row of S), S DEV double [F][9]
 */
int evz_remap(evz_handle* h, const double* pts_in, const int32_t* frame_idx, int64_t n,
              const double* S, int n_frames, double sx, double sy, int inverse,
              double* pts_out, void* stream);

/* ---- dense remap + max-movement metric (SURVEY 8f-2).  Replaces the per-pixel
 * np.apply_along_axis(homography_transformation, ...) of heatmap_video_processing
 * (visualization/processing_visualization.py:404-418): max over the first n_frames rows of S
 * and all pixels of the w x h grid of max(x', y').
 *   out_max DEV double [1]
 */
int evz_max_movement(evz_handle* h, const double* S, int n_frames, int height, int width,
                     double* out_max, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EVZ_H */
