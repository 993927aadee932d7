"""Video driver (reference evenvizion/processing/video_processing.py:27-108) with the geometry on the GPU.

    get_homography_dict(capture, resize_width=400, matching_path=None, none_H_processing=True)
        -> {2: {"H": 3x3 list}, ..., F: {"H": ...}, "resize_info": {"h": int, "w": int}}

Frames are decoded / resized / described by OpenCV on the CPU (once per frame; the reference
describes every frame twice), then ALL consecutive pairs are matched, RANSAC'd and static-filtered
in batched kernel launches.  One video is a batch of one (`geometry_from_features_batch`).  Two
formulations of the second RANSAC:

  mode="reference" (default)  points are pre-transformed by the running superposition exactly as
      compute_homography(matrix_H_prev) does (utils.py:351-355), so H_k lives in the fixed plane
      and pair k depends on all earlier pairs: the chains advance in lockstep on the device, one
      RANSAC launch and one chain-step launch per step, with no host round trip inside the loop;
  mode="parallel"  every pair is solved in its own frame plane, then None-H forward fill and the
      cumulative product run as a parallel prefix scan and H_k = S_k . S_{k-1}^-1 is emitted, so
      that the reference's `superposition_dict` reproduces S.  The RANSAC threshold then acts in
      frame pixels instead of fixed-plane pixels (documented deviation, DESIGN.md).
"""
import numpy as np
import torch

from .. import _lib
from .._lib import EVZ_MAX_KP
from .constants import RANSAC_HYPOTHESES, RANSAC_SEED, THRESHOLD_FOR_FIND_HOMOGRAPHY, LENGTH_ACCOUNTED_POINTS
from .frame_processing import FrameProcessing, resize, DEFAULT_FEATURES


def read_and_describe(capture, resize_width=400, features_type_list=None):
    """Decode, resize and describe every frame (OpenCV, CPU).  Returns (features, shape) where
    features[type] = list over frames of (coords (N,2) f32, desc (N,D))."""
    feats = {t: [] for t in (features_type_list or DEFAULT_FEATURES)}
    success, image = capture.read()
    if not success:
        raise ValueError("Problem with video! Can't read first frame")
    shape = None
    while success:
        image = resize(image, width=resize_width)
        shape = image.shape[:2]
        fp = FrameProcessing(image, list(feats))
        for t in feats:
            feats[t].append(fp.detect_and_describe_features(t))
        success, image = capture.read()
    return feats, shape


def geometry_from_features(feats, none_H_processing=True, mode="reference", n_hyp=None, seed=None, engine=None):
    """The hot path for a whole video given per-frame features: `geometry_from_features_batch` of one video.  Returns
    (H_list, status): H_list[k] is the 3x3 matrix stored under frame k+2, after the None-H policy (identity where the
    policy leaves it undefined); status int32 [F-1]."""
    return geometry_from_features_batch([feats], none_H_processing, mode, n_hyp, seed, engine)[0]


class PairLayout:
    """Where the pairs of several videos sit in one batched call.  Video v has n_pairs[v] pairs; pair (v, k) is frame
    pair (k + 1, k) of video v.
      video, k   int64 [P]  video and within-video pair index of every pair, in processing order
      inverse    int64 [P]  processing position of every pair in input order (video-major, videos in input order), so that
                            per_pair_result[inverse] lists video 0's pairs, then video 1's, ...
      seg_off    int64 [V+1] first input-order position of every video's pairs (the split of per_pair_result[inverse])
      step_off   int64 [K+1] step-major only: step k = pairs [step_off[k], step_off[k+1]) = pair k of the n_k longest videos
    Step-major order (the lockstep reference chain) sorts the videos by pair count, longest first (ties in input order),
    so the chains still running at step k are a prefix; otherwise the order is video-major in input order, which is what
    the segmented scan wants."""

    def __init__(self, n_pairs, step_major):
        n = np.asarray(n_pairs, np.int64).reshape(-1)
        self.seg_off = np.zeros(len(n) + 1, np.int64)
        np.cumsum(n, out=self.seg_off[1:])
        video_in = np.repeat(np.arange(len(n), dtype=np.int64), n)        # input order
        k_in = np.arange(int(self.seg_off[-1]), dtype=np.int64) - self.seg_off[video_in]
        if step_major:
            rank = np.empty(len(n), np.int64)
            rank[np.argsort(-n, kind="stable")] = np.arange(len(n))
            order = np.lexsort((rank[video_in], k_in))                    # by step, then by rank of the video
            self.step_off = np.searchsorted(k_in[order], np.arange(int(n.max(initial=0)) + 1), side="left").astype(np.int64)
        else:
            order = np.arange(len(video_in), dtype=np.int64)
            self.step_off = None
        self.video, self.k = video_in[order], k_in[order]
        self.inverse = np.empty(len(order), np.int64)
        self.inverse[order] = np.arange(len(order), dtype=np.int64)

    def split(self, per_pair):
        """per-pair values in processing order -> list over videos (input order) of their pairs in order."""
        x = np.asarray(per_pair)[self.inverse]
        return [x[a:b] for a, b in zip(self.seg_off[:-1], self.seg_off[1:])]


def _ingest_frames(eng, frames_per_video, d):
    """One frame store over the frames of every video, concatenated; d = descriptor width of the feature type.  A frame
    without descriptors becomes an empty frame: it fails every pair it belongs to (matching.py:104-107)."""
    frames = [(c if dd is not None else np.zeros((0, 2), np.float32), dd if dd is not None else np.zeros((0, d), np.uint8))
              for fr in frames_per_video for c, dd in fr]
    dtype = np.uint8 if all(dd.dtype == np.uint8 for _, dd in frames) else np.float32
    desc = np.concatenate([np.asarray(dd, dtype).reshape(len(c), d) for c, dd in frames])
    coords = np.concatenate([np.asarray(c, np.float32).reshape(-1, 2) for c, _ in frames])
    return eng.ingest(desc, coords, [len(c) for c, _ in frames])


def _level2_bound(feats_list, types):
    """Upper bound of the point count of a pair at RANSAC #2, known before anything is launched: over the videos with a
    pair, the sum over the feature types of the video's largest frame (the static points of every type are concatenated,
    frame_processing.py:91-104).  Raises ValueError when it exceeds EVZ_MAX_KP, the most that RANSAC and the de-dup take."""
    kp = lambda frames: max((len(c) for c, dd in frames if dd is not None), default=0)
    bound = max((sum(kp(f[t]) for t in types) for f in feats_list if len(f[types[0]]) > 1), default=0)
    if bound > EVZ_MAX_KP:
        raise ValueError(f"frames of {' + '.join(types)} features reach {bound} points per pair after concatenation; "
                         f"at most EVZ_MAX_KP = {EVZ_MAX_KP} are supported")
    return bound


def _level2_input(eng, feats_list, lay, ids, n_hyp, seed):
    """Match, RANSAC #1 (pair p seeded with ids[p]) and the static filter of every pair of `lay`, for every feature type,
    then the input of RANSAC #2: the static points of all types concatenated and de-duplicated per pair
    (frame_processing.py:91-104).  Returns (pts, off, cnt, status, max_cnt); a pair that failed for any type has status
    != 0, and max_cnt is `_level2_bound` (checked before anything is launched)."""
    types = list(feats_list[0])
    max_cnt = _level2_bound(feats_list, types)
    F = np.array([len(f[types[0]]) for f in feats_list], np.int64)
    P = len(lay.k)
    f0 = np.zeros(len(F), np.int64)
    np.cumsum(F[:-1], out=f0[1:])
    pq = f0[lay.video] + lay.k + 1
    pt = f0[lay.video] + lay.k
    status = torch.zeros(P, dtype=torch.int32, device=eng.device)
    per_type = []
    for t in types:
        d = next((dd.shape[1] for f in feats_list for _, dd in f[t] if dd is not None), 128)
        st = _ingest_frames(eng, [f[t] for f in feats_list], d)
        r = eng.match(st, pq, pt)
        h1 = eng.find_homography(r.m_pts, r.out_off, r.m_cnt, r.status, st.max_kp, n_hyp, seed, 0, 1,
                                 THRESHOLD_FOR_FIND_HOMOGRAPHY, 0.0, _lib.ST_NO_MODEL_1, pair_ids=ids)
        sp, sc, _, _ = eng.static_filter(r.m_pts, r.out_off, r.m_cnt, h1["H"], r.status, max_cnt=st.max_kp)
        status = torch.where(status == 0, r.status, status)      # any failing feature type fails the pair
        per_type.append((st, r, sp, sc))
    if len(types) == 1:
        st, r, pts2, cnt2 = per_type[0]
        return pts2, r.out_off, torch.where(status == 0, cnt2, torch.zeros_like(cnt2)), status, max_cnt
    # evz_concat_dedup: pair p may hold up to the sum over the types of the query frame's keypoints -- known on the host,
    # so the layout needs no read-back
    cap = np.zeros(P, np.int64)
    for st, _, _, _ in per_type:
        cap += st.n_kp_h[pq].astype(np.int64)
    cap = (cap + 3) // 4 * 4 + 4
    off_h = np.zeros(P, np.int64)
    np.cumsum(cap[:-1], out=off_h[1:])
    off2 = torch.from_numpy(off_h.astype(np.int32)).to(eng.device)
    pts2, cnt2 = eng.concat_dedup([(sp, r.out_off, sc) for _, r, sp, sc in per_type], status, off2, int(cap.sum()), max_cnt)
    return pts2, off2, cnt2, status, max_cnt


def geometry_from_features_batch(feats_list, none_H_processing=True, mode="reference", n_hyp=None, seed=None, engine=None):
    """The geometry of many videos in one call: returns [(H_list, status)] in input order, entry i the same as for
    feats_list[i] alone.  All videos share one frame store per feature type and one launch of every per-pair stage;
    pair k of every video keeps RANSAC id k.  mode="parallel" ends in one segmented scan;
    mode="reference" runs the reference-exact chains of all videos in lockstep on the device (one RANSAC #2 launch and
    one chain-step launch per step, no host round trip inside the loop)."""
    from .. import default_engine
    eng = engine or default_engine()
    n_hyp = RANSAC_HYPOTHESES if n_hyp is None else n_hyp
    seed = RANSAC_SEED if seed is None else seed
    if mode not in ("reference", "parallel"):
        raise ValueError("mode must be 'reference' or 'parallel'")
    if not feats_list:
        return []
    types = list(feats_list[0])
    if any(list(f) != types for f in feats_list):
        raise ValueError("every video must list the same feature types")
    lay = PairLayout(np.maximum([len(f[types[0]]) - 1 for f in feats_list], 0), step_major=(mode == "reference"))
    P = len(lay.k)
    if P == 0:
        return [([], np.zeros(0, np.int32)) for _ in feats_list]
    _level2_bound(feats_list, types)                 # an unsupported size is refused before the engine is used
    dev = eng.device
    ids = torch.from_numpy(lay.k).to(dev)
    pts2, off2, cnt2, status, max_cnt = _level2_input(eng, feats_list, lay, ids, n_hyp, seed)
    if mode == "parallel":
        h2 = eng.find_homography(pts2, off2, cnt2, status, max_cnt, n_hyp, seed, 0, 2, THRESHOLD_FOR_FIND_HOMOGRAPHY,
                                 LENGTH_ACCOUNTED_POINTS, _lib.ST_NO_MODEL_2, pair_ids=ids)
        seg_off = torch.from_numpy(lay.seg_off.astype(np.int32)).to(dev)
        _, H = eng.chain_scan_segments(h2["H"], status, seg_off, none_H_processing)
    else:
        H = eng.reference_chains(pts2, off2, cnt2, status, max_cnt, lay.step_off, n_hyp, seed, none_H_processing,
                                 THRESHOLD_FOR_FIND_HOMOGRAPHY, LENGTH_ACCOUNTED_POINTS, _lib.ST_NO_MODEL_2)
    H = H.cpu().numpy().reshape(P, 3, 3)
    st_h = status.cpu().numpy()
    return [([Hv[k] for k in range(len(Hv))], sv) for Hv, sv in zip(lay.split(H), lay.split(st_h))]


def get_homography_dict(capture, resize_width=400, matching_path=None, none_H_processing=True,
                        features_type_list=None, mode="reference", n_hyp=None, seed=None):
    """reference video_processing.py:27-108.  `matching_path` (match visualisation PNGs) belongs to the
    out-of-scope visualisation layer and is ignored."""
    return get_homography_dicts([capture], resize_width, matching_path, none_H_processing, features_type_list, mode,
                                n_hyp, seed)[0]


def get_homography_dicts(captures, resize_width=400, matching_path=None, none_H_processing=True,
                         features_type_list=None, mode="reference", n_hyp=None, seed=None):
    """`get_homography_dict` for several captures: every capture is decoded and described (`read_and_describe`), then
    the geometry of all of them runs in one `geometry_from_features_batch` call.  Returns one dict per capture, in order."""
    described = [read_and_describe(c, resize_width, features_type_list) for c in captures]
    results = geometry_from_features_batch([f for f, _ in described], none_H_processing, mode, n_hyp, seed)
    out = []
    for (_, shape), (H_list, _) in zip(described, results):
        homography_dict = {k + 2: {"H": np.asarray(H, np.float64).tolist()} for k, H in enumerate(H_list)}
        homography_dict["resize_info"] = {"h": int(shape[0]), "w": int(shape[1])}
        out.append(homography_dict)
    return out
