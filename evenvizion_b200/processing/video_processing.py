"""Video driver (reference evenvizion/processing/video_processing.py:27-108) with the geometry on the GPU.

    get_homography_dict(capture, resize_width=400, matching_path=None, none_H_processing=True)
        -> {2: {"H": 3x3 list}, ..., F: {"H": ...}, "resize_info": {"h": int, "w": int}}

Frames are decoded / resized / described by OpenCV on the CPU (once per frame; the reference
describes every frame twice), then ALL consecutive pairs are matched, RANSAC'd and static-filtered
in batched kernel launches.  Two formulations of the second RANSAC:

  mode="reference" (default)  points are pre-transformed by the running superposition exactly as
      compute_homography(matrix_H_prev) does (utils.py:351-355), so H_k lives in the fixed plane
      and pair k depends on all earlier pairs: a serial chain of single-pair launches;
  mode="parallel"  every pair is solved in its own frame plane, then None-H forward fill and the
      cumulative product run as a parallel prefix scan and H_k = S_k . S_{k-1}^-1 is emitted, so
      that the reference's `superposition_dict` reproduces S.  The RANSAC threshold then acts in
      frame pixels instead of fixed-plane pixels (documented deviation, DESIGN.md).
"""
import logging

import numpy as np
import torch

from .. import _lib
from .constants import RANSAC_HYPOTHESES, RANSAC_SEED, THRESHOLD_FOR_FIND_HOMOGRAPHY, LENGTH_ACCOUNTED_POINTS
from .frame_processing import FrameProcessing, resize, DEFAULT_FEATURES

log = logging.getLogger(__name__)


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
    """The hot path for a whole video given per-frame features.  Returns (H_list, status): H_list[k]
    is the 3x3 matrix stored under frame k+2 (None only when the policy leaves it undefined)."""
    from .. import default_engine
    eng = engine or default_engine()
    n_hyp = RANSAC_HYPOTHESES if n_hyp is None else n_hyp
    seed = RANSAC_SEED if seed is None else seed
    types = list(feats)
    F = len(feats[types[0]])
    P = F - 1
    if P <= 0:
        return [], np.zeros(0, np.int32)
    dev = eng.device
    status = torch.zeros(P, dtype=torch.int32, device=dev)
    per_type = []
    for t in types:
        st = _ingest_frames(eng, [feats[t]], frames_d(feats[t]))
        r = eng.match(st, np.arange(1, F), np.arange(0, F - 1))
        h1 = eng.find_homography(r.m_pts, r.out_off, r.m_cnt, r.status, st.max_kp, n_hyp, seed, 0, 1,
                                 THRESHOLD_FOR_FIND_HOMOGRAPHY, 0.0, _lib.ST_NO_MODEL_1)
        sp, sc, _, _ = eng.static_filter(r.m_pts, r.out_off, r.m_cnt, h1["H"], r.status, max_cnt=st.max_kp)
        status = torch.where(status == 0, r.status, status)      # any failing feature type fails the pair
        per_type.append((st, r, sp, sc))
    # level-2 input: static points of all feature types, concatenated + de-duplicated per pair
    if len(types) == 1:
        st, r, pts2, cnt2 = per_type[0]
        off2 = r.out_off
        max_cnt = st.max_kp
        cnt2 = torch.where(status == 0, cnt2, torch.zeros_like(cnt2))
    else:
        # frame_processing.py:91-104 on the device (evz_concat_dedup): pair p may hold up to the sum over the types
        # of the query frame's keypoints -- known on the host, so the layout needs no read-back
        cap = np.zeros(P, np.int64)
        for st, _, _, _ in per_type:
            cap += st.n_kp_h[1:].astype(np.int64)
        cap = (cap + 3) // 4 * 4 + 4
        off_h = np.zeros(P, np.int64)
        np.cumsum(cap[:-1], out=off_h[1:])
        max_cnt = max(int(sum(st.max_kp for st, _, _, _ in per_type)), 4)
        off2 = torch.from_numpy(off_h.astype(np.int32)).to(dev)
        pts2, cnt2 = eng.concat_dedup([(sp, r.out_off, sc) for _, r, sp, sc in per_type], status, off2,
                                      int(cap.sum()), max_cnt)
    if mode == "parallel":
        h2 = eng.find_homography(pts2, off2, cnt2, status, max_cnt, n_hyp, seed, 0, 2, THRESHOLD_FOR_FIND_HOMOGRAPHY,
                                 LENGTH_ACCOUNTED_POINTS, _lib.ST_NO_MODEL_2)
        S, Hf, _ = eng.chain_scan(h2["H"], status, none_H_processing)
        st_h = status.cpu().numpy()
        Hf = Hf.cpu().numpy().reshape(P, 3, 3)
        return [Hf[k] for k in range(P)], st_h
    if mode != "reference":
        raise ValueError("mode must be 'reference' or 'parallel'")
    # reference-exact serial chain (video_processing.py:67-105): RANSAC #2 of pair k sees its points through the
    # running superposition, so the pairs go one by one.  Everything a pair needs is allocated once (single-pair
    # views of the point store); per pair: one launch pair and one small read-back (status + H).
    H_list, st_out = [], np.zeros(P, np.int32)
    st_in = status.cpu().numpy()
    S, H_prev, first = None, None, True
    pre = torch.zeros((1, 9), dtype=torch.float64, device=dev)
    pre_h = torch.zeros((1, 9), dtype=torch.float64).pin_memory()
    res = torch.zeros((1, 10), dtype=torch.float64, device=dev)          # H (9) + status
    res_h = torch.zeros((1, 10), dtype=torch.float64).pin_memory()
    s_k = torch.zeros(1, dtype=torch.int32, device=dev)
    for k in range(P):
        H = None
        st_out[k] = st_in[k]
        if st_in[k] == 0:
            s_k.zero_()
            if S is not None:
                pre_h.copy_(torch.from_numpy(np.asarray(S, np.float64).reshape(1, 9)))
                pre.copy_(pre_h, non_blocking=True)
            h2 = eng.find_homography(pts2, off2[k:k + 1], cnt2[k:k + 1], s_k, max_cnt, n_hyp, seed, k, 2,
                                     THRESHOLD_FOR_FIND_HOMOGRAPHY, LENGTH_ACCOUNTED_POINTS, _lib.ST_NO_MODEL_2,
                                     pre_H=None if S is None else pre, light=True)
            res[0, :9] = h2["H"][0]
            res[0, 9] = s_k[0]
            res_h.copy_(res)                                         # one synchronising read-back per pair
            st_out[k] = int(res_h[0, 9])
            if st_out[k] == 0:
                H = res_h[0, :9].numpy().reshape(3, 3).copy()
        if H is None:
            if none_H_processing:
                H = H_prev                       # the reference reuses the previous pair's matrix (:95-96)
            if H is None:
                # none_H_processing=False, or no previous matrix yet.  The reference crashes here
                # (video_processing.py:98-101); README.md:45 documents "no transformation on this frame".
                H = np.eye(3)
                log.info("pair %d: no homography (status %d), identity step", k + 2, st_out[k])
        H_list.append(H)
        if first:
            S, first = H, False
        else:
            S = np.dot(H, S)
            S = S / S[2][2]
        H_prev = H
    return H_list, st_out


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


def geometry_from_features_batch(feats_list, none_H_processing=True, mode="reference", n_hyp=None, seed=None, engine=None):
    """`geometry_from_features` for many videos in one call: returns [(H_list, status)] in input order, entry i equal to
    geometry_from_features(feats_list[i], ...).  All videos share one frame store per feature type and one launch of
    every per-pair stage; pair k of every video keeps RANSAC id k.  mode="parallel" ends in one segmented scan;
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
    F = np.array([len(f[types[0]]) for f in feats_list], np.int64)
    n_pairs = np.maximum(F - 1, 0)
    lay = PairLayout(n_pairs, step_major=(mode == "reference"))
    P = len(lay.k)
    if P == 0:
        return [([], np.zeros(0, np.int32)) for _ in feats_list]
    dev = eng.device
    f0 = np.zeros(len(F), np.int64)
    np.cumsum(F[:-1], out=f0[1:])
    pq = f0[lay.video] + lay.k + 1
    pt = f0[lay.video] + lay.k
    ids = torch.from_numpy(lay.k).to(dev)
    status = torch.zeros(P, dtype=torch.int32, device=dev)
    per_type, video_kp = [], []
    for t in types:
        d = next((dd.shape[1] for f in feats_list for _, dd in f[t] if dd is not None), 128)
        st = _ingest_frames(eng, [f[t] for f in feats_list], d)
        kp = st.n_kp_h.astype(np.int64)
        video_kp.append([int(kp[a:b].max(initial=0)) for a, b, n in zip(f0, f0 + F, n_pairs) if n])   # each video's store max_kp
        r = eng.match(st, pq, pt)
        h1 = eng.find_homography(r.m_pts, r.out_off, r.m_cnt, r.status, st.max_kp, n_hyp, seed, 0, 1,
                                 THRESHOLD_FOR_FIND_HOMOGRAPHY, 0.0, _lib.ST_NO_MODEL_1, pair_ids=ids)
        sp, sc, _, _ = eng.static_filter(r.m_pts, r.out_off, r.m_cnt, h1["H"], r.status, max_cnt=st.max_kp)
        status = torch.where(status == 0, r.status, status)
        per_type.append((st, r, sp, sc))
    # level-2 input, as geometry_from_features builds it; max_cnt = the largest of the per-video bounds it would use
    if len(types) == 1:
        st, r, pts2, cnt2 = per_type[0]
        off2 = r.out_off
        max_cnt = max(video_kp[0])
        cnt2 = torch.where(status == 0, cnt2, torch.zeros_like(cnt2))
    else:
        cap = np.zeros(P, np.int64)
        for st, _, _, _ in per_type:
            cap += st.n_kp_h[pq].astype(np.int64)
        cap = (cap + 3) // 4 * 4 + 4
        off_h = np.zeros(P, np.int64)
        np.cumsum(cap[:-1], out=off_h[1:])
        max_cnt = max(max(sum(v), 4) for v in zip(*video_kp))
        off2 = torch.from_numpy(off_h.astype(np.int32)).to(dev)
        pts2, cnt2 = eng.concat_dedup([(sp, r.out_off, sc) for _, r, sp, sc in per_type], status, off2,
                                      int(cap.sum()), max_cnt)
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


def frames_d(frames):
    for _, d in frames:
        if d is not None:
            return d.shape[1]
    return 128


def get_homography_dict(capture, resize_width=400, matching_path=None, none_H_processing=True,
                        features_type_list=None, mode="reference", n_hyp=None, seed=None):
    """reference video_processing.py:27-108.  `matching_path` (match visualisation PNGs) belongs to the
    out-of-scope visualisation layer and is ignored."""
    feats, shape = read_and_describe(capture, resize_width, features_type_list)
    H_list, _ = geometry_from_features(feats, none_H_processing, mode, n_hyp, seed)
    homography_dict = {}
    for k, H in enumerate(H_list):
        homography_dict[k + 2] = {"H": np.asarray(H, np.float64).tolist()}
    homography_dict["resize_info"] = {"h": int(shape[0]), "w": int(shape[1])}
    return homography_dict


def get_homography_dicts(captures, resize_width=400, matching_path=None, none_H_processing=True,
                         features_type_list=None, mode="reference", n_hyp=None, seed=None):
    """`get_homography_dict` for several captures: every capture is decoded and described as there, then the geometry
    of all of them runs in one `geometry_from_features_batch` call.  Returns one dict per capture, in order."""
    described = [read_and_describe(c, resize_width, features_type_list) for c in captures]
    results = geometry_from_features_batch([f for f, _ in described], none_H_processing, mode, n_hyp, seed)
    out = []
    for (_, shape), (H_list, _) in zip(described, results):
        homography_dict = {k + 2: {"H": np.asarray(H, np.float64).tolist()} for k, H in enumerate(H_list)}
        homography_dict["resize_info"] = {"h": int(shape[0]), "w": int(shape[1])}
        out.append(homography_dict)
    return out
