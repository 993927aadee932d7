"""Descriptor matching on the GPU behind the reference's `matching.py` API
(reference evenvizion/processing/matching.py:22-239).

`KeyPoints.match_kps` / `match_static_kps` run the tcgen05 matcher, the ratio / many-to-one /
de-dup filter, the seeded RANSAC + LM refit and the static-point filter of libevz.so on the
current CUDA device.  There is no CPU fallback.
"""
import numpy as np
import torch

from .. import _lib
from .constants import THRESHOLD_FOR_FIND_HOMOGRAPHY, LOWES_RATIO, MINIMUM_MATCHING_POINTS, \
    RANSAC_HYPOTHESES, RANSAC_SEED


class NoMatchesException(Exception):
    """reference matching.py:22-44: `str(e)` is "reason -> description"."""

    def __init__(self, reason, description="no matches found"):
        self.reason = reason
        self.description = description
        super().__init__(description)

    def __str__(self):
        return f'{self.reason} -> {self.description}'


def _engine():
    from .. import default_engine
    return default_engine()


def _two_frame_store(eng, q_kps, t_kps):
    """frame 0 = acceding (train), frame 1 = self (query)."""
    qd, td = np.asarray(q_kps.descriptors), np.asarray(t_kps.descriptors)
    if qd.ndim != 2 or td.ndim != 2 or qd.shape[1] != td.shape[1]:
        raise ValueError("descriptor arrays must be 2-D with the same width")
    dt = np.float32 if (qd.dtype != np.uint8 or td.dtype != np.uint8) else np.uint8
    desc = np.concatenate([td.astype(dt, copy=False), qd.astype(dt, copy=False)])
    coords = np.concatenate([np.asarray(t_kps.coordinates, np.float32).reshape(-1, 2),
                             np.asarray(q_kps.coordinates, np.float32).reshape(-1, 2)])
    return eng.ingest(desc, coords, [len(td), len(qd)])


class KeyPoints:
    """reference matching.py:47-163.  coordinates: (N,2) float32; descriptors: (N,D) SIFT (float32,
    integer-valued) or ORB (uint8) descriptors, or None."""

    def __init__(self, coordinates, descriptors):
        self.coordinates = coordinates
        self.descriptors = descriptors

    # -- device-side core shared by match_kps / match_static_kps
    def _match_device(self, acceding_kps, ratio, min_matching_pts):
        if self.descriptors is None:
            raise NoMatchesException("self.descriptors is None", "couldn't process")
        if acceding_kps.descriptors is None:
            raise NoMatchesException("kps.descriptors is None", "couldn't process")
        eng = _engine()
        st = _two_frame_store(eng, self, acceding_kps)
        r = eng.match(st, [1], [0], ratio, min_matching_pts)
        if int(r.status[0]) == _lib.ST_FEW_MATCHES:
            raise NoMatchesException("len(matches) {} < min_matching_pts {}".format(int(r.n_filtered[0]), min_matching_pts),
                                     "couldn't process")
        return eng, st, r

    def match_kps(self, acceding_kps, ratio=LOWES_RATIO, min_matching_pts=MINIMUM_MATCHING_POINTS):
        """2-NN brute-force match, Lowe ratio test, many-to-one filter, coordinate de-dup
        (reference matching.py:75-129).  Returns (pts_a, pts_b): lists of float32 (x, y) arrays,
        pts_a from self, pts_b from acceding_kps."""
        eng, st, r = self._match_device(acceding_kps, ratio, min_matching_pts)
        o, m = int(st.row_off_h[1]), int(r.m_cnt[0])
        pts = r.m_pts[o:o + m].cpu().numpy()
        return [p for p in pts[:, :2].copy()], [p for p in pts[:, 2:].copy()]

    def match_static_kps(self, acceding_kps, reproj_thresh=THRESHOLD_FOR_FIND_HOMOGRAPHY,
                         n_hyp=None, seed=None, pair_id=0, confidence=None):
        """Matches that lie on static objects (reference matching.py:131-163): RANSAC homography,
        then the largest group of equal rounded displacement.  Returns two (Ms,2) float32 arrays.
        confidence: None scores n_hyp hypotheses; a float in (0, 1) stops where cv2's RANSAC would (n_hyp = maxIters)."""
        eng, st, r = self._match_device(acceding_kps, LOWES_RATIO, MINIMUM_MATCHING_POINTS)
        n_hyp = RANSAC_HYPOTHESES if n_hyp is None else n_hyp
        seed = RANSAC_SEED if seed is None else seed
        h1 = eng.find_homography(r.m_pts, r.out_off, r.m_cnt, r.status, st.max_kp, n_hyp, seed, pair_id, 1,
                                 reproj_thresh, 0.0, _lib.ST_NO_MODEL_1, confidence=confidence)
        s = int(r.status[0])
        if s == _lib.ST_FEW_POINTS:
            raise NoMatchesException("fewer than 4 matching points after de-duplication", "couldn't process")
        if s != 0:
            raise NoMatchesException("can't find homography matrix", "couldn't process")
        sp, sc, _, _ = eng.static_filter(r.m_pts, r.out_off, r.m_cnt, h1["H"], r.status, max_cnt=st.max_kp)
        o, m = int(st.row_off_h[1]), int(sc[0])
        pts = sp[o:o + m].cpu().numpy()
        return pts[:, :2].copy(), pts[:, 2:].copy()


def lowes_ratio_test(raw_matches, ratio=LOWES_RATIO):
    """reference matching.py:166-198 on a list of cv2 DMatch tuples.  Host-side structural helper
    kept for API compatibility only: the device pipeline (`KeyPoints.match_kps`) fuses this test
    into the matcher's filter kernel and never calls it."""
    train_idx_dict = {}
    query_idx_dict = {}
    for m in raw_matches:
        if len(m) == 2 and m[0].distance < m[1].distance * ratio:
            train_idx_dict.setdefault(m[0].trainIdx, []).append(m[0].queryIdx)
            query_idx_dict.setdefault(m[0].queryIdx, []).append(m[0].trainIdx)
    return filter_corresponding_points(train_idx_dict, query_idx_dict)


def filter_corresponding_points(train_idx_dict, query_idx_dict):
    """reference matching.py:201-239: a train point claimed by several query points is dropped."""
    dead = {k for k, v in train_idx_dict.items() if len(v) > 1}
    for v in query_idx_dict.values():
        if len(v) > 1:
            dead.update(v)
    for k in dead:
        train_idx_dict.pop(k, None)
    return [(t, q[0]) for t, q in train_idx_dict.items()]
