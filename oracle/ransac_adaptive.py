"""Oracle: OpenCV's confidence-bounded RANSAC stop on the seeded hypothesis stream of oracle/ransac.py
(evz_find_homography_adaptive, include/evz.h), and the multi-feature video chain of oracle/pipeline.py with that stop at
both RANSAC levels.

Test infrastructure only -- see oracle/__init__.py.

The rule is OpenCV's RANSACPointSetRegistrator::run / RANSACUpdateNumIters (ptsetreg.cpp, recalled), applied to the
hypotheses 0, 1, .., n_hyp - 1 of `ransac.hyp_indices` in index order:
  * a hypothesis that fails `solve4`'s validity test consumes no iteration (cv2's getSubset draws again);
  * state: best = 0, niters = n_hyp, it = 0;
  * after each valid hypothesis with count c: it += 1; if c > max(best, 3): best = c and
    niters = update_num_iters(confidence, (m - c) / m, niters);
  * stop when it >= niters or when the stream ends; n_used = one past the last hypothesis consumed.
The winner is the (count desc, index asc) arg-max over the consumed prefix, so the whole result is
`ransac.find_homography_seeded` at n_hyp = n_used.
"""
import math

import numpy as np

from . import chain, matching, ransac, static_filter
from .pipeline import (LENGTH_ACCOUNTED_POINTS, ST_FEW_INLIERS, ST_FEW_MATCHES, ST_FEW_POINTS, ST_NO_MODEL_1,
                       ST_NO_MODEL_2, ST_OK)

TIE_REL = 1e-9    # a bound this close to a rounding or cap boundary may come out either way with another libm
DBL_MIN = np.finfo(np.float64).tiny


def update_num_iters(p, ep, max_iters, model_points=4, flag=False):
    """OpenCV's RANSACUpdateNumIters(p, ep, modelPoints, maxIters), literally.  With flag=True returns
    (bound, near_tie): near_tie marks a num/denom within TIE_REL (relative) of a half-integer, or a cap comparison
    within TIE_REL of equality, where a libm that differs in the last ulp could give the other answer."""
    p = min(max(p, 0.0), 1.0)
    ep = min(max(ep, 0.0), 1.0)
    num = max(1.0 - p, DBL_MIN)
    denom = 1.0 - math.pow(1.0 - ep, model_points)
    if denom < DBL_MIN:
        return (0, False) if flag else 0
    num = math.log(num)
    denom = math.log(denom)
    cap = max_iters * (-denom)
    if denom >= 0 or -num >= cap:
        r = max_iters
    else:
        r = int(np.rint(num / denom))            # cvRound: round half to even
    if not flag:
        return r
    near = denom < 0 and abs(-num - cap) <= TIE_REL * abs(cap)
    if denom < 0:
        q = num / denom
        near = near or abs(q - (np.floor(q) + 0.5)) <= TIE_REL * abs(q)
    return r, bool(near)


def adaptive_stop(counts, ok, m, n_hyp, confidence):
    """The stop rule over the hypothesis stream (module docstring).  counts / ok: per hypothesis, as
    `ransac.ransac_hypotheses` returns them.  Returns (n_used, near_tie)."""
    best, niters, it, tie = 0, n_hyp, 0, False
    for h in range(n_hyp):
        if not ok[h]:
            continue
        it += 1
        c = int(counts[h])
        if c > max(best, 3):
            best = c
            niters, near = update_num_iters(confidence, float(m - c) / m, niters, flag=True)
            tie = tie or near
        if it >= niters:
            return h + 1, tie
    return n_hyp, tie


def find_homography_seeded(a, b, n_hyp=1024, seed=0, pair_id=0, level=1, thresh=3.0, confidence=0.995):
    """`ransac.find_homography_seeded` with the stop rule: n_hyp is cv2's maxIters.  The result is that of
    `ransac.find_homography_seeded` at n_hyp = n_used, plus n_used (0 when m <= 4: such a pair never samples) and tie
    (the stop lies within TIE_REL of a libm-dependent boundary)."""
    if not 0.0 < confidence < 1.0:
        raise ValueError("confidence must lie in (0, 1)")
    a = np.ascontiguousarray(a, np.float32).reshape(-1, 2)
    b = np.ascontiguousarray(b, np.float32).reshape(-1, 2)
    m = len(a)
    n_used, tie = 0, False
    if m > 4:
        hyp = ransac.ransac_hypotheses(a, b, n_hyp, seed, pair_id, level, thresh)
        n_used, tie = adaptive_stop(hyp["counts"], hyp["ok_all"], m, n_hyp, confidence)
    # (the hypotheses of a prefix do not depend on n_hyp)
    out = ransac.find_homography_seeded(a, b, max(n_used, 1), seed, pair_id, level, thresh)
    out.update(n_used=n_used, tie=tie)
    return out


def _status(r, fail):
    return ST_FEW_POINTS if r["status"] == ransac.ST_TOO_FEW else fail


def pair_static_multi(frames_q, frames_t, n_hyp=1024, seed=0, pair_id=0, ratio=0.5, thresh=3.0, confidence=0.995):
    """`pipeline.pair_static_multi` with the stop rule at RANSAC #1."""
    all_a, all_b = [], []
    for (qc, qd), (tc, td) in zip(frames_q, frames_t):
        if qd is None or td is None:
            return ST_FEW_MATCHES, None, None
        mk = matching.match_kps(qc, qd, tc, td, ratio)
        if mk["status"] != 0:
            return ST_FEW_MATCHES, None, None
        r1 = find_homography_seeded(mk["pts_a"], mk["pts_b"], n_hyp, seed, pair_id, 1, thresh, confidence)
        if r1["status"] != 0:
            return _status(r1, ST_NO_MODEL_1), None, None
        keep, _, _ = static_filter.static_points(r1["H"], mk["pts_a"], mk["pts_b"])
        all_a.append(mk["pts_a"][keep]); all_b.append(mk["pts_b"][keep])
    sa, sb, _, _ = matching.remove_double_matching(np.concatenate(all_a), np.concatenate(all_b))
    return ST_OK, sa, sb


def video_chain_multi(feats, n_hyp=1024, seed=0, none_h_processing=True, reference_exact=False,
                      ratio=0.5, thresh=3.0, confidence=0.995):
    """`pipeline.video_chain_multi` with the stop rule at both RANSAC levels; same return value."""
    types = list(feats)
    P = len(feats[types[0]]) - 1
    status = np.zeros(P, np.int32)
    G = np.tile(np.eye(3), (P, 1, 1))
    valid = np.zeros(P, bool)
    Hs, sup = [], [np.eye(3)]
    S, Hprev, first = None, None, True
    for p in range(P):
        st, sa, sb = pair_static_multi([feats[t][p + 1] for t in types], [feats[t][p] for t in types],
                                       n_hyp, seed, p, ratio, thresh, confidence)
        H = None
        if st == ST_OK:
            if reference_exact and S is not None:
                Sp = np.asarray(S, np.float64)
                sa = np.array([chain.homography_transformation(q, Sp) for q in sa]).reshape(-1, 2)
                sb = np.array([chain.homography_transformation(q, Sp) for q in sb]).reshape(-1, 2)
            r2 = find_homography_seeded(sa, sb, n_hyp, seed, p, 2, thresh, confidence)
            if r2["status"] != 0:
                st = _status(r2, ST_NO_MODEL_2)
            elif int(r2["mask"].sum()) < LENGTH_ACCOUNTED_POINTS * len(r2["mask"]):
                st = ST_FEW_INLIERS
            else:
                H = r2["H"]
        status[p] = st
        valid[p] = H is not None
        if not reference_exact:
            if H is not None:
                G[p] = H
            continue
        if H is None:
            H = Hprev if none_h_processing else None
        Hs.append(H)
        S = chain.matrix_superposition(H, S, first) if H is not None or S is not None else S
        if H is not None:
            first = False
            Hprev = H
        sup.append(np.eye(3) if S is None else np.asarray(S, np.float64))
    if not reference_exact:
        Gf = chain.fill_none(G, valid, none_h_processing)
        Sx = chain.chain_products(Gf)
        return dict(G=G, valid=valid, S=Sx, status=status, H_fixed=chain.fixed_plane_H(Sx))
    return dict(H_fixed=Hs, valid=valid, S=np.array(sup), status=status)
