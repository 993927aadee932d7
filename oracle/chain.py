"""Oracle: None-H fallback, cumulative superposition, object-coordinate remap
(reference video_processing.py:94-105, utils.py:71-145,184-211, fixed_coordinate_system.py:19-122).

Test infrastructure only -- see oracle/__init__.py.
"""
import numpy as np


def matrix_superposition(H, S, first=False):
    """reference utils.py:118-145."""
    if H is not None:
        if first:
            S = H
        else:
            S = np.dot(H, S)
            S = np.divide(S, S[2][2])
    return S


def superposition_dict(homography_dict):
    """reference utils.py:184-211 (left fold, frame 1 -> identity)."""
    out = {1: [[1, 0, 0], [0, 1, 0], [0, 0, 1]]}
    S = None
    first = True
    for frame_no, frame_H in homography_dict.items():
        S = matrix_superposition(frame_H["H"], S, first)
        first = False
        out[frame_no] = S
    return out


def homography_transformation(vec, H):
    """reference utils.py:71-92."""
    v = np.append(np.asarray(vec, np.float64), [1.0])[:3]
    nv = np.dot(np.asarray(H, np.float64), v)
    return nv[:-1] / nv[-1]


def fill_none(G, valid, policy_prev=True):
    """None-H policy on frame-plane matrices G (P,3,3).  policy_prev=True: reuse the previous
    pair's matrix (reference video_processing.py:95-96; equivalent in the frame plane, see
    DESIGN.md); False: identity step.  Leading invalid pairs -> identity (the reference crashes)."""
    G = np.array(G, np.float64).reshape(-1, 3, 3)
    out = np.empty_like(G)
    prev = np.eye(3)
    for k in range(len(G)):
        if valid[k]:
            prev = G[k]
            out[k] = G[k]
        else:
            out[k] = prev if policy_prev else np.eye(3)
    return out


def chain_products(G, dtype=np.float64):
    """S_k = normalise(S_{k-1} . G_k), S_0 = I: frame-plane step matrices (new frame -> previous
    frame) to cumulative superposition (frame k -> frame 1).  Returns (P+1,3,3) with S[0]=I.
    dtype=np.longdouble folds in extended precision (80-bit on x86-64: eps 1.1e-19), a reference
    whose own rounding is far below that of any f64 evaluation order."""
    G = np.asarray(G, np.float64).reshape(-1, 3, 3).astype(dtype, copy=False)
    S = np.empty((len(G) + 1, 3, 3), dtype)
    S[0] = np.eye(3)
    for k in range(len(G)):
        T = S[k] @ G[k]
        S[k + 1] = T / T[2, 2]
    return S


def adjugate(M):
    """adj(M) = det(M) . M^-1 for (...,3,3) arrays of any float dtype (np.linalg.inv has no long double)."""
    M = np.asarray(M)
    a, b, c = M[..., 0, 0], M[..., 0, 1], M[..., 0, 2]
    d, e, f = M[..., 1, 0], M[..., 1, 1], M[..., 1, 2]
    g, h, i = M[..., 2, 0], M[..., 2, 1], M[..., 2, 2]
    return np.stack([np.stack([e * i - f * h, c * h - b * i, b * f - c * e], -1),
                     np.stack([f * g - d * i, a * i - c * g, c * d - a * f], -1),
                     np.stack([d * h - e * g, b * g - a * h, a * e - b * d], -1)], -2)


def fixed_plane_H(S):
    """H_k = S_k . S_{k-1}^{-1} (normalised): the matrices the reference stores in
    dict_with_homography_matrix.json, so that its `superposition_dict` (a LEFT fold)
    reproduces S.  Computed in S's dtype; a long double S uses the adjugate (the scale of the
    inverse cancels in the normalisation)."""
    if np.asarray(S).dtype == np.longdouble:
        T = S[1:] @ adjugate(S[:-1])
        return T / T[:, 2:3, 2:3]
    out = np.empty((len(S) - 1, 3, 3))
    for k in range(1, len(S)):
        T = S[k] @ np.linalg.inv(S[k - 1])
        out[k - 1] = T / T[2, 2]
    return out


def from_original_to_fix(original_coordinates, sup, original_shape, resize_shape):
    """reference fixed_coordinate_system.py:19-69."""
    oh, ow = original_shape
    rh, rw = resize_shape
    hc = int(rh) / oh
    wc = int(rw) / ow
    out = {}
    for frame_no, rects in original_coordinates.items():
        out[frame_no] = []
        for rect in rects:
            nr = dict(rect)
            nr["x1"], nr["y1"] = np.around(
                homography_transformation([wc * rect["x1"], hc * rect["y1"]], sup[frame_no]), decimals=2)
            out[frame_no].append(nr)
    return out


def from_fix_to_original(fix_coordinates, sup, original_shape, resize_shape):
    """reference fixed_coordinate_system.py:72-122 (scales BEFORE the inverse transform, as the
    reference does)."""
    oh, ow = original_shape
    rh, rw = resize_shape
    hc = oh / rh
    wc = ow / rw
    out = {}
    for frame_no, rects in fix_coordinates.items():
        out[frame_no] = []
        Hi = np.linalg.inv(np.asarray(sup[frame_no], np.float64))
        for rect in rects:
            nr = dict(rect)
            nr["x1"], nr["y1"] = np.around(
                homography_transformation([wc * rect["x1"], hc * rect["y1"]], Hi), decimals=2)
            out[frame_no].append(nr)
    return out


def max_movement(sup, h, w):
    """reference processing_visualization.py:404-418 (`heatmap_video_processing`): the maximum
    transformed coordinate over the h x w pixel grid and all frames except the last dict entry."""
    ys, xs = np.mgrid[0:h, 0:w]
    p = np.stack([xs.ravel(), ys.ravel(), np.ones(h * w)], 0).astype(np.float64)
    best = -np.inf
    keys = list(sup.keys())
    for k in keys[:-1]:
        q = np.asarray(sup[k], np.float64) @ p
        best = max(best, float((q[:2] / q[2]).max()))
    return best


# ---------------------------------------------------------------------------------- exact references
REMAP_TIE_WINDOW = 1e-6


def _frac_adjugate(T):
    (a, b, c), (d, e, f), (g, h, i) = T
    return [[e * i - f * h, c * h - b * i, b * f - c * e],
            [f * g - d * i, a * i - c * g, c * d - a * f],
            [d * h - e * g, b * g - a * h, a * e - b * d]]


def remap_exact(pts, frame_idx, S, sx, sy, inverse=False, exact=False):
    """What `around(T . (sx x, sy y, 1), 2)` (reference fixed_coordinate_system.py:19-122, evz_remap) is
    without rounding error in the transform: p = (fl(sx x), fl(sy y)) -- the one rounding the reference and
    the kernel both do --, e = (T p) / W exactly, output float64(round_half_even(100 e)) / 100.
    T = S[frame_idx], or for `inverse` the inverse of S[frame_idx] (its adjugate: the scale cancels in e).
    exact=True evaluates e in fractions.Fraction (slow, for samples); otherwise in long double.
    Returns (out [n,2] f64, tie [n] bool): tie marks points where 100 e lies within REMAP_TIE_WINDOW of a
    half-integer, where the f64 evaluation order of an implementation may legitimately decide the rounding."""
    pts = np.asarray(pts, np.float64).reshape(-1, 2)
    fi = np.asarray(frame_idx, np.int64).reshape(-1)
    S = np.asarray(S, np.float64).reshape(-1, 3, 3)
    x = np.float64(sx) * pts[:, 0]
    y = np.float64(sy) * pts[:, 1]
    if exact:
        from fractions import Fraction
        out = np.empty((len(pts), 2))
        tie = np.zeros(len(pts), bool)
        cache = {}
        half = Fraction(1, 2)
        for n in range(len(pts)):
            f = int(fi[n])
            if f not in cache:
                T = [[Fraction(float(v)) for v in row] for row in S[f]]
                cache[f] = _frac_adjugate(T) if inverse else T
            T = cache[f]
            px, py = Fraction(float(x[n])), Fraction(float(y[n]))
            X, Y, W = (r[0] * px + r[1] * py + r[2] for r in T)
            for j, v in enumerate((X / W * 100, Y / W * 100)):
                out[n, j] = np.float64(round(v)) / 100          # Fraction.__round__: half to even, exact
                d = v - (v.numerator // v.denominator) - half
                tie[n] |= abs(d) < REMAP_TIE_WINDOW
        return out, tie
    T = S[fi].astype(np.longdouble)
    if inverse:
        T = adjugate(T)
    xl, yl = x.astype(np.longdouble), y.astype(np.longdouble)
    X = T[:, 0, 0] * xl + T[:, 0, 1] * yl + T[:, 0, 2]
    Y = T[:, 1, 0] * xl + T[:, 1, 1] * yl + T[:, 1, 2]
    W = T[:, 2, 0] * xl + T[:, 2, 1] * yl + T[:, 2, 2]
    v = np.stack([X / W, Y / W], -1) * 100
    out = np.rint(v).astype(np.float64) / 100                     # rint: half to even
    tie = (np.abs(v - np.floor(v) - np.longdouble(0.5)) < REMAP_TIE_WINDOW).any(-1)
    return out, tie


def max_movement_corners(S, n_frames, h, w):
    """Exact max over frames [0, n_frames) of max(X/W, Y/W) over the pixel lattice [0, w-1] x [0, h-1], the
    quantity evz_max_movement computes by brute force.  While W > 0 on the whole rectangle a linear-fractional
    function is largest at a corner, and the corners are lattice points, so four corners per frame give the
    exact grid maximum.  Frames are screened in long double; the leading ones are evaluated in
    fractions.Fraction.  Returns (max rounded to nearest f64, its frame, smallest corner W)."""
    from fractions import Fraction
    S = np.asarray(S, np.float64).reshape(-1, 3, 3)[:n_frames]
    corners = [(0, 0), (w - 1, 0), (0, h - 1), (w - 1, h - 1)]
    q = S.astype(np.longdouble) @ np.array([[cx, cy, 1] for cx, cy in corners], np.longdouble).T      # [F,3,4]
    W = q[:, 2, :]
    assert (W > 0).all(), "W <= 0 at a corner: the corner maximum does not apply"
    val = np.maximum(q[:, 0, :] / W, q[:, 1, :] / W).max(1)
    top = val.max()
    best, arg = None, -1
    for f in np.nonzero(val >= top - abs(top) * 1e-12)[0]:
        T = [[Fraction(float(v)) for v in row] for row in S[f]]
        for cx, cy in corners:
            X, Y, Wf = (r[0] * cx + r[1] * cy + r[2] for r in T)
            assert Wf > 0
            m = max(X / Wf, Y / Wf)
            if best is None or m > best:
                best, arg = m, int(f)
    return float(best), arg, float(W.min())
