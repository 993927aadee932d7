"""Oracle: seeded RANSAC homography (replaces `cv2.findHomography(a, b, cv2.RANSAC, 3.0)`
called at reference matching.py:156-157 and utils.py:356-358).

Test infrastructure only -- see oracle/__init__.py.

What is pinned against OpenCV 4.13 (the algorithm lives in OpenCV, which is not
vendored in /root/reference; recalled from modules/calib3d/src/{fundam,ptsetreg}.cpp):
  * `reproj_err32`   == HomographyEstimatorCallback::computeError  (bit-exact, SURVEY P3)
  * `refit`          == runKernel (normalised DLT) + LMSolver(10) on the inlier set
  * final mask       == reproj_err32(refined H) <= thresh^2        (bit-exact, SURVEY P3)
What is *defined here* (OpenCV's internal RNG/sample stream cannot be injected, so
criterion (b) "identical seeded hypotheses -> bit-exact masks" is against this file):
  * `hyp_indices`    counter-based PCG sampler, 4 distinct indices per hypothesis
  * `solve4`         closed-form 4-point homography in f64 (no FMA contraction)
  * `subset_ok`      orientation / collinearity test (after checkSubset)
  * best hypothesis  = max inlier count, ties -> lowest hypothesis index
"""
import numpy as np

U32 = np.uint32
_M32 = 0xFFFFFFFF


# ----------------------------------------------------------------------------- RNG
def _mix32(x):
    x = np.asarray(x, np.uint64) & _M32
    x ^= x >> np.uint64(16)
    x = (x * np.uint64(0x85EBCA6B)) & _M32
    x ^= x >> np.uint64(13)
    x = (x * np.uint64(0xC2B2AE35)) & _M32
    x ^= x >> np.uint64(16)
    return x


def _pcg_next(s):
    """PCG-RXS-M-XS-32 step; s uint64 array holding u32 values."""
    s = (s * np.uint64(747796405) + np.uint64(2891336453)) & _M32
    sh = (s >> np.uint64(28)) + np.uint64(4)
    w = (((s >> sh) ^ s) * np.uint64(277803737)) & _M32
    return s, ((w >> np.uint64(22)) ^ w) & _M32


def hyp_indices(seed, pair_id, level, n_hyp, m):
    """(n_hyp, 4) int32 distinct indices in [0, m), m >= 4."""
    h = np.arange(n_hyp, dtype=np.uint64)
    base = _mix32(np.uint64(seed & _M32) ^ _mix32(np.uint64((pair_id * 2 + level + 0x9E3779B9) & _M32)))
    s = _mix32((base + h * np.uint64(0x9E3779B9)) & _M32)
    picks = []
    for k in range(4):
        s, r = _pcg_next(s)
        c = ((r * np.uint64(m - k)) >> np.uint64(32)).astype(np.int64)   # Lemire, no rejection
        prev = np.sort(np.stack(picks, 1), axis=1) if picks else None
        if prev is not None:
            for j in range(prev.shape[1]):
                c = c + (c >= prev[:, j])
        picks.append(c)
    return np.stack(picks, 1).astype(np.int32)


# ----------------------------------------------------------------------------- 4-point solve
def _area(ax, ay, bx, by, cx, cy):
    return (bx - ax) * (cy - ay) - (by - ay) * (cx - ax)


def solve4(src, dst):
    """src, dst: (n,4,2) float32.  Returns H (n,9) float64 with H[8]==1 and ok (n,) bool.
    Projective-basis closed form; every operation is an individually rounded f64 op in
    exactly this order (the CUDA kernel is compiled with --fmad=false and mirrors it)."""
    s = src.astype(np.float64)
    d = dst.astype(np.float64)
    x0, y0, x1, y1, x2, y2, x3, y3 = [s[:, i, j] for i in range(4) for j in range(2)]
    u0, v0, u1, v1, u2, v2, u3, v3 = [d[:, i, j] for i in range(4) for j in range(2)]
    with np.errstate(all="ignore"):
        l0 = _area(x3, y3, x1, y1, x2, y2)
        l1 = _area(x0, y0, x3, y3, x2, y2)
        l2 = _area(x0, y0, x1, y1, x3, y3)
        lt = _area(x0, y0, x1, y1, x2, y2)
        m0 = _area(u3, v3, u1, v1, u2, v2)
        m1 = _area(u0, v0, u3, v3, u2, v2)
        m2 = _area(u0, v0, u1, v1, u3, v3)
        mt = _area(u0, v0, u1, v1, u2, v2)
        eps = 1e-6
        neg = ((lt * mt < 0).astype(np.int32) + (l0 * m0 < 0) + (l1 * m1 < 0) + (l2 * m2 < 0))
        big = ((np.abs(lt) > eps) & (np.abs(l0) > eps) & (np.abs(l1) > eps) & (np.abs(l2) > eps) &
               (np.abs(mt) > eps) & (np.abs(m0) > eps) & (np.abs(m1) > eps) & (np.abs(m2) > eps))
        ok = big & ((neg == 0) | (neg == 4))
        w0 = m0 * (l1 * l2)
        w1 = m1 * (l0 * l2)
        w2 = m2 * (l0 * l1)
        c0 = (y1 - y2, x2 - x1, x1 * y2 - y1 * x2)
        c1 = (y2 - y0, x0 - x2, x2 * y0 - y2 * x0)
        c2 = (y0 - y1, x1 - x0, x0 * y1 - y0 * x1)
        one = np.ones_like(u0)
        H = np.empty((len(x0), 9), np.float64)
        for r, (q0, q1, q2) in enumerate(((u0, u1, u2), (v0, v1, v2), (one, one, one))):
            a0 = w0 * q0
            a1 = w1 * q1
            a2 = w2 * q2
            for j in range(3):
                H[:, 3 * r + j] = (a0 * c0[j] + a1 * c1[j]) + a2 * c2[j]
        inv = 1.0 / H[:, 8]
        ok &= np.isfinite(inv)
        H[:, :8] = H[:, :8] * inv[:, None]
        H[:, 8] = 1.0
    return H, ok


# ----------------------------------------------------------------------------- scoring
def reproj_err32(H, a, b):
    """OpenCV HomographyEstimatorCallback::computeError: H cast f64->f32, all f32 ops
    individually rounded, IEEE reciprocal, no FMA.  H: (...,9) f64; a,b: (M,2) f32.
    Returns (..., M) f32."""
    Hf = np.asarray(H, np.float64).astype(np.float32)
    x = a[:, 0].astype(np.float32)
    y = a[:, 1].astype(np.float32)
    one = np.float32(1.0)
    h = [Hf[..., i, None] for i in range(8)]
    with np.errstate(all="ignore"):
        ww = one / ((h[6] * x + h[7] * y) + one)
        dx = ((h[0] * x + h[1] * y) + h[2]) * ww - b[:, 0]
        dy = ((h[3] * x + h[4] * y) + h[5]) * ww - b[:, 1]
        return dx * dx + dy * dy


# ----------------------------------------------------------------------------- fused count bounds
# Restatements of the device's fast classification (csrc/ransac_device.cuh): the fused evaluation reproj_err_fused (FFMA
# and rcp.approx), the cuts fused_thresholds and the den_safe test.  The scoring kernels count a match as a sure inlier
# when its fused error is <= tlo and as a sure outlier when it is >= thi; both rest on the bound proved in the header.
F32 = np.float32
U = F32(2.0 ** -24)
DEN_MIN = F32(0.0625)          # kDenMin


def reproj_err32_pairs(h, a, b):
    """reproj_err32 with one f32 model per point: h (N,8) f32, a, b (N,2) f32 -> (N,) f32."""
    h = np.asarray(h, F32)
    x, y, z, w = a[:, 0].astype(F32), a[:, 1].astype(F32), b[:, 0].astype(F32), b[:, 1].astype(F32)
    with np.errstate(all="ignore"):
        ww = F32(1) / ((h[:, 6] * x + h[:, 7] * y) + F32(1))
        dx = ((h[:, 0] * x + h[:, 1] * y) + h[:, 2]) * ww - z
        dy = ((h[:, 3] * x + h[:, 4] * y) + h[:, 5]) * ww - w
        return dx * dx + dy * dy


def fma32(a, b, c):
    """Correctly rounded f32 fma(a, b, c) of f32 arrays (round to nearest even).  The product is exact in f64; the f64
    sum s and its error e (TwoSum) hold a*b + c exactly, and rounding s to f32 is wrong only when s is an f32 midpoint
    and e != 0 (double rounding), where e decides the side.  Overflow and subnormal results are not handled."""
    a, b, c = (np.asarray(v, F32).astype(np.float64) for v in (a, b, c))
    p = a * b
    s = p + c
    bb = s - p
    e = (p - (s - bb)) + (c - bb)
    r = s.astype(F32)
    other = np.nextafter(r, np.where(s > r, F32(np.inf), F32(-np.inf)).astype(F32))
    mid = (r.astype(np.float64) + other.astype(np.float64)) * 0.5
    fix = (s == mid) & (e != 0) & (s != r.astype(np.float64))
    side = np.where(e > 0, np.maximum(r, other), np.minimum(r, other))
    return np.where(fix, side, r).astype(F32)


def fused_den32(h, a):
    """den of reproj_err_fused: fma(h6, x, fma(h7, y, 1))."""
    h = np.asarray(h, F32)
    return fma32(h[:, 6], a[:, 0], fma32(h[:, 7], a[:, 1], np.ones(len(a), F32)))


def reproj_err_fused32(h, a, b, ww):
    """reproj_err_fused with the reciprocal given: h (N,8), a, b (N,2), ww (N,) f32 -> (N,) f32."""
    h = np.asarray(h, F32)
    x, y = a[:, 0].astype(F32), a[:, 1].astype(F32)
    X = fma32(h[:, 0], x, fma32(h[:, 1], y, h[:, 2]))
    Y = fma32(h[:, 3], x, fma32(h[:, 4], y, h[:, 5]))
    dx = fma32(X, ww, -b[:, 0].astype(F32))
    dy = fma32(Y, ww, -b[:, 1].astype(F32))
    with np.errstate(all="ignore"):
        return fma32(dx, dx, dy * dy)


def rcp_candidates(den, k=4):
    """Every f32 within 2^-23 relative of 1/den (what the bound assumes of rcp.approx): (N, 2k+1) f32 candidates and a
    mask of the admissible ones.  |w - 1/den| <= 2^-23 |1/den|  <=>  |w den - 1| <= 2^-23, exact in f64."""
    den = np.asarray(den, F32)
    with np.errstate(all="ignore"):
        w0 = (1.0 / den.astype(np.float64)).astype(F32)
    cand = [w0]
    lo = hi = w0
    for _ in range(k):
        lo = np.nextafter(lo, F32(-np.inf))
        hi = np.nextafter(hi, F32(np.inf))
        cand = [lo] + cand + [hi]
    w = np.stack(cand, 1)
    with np.errstate(all="ignore"):
        ok = np.abs(w.astype(np.float64) * den.astype(np.float64)[:, None] - 1.0) <= 2.0 ** -23
    return w, ok


def fused_err_range32(h, a, b):
    """(min, max) of reproj_err_fused over every admissible reciprocal, and the fused denominator."""
    den = fused_den32(h, a)
    w, ok = rcp_candidates(den)
    e = np.stack([reproj_err_fused32(h, a, b, w[:, j]) for j in range(w.shape[1])], 1)
    with np.errstate(all="ignore"):
        emin = np.where(ok, e, F32(np.inf)).min(1)
        emax = np.where(ok, e, F32(-np.inf)).max(1)
    return emin, emax, den


def _bound_terms32(h, cmax):
    h = np.abs(np.asarray(h, F32))
    cmax = np.asarray(cmax, F32)
    with np.errstate(all="ignore"):
        a6 = h[:, 6] + h[:, 7]
        Bd = a6 * cmax + F32(1)
        Bx = (h[:, 0] + h[:, 1]) * cmax + h[:, 2]
        By = (h[:, 3] + h[:, 4]) * cmax + h[:, 5]
        lim = (F32(8) * U) * Bd <= F32(0.1) * DEN_MIN
        dm = np.fmax(F32(0.9) * DEN_MIN, ((F32(1) - a6 * cmax) - (F32(8) * U) * Bd) * F32(0.999999))
        rho = ((F32(4) * U) * Bd) / dm + F32(2) * U
        dX = F32(2.5) * ((Bx / dm) * (F32(6) * U + rho) + U * cmax)
        dY = F32(2.5) * ((By / dm) * (F32(6) * U + rho) + U * cmax)
        return a6, Bd, lim, dX + dY


def fused_D32(h, cmax):
    """D of fused_thresholds (bound on |dx_exact - dx_fused| + |dy_exact - dy_fused|)."""
    return _bound_terms32(h, cmax)[3]


def den_safe32(h, cmax):
    """den_safe(h6, h7, cmax) in the device's operation order: h (N,8) f32."""
    a6, Bd, lim, _ = _bound_terms32(h, cmax)
    cmax = np.asarray(cmax, F32)
    with np.errstate(all="ignore"):
        return lim & (((F32(1) - a6 * cmax) - (F32(8) * U) * Bd) * F32(0.999999) >= DEN_MIN)


def fused_thresholds32(h, cmax, t, exact_only=False):
    """(tlo, thi) of fused_thresholds in the device's operation order: h (N,8) f32, cmax and t scalars or (N,) f32."""
    _, _, lim, D = _bound_terms32(h, cmax)
    t = np.broadcast_to(np.asarray(t, F32), D.shape)
    tlo = np.full(D.shape, -np.inf, F32)
    thi = np.full(D.shape, np.inf, F32)
    use = lim & (D < F32(1e6)) & (not exact_only)
    with np.errstate(all="ignore"):
        s = np.sqrt(t)
        rnd = np.fmax(F32(1e-4), (F32(8) * U) * t)
        th = (t + F32(1.25) * ((F32(2) * D) * D + (F32(2) * D) * np.sqrt(D * D + t))) + rnd
        tl = (t - (F32(2.5) * s) * D) - rnd
    thi = np.where(use, th, thi)
    tlo = np.where(use & (D < s), tl, tlo)
    return tlo.astype(F32), thi.astype(F32)


FUSED_BOUND_THRESHOLDS = (0.5, 0.75, 1.0, 3.0, 5.0, 12.5, 32.0, 64.0, 100.0, 256.0)


def fused_bound_family(rng, name, n):
    """Parameters of near_threshold_cases for the families the fused bound is tested on (n base points)."""
    pick = lambda: rng.choice(FUSED_BOUND_THRESHOLDS, n)
    if name.startswith("thresh_"):                  # one threshold, near-identity models on a 1920 x 1080 frame
        return dict(thresh=np.full(n, float(name[7:])))
    if name == "scale":                             # frames of 0.05x to 100x 1920 x 1080
        s = 10.0 ** rng.uniform(np.log10(0.05), 2.0, n)
        return dict(thresh=pick(), scale=s, trans=8.0 * s)
    if name == "translation":                       # translations up to 8 000 px
        return dict(thresh=pick(), trans=rng.uniform(-8000, 8000, (n, 2)))
    if name == "perspective":                       # (|h6| + |h7|) 1920 up to and just past the den_safe limit 15/16
        return dict(thresh=pick(), persp_sum=rng.uniform(0.5, 1.0, n) * 0.9375 / 1920)
    if name == "low_den":                           # denominators in [1, 1.5] kDenMin of either sign (dm floor)
        return dict(thresh=pick(), persp_sum=rng.uniform(1.0, 3.0, n) / 1920, low_den=True)
    if name == "small_coords":                      # points within 16 px, 100 px threshold
        return dict(thresh=np.full(n, 100.0), scale=np.full(n, 16 / 1920), trans=rng.uniform(-1, 1, (n, 2)))
    if name == "D_both_sides":                      # D on both sides of sqrt(t), the condition of the sure-inlier cut
        s = 10.0 ** rng.uniform(1.0, 2.0, n)
        return dict(thresh=rng.choice([0.5, 0.75], n), scale=s, trans=8.0 * s)
    raise ValueError(name)


FUSED_BOUND_FAMILIES = tuple(f"thresh_{t:g}" for t in FUSED_BOUND_THRESHOLDS) + (
    "scale", "translation", "perspective", "low_den", "small_coords", "D_both_sides")


def near_threshold_b(h, a, thresh, phi, walk=3):
    """b = f32(pi(h a) + thresh (cos phi, sin phi)), projected in f64, and its f32 neighbours within `walk` ulps in each
    coordinate: h (n,8) f32, a (n,2) f32 -> (n, (2 walk + 1)^2, 2) f32."""
    n = len(h)
    h64, a64 = h.astype(np.float64), a.astype(np.float64)
    den = h64[:, 6] * a64[:, 0] + h64[:, 7] * a64[:, 1] + 1.0
    px = (h64[:, 0] * a64[:, 0] + h64[:, 1] * a64[:, 1] + h64[:, 2]) / den
    py = (h64[:, 3] * a64[:, 0] + h64[:, 4] * a64[:, 1] + h64[:, 5]) / den
    with np.errstate(all="ignore"):
        b0 = np.stack([px + thresh * np.cos(phi), py + thresh * np.sin(phi)], 1).astype(F32)
    k = 2 * walk + 1
    bz = np.repeat(b0[:, 0], k * k).reshape(n, k, k)
    bw = np.repeat(b0[:, 1], k * k).reshape(n, k, k)
    for s in range(1, walk + 1):       # bz[:, i, :] = b0.x moved i - walk ulps, bw[:, :, j] = b0.y moved j - walk ulps
        for arr, ax in ((bz, 1), (bw, 2)):
            for sgn, idx in ((1, walk + s), (-1, walk - s)):
                sl = [slice(None)] * 3
                sl[ax] = idx
                prev = [slice(None)] * 3
                prev[ax] = idx - sgn
                arr[tuple(sl)] = np.nextafter(arr[tuple(prev)], F32(sgn * np.inf))
    return np.stack([bz.reshape(n, -1), bw.reshape(n, -1)], 2).astype(F32)


def near_threshold_cases(rng, n, thresh, scale=1.0, trans=8.0, persp=1e-5, persp_sum=None, low_den=False, walk=3):
    """Point pairs whose exact error lies within a few ulps of thresh^2 on both sides, under random f32 models.

    n base points (every argument a scalar or one value per base point): a near-identity model h (rotation ~0.02 rad,
    scale ~1e-3; translation ~N(0, trans), or trans itself when it has shape (n, 2); perspective ~N(0, persp / scale),
    or of random signs with |h6| + |h7| = persp_sum), a point a in the frame [0, 1920 scale] x [0, 1080 scale] (low_den:
    moved to where the f64 denominator lies in [1, 1.5] kDenMin, of either sign), b = f32(pi(h a) + thresh (cos phi,
    sin phi)) in f64, then every f32 neighbour of b within `walk` ulps in each coordinate.  Returns h (N,8) f32, a, b
    (N,2) f32, t = f32(thresh^2) and cmax (N,) f32 (the frame, or the largest |coordinate| of the pair when larger) with
    N = n (2 walk + 1)^2."""
    thresh = np.broadcast_to(np.asarray(thresh, np.float64), (n,))
    scale = np.broadcast_to(np.asarray(scale, np.float64), (n,))
    th = rng.normal(size=n) * 0.02
    sc = 1 + rng.normal(size=n) * 1e-3
    tr = np.asarray(trans, np.float64)
    tr = tr if tr.shape == (n, 2) else rng.normal(size=(n, 2)) * np.broadcast_to(tr, (n,))[:, None]
    if persp_sum is None:
        pp = rng.normal(size=(n, 2)) * (np.broadcast_to(np.asarray(persp, np.float64), (n,)) / scale)[:, None]
    else:
        f = rng.random(n)
        pp = np.stack([f, 1 - f], 1) * np.broadcast_to(np.asarray(persp_sum, np.float64), (n,))[:, None]
        pp *= rng.choice([-1.0, 1.0], (n, 2))
    h = np.stack([sc * np.cos(th), -sc * np.sin(th), tr[:, 0], sc * np.sin(th), sc * np.cos(th), tr[:, 1],
                  pp[:, 0], pp[:, 1]], 1).astype(F32)
    frame = np.array([1920.0, 1080.0]) * scale[:, None]
    a = rng.random((n, 2)) * frame
    if low_den:
        # move a along the gradient of the denominator until den = target (in f64), inside the frame when possible
        g = h[:, 6:8].astype(np.float64)
        target = rng.uniform(1.0, 1.5, n) * float(DEN_MIN) * rng.choice([-1.0, 1.0], n)
        d0 = 1.0 + (g * a).sum(1)
        a = a + ((target - d0) / (g * g).sum(1))[:, None] * g
    a = a.astype(F32)
    b = near_threshold_b(h, a, thresh, rng.uniform(0, 2 * np.pi, n), walk).reshape(-1, 2)
    k = 2 * walk + 1
    a = np.repeat(a, k * k, 0)
    h = np.repeat(h, k * k, 0)
    t = np.repeat((thresh * thresh).astype(F32), k * k)
    with np.errstate(all="ignore"):
        cmax = np.maximum(np.repeat(frame.max(1), k * k).astype(F32), np.maximum(np.abs(a).max(1), np.abs(b).max(1)))
    return h, a, b, t, cmax.astype(F32)


# ----------------------------------------------------------------------------- refit
def dlt_normalised(a, b):
    """OpenCV HomographyEstimatorCallback::runKernel: per-axis mean-abs-deviation
    normalisation, 9x9 LtL, eigenvector of the smallest eigenvalue, de-normalise, /h22.
    Returns H (9,) f64 or None."""
    a = a.astype(np.float64)
    b = b.astype(np.float64)
    n = len(a)
    cM = a.mean(0)
    cm = b.mean(0)
    sM = np.abs(a - cM).sum(0)
    sm = np.abs(b - cm).sum(0)
    if (sM < np.finfo(np.float64).eps).any() or (sm < np.finfo(np.float64).eps).any():
        return None
    sM = n / sM
    sm = n / sm
    X = (a[:, 0] - cM[0]) * sM[0]
    Y = (a[:, 1] - cM[1]) * sM[1]
    x = (b[:, 0] - cm[0]) * sm[0]
    y = (b[:, 1] - cm[1]) * sm[1]
    z = np.zeros(n)
    o = np.ones(n)
    Lx = np.stack([X, Y, o, z, z, z, -x * X, -x * Y, -x], 1)
    Ly = np.stack([z, z, z, X, Y, o, -y * X, -y * Y, -y], 1)
    LtL = Lx.T @ Lx + Ly.T @ Ly
    w, v = np.linalg.eigh(LtL)
    h0 = v[:, 0].reshape(3, 3)
    inv_hnorm = np.array([[1.0 / sm[0], 0, cm[0]], [0, 1.0 / sm[1], cm[1]], [0, 0, 1]])
    hnorm2 = np.array([[sM[0], 0, -cM[0] * sM[0]], [0, sM[1], -cM[1] * sM[1]], [0, 0, 1]])
    H = inv_hnorm @ h0 @ hnorm2
    with np.errstate(all="ignore"):
        H = H * (1.0 / H[2, 2])
    if not np.isfinite(H).all():
        return None
    return H.ravel()


def _lm_residual_jac(h, a, b, want_j=True):
    """OpenCV HomographyRefineCallback::compute."""
    Mx = a[:, 0].astype(np.float64)
    My = a[:, 1].astype(np.float64)
    ww = h[6] * Mx + h[7] * My + 1.0
    ww = np.where(np.abs(ww) > np.finfo(np.float64).eps, 1.0 / np.where(ww == 0, 1, ww), 0.0)
    xi = (h[0] * Mx + h[1] * My + h[2]) * ww
    yi = (h[3] * Mx + h[4] * My + h[5]) * ww
    r = np.empty(2 * len(a))
    r[0::2] = xi - b[:, 0]
    r[1::2] = yi - b[:, 1]
    if not want_j:
        return r, None
    J = np.zeros((2 * len(a), 8))
    J[0::2, 0] = Mx * ww
    J[0::2, 1] = My * ww
    J[0::2, 2] = ww
    J[0::2, 6] = -Mx * ww * xi
    J[0::2, 7] = -My * ww * xi
    J[1::2, 3] = Mx * ww
    J[1::2, 4] = My * ww
    J[1::2, 5] = ww
    J[1::2, 6] = -Mx * ww * yi
    J[1::2, 7] = -My * ww * yi
    return r, J


def lm_refine(H, a, b, max_iters=10):
    """cv::LMSolver (calib3d/src/levmarq.cpp) as driven by findHomography: 8 parameters
    (h22 pinned to 1), lambda0 = 1 on diag(JtJ), Rlo/Rhi = 0.25/0.75, eps = FLT_EPSILON."""
    eps = float(np.finfo(np.float32).eps)
    deps = float(np.finfo(np.float64).eps)
    x = np.array(H[:8], np.float64)
    r, J = _lm_residual_jac(x, a, b)
    S = float(r @ r)
    A = J.T @ J
    v = J.T @ r
    D = np.diag(A).copy()
    lam, lc = 1.0, 0.75
    it = 0
    while True:
        Ap = A + np.diag(lam * D)
        try:
            d = np.linalg.solve(Ap, v)
        except np.linalg.LinAlgError:
            d = np.linalg.lstsq(Ap, v, rcond=None)[0]
        xd = x - d
        rd, _ = _lm_residual_jac(xd, a, b, want_j=False)
        Sd = float(rd @ rd)
        temp_d = 2 * v - A @ d
        dS = float(d @ temp_d)
        R = (S - Sd) / (dS if abs(dS) > deps else 1.0)
        if R > 0.75:
            lam *= 0.5
            if lam < lc:
                lam = 0.0
        elif R < 0.25:
            t = float(d @ v)
            nu = (Sd - S) / (t if abs(t) > deps else 1.0) + 2
            nu = min(max(nu, 2.0), 10.0)
            if lam == 0:
                Ainv = np.linalg.pinv(A)
                maxval = max(deps, float(np.abs(np.diag(Ainv)).max()))
                lam = lc = 1.0 / maxval
                nu *= 0.5
            lam *= nu
        if Sd < S:
            S = Sd
            x = xd
            r, J = _lm_residual_jac(x, a, b)
            A = J.T @ J
            v = J.T @ r
        it += 1
        if not (it < max_iters and np.abs(d).max() >= eps and np.abs(r).max() >= eps):
            break
    return np.append(x, 1.0)


def refit(a, b):
    """findHomography(method=0) on a point set == DLT (+ LM when n > 4)."""
    H = dlt_normalised(a, b)
    if H is None:
        return None
    if len(a) > 4:
        H = lm_refine(H, a, b)
    return H


# ----------------------------------------------------------------------------- least-squares optimum
def _project(H, p):
    """pi(H p) for (N,2) points in the dtype of p (H is cast to it)."""
    H = np.asarray(H).reshape(3, 3).astype(p.dtype)
    w = H[2, 0] * p[:, 0] + H[2, 1] * p[:, 1] + H[2, 2]
    return np.stack([(H[0, 0] * p[:, 0] + H[0, 1] * p[:, 1] + H[0, 2]) / w,
                     (H[1, 0] * p[:, 0] + H[1, 1] * p[:, 1] + H[1, 2]) / w], 1)


def probe_points(a):
    """The points of a set plus the four corners of its bounding box (f64)."""
    a = np.asarray(a, np.float64).reshape(-1, 2)
    lo, hi = a.min(0), a.max(0)
    corners = np.array([[lo[0], lo[1]], [hi[0], lo[1]], [lo[0], hi[1]], [hi[0], hi[1]]])
    return np.concatenate([a, corners])


def max_px_dist(H1, H2, a):
    """Largest distance in pixels between pi(H1 p) and pi(H2 p) over the points of `a` and the corners of their
    bounding box, evaluated in long double."""
    p = probe_points(a).astype(np.longdouble)
    return float(np.sqrt(((_project(H1, p) - _project(H2, p)) ** 2).sum(1)).max())


def sum_sq(H, a, b):
    """S(H) = sum |pi(H a) - b|^2 in long double (a, b as given, usually f32)."""
    a = np.asarray(a).astype(np.longdouble).reshape(-1, 2)
    b = np.asarray(b).astype(np.longdouble).reshape(-1, 2)
    return float(((_project(H, a) - b) ** 2).sum())


def _normalise(p):
    """(T, p') for the similarity T that moves the centroid of p to the origin and scales the mean distance from it
    to 1, and p' = T p."""
    c = p.mean(0)
    s = np.sqrt(((p - c) ** 2).sum(1)).mean()
    s = s if s > 0 else 1.0
    return np.array([[1 / s, 0, -c[0] / s], [0, 1 / s, -c[1] / s], [0, 0, 1.0]]), (p - c) / s


def _gauss_newton(g, an, bn, probe, sb, max_iters=200, tol_px=1e-12):
    """Gauss-Newton on the 8 free entries of g (g22 = 1) in normalised coordinates.  Far from the optimum a step is
    halved until S does not grow; a step that moves no probe point by more than 1e-6 px of b is taken as it is (S cannot
    resolve such steps in f64; Gauss-Newton converges there).  Stops when a step moves no probe point by more than
    tol_px pixels of b.  Returns (g (9,), converged)."""
    x = np.asarray(g, np.float64).ravel()[:8] / g.ravel()[8]
    def move_px(x1, x0):
        return sb * np.sqrt(((_project(np.append(x1, 1.0), probe) - _project(np.append(x0, 1.0), probe)) ** 2).sum(1)).max()
    for _ in range(max_iters):
        r, J = _lm_residual_jac(x, an, bn)
        S = float(r @ r)
        d = np.linalg.lstsq(J, r, rcond=None)[0]
        t = 1.0
        while True:
            xt = x - t * d
            mv = move_px(xt, x)
            if mv <= 1e-6:
                break
            rt, _ = _lm_residual_jac(xt, an, bn, want_j=False)
            if float(rt @ rt) <= S:
                break
            t *= 0.5
        x = xt
        if t == 1.0 and mv <= tol_px:
            return np.append(x, 1.0), True
    return np.append(x, 1.0), False


def ls_optimum(a, b, H0):
    """Minimiser of S(H) = sum |pi(H a) - b|^2 over the point set (a, b), h22 = 1.

    Solved by Gauss-Newton with a backtracking line search in coordinates where a and b are moved to their centroids and
    scaled by a similarity to unit mean distance: the residuals are those in pixels of b divided by one constant, so the
    minimiser is unchanged, and J^T J is well conditioned even for a small patch far from the origin.  Iterates until a
    step moves no point of a (nor a corner of its bounding box) by more than 1e-12 px.

    Runs from H0 (the winning 4-point model), from the normalised DLT and from `refit` and keeps the lowest S.
    Returns (H (9,) f64 with H[8] == 1, cert) where cert holds
      grad_rel   max |J^T r| / (||J||_F (||r|| + ||J||_F ||x||)) at the optimum x in normalised coordinates, J^T r
                 evaluated in long double (rounding x to f64 alone leaves ~1e-16 here; the ||J|| ||x|| term keeps the
                 measure meaningful for exact fits, where r is rounding noise);
      cond       condition number of the normalised J^T J (positive definite when finite and min_eig > 0);
      min_eig    its smallest eigenvalue;
      spread_px  largest max_px_dist between the optima reached from the different starts;
      converged  every start met the 1e-12 px stop rule;
      S          S at the optimum (long double, pixels)."""
    a = np.asarray(a, np.float32).reshape(-1, 2)
    b = np.asarray(b, np.float32).reshape(-1, 2)
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    Ta, an = _normalise(a64)
    Tb, bn = _normalise(b64)
    sb = 1.0 / Tb[0, 0]                 # pixels of b per normalised unit
    Tb_inv = np.linalg.inv(Tb)
    probe = probe_points(an)
    starts = [np.asarray(H0, np.float64).reshape(3, 3)]
    for H in (dlt_normalised(a, b), refit(a, b)):
        if H is not None and np.isfinite(H).all():
            starts.append(H.reshape(3, 3))
    sols, conv = [], True
    for H in starts:
        g = Tb @ H @ np.linalg.inv(Ta)
        g, ok = _gauss_newton(g / g[2, 2], an, bn, probe, sb)
        conv = conv and ok
        Hp = Tb_inv @ g.reshape(3, 3) @ Ta
        Hp = Hp / Hp[2, 2]
        sols.append((sum_sq(Hp, a, b), Hp.ravel(), g))
    S, H, g = min(sols, key=lambda s: s[0])
    spread = max(max_px_dist(H, s[1], a) for s in sols)
    # certificate in the normalised parametrisation: gradient in long double, curvature of the normal equations
    an_l, bn_l = an.astype(np.longdouble), bn.astype(np.longdouble)
    gl = np.asarray(g, np.float64).astype(np.longdouble)
    w = gl[6] * an_l[:, 0] + gl[7] * an_l[:, 1] + 1
    xi = (gl[0] * an_l[:, 0] + gl[1] * an_l[:, 1] + gl[2]) / w
    yi = (gl[3] * an_l[:, 0] + gl[4] * an_l[:, 1] + gl[5]) / w
    r = np.empty(2 * len(a), np.longdouble)
    r[0::2] = xi - bn_l[:, 0]
    r[1::2] = yi - bn_l[:, 1]
    J = np.zeros((2 * len(a), 8), np.longdouble)
    J[0::2, 0] = an_l[:, 0] / w; J[0::2, 1] = an_l[:, 1] / w; J[0::2, 2] = 1 / w
    J[1::2, 3] = an_l[:, 0] / w; J[1::2, 4] = an_l[:, 1] / w; J[1::2, 5] = 1 / w
    J[0::2, 6] = -an_l[:, 0] * xi / w; J[0::2, 7] = -an_l[:, 1] * xi / w
    J[1::2, 6] = -an_l[:, 0] * yi / w; J[1::2, 7] = -an_l[:, 1] * yi / w
    grad = J.T @ r
    nJ = np.sqrt(float((J.astype(np.float64) ** 2).sum()))
    scale = nJ * (np.sqrt(float(r @ r)) + nJ * np.linalg.norm(np.asarray(g, np.float64)[:8]))
    eig = np.linalg.eigvalsh((J.T @ J).astype(np.float64))
    cert = dict(grad_rel=float(np.abs(grad).max()) / scale, min_eig=float(eig[0]),
                cond=float(eig[-1] / eig[0]) if eig[0] > 0 else float("inf"),
                spread_px=spread, converged=conv, S=S)
    return H, cert


# ----------------------------------------------------------------------------- driver
ST_OK = 0
ST_TOO_FEW = 3        # < 4 points: cv2.error in the reference (uncaught)
ST_NO_MODEL = 4       # findHomography returned None -> NoMatchesException / HomographyException


def ransac_hypotheses(a, b, n_hyp, seed, pair_id, level, thresh=3.0):
    """Phase 1 only: returns dict(best, best_count, counts, H_all, ok_all, mask_best)."""
    m = len(a)
    idx = hyp_indices(seed, pair_id, level, n_hyp, m)
    H, ok = solve4(a[idx], b[idx])
    t = np.float32(thresh * thresh)
    counts = np.zeros(n_hyp, np.int32)
    step = max(1, (1 << 22) // max(m, 1))
    for s in range(0, n_hyp, step):
        e = min(n_hyp, s + step)
        err = reproj_err32(H[s:e], a, b)
        counts[s:e] = (err <= t).sum(1)
    counts[~ok] = 0
    best = int(np.argmax(counts))              # first maximum -> lowest hypothesis index
    return dict(best=best, best_count=int(counts[best]), counts=counts, H_all=H, ok_all=ok,
                idx=idx, mask_best=(reproj_err32(H[best], a, b) <= t))


def find_homography_seeded(a, b, n_hyp=1024, seed=0, pair_id=0, level=1, thresh=3.0):
    """Full replacement of cv2.findHomography(a, b, RANSAC, thresh) with seeded hypotheses.
    Returns dict(status, H (3,3) f64 or None, mask (M,) uint8, hyp=phase-1 dict)."""
    a = np.ascontiguousarray(a, np.float32).reshape(-1, 2)
    b = np.ascontiguousarray(b, np.float32).reshape(-1, 2)
    m = len(a)
    out = dict(status=ST_OK, H=None, mask=np.zeros(m, np.uint8), hyp=None, mask_best=np.zeros(m, bool))
    if m < 4:
        out["status"] = ST_TOO_FEW
        return out
    t = np.float32(thresh * thresh)
    if m == 4:
        H = dlt_normalised(a, b)         # findHomography: npoints == 4 -> runKernel only, mask = ones
        if H is None:
            out["status"] = ST_NO_MODEL
            return out
        out.update(H=H.reshape(3, 3), mask=np.ones(4, np.uint8), mask_best=np.ones(4, bool))
        return out
    hyp = ransac_hypotheses(a, b, n_hyp, seed, pair_id, level, thresh)
    out["hyp"] = hyp
    if hyp["best_count"] < 4:
        out["status"] = ST_NO_MODEL
        return out
    inl = hyp["mask_best"]
    out["mask_best"] = inl
    H = refit(a[inl], b[inl])
    if H is None:
        out["status"] = ST_NO_MODEL
        return out
    out["H"] = H.reshape(3, 3)
    out["mask"] = (reproj_err32(H, a, b) <= t).astype(np.uint8)
    return out
