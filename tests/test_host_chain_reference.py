"""The extended-precision references of oracle/chain.py (long double fold, exact remap, corner maximum) against the
reference's own bundled outputs.  No GPU needed."""
import numpy as np
import pytest

from oracle import chain


def _bundled_S(bundled):
    sup = {int(k): np.asarray(v, np.float64) for k, v in bundled["superposition"].items()}
    keys = sorted(sup)
    return keys, np.array([sup[k] for k in keys])


def _bundled_points(bundled, keys):
    pts, fidx, fixed, back = [], [], [], []
    for k, rects in bundled["original_coordinates"].items():
        for r, e, bk in zip(rects, bundled["fixed_coordinates"][k], bundled["back_to_original"][k]):
            pts.append([r["x1"], r["y1"]]); fidx.append(keys.index(int(k)))
            fixed.append([e["x1"], e["y1"]]); back.append([bk["x1"], bk["y1"]])
    return np.array(pts), np.array(fidx), np.array(fixed), np.array(back)


def test_long_double_fold_agrees_with_f64_fold(bundled):
    """The long double fold is the same computation as the f64 fold, to f64 rounding: at most one f64 eps of max|S| per
    step of the chain (the bundled chain measures 6 eps after 120 steps)."""
    keys, S = _bundled_S(bundled)
    G = np.array([np.linalg.inv(S[i]) @ S[i + 1] for i in range(len(S) - 1)])
    G /= G[:, 2:3, 2:3]
    a, l = chain.chain_products(G), chain.chain_products(G, np.longdouble)
    assert l.dtype == np.longdouble and a.dtype == np.float64
    assert np.array_equal(a, chain.chain_products(G, np.float64))
    bound = len(G) * np.finfo(np.float64).eps
    assert float(np.abs(a - l).max()) <= bound * float(np.abs(l).max())
    ha, hl = chain.fixed_plane_H(a), chain.fixed_plane_H(l)
    assert hl.dtype == np.longdouble
    assert float(np.abs(ha - hl).max()) <= bound * float(np.abs(hl).max())
    # and both reproduce the reference's stored matrices, the long double one from the adjugate
    hd = bundled["homography_dict"]
    want = np.array([hd[str(k)]["H"] for k in keys[1:]])
    assert float(np.abs(hl - want).max()) <= bound * float(np.abs(want).max())


@pytest.mark.parametrize("exact", [True, False])
def test_exact_remap_reproduces_bundled_coordinates(bundled, exact):
    """All 3 664 coordinates of fixed_coordinates and back_to_original, forward and back, bit for bit; none of them
    lies in the tie window, so an implementation can be held to every one of them."""
    keys, S = _bundled_S(bundled)
    pts, fidx, fixed, back = _bundled_points(bundled, keys)
    oh, ow = bundled["original_shape"]; ri = bundled["resize_info"]
    out, tie = chain.remap_exact(pts, fidx, S, int(ri["w"]) / ow, int(ri["h"]) / oh, False, exact=exact)
    assert out.size + fixed.size == 3664 and np.array_equal(out, fixed) and not tie.any()
    out2, tie2 = chain.remap_exact(fixed, fidx, S, ow / ri["w"], oh / ri["h"], True, exact=exact)
    assert np.array_equal(out2, back) and not tie2.any()


def test_long_double_remap_agrees_with_fractions():
    """The bulk (long double) remap gives the exact answer outside the tie window, also for points built to land within
    1e-12 of a half-cent, which both evaluations must flag."""
    rng = np.random.default_rng(1)
    F = 40
    S = np.tile(np.eye(3), (F, 1, 1)) + rng.normal(size=(F, 3, 3)) * [[3e-2, 3e-2, 40], [3e-2, 3e-2, 40], [2e-5, 2e-5, 0]]
    n = 600
    fidx = rng.integers(0, F, n)
    pts = rng.random((n, 2)) * [1170, 658]
    sx, sy = 400 / 1170, 224 / 658
    # the last 100 points: x solved in long double so that X/W is a half-cent
    for i in range(n - 100, n):
        T = S[fidx[i]].astype(np.longdouble)
        y = np.longdouble(np.float64(sy) * pts[i, 1])
        t = (np.floor(np.longdouble(rng.random() * 30000)) + np.longdouble(0.5)) / 100
        x = (t * (T[2, 1] * y + T[2, 2]) - T[0, 1] * y - T[0, 2]) / (T[0, 0] - t * T[2, 0])
        pts[i, 0] = float(x / np.longdouble(sx))
    for inverse in (False, True):
        ex, tie_ex = chain.remap_exact(pts, fidx, S, sx, sy, inverse, exact=True)
        ld, tie_ld = chain.remap_exact(pts, fidx, S, sx, sy, inverse)
        assert np.array_equal(tie_ex, tie_ld)
        assert np.array_equal(ex[~tie_ex], ld[~tie_ld])
        assert tie_ex.mean() < 0.5
    assert tie_ex[:n - 100].sum() == 0
    _, tie_fwd = chain.remap_exact(pts, fidx, S, sx, sy, False, exact=True)
    assert tie_fwd[n - 100:].all()


def test_corner_max_equals_metrics_file(bundled):
    """The exact grid maximum over frames 1 .. 120 (the reference's loop drops the last entry) is within one ulp of
    metrics_file.txt (863.0428982580879, the reference's own f64 evaluation; the exact value rounds to ...878)."""
    keys, S = _bundled_S(bundled)
    ri = bundled["resize_info"]
    mm, frame, w_min = chain.max_movement_corners(S, len(S) - 1, ri["h"], ri["w"])
    golden = bundled["max_movement"]
    assert abs(mm - golden) <= np.spacing(golden)
    assert 0 <= frame < len(S) - 1 and w_min > 0.9
    sup = {k: S[i] for i, k in enumerate(keys)}
    assert abs(mm - chain.max_movement(sup, ri["h"], ri["w"])) <= np.spacing(golden)


def test_corner_max_refuses_a_sign_change_of_W():
    S = np.tile(np.eye(3), (3, 1, 1))
    S[2, 2, 0] = -0.01                       # W = 1 - 0.01 x changes sign inside a 400-wide grid
    with pytest.raises(AssertionError):
        chain.max_movement_corners(S, 3, 224, 400)
    mm, frame, _ = chain.max_movement_corners(S, 2, 224, 400)
    assert mm == 399.0 and frame == 0
