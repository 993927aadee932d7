"""The fused count bounds of the RANSAC scoring kernels (csrc/ransac_device.cuh fused_thresholds, den_safe), checked point
by point on the CPU against the exact f32 error on pairs built to lie within a few ulps of the threshold.

A match counts as a sure inlier when its fused error (FFMA, rcp.approx) is <= tlo and as a sure outlier when it is
>= thi, and a den_safe hypothesis skips the |den| test.  The kernels trust three implications:
  fused <= tlo  =>  reproj_err32 <= t;   fused >= thi  =>  reproj_err32 > t;
  den_safe(h, cmax)  =>  |den| >= kDenMin on both paths wherever |x|, |y| <= cmax.
The fused error is emulated exactly (correctly rounded f32 fma) for every f32 reciprocal within 2^-23 of 1/den, the
accuracy the bound assumes of rcp.approx; the implications must hold for all of them."""
from fractions import Fraction

import numpy as np
import pytest

from oracle import ransac as R

F32 = np.float32
N_BASE = 4000                  # x 49 f32 neighbours of b: ~200 000 pairs per family


def check_implications(h, a, b, t, cmax, emin, emax, den_f):
    """Violations of the two cut implications among the classified evaluations (|den_fused| >= kDenMin); returns
    (n_sure_in_wrong, n_sure_out_wrong, n_classified, exact errors, tlo, thi)."""
    tlo, thi = R.fused_thresholds32(h, cmax, t)
    ee = R.reproj_err32_pairs(h, a, b)
    cls = np.abs(den_f) >= R.DEN_MIN
    bad_in = cls & (emin <= tlo) & ~(ee <= t)
    bad_out = cls & (emax >= thi) & (ee <= t)
    return int(bad_in.sum()), int(bad_out.sum()), int(cls.sum()), ee, tlo, thi


def test_fma32_is_correctly_rounded():
    rng = np.random.default_rng(1)
    n = 3000
    x = (rng.normal(size=n) * rng.choice([1.0, 1e3, 1e-3], n)).astype(F32)
    y = rng.normal(size=n).astype(F32)
    z = (-(x.astype(np.float64) * y) * rng.choice([1.0, 1.0 + 1e-7], n) + rng.normal(size=n) * 1e-9).astype(F32)
    # products on an f32 midpoint: (1 + 2^-12)^2 = 1 + 2^-11 + 2^-24; an addend far below the f64 ulp decides the side
    one = F32(1 + 2.0 ** -12)
    x = np.r_[x, one, one, one, -one]
    y = np.r_[y, one, one, one, one]
    z = np.r_[z, F32(2.0 ** -60), F32(-2.0 ** -60), F32(0), F32(2.0 ** -60)]
    r = R.fma32(x, y, z)
    for i in range(len(x)):
        ex = Fraction(float(x[i])) * Fraction(float(y[i])) + Fraction(float(z[i]))
        c = F32(float(ex))
        cands = [np.nextafter(c, F32(-np.inf)), c, np.nextafter(c, F32(np.inf))]
        want = min(cands, key=lambda v: (abs(Fraction(float(v)) - ex), int(v.view(np.uint32)) & 1))
        assert r[i] == want, (i, x[i], y[i], z[i], r[i], want)
    assert r[-4] == F32(1 + 2.0 ** -11 + 2.0 ** -23) and r[-3] == F32(1 + 2.0 ** -11) and r[-2] == F32(1 + 2.0 ** -11)


def test_pointwise_err32_equals_reproj_err32():
    rng = np.random.default_rng(2)
    h, a, b, t, cmax = R.near_threshold_cases(rng, 50, 3.0)
    for i in range(0, len(h), 97):
        H = np.append(h[i].astype(np.float64), 1.0)
        assert R.reproj_err32(H, a[i:i + 1], b[i:i + 1])[0] == R.reproj_err32_pairs(h[i:i + 1], a[i:i + 1], b[i:i + 1])[0]


def test_seed_case_100px():
    """An outlier whose exact error is 10000.002 > 100^2 while the fused value 9999.92 lay below the cut
    t - 7.5 D - 1e-4 = 9999.94 (D = 0.008): the sure-inlier cut written for 3 px, applied at 100 px."""
    h = np.array([[1.0008821487, -0.0153469807, -2.3652982712, 0.0153469807, 0.9998822212, -15.6064453125,
                   -9.983219570e-06, -8.309625627e-06]], F32)
    a = np.array([[1657.9595947, 925.5112915]], F32)
    b = np.array([[1778.9494629, 988.8345337]], F32)
    t, cmax = F32(10000), np.array([1920], F32)
    emin, emax, den = R.fused_err_range32(h, a, b)
    assert R.reproj_err32_pairs(h, a, b)[0] > t and emin[0] < F32(9999.93)
    assert abs(float(R.fused_D32(h, cmax)[0]) - 0.00801) < 1e-5
    bi, bo, ncls, _, tlo, _ = check_implications(h, a, b, t, cmax, emin, emax, den)
    assert ncls == 1 and bo == 0
    assert bi == 0, (float(emin[0]), float(tlo[0]))


@pytest.mark.parametrize("family", R.FUSED_BOUND_FAMILIES)
def test_fused_cuts_hold_near_the_threshold(family):
    rng = np.random.default_rng(R.FUSED_BOUND_FAMILIES.index(family) + 100)
    h, a, b, t, cmax = R.near_threshold_cases(rng, N_BASE, **R.fused_bound_family(rng, family, N_BASE))
    emin, emax, den = R.fused_err_range32(h, a, b)
    bi, bo, ncls, ee, tlo, thi = check_implications(h, a, b, t, cmax, emin, emax, den)
    assert bi == 0 and bo == 0, (family, bi, bo)
    # the pairs straddle the threshold, and the cuts are in use (tlo finite: with the dm floor of low_den, only at the
    # larger thresholds)
    assert ncls > 0.5 * len(h)
    assert ((ee > t) & (ee < t * F32(1 + 1e-3))).sum() > 1000 and ((ee <= t) & (ee > t * F32(1 - 1e-3))).sum() > 1000
    D = R.fused_D32(h, cmax)
    if family == "D_both_sides":
        assert (D < np.sqrt(t)).sum() > 1000 and (D >= np.sqrt(t)).sum() > 1000
        assert np.isneginf(tlo[D >= np.sqrt(t)]).all()
    else:
        assert np.isfinite(tlo).sum() > 10000


def test_den_safe_implies_den_min_on_both_paths():
    """den_safe(h6, h7, cmax) with |h6| + |h7| on both sides of the limit (1 - kDenMin) / cmax, at the corner where the
    denominator is smallest and at random points of the square |x|, |y| <= cmax."""
    rng = np.random.default_rng(3)
    n = 20000
    cmax = (10.0 ** rng.uniform(np.log10(16), np.log10(192000), n)).astype(F32)
    s = (0.9375 / cmax.astype(np.float64)) * (1 + rng.uniform(-2e-5, 2e-5, n) * rng.choice([1, 100], n))
    f = rng.random(n)
    sg = rng.choice([-1.0, 1.0], (n, 2))
    h = np.zeros((n, 8), F32)
    h[:, 6] = (f * s * sg[:, 0]).astype(F32)
    h[:, 7] = ((1 - f) * s * sg[:, 1]).astype(F32)
    safe = R.den_safe32(h, cmax)
    assert 0.2 < safe.mean() < 0.8
    for k in range(8):
        if k == 0:                                     # the corner of the smallest denominator
            x, y = -np.sign(h[:, 6]) * cmax, -np.sign(h[:, 7]) * cmax
        else:
            x, y = (rng.uniform(-1, 1, (2, n)) * cmax).astype(F32)
        a = np.stack([x, y], 1).astype(F32)
        den_e = (h[:, 6] * a[:, 0] + h[:, 7] * a[:, 1]) + F32(1)
        den_f = R.fused_den32(h, a)
        assert (np.abs(den_e[safe]) >= R.DEN_MIN).all() and (np.abs(den_f[safe]) >= R.DEN_MIN).all(), k
        if k == 0:      # at the corner, the test is tight: den_safe is false well before |den| reaches kDenMin
            assert (np.abs(den_e[~safe]) < F32(0.0626)).mean() > 0.5


def test_cut_at_3px_keeps_its_value():
    """At t = 9 the general cut t - 2.5 sqrt(t) D - max(1e-4, 8u t) is t - 7.5 D - 1e-4, bit for bit."""
    rng = np.random.default_rng(4)
    h, a, b, t, cmax = R.near_threshold_cases(rng, 3000, 3.0, scale=10.0 ** rng.uniform(-1.3, 1, 3000), walk=0)
    tlo, thi = R.fused_thresholds32(h, cmax, F32(9))
    D = R.fused_D32(h, cmax)
    old_lo = np.where(D < F32(2), (F32(9) - F32(7.5) * D) - F32(1e-4), F32(-np.inf))
    old_hi = (F32(9) + F32(1.25) * ((F32(2) * D) * D + (F32(2) * D) * np.sqrt(D * D + F32(9)))) + F32(1e-4)
    assert np.array_equal(tlo[tlo >= 0], old_lo[tlo >= 0]) and np.array_equal(tlo >= 0, old_lo >= 0)
    assert np.array_equal(thi, old_hi)
