"""The oracle's confidence-bounded RANSAC stop (oracle/ransac_adaptive.py update_num_iters / adaptive_stop): OpenCV's iteration
bound, and the key property that an adaptive result is the fixed-count result at n_hyp = n_used.  CPU only."""
import math

import numpy as np
import pytest

from oracle import ransac, ransac_adaptive


@pytest.mark.parametrize("w,bound", [(0.99, 2), (0.9, 5), (0.8, 10), (0.5, 82), (0.3, 651), (0.2, 1024), (1.0, 0)])
def test_update_num_iters_known_answers(w, bound):
    m = 1000
    c = int(round(w * m))
    assert ransac_adaptive.update_num_iters(0.995, (m - c) / m, 1024) == bound


def test_update_num_iters_edges():
    u = ransac_adaptive.update_num_iters
    assert u(0.995, 0.0, 1024) == 0                      # every point an inlier: denom = 0 < DBL_MIN
    assert u(0.995, 1.0, 1024) == 1024                   # no inlier: log(1) = 0 -> denom >= 0 -> the cap
    assert u(1 - 1e-300, 0.5, 1024) == 1024              # confidence near 1: -num huge -> the cap
    assert u(1e-12, 0.5, 1024) == 0                      # confidence near 0: log(1 - p) ~ -1e-12 -> rounds to 0
    assert u(0.995, 0.5, 50) == 50                       # the bound (82) is above maxIters: the cap
    assert u(0.995, -1.0, 7) == 0 and u(2.0, 0.5, 7) == 7   # OpenCV clamps p and ep to [0, 1]


def test_update_num_iters_cap_comparison_and_rounding():
    # ep with (1 - ep)^4 = 1/2: denom = log(1/2); the cap comparison is -num >= maxIters * (-denom)
    ep = 1 - 0.5 ** 0.25
    p = 1 - 0.5 ** 10                                    # num = log(2^-10) = 10 log(1/2): bound 10 (up to ulps)
    assert ransac_adaptive.update_num_iters(p, ep, 11) == 10
    assert ransac_adaptive.update_num_iters(p, ep, 10) == 10      # at the cap (either branch gives 10)
    assert ransac_adaptive.update_num_iters(p, ep, 9) == 9
    # half-integers round to even: num / denom = 2.5 -> 2, 3.5 -> 4 (bounds flagged as near ties)
    for q, want in ((2.5, 2), (3.5, 4)):
        p = 1 - 0.5 ** q
        r, tie = ransac_adaptive.update_num_iters(p, ep, 1024, flag=True)
        assert tie
        assert r in (want, want + (1 if want == 2 else -1))
        assert abs(math.log(1 - p) / math.log(1 - (1 - ep) ** 4) - q) < 1e-9
    # well away from a boundary: not flagged
    assert ransac_adaptive.update_num_iters(0.995, 0.2, 1024, flag=True) == (10, False)


def _mk(rng, n, out_frac, noise=0.5):
    a = (rng.random((n, 2)) * [1920, 1080]).astype(np.float32)
    th = rng.normal() * 0.01
    Ht = np.array([[np.cos(th), -np.sin(th), rng.normal() * 8], [np.sin(th), np.cos(th), rng.normal() * 8],
                   [rng.normal() * 1e-5, rng.normal() * 1e-5, 1]])
    p = np.c_[a, np.ones(n)] @ Ht.T
    b = (p[:, :2] / p[:, 2:] + rng.normal(size=(n, 2)) * noise).astype(np.float32)
    o = rng.random(n) < out_frac
    b[o] = (rng.random((int(o.sum()), 2)) * [1920, 1080]).astype(np.float32)
    return a, b


def _same(r, f):
    assert r["status"] == f["status"]
    assert np.array_equal(r["mask"], f["mask"]) and np.array_equal(r["mask_best"], f["mask_best"])
    if r["H"] is None:
        assert f["H"] is None
    else:
        assert np.array_equal(r["H"], f["H"])
    if r["hyp"] is not None:
        assert r["hyp"]["best"] == f["hyp"]["best"] and r["hyp"]["best_count"] == f["hyp"]["best_count"]


def _point_sets(golden):
    rng = np.random.default_rng(5)
    sets = [(golden[f"fh{i}_a"], golden[f"fh{i}_b2"]) for i in range(1, int(golden["fh_n"]))]
    sets += [_mk(rng, n, of) for n, of in ((300, 0.01), (300, 0.2), (500, 0.5), (200, 0.7), (120, 0.8), (5, 0.0), (4, 0.0))]
    return sets


@pytest.mark.parametrize("conf", [0.5, 0.995, 0.999999])
@pytest.mark.parametrize("level", [1, 2])
def test_adaptive_equals_fixed_at_n_used(golden, conf, level):
    used = []
    for i, (a, b) in enumerate(_point_sets(golden)):
        r = ransac_adaptive.find_homography_seeded(a, b, 1024, 3, 40 + i, level, 3.0, confidence=conf)
        n = r["n_used"]
        if len(a) <= 4:
            assert n == 0
            continue
        assert 1 <= n <= 1024
        used.append(n)
        _same(r, ransac.find_homography_seeded(a, b, n, 3, 40 + i, level, 3.0))
    assert min(used) < 1024                                   # the stop fired somewhere


def test_adaptive_walk_matches_the_rule_by_hand():
    # counts / validity chosen by hand: m = 100, confidence 0.995
    ok = np.array([0, 1, 1, 1, 1, 1, 1, 1], bool)
    counts = np.array([99, 3, 50, 50, 80, 10, 80, 90])
    # h1: c = 3 (not > 3); h2: best = 50, bound 82; h3: tie, no update; h4: best = 80, bound 10 (it = 4); ...
    n, tie = ransac_adaptive.adaptive_stop(counts, ok, 100, 8, 0.995)
    assert n == 8 and not tie                                 # niters 10 > 7 valid hypotheses: the stream ends
    n, _ = ransac_adaptive.adaptive_stop(counts, ok, 100, 8, 0.9)      # at 0.9 and w = 0.8 the bound is 4 = it at h4: stop there
    assert n == 5
    n, _ = ransac_adaptive.adaptive_stop(np.array([100, 100]), np.ones(2, bool), 100, 2, 0.5)   # c = m: bound 0
    assert n == 1


def test_adaptive_without_a_binding_bound_is_the_fixed_route(golden):
    # the bound only falls as the best count grows: when even the final winner's count leaves it at n_hyp, the adaptive
    # route scores the whole stream and is the fixed route
    checked = 0
    for i, (a, b) in enumerate(_point_sets(golden)):
        f = ransac.find_homography_seeded(a, b, 16, 1, i, 1, 3.0)
        if f["hyp"] is None or f["hyp"]["best_count"] < 4:
            continue
        m, c = len(a), f["hyp"]["best_count"]
        if ransac_adaptive.update_num_iters(0.999999, (m - c) / m, 16) < 16:
            continue
        r = ransac_adaptive.find_homography_seeded(a, b, 16, 1, i, 1, 3.0, confidence=0.999999)
        assert r["n_used"] == 16
        _same(r, f)
        checked += 1
    assert checked >= 3


@pytest.mark.parametrize("bad", [0.0, 1.0, -0.1, float("nan")])
def test_oracle_refuses_confidence_out_of_range(bad):
    with pytest.raises(ValueError):
        ransac_adaptive.find_homography_seeded(np.zeros((10, 2)), np.zeros((10, 2)), 16, confidence=bad)


@pytest.mark.parametrize("reference_exact", [False, True])
def test_restated_chain_equals_pipeline_when_the_bound_cannot_bind(reference_exact):
    # at the largest confidence below 1 the bound stays >= 4 unless a model counts every point, and a model that does
    # is the fixed arg-max as well: with n_hyp = 4 the restated multi-feature chain is pipeline.video_chain_multi
    import os
    from oracle import pipeline
    clip = np.load(os.path.join(os.path.dirname(__file__), "golden", "clip_full.npz"))
    feats = {t: [(clip[f"{t.lower()}{f}_c"], clip[f"{t.lower()}{f}_d"]) for f in range(0, 6)] for t in ("SIFT", "ORB")}
    conf = float(np.nextafter(1.0, 0.0))
    got = ransac_adaptive.video_chain_multi(feats, 4, 0, True, reference_exact, confidence=conf)
    want = pipeline.video_chain_multi(feats, 4, 0, True, reference_exact)
    assert np.array_equal(got["status"], want["status"])
    assert np.array_equal(got["S"], want["S"])
