"""CPU: `oracle.ransac.ls_optimum`, the least-squares optimum the refit kernel is held to, pinned to `ransac.refit`, to
live and frozen `cv2.findHomography(method=0)` and to its own certificate, on the golden sets and the bundled clip."""
import numpy as np
import pytest

from oracle import ransac


def _clip_sets(golden):
    """(name, a, b, H_start): the winning inlier sets of the seeded RANSAC on the golden synthetic pairs and on the
    bundled clip's match lists (level 1) and static sets (level 2), with the winning 4-point model."""
    out = []
    def add(name, a, b, pair_id, level):
        r = ransac.find_homography_seeded(a, b, 1024, 0, pair_id, level, 3.0)
        if r["status"] != ransac.ST_OK or r["hyp"] is None:
            return
        mb = r["mask_best"]
        out.append((name, a[mb], b[mb], r["hyp"]["H_all"][r["hyp"]["best"]]))
    for i in range(int(golden["fh_n"])):
        add(f"fh{i}", golden[f"fh{i}_a"], golden[f"fh{i}_b2"], i, 1)
    for p in range(int(golden["clip_n"]) - 1):
        if f"clip{p}_pts_a" in golden.files:
            add(f"clip{p}_match", golden[f"clip{p}_pts_a"], golden[f"clip{p}_pts_b"], p, 1)
            add(f"clip{p}_static", golden[f"clip{p}_static_a"], golden[f"clip{p}_static_b"], p, 2)
    return out


@pytest.fixture(scope="module")
def sets(golden):
    s = _clip_sets(golden)
    assert len(s) >= 20
    return s


def _check_certificate(cert, name):
    assert cert["converged"], name
    assert cert["grad_rel"] < 1e-12, (name, cert)
    assert cert["min_eig"] > 0 and cert["cond"] < 1e8, (name, cert)
    assert cert["spread_px"] < 1e-9, (name, cert)


def test_optimum_agrees_with_refit_and_certificate(sets):
    for name, a, b, H0 in sets:
        H, cert = ransac.ls_optimum(a, b, H0)
        _check_certificate(cert, name)
        assert H[8] == 1.0 and np.isfinite(H).all(), name
        Hr = ransac.refit(a, b)
        d = ransac.max_px_dist(H, Hr, a)
        assert d <= 1e-6, (name, d)
        # no start does better: S at the optimum is not above S at the refit or at the winning 4-point model
        assert cert["S"] <= ransac.sum_sq(Hr, a, b) * (1 + 1e-12), name
        assert cert["S"] <= ransac.sum_sq(H0, a, b), name


def test_optimum_agrees_with_frozen_opencv_method0(golden):
    """fh*_H0 is cv2.findHomography(a, b, 0) frozen when the golden file was made (all points of the set)."""
    for i in range(int(golden["fh_n"])):
        a, b = golden[f"fh{i}_a"], golden[f"fh{i}_b"]
        H, cert = ransac.ls_optimum(a, b, golden[f"fh{i}_H0"])
        _check_certificate(cert, i)
        d = ransac.max_px_dist(H, golden[f"fh{i}_H0"], a)
        assert d <= 1e-6, (i, d)


def test_optimum_agrees_with_live_opencv(sets):
    cv2 = pytest.importorskip("cv2")
    for name, a, b, H0 in sets:
        H, _ = ransac.ls_optimum(a, b, H0)
        Hcv, _ = cv2.findHomography(a, b, 0)
        d = ransac.max_px_dist(H, Hcv, a)
        assert d <= 1e-6, (name, d)


def test_optimum_is_invariant_under_a_shift(sets):
    """Moving a and b by (8000, 5000) px moves the optimum by the same conjugation.  The shifted f32 points are formed
    first and the unshifted set is recovered from them exactly, so both problems hold the same points."""
    sh = np.array([8000.0, 5000.0])
    T = np.array([[1, 0, sh[0]], [0, 1, sh[1]], [0, 0, 1.0]])
    Ti = np.linalg.inv(T)
    for name, a, b, H0 in sets:
        a_s = (a.astype(np.float64) + sh).astype(np.float32)
        b_s = (b.astype(np.float64) + sh).astype(np.float32)
        a0 = (a_s.astype(np.float64) - sh).astype(np.float32)
        b0 = (b_s.astype(np.float64) - sh).astype(np.float32)
        assert np.array_equal(a0.astype(np.float64) + sh, a_s.astype(np.float64)), name      # exact round trip
        H, c0 = ransac.ls_optimum(a0, b0, H0)
        G0 = T @ np.asarray(H0).reshape(3, 3) @ Ti
        G, c1 = ransac.ls_optimum(a_s, b_s, G0 / G0[2, 2])
        _check_certificate(c1, name)
        Gb = Ti @ G.reshape(3, 3) @ T
        d = ransac.max_px_dist(H, Gb / Gb[2, 2], a0)
        assert d <= 1e-9, (name, d)
        assert abs(c1["S"] - c0["S"]) <= 1e-9 * c0["S"] + 1e-18, name


def test_max_px_dist_known_answers():
    """A translation moves every point by its length; a scale about the first point moves the far corner the most."""
    a = np.array([[10, 10], [20, 10], [10, 20], [20, 20], [15, 15]], np.float32)
    H1 = np.eye(3).ravel()
    assert ransac.max_px_dist(H1, H1, a) == 0.0
    H2 = np.array([[1, 0, 1e-3], [0, 1, 0], [0, 0, 1.0]]).ravel()
    assert abs(ransac.max_px_dist(H1, H2, a) - 1e-3) < 1e-12
    H3 = np.array([[1.001, 0, -0.01], [0, 1.001, -0.01], [0, 0, 1.0]]).ravel()         # scale 1.001 about (10, 10)
    assert abs(ransac.max_px_dist(H1, H3, a) - 0.01 * np.sqrt(2)) < 1e-12
    assert abs(ransac.max_px_dist(H1, H3, a[[0, 4]]) - 0.005 * np.sqrt(2)) < 1e-12       # bounding box (10..15)
