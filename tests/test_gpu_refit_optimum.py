"""K4: the refit of `ransac_refit_kernel` against the exact least-squares optimum (`oracle.ransac.ls_optimum`) on the
winner's inlier set, over point sets spread over the frame, clustered in small patches near and far from the origin
(also with outliers spread over the whole frame), offset by thousands of pixels, strongly perspective, tiny and at the
12 288-point limit, at both levels and at thresholds 1 and 3.  For every pair with a model:
  * winner, its f64 model and its inlier mask equal the oracle bit for bit (the refit sees the reference's inlier set);
  * H is within 1e-5 px of the optimum on that set (its points and the corners of their bounding box), ten times the
    kernel's own 1e-6 px stop rule, and S(H) <= S_opt (1 + 1e-9);
  * the final mask is the f32 mask of H bit for bit, and equals the f32 mask of the optimum except where the f32 error
    lies within the distance between the two models plus the rounding of the f32 formula;
  * the inlier count is the sum of the mask and the 70 % gate follows it.
Needs a B200."""
import numpy as np
import pytest
import torch

from oracle import ransac

pytestmark = pytest.mark.gpu

PX_TOL = 1e-5            # distance to the optimum, px
S_REL = 1e-9             # excess of the sum of squares over the optimum
GATE = 0.7
N_HYP = 1024
SEED = 0
U32 = 2.0 ** -24


def _pack(sets, dev):
    cnt = np.array([len(a) for a, _ in sets], np.int32)
    cap = (cnt + 3) // 4 * 4 + 4
    off = np.zeros(len(sets), np.int32)
    off[1:] = np.cumsum(cap)[:-1]
    pts = np.zeros((int(cap.sum()), 4), np.float32)
    for i, (a, b) in enumerate(sets):
        pts[off[i]:off[i] + cnt[i], :2] = a
        pts[off[i]:off[i] + cnt[i], 2:] = b
    return (torch.from_numpy(pts).to(dev), torch.from_numpy(off).to(dev), torch.from_numpy(cnt).to(dev), off, cnt)


def _make(rng, n, region, noise, out_frac, persp, rot=0.05, shift=8.0, out_region=None):
    """n correspondences uniform in region = (x0, y0, w, h); b = pi(Ht a) + N(0, noise) with a rotation N(0, rot) rad,
    a translation N(0, shift) px and perspective N(0, persp) about the origin; a fraction out_frac of b replaced by
    uniform points over the bounding box of the true b, or, with out_region, both a and b of those correspondences
    replaced by uniform points over out_region (a static patch in a busy frame)."""
    x0, y0, w, h = region
    a = (rng.random((n, 2)) * [w, h] + [x0, y0]).astype(np.float32)
    th = rng.normal() * rot
    Ht = np.array([[np.cos(th), -np.sin(th), rng.normal() * shift], [np.sin(th), np.cos(th), rng.normal() * shift],
                   [rng.normal() * persp, rng.normal() * persp, 1.0]])
    p = np.c_[a.astype(np.float64), np.ones(n)] @ Ht.T
    t = p[:, :2] / p[:, 2:]
    b = (t + rng.normal(size=(n, 2)) * noise).astype(np.float32)
    o = rng.random(n) < out_frac
    lo, hi = t.min(0), t.max(0)
    if out_region is None:
        b[o] = (lo + rng.random((int(o.sum()), 2)) * (hi - lo)).astype(np.float32)
    else:
        ox, oy, ow, oh = out_region
        a[o] = (rng.random((int(o.sum()), 2)) * [ow, oh] + [ox, oy]).astype(np.float32)
        b[o] = (rng.random((int(o.sum()), 2)) * [ow, oh] + [ox, oy]).astype(np.float32)
    return a, b


FULL, P96, P384 = (0, 0, 1920, 1080), (96, 54), (384, 216)
NOISE = [0.1, 0.5, 1.0, 2.5]
OUT = [0.0, 0.2, 0.5]


def _families(seed):
    """name -> list of (a, b) (pre-transform applied later where the family asks for one)."""
    rng = np.random.default_rng(seed)
    fam = {}
    def add(name, k, **kw):
        fam[name] = [_make(rng, noise=NOISE[i % 4], out_frac=OUT[i % 3], **{**dict(persp=1e-5), **kw}) for i in range(k)]
    add("full", 6, n=600, region=FULL)
    add("patch96@0", 6, n=200, region=(0, 0) + P96)
    add("patch96@1500,800", 8, n=200, region=(1500, 800) + P96)
    add("patch384@0", 6, n=400, region=(0, 0) + P384)
    add("patch384@1500,800", 6, n=400, region=(1500, 800) + P384)
    add("full+8000", 6, n=600, region=(8000, 8000, 1920, 1080), persp=1e-6)
    add("persp5e-4 patch384@0", 4, n=400, region=(0, 0) + P384, persp=5e-4)
    add("persp1e-4 full", 4, n=600, region=FULL, persp=1e-4)
    for name, reg in (("patch96@1500,800 + frame outliers", (1500, 800) + P96),
                      ("patch384@1500,800 + frame outliers", (1500, 800) + P384)):
        fam[name] = [_make(rng, 350, reg, NOISE[i % 4], [0.2, 0.45][i % 2], 1e-5, out_region=FULL) for i in range(8)]
    fam["5-8 points"] = [_make(rng, n, FULL, [0.1, 0.5][k % 2], 0.0, 1e-5) for k, n in enumerate([5, 6, 7, 8, 5, 8])]
    fam["5-8 points patch96@1500,800"] = [_make(rng, n, (1500, 800) + P96, 0.1, 0.0, 1e-5) for n in (5, 6, 7, 8)]
    return fam


# pre-transform of reference mode: the running superposition, here a translation by thousands of pixels with a small
# rotation and perspective; the kernel maps both point lists through it (f64, rounded to f32) before RANSAC
PRE_H = np.array([[0.999, 0.02, 3000.0], [-0.02, 0.999, -2500.0], [1e-6, -2e-6, 1.0]])


def _pre_map(T, p):
    """pre_map of ransac_kernels.cu: f64 operations in the kernel's order, f32 result."""
    q = p.astype(np.float64)
    X = (T[0, 0] * q[:, 0] + T[0, 1] * q[:, 1]) + T[0, 2]
    Y = (T[1, 0] * q[:, 0] + T[1, 1] * q[:, 1]) + T[1, 2]
    W = (T[2, 0] * q[:, 0] + T[2, 1] * q[:, 1]) + T[2, 2]
    return np.stack([X / W, Y / W], 1).astype(np.float32)


def _f32_slack(H, a, b):
    """Bound (px) on |sqrt(reproj_err32(H)) - exact distance| per point: H rounded to f32 and every f32 operation of
    the formula rounded once, with a factor 2 of margin."""
    h = np.asarray(H, np.float64).ravel()
    x, y = a[:, 0].astype(np.float64), a[:, 1].astype(np.float64)
    den = h[6] * x + h[7] * y + 1.0
    Bd = np.abs(h[6] * x) + np.abs(h[7] * y) + 1.0
    X = h[0] * x + h[1] * y + h[2]
    Y = h[3] * x + h[4] * y + h[5]
    Bx = np.abs(h[0] * x) + np.abs(h[1] * y) + np.abs(h[2])
    By = np.abs(h[3] * x) + np.abs(h[4] * y) + np.abs(h[5])
    rel_w = 4 * U32 * Bd / np.abs(den) + 2 * U32
    ex = (4 * U32 * Bx + np.abs(X) * rel_w) / np.abs(den) + 2 * U32 * (np.abs(X / den) + np.abs(b[:, 0]))
    ey = (4 * U32 * By + np.abs(Y) * rel_w) / np.abs(den) + 2 * U32 * (np.abs(Y / den) + np.abs(b[:, 1]))
    dist = np.hypot(X / den - b[:, 0], Y / den - b[:, 1])
    return 2 * (ex + ey + 4 * U32 * dist)


def _point_dist(H1, H2, a):
    p = np.c_[a.astype(np.float64), np.ones(len(a))]
    q1 = p @ np.asarray(H1, np.float64).reshape(3, 3).T
    q2 = p @ np.asarray(H2, np.float64).reshape(3, 3).T
    return np.hypot(q1[:, 0] / q1[:, 2] - q2[:, 0] / q2[:, 2], q1[:, 1] / q1[:, 2] - q2[:, 1] / q2[:, 2])


def _check_pair(got, a, b, level, pair_id, thresh, fail_status, n_hyp):
    """Checks one pair against the oracle and the optimum; returns None (no model) or (distance px, S excess).
    got: dict of host arrays of this pair (status, H, mask, inl_cnt, best_hyp, best_cnt, H_best, mask_best)."""
    m = len(a)
    ref = ransac.find_homography_seeded(a, b, n_hyp, SEED, pair_id, level, thresh)
    if ref["status"] != ransac.ST_OK:
        want = {ransac.ST_TOO_FEW: 3, ransac.ST_NO_MODEL: fail_status}[ref["status"]]
        assert got["status"] == want, (got["status"], want)
        return None
    inl = int(got["mask"].sum())
    assert got["inl_cnt"] == inl
    assert got["status"] == (6 if inl < GATE * m else 0), (got["status"], inl, m)      # the 70 % gate follows the count
    hyp = ref["hyp"]
    assert got["best_hyp"] == hyp["best"] and got["best_cnt"] == hyp["best_count"]
    assert np.array_equal(got["H_best"], hyp["H_all"][hyp["best"]])
    mb = ref["mask_best"]
    assert np.array_equal(got["mask_best"], mb)
    H = got["H"]
    assert H[8] == 1.0 and np.isfinite(H).all()
    H_opt, cert = ransac.ls_optimum(a[mb], b[mb], got["H_best"])
    assert cert["converged"] and cert["grad_rel"] < 1e-12 and cert["min_eig"] > 0 and cert["spread_px"] < 1e-9, cert
    dist = ransac.max_px_dist(H, H_opt, a[mb])
    S = ransac.sum_sq(H, a[mb], b[mb])
    excess = (S - cert["S"]) / max(cert["S"], 1e-300)
    # final mask: bit for bit the f32 formula at H (phase 4) ...
    t = np.float32(thresh * thresh)
    assert np.array_equal(got["mask"], ransac.reproj_err32(H, a, b) <= t)
    # ... and the f32 mask of the optimum except within the distance between the models plus the f32 rounding
    e_opt = ransac.reproj_err32(H_opt, a, b)
    diff = got["mask"] != (e_opt <= t)
    win = np.maximum(_point_dist(H, H_opt, a), PX_TOL) + _f32_slack(H_opt, a, b) + _f32_slack(H, a, b)
    assert (np.abs(np.sqrt(e_opt[diff].astype(np.float64)) - thresh) <= win[diff]).all(), np.flatnonzero(diff)
    return dist, excess, S, cert["S"], int(mb.sum())


def _run_and_check(engine, groups, level, thresh, pre_H=None, n_hyp=N_HYP):
    """groups: name -> list of (a, b).  One batched call over every pair; per-family maxima of the distance to the
    optimum and of the S excess; asserts the bounds after every pair has been looked at, so that a failure reports
    every family."""
    names, sets = [], []
    for name, ss in groups.items():
        for s in ss:
            names.append(name)
            sets.append(s)
    pts, off, cnt, off_h, cnt_h = _pack(sets, engine.device)
    P = len(sets)
    status = torch.zeros(P, dtype=torch.int32, device=engine.device)
    pre = None
    if pre_H is not None:
        pre = torch.from_numpy(np.tile(pre_H.ravel(), (P, 1))).to(engine.device)
    fail_status = 4 if level == 1 else 5
    out = engine.find_homography(pts, off, cnt, status, int(cnt_h.max()), n_hyp, SEED, 0, level, thresh, GATE,
                                 fail_status, pre_H=pre)
    torch.cuda.synchronize()
    h = {k: v.cpu().numpy() for k, v in out.items()}
    st = status.cpu().numpy()
    stats, bad = {}, []
    for i, (a, b) in enumerate(sets):
        o, m = off_h[i], cnt_h[i]
        if pre_H is not None:
            a, b = _pre_map(pre_H, a), _pre_map(pre_H, b)
        got = dict(status=int(st[i]), H=h["H"][i], mask=h["mask"][o:o + m].astype(bool), inl_cnt=int(h["inl_cnt"][i]),
                   best_hyp=int(h["best_hyp"][i]), best_cnt=int(h["best_cnt"][i]), H_best=h["H_best"][i],
                   mask_best=h["mask_best"][o:o + m].astype(bool))
        r = _check_pair(got, a, b, level, i, thresh, fail_status, n_hyp)
        s = stats.setdefault(names[i], dict(pairs=0, checked=0, dist=0.0, excess=-np.inf))
        s["pairs"] += 1
        if r is None:
            continue
        dist, excess, S, S_opt, n_in = r
        s["checked"] += 1
        s["dist"] = max(s["dist"], dist)
        s["excess"] = max(s["excess"], excess)
        if not (dist <= PX_TOL and S <= S_opt * (1 + S_REL) + n_in * 1e-24):
            bad.append((names[i], i, dist, excess))
    table = "\n".join(f"  {k:36s} pairs {v['pairs']:2d} with a model {v['checked']:2d}  max px to optimum {v['dist']:.3e}"
                      f"  max S excess {v['excess']:.3e}" for k, v in stats.items())
    print(f"\nlevel {level} thresh {thresh} pre_H {pre_H is not None}\n{table}")
    assert not bad, f"{len(bad)} pairs off the optimum (family, pair, px, S excess): {bad}\n{table}"
    for k, v in stats.items():
        assert v["checked"] >= max(1, v["pairs"] // 2), (k, v)           # every family reaches the refit
    return stats


@pytest.fixture(scope="module")
def families():
    return _families(2024)


@pytest.mark.parametrize("level", [1, 2])
@pytest.mark.parametrize("thresh", [1.0, 3.0])
def test_refit_reaches_least_squares_optimum(engine, families, level, thresh):
    _run_and_check(engine, families, level, thresh)


@pytest.mark.parametrize("level", [1, 2])
def test_refit_optimum_at_the_point_limit(engine, level):
    """12 288 points, the largest supported set (512 hypotheses: the scoring kernel's shared-memory tables for 12 288
    points leave no room for 1 024)."""
    rng = np.random.default_rng(12288 + level)
    groups = {"12288 points": [_make(rng, 12288, FULL, 0.5, 0.3, 1e-5)],
              "12288 points patch384@1500,800": [_make(rng, 12288, (1500, 800) + P384, 1.0, 0.2, 1e-5)]}
    _run_and_check(engine, groups, level, 3.0, n_hyp=512)


@pytest.mark.parametrize("level", [1, 2])
def test_refit_optimum_with_reference_mode_pre_transform(engine, level):
    """pre_H as reference mode passes it: the running superposition, thousands of pixels of translation."""
    fam = _families(77)
    groups = {k: fam[k] for k in ("full", "patch96@1500,800", "patch384@0", "5-8 points")}
    _run_and_check(engine, groups, level, 3.0, pre_H=PRE_H)


def test_refit_optimum_on_bench_config2_shape(engine):
    """The point sets of one bench.py config-2 step (synth.make_chain, 2048 keypoints): RANSAC #1 on the match lists,
    RANSAC #2 on the static sets, as the oracle pipeline forms them."""
    from evenvizion_b200 import synth
    from oracle import pipeline
    ch = synth.make_chain(4, 2048, seed=5, device="cpu")
    frames = [(ch["coords"][i].numpy(), ch["desc"][i].numpy()) for i in range(4)]
    l1, l2 = [], []
    for p in range(3):
        r = pipeline.pair_geometry(*frames[p + 1], *frames[p], n_hyp=N_HYP, seed=SEED, pair_id=p)
        l1.append((r["match"]["pts_a"], r["match"]["pts_b"]))
        l2.append((r["static_a"], r["static_b"]))
    st1 = _run_and_check(engine, {"config-2 match lists": l1}, 1, 3.0)
    st2 = _run_and_check(engine, {"config-2 static sets": l2}, 2, 3.0)
    assert st1["config-2 match lists"]["checked"] == 3 and st2["config-2 static sets"]["checked"] == 3
