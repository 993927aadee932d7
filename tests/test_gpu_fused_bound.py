"""The fused count bounds of the RANSAC scoring kernels on the device.  Needs a B200.

tests/probes/libfused_bound_probe.so (built with the library) evaluates reproj_err_fused, reproj_err32, fused_thresholds,
den_safe and the raw rcp.approx.ftz of ransac_device.cuh as the kernels compile them.  Against the restatements of
oracle/ransac.py and the exact f32 error, on pairs within a few ulps of the threshold (the families of
test_host_fused_bound.py, 10^7 pairs each), and end to end: sets whose matches sit on the threshold of the winning and
leading models must give the same result on the fused route, the exact route and the oracle."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import ransac as R
from oracle import ransac_adaptive

pytestmark = pytest.mark.gpu

F32 = np.float32
PROBE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "probes", "libfused_bound_probe.so")
N_SAMPLES = 10 ** 7
_lib = []


def _probe_lib():
    if not _lib:
        if not os.path.exists(PROBE):
            pytest.fail(f"{PROBE} is missing: build it with `make -C evenvizion_b200/csrc` (part of build())")
        lib = ctypes.CDLL(PROBE)
        lib.fused_bound_probe.restype = ctypes.c_int
        lib.fused_bound_probe.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_int64] + [ctypes.c_void_p] * 9
        _lib.append(lib)
    return _lib[0]


def probe(h, a, b, t, cmax, dev="cuda:0"):
    """Device values for every (h, a, b, t, cmax): numpy arrays e_fused, e_exact, tlo, thi, safe, rcp, den_f, den_e."""
    lib = _probe_lib()
    n = len(h)
    hd = torch.from_numpy(np.ascontiguousarray(h, F32)).to(dev)
    pd = torch.from_numpy(np.ascontiguousarray(np.concatenate([a, b], 1), F32)).to(dev)
    td = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(np.asarray(t, F32), (n,)))).to(dev)
    cd = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(np.asarray(cmax, F32), (n,)))).to(dev)
    names = ("e_fused", "e_exact", "tlo", "thi", "safe", "rcp", "den_f", "den_e")
    out = {k: torch.empty(n, dtype=torch.uint8 if k == "safe" else torch.float32, device=dev) for k in names}
    err = lib.fused_bound_probe(hd.data_ptr(), pd.data_ptr(), td.data_ptr(), cd.data_ptr(), n,
                                *[out[k].data_ptr() for k in names], torch.cuda.current_stream(dev).cuda_stream)
    assert err == 0, err
    torch.cuda.synchronize(dev)
    return {k: v.cpu().numpy() for k, v in out.items()}


def _bits_equal(x, y):
    return np.array_equal(np.asarray(x, F32).view(np.uint32), np.asarray(y, F32).view(np.uint32))


def old_tlo(h, cmax, t):
    """The parent's sure-inlier cut t - 7.5 D - 1e-4 (D < 2), written for 3 px."""
    D = R.fused_D32(h, cmax)
    with np.errstate(all="ignore"):
        return np.where(D < F32(2), (t - F32(7.5) * D) - F32(1e-4), F32(-np.inf)).astype(F32)



@pytest.mark.parametrize("family", R.FUSED_BOUND_FAMILIES)
def test_device_fused_bound(family):
    rng = np.random.default_rng(R.FUSED_BOUND_FAMILIES.index(family) + 1000)
    n_base = -(-N_SAMPLES // 49)
    h, a, b, t, cmax = R.near_threshold_cases(rng, n_base, **R.fused_bound_family(rng, family, n_base))
    d = probe(h, a, b, t, cmax)
    # (a) the exact error of the kernels' rescoring, bit for bit
    assert _bits_equal(d["e_exact"], R.reproj_err32_pairs(h, a, b))
    # (b) the cuts and den_safe, bit for bit
    tlo, thi = R.fused_thresholds32(h, cmax, t)
    assert _bits_equal(d["tlo"], tlo) and _bits_equal(d["thi"], thi)
    assert np.array_equal(d["safe"].astype(bool), R.den_safe32(h, cmax))
    # the emulated fused evaluation, given the device's reciprocal, is the device's value bit for bit
    assert _bits_equal(d["den_f"], R.fused_den32(h, a))
    assert _bits_equal(d["e_fused"], R.reproj_err_fused32(h, a, b, d["rcp"]))
    # (c) the implications on the device's own fused values, where the kernels classify (|den| >= kDenMin)
    ee, ef = d["e_exact"], d["e_fused"]
    cls = np.abs(d["den_f"]) >= R.DEN_MIN
    bad_in = cls & (ef <= tlo) & ~(ee <= t)
    bad_out = cls & (ef >= thi) & (ee <= t)
    assert not bad_in.any() and not bad_out.any(), (int(bad_in.sum()), int(bad_out.sum()))
    sf = d["safe"].astype(bool)
    assert (np.abs(d["den_f"][sf]) >= R.DEN_MIN).all() and (np.abs(d["den_e"][sf]) >= R.DEN_MIN).all()
    # (d) rcp.approx.ftz within 2^-23 relative over the classified denominators
    rel = np.abs(d["rcp"][cls].astype(np.float64) * d["den_f"][cls].astype(np.float64) - 1.0)
    assert rel.max() <= 2.0 ** -23, rel.max()
    n_old = int((cls & (ef <= old_tlo(h, cmax, t)) & (ee > t)).sum())
    print(f"{family}: {len(h)} pairs, {int(cls.sum())} classified, max rcp rel. error {rel.max() / 2.0 ** -23:.3f} x 2^-23, "
          f"{n_old} device-level violators of the old cut t - 7.5 D - 1e-4")


def test_device_den_safe_at_the_limit():
    """den_safe with |h6| + |h7| on both sides of (1 - kDenMin) / cmax, at the corner of the smallest denominator and at
    random points of |x|, |y| <= cmax: both paths' denominators stay >= kDenMin on every safe model."""
    rng = np.random.default_rng(7)
    n = N_SAMPLES
    cmax = (10.0 ** rng.uniform(np.log10(16), np.log10(192000), n)).astype(F32)
    s = (0.9375 / cmax.astype(np.float64)) * (1 + rng.uniform(-2e-5, 2e-5, n) * rng.choice([1, 100], n))
    f = rng.random(n)
    sg = rng.choice([-1.0, 1.0], (n, 2))
    h = np.zeros((n, 8), F32)
    h[:, 0] = h[:, 4] = 1
    h[:, 6] = (f * s * sg[:, 0]).astype(F32)
    h[:, 7] = ((1 - f) * s * sg[:, 1]).astype(F32)
    corner = rng.random(n) < 0.5
    x = np.where(corner, -np.sign(h[:, 6]) * cmax, rng.uniform(-1, 1, n) * cmax).astype(F32)
    y = np.where(corner, -np.sign(h[:, 7]) * cmax, rng.uniform(-1, 1, n) * cmax).astype(F32)
    a = np.stack([x, y], 1)
    d = probe(h, a, a, F32(9), cmax)
    safe = d["safe"].astype(bool)
    assert np.array_equal(safe, R.den_safe32(h, cmax)) and 0.2 < safe.mean() < 0.8
    assert (np.abs(d["den_f"][safe]) >= R.DEN_MIN).all() and (np.abs(d["den_e"][safe]) >= R.DEN_MIN).all()


# ----------------------------------------------------------------------------- end to end
def _mk(rng, n, w, thresh):
    """n pairs on a near-identity homography, noise thresh / 6, a fraction 1 - w of them uniform outliers."""
    a = (rng.random((n, 2)) * [1920, 1080]).astype(np.float32)
    th = rng.normal() * 0.01
    s = 1 + rng.normal() * 0.01
    Ht = np.array([[s * np.cos(th), -s * np.sin(th), rng.normal() * 8], [s * np.sin(th), s * np.cos(th), rng.normal() * 8],
                   [rng.normal() * 1e-5, rng.normal() * 1e-5, 1]])
    p = np.c_[a, np.ones(n)] @ Ht.T
    b = (p[:, :2] / p[:, 2:] + rng.normal(size=(n, 2)) * thresh / 6).astype(np.float32)
    o = rng.permutation(n)[:int(round(n * (1 - w)))]
    b[o] = (rng.random((len(o), 2)) * [1920, 1080]).astype(np.float32)
    return a, b


def _leader(hyp, cmax):
    """The kernel's level-1 leader, up to the fused-versus-exact difference: the first valid hypothesis with the largest
    count among the first 32 slots (den_safe hypotheses first, in index order)."""
    ok = hyp["ok_all"]
    h32 = hyp["H_all"][:, :8].astype(F32)
    safe = R.den_safe32(h32, np.full(len(h32), cmax, F32)) & ok
    order = np.r_[np.flatnonzero(safe), np.flatnonzero(ok & ~safe)][:32]
    return int(order[np.argmax(hyp["counts"][order])])


def _place(a, b, idx, h32, thresh, rng, mode, cmax):
    """Moves b[idx] to within a few ulps of thresh^2 under the f32 model h32: a device-level violator of the old cut
    when the 7 x 7 walk holds one, else the nearest f32 neighbour just outside (mode 'out'), just inside ('in') or
    alternately.  Returns the number of old-cut violators placed."""
    n = len(idx)
    H = np.repeat(h32[None], n, 0)
    cand = R.near_threshold_b(H, a[idx], thresh, rng.uniform(0, 2 * np.pi, n))          # (n, 49, 2)
    k = cand.shape[1]
    t = F32(thresh * thresh)
    d = probe(np.repeat(H, k, 0), np.repeat(a[idx], k, 0), cand.reshape(-1, 2), t, cmax)
    ee, ef = d["e_exact"].reshape(n, k), d["e_fused"].reshape(n, k)
    cls = (np.abs(d["den_f"]) >= R.DEN_MIN).reshape(n, k)
    viol = cls & (ef <= old_tlo(np.repeat(H, k, 0), F32(cmax), t).reshape(n, k)) & (ee > t)
    n_viol = 0
    for j in range(n):
        want_out = mode == "out" or (mode == "alt" and j % 2 == 0)
        if viol[j].any() and mode != "in":
            c = int(np.flatnonzero(viol[j])[0]); n_viol += 1
        elif want_out:
            c = int(np.argmin(np.where(ee[j] > t, ee[j], np.inf)))
        else:
            c = int(np.argmax(np.where(ee[j] <= t, ee[j], -np.inf)))
        b[idx[j]] = cand[j, c]
    return n_viol


def _near_sets(rng, thresh, level, n_hyp, seed, base):
    """Sets whose matches (outside the models' samples) lie on the threshold of the oracle's winner and leader (level 1)
    or of its winner and first valid hypothesis (level 2)."""
    sets, n_viol = [], 0
    specs = [(700, 0.6), (900, 0.45), (500, 0.8), (1200, 0.35)] if level == 1 else [(400, 1.0), (600, 1.0), (300, 1.0), (800, 0.97)]
    for i, (n, w) in enumerate(specs):
        a, b = _mk(rng, n, w, thresh)
        cmax = float(max(np.abs(a).max(), np.abs(b).max()) + thresh + 1)
        hyp = R.ransac_hypotheses(a, b, n_hyp, seed, base + i, level, thresh)
        win = hyp["best"]
        other = _leader(hyp, cmax) if level == 1 else int(np.flatnonzero(hyp["ok_all"])[0])
        fixed = set(hyp["idx"][win].tolist()) | set(hyp["idx"][other].tolist())
        free = np.array([j for j in rng.permutation(n) if j not in fixed])
        inl = R.reproj_err32(hyp["H_all"][win], a, b) <= F32(thresh * thresh)
        free = free[inl[free]]                                   # inliers of the winner go on its threshold
        q = len(free) // 3
        if level == 1:
            n_viol += _place(a, b, free[:q], hyp["H_all"][win][:8].astype(F32), thresh, rng, "alt", cmax)
            if other != win:
                n_viol += _place(a, b, free[q:2 * q], hyp["H_all"][other][:8].astype(F32), thresh, rng, "alt", cmax)
        else:
            # just inside the winner's threshold (unsure for the fused test: the search must rescore them), and on
            # alternate sets just outside that of the first valid hypothesis (a wrong cut would make it "perfect")
            n_viol += _place(a, b, free[:q], hyp["H_all"][win][:8].astype(F32), thresh, rng, "in", cmax)
            if i % 2 and other != win:
                n_viol += _place(a, b, free[q:q + 8], hyp["H_all"][other][:8].astype(F32), thresh, rng, "out", cmax)
        sets.append((a, b))
    return sets, n_viol


def _pack(sets, dev):
    cnt = np.array([len(a) for a, _ in sets], np.int32)
    cap = (cnt + 3) // 4 * 4 + 4
    off = np.zeros(len(sets), np.int32)
    off[1:] = np.cumsum(cap)[:-1]
    pts = np.zeros((int(cap.sum()), 4), np.float32)
    for i, (a, b) in enumerate(sets):
        pts[off[i]:off[i] + cnt[i], :2] = a
        pts[off[i]:off[i] + cnt[i], 2:] = b
    return torch.from_numpy(pts).to(dev), torch.from_numpy(off).to(dev), torch.from_numpy(cnt).to(dev), off, cnt


def _run(engine, packed, n_hyp, seed, base, level, thresh, conf, exact):
    pts, off, cnt, off_h, cnt_h = packed
    engine.set_option(1, exact)
    try:
        status = torch.zeros(len(cnt_h), dtype=torch.int32, device=engine.device)
        out = engine.find_homography(pts, off, cnt, status, int(cnt_h.max()), n_hyp, seed, base, level, thresh, 0.0, 4,
                                     confidence=conf)
        o = {k: v.cpu().numpy() for k, v in out.items() if v is not None}
        o["status"] = status.cpu().numpy()
        return o
    finally:
        engine.set_option(1, 0)


@pytest.mark.parametrize("route", ["level1", "level2", "adaptive"])
@pytest.mark.parametrize("thresh", [3.0, 100.0])
def test_near_threshold_sets_fused_equals_exact_and_oracle(engine, thresh, route):
    """Level 1 (leader partition, staged scoring, the sliced partial row: 336 hypotheses = 32 + 256 + 48), level 2 (the
    first-perfect search) and the confidence-bounded route on sets built on the threshold: status, winner, count, f64
    model, both masks and n_used equal on the fused route, the exact route (EVZ_OPT_RANSAC_EXACT) and the oracle."""
    level = 2 if route == "level2" else 1
    conf = 0.995 if route == "adaptive" else None
    n_hyp, seed, base = (336 if route == "level1" else 512), 21, 40
    rng = np.random.default_rng(int(thresh) * 10 + level + (5 if conf else 0))
    sets, n_viol = _near_sets(rng, thresh, level, n_hyp, seed, base)
    print(f"{route} at {thresh:g} px: {n_viol} device-level violators of the old cut placed")
    packed = _pack(sets, engine.device)
    f = _run(engine, packed, n_hyp, seed, base, level, thresh, conf, 0)
    e = _run(engine, packed, n_hyp, seed, base, level, thresh, conf, 1)
    for k in f:
        assert np.array_equal(f[k], e[k]), k
    _, _, _, off_h, cnt_h = packed
    t = F32(thresh * thresh)
    for i, (a, b) in enumerate(sets):
        if conf is None:
            ref = R.find_homography_seeded(a, b, n_hyp, seed, base + i, level, thresh)
        else:
            ref = ransac_adaptive.find_homography_seeded(a, b, n_hyp, seed, base + i, level, thresh, confidence=conf)
            if ref["tie"] and int(f["n_used"][i]) != ref["n_used"]:
                continue                                         # a stop on a libm-dependent boundary
            assert int(f["n_used"][i]) == ref["n_used"], i
        assert f["status"][i] == ref["status"] == 0, i
        assert int(f["best_hyp"][i]) == ref["hyp"]["best"] and int(f["best_cnt"][i]) == ref["hyp"]["best_count"], i
        assert np.array_equal(f["H_best"][i], ref["hyp"]["H_all"][ref["hyp"]["best"]]), i
        o, m = off_h[i], cnt_h[i]
        assert np.array_equal(f["mask_best"][o:o + m].astype(bool), ref["mask_best"]), i
        # final mask: the refit H agrees with the oracle's to ~1e-6 px, so only errors on the threshold may differ
        diff = f["mask"][o:o + m] != ref["mask"]
        er = R.reproj_err32(ref["H"].ravel(), a, b)
        assert (np.abs(er[diff] - t) < 1e-3 * t).all(), i
        assert int(f["inl_cnt"][i]) == int(f["mask"][o:o + m].sum()), i
