"""evz_find_homography_adaptive: OpenCV's confidence-bounded RANSAC stop on the seeded hypothesis stream, against the
oracle (oracle/ransac_adaptive.py) and against evz_find_homography at n_hyp = n_used.  Needs a B200.

Where the oracle flags a bound within 1e-9 of a libm-dependent boundary (`tie`), either n_used is accepted; the tests
print how many such pairs they met."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import chain, ransac, ransac_adaptive

pytestmark = pytest.mark.gpu

MAX_KP = 12288
OPT_EXACT, OPT_NO_PRUNE = 1, 3
E_ARG = -2
RATIOS = (0.99, 0.8, 0.5, 0.3, 0.2)
_ties = [0]


def _mk(rng, n, w, noise=0.5):
    """n point pairs, a fraction w of them inliers of a near-identity homography."""
    a = (rng.random((n, 2)) * [1920, 1080]).astype(np.float32)
    th = rng.normal() * 0.01
    s = 1 + rng.normal() * 0.01
    Ht = np.array([[s * np.cos(th), -s * np.sin(th), rng.normal() * 8], [s * np.sin(th), s * np.cos(th), rng.normal() * 8],
                   [rng.normal() * 1e-5, rng.normal() * 1e-5, 1]])
    p = np.c_[a, np.ones(n)] @ Ht.T
    b = (p[:, :2] / p[:, 2:] + rng.normal(size=(n, 2)) * noise).astype(np.float32)
    o = rng.permutation(n)[:int(round(n * (1 - w)))]
    b[o] = (rng.random((len(o), 2)) * [1920, 1080]).astype(np.float32)
    return a, b


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


def _px(H, a):
    p = np.c_[a.astype(np.float64), np.ones(len(a))] @ np.asarray(H, np.float64).reshape(3, 3).T
    return p[:, :2] / p[:, 2:]


def _pre_map(T, p):
    q = p.astype(np.float64)
    X = (T[0, 0] * q[:, 0] + T[0, 1] * q[:, 1]) + T[0, 2]
    Y = (T[1, 0] * q[:, 0] + T[1, 1] * q[:, 1]) + T[1, 2]
    W = (T[2, 0] * q[:, 0] + T[2, 1] * q[:, 1]) + T[2, 2]
    return np.stack([X / W, Y / W], 1).astype(np.float32)


def _host(out):
    return {k: v.cpu().numpy() for k, v in out.items() if v is not None}


def _run(engine, sets, n_hyp, seed, base, level, conf, thresh=3.0, pre=None, max_cnt=None, status0=None, frac=0.0):
    pts, off, cnt, off_h, cnt_h = _pack(sets, engine.device)
    P = len(sets)
    status = torch.zeros(P, dtype=torch.int32, device=engine.device) if status0 is None else \
        torch.from_numpy(np.asarray(status0, np.int32)).to(engine.device)
    pre_d = None if pre is None else torch.from_numpy(np.tile(pre.reshape(1, 9), (P, 1))).to(engine.device)
    mc = max(4, int(cnt_h.max())) if max_cnt is None else max_cnt
    out = engine.find_homography(pts, off, cnt, status, mc, n_hyp, seed, base, level, thresh, frac, 4, pre_H=pre_d,
                                 confidence=conf)
    o = _host(out)
    o["status"] = status.cpu().numpy()
    return o, (pts, off, cnt, off_h, cnt_h, pre_d, mc)


def _check_oracle(o, packed, sets, n_hyp, seed, base, level, conf, thresh=3.0, pre=None):
    """n_used, winner, its count and 4-point model, both masks and status bit-exact; H within 1e-3 px on the inliers."""
    _, _, _, off_h, cnt_h, _, _ = packed
    for i, (a, b) in enumerate(sets):
        if pre is not None:
            a, b = _pre_map(pre, a), _pre_map(pre, b)
        ref = ransac_adaptive.find_homography_seeded(a, b, n_hyp, seed, base + i, level, thresh, confidence=conf)
        if ref["tie"] and int(o["n_used"][i]) != ref["n_used"]:
            _ties[0] += 1
            print(f"near-tie bound: pair {i} n_used {int(o['n_used'][i])} (oracle {ref['n_used']})")
            continue
        assert int(o["n_used"][i]) == ref["n_used"], (i, int(o["n_used"][i]), ref["n_used"])
        assert o["status"][i] == ref["status"], i
        om, m = off_h[i], cnt_h[i]
        if ref["hyp"] is not None:
            assert int(o["best_cnt"][i]) == ref["hyp"]["best_count"], i
            if ref["hyp"]["best_count"] > 0:                    # (no inlier at all: the device reports -1)
                assert int(o["best_hyp"][i]) == ref["hyp"]["best"], i
            if ref["hyp"]["best_count"] >= 4:
                assert np.array_equal(o["H_best"][i], ref["hyp"]["H_all"][ref["hyp"]["best"]]), i
        if ref["status"] != 0:
            continue
        assert np.array_equal(o["mask_best"][om:om + m].astype(bool), ref["mask_best"]), i
        assert np.array_equal(o["mask"][om:om + m], ref["mask"]), i
        inl = ref["mask_best"]
        err = np.linalg.norm(_px(o["H"][i], a[inl]) - _px(ref["H"], a[inl]), axis=1).max()
        assert err < 1e-3, (i, err)


def _check_fixed(engine, o, packed, n_hyp, seed, base, level, thresh=3.0, frac=0.0, status0=None):
    """Every output of pair p equals evz_find_homography_ids' at n_hyp = n_used[p], pair by pair."""
    pts, off, cnt, off_h, cnt_h, pre_d, mc = packed
    for p in range(len(cnt_h)):
        n = int(o["n_used"][p])
        st = torch.tensor([0 if status0 is None else status0[p]], dtype=torch.int32, device=engine.device)
        ids = torch.tensor([base + p], dtype=torch.int64, device=engine.device)
        f = engine.find_homography(pts, off[p:p + 1], cnt[p:p + 1], st, mc, max(n, 1), seed, 0, level, thresh, frac, 4,
                                   pre_H=None if pre_d is None else pre_d[p:p + 1], pair_ids=ids)
        f = _host(f)
        assert int(st[0]) == o["status"][p], p
        for k in ("H", "inl_cnt", "best_hyp", "best_cnt", "H_best"):
            assert np.array_equal(f[k][0], o[k][p]), (p, k)
        om, m = off_h[p], cnt_h[p]
        for k in ("mask", "mask_best"):
            assert np.array_equal(f[k][om:om + m], o[k][om:om + m]), (p, k)


@pytest.mark.parametrize("conf", [0.5, 0.9, 0.995, 0.999999])
@pytest.mark.parametrize("thresh", [1.0, 3.0])
@pytest.mark.parametrize("level", [1, 2])
def test_adaptive_vs_oracle_and_fixed(engine, level, thresh, conf):
    rng = np.random.default_rng(int(conf * 1e6) + 17 * level + int(thresh))
    sets = [_mk(rng, n, w, noise=0.4 * thresh / 3) for w in RATIOS for n in (150, 600)]
    for pre in (None, np.array([[1.01, 0.02, 5.0], [-0.01, 0.99, -3.0], [1e-5, -2e-5, 1.0]])):
        o, packed = _run(engine, sets, 1024, 5, 300, level, conf, thresh, pre=pre)
        _check_oracle(o, packed, sets, 1024, 5, 300, level, conf, thresh, pre=pre)
        _check_fixed(engine, o, packed, 1024, 5, 300, level, thresh)
    print("near-tie pairs so far:", _ties[0])


@pytest.mark.parametrize("n_hyp", [1, 31, 32, 33, 255, 256, 257, 1024, 4096, 65535])
def test_adaptive_hypothesis_counts(engine, n_hyp):
    rng = np.random.default_rng(n_hyp)
    sets = [_mk(rng, 300, w) for w in RATIOS] + [_mk(rng, 257, 0.25, noise=0.2)]
    for conf in (0.995, 0.999999):
        o, packed = _run(engine, sets, n_hyp, 9, 1000, 1, conf)
        _check_oracle(o, packed, sets, n_hyp, 9, 1000, 1, conf)
        _check_fixed(engine, o, packed, n_hyp, 9, 1000, 1)


def test_adaptive_stops_on_group_boundaries(engine):
    """Crafted confidences whose stop lands on the last hypothesis of a group (32, 160 = 32 + 128, 672 = 160 + 512) and
    on the first of the next."""
    rng = np.random.default_rng(3)
    targets = (32, 33, 160, 161, 672, 673)
    found = {}
    for k in range(60):
        a, b = _mk(rng, 400, rng.uniform(0.15, 0.45))
        hyp = ransac.ransac_hypotheses(a, b, 1024, 2, k, 1)
        ok, counts = hyp["ok_all"], hyp["counts"]
        for n in targets:
            # the bound of the best count in [0, n) equal to the valid hypotheses in [0, n): stop at hypothesis n - 1
            c = int(counts[:n][ok[:n]].max(initial=0))
            if n in found or not ok[n - 1] or c < 4:
                continue
            conf = 1 - (1 - (c / 400) ** 4) ** int(ok[:n].sum())
            if 0 < conf < 1 and ransac_adaptive.adaptive_stop(counts, ok, 400, 1024, conf) == (n, False):
                found[n] = ((a, b), k, conf)
        if len(found) == len(targets):
            break
    print("group-boundary stops crafted:", sorted(found))
    assert set(found) == set(targets)
    for n, ((a, b), k, conf) in sorted(found.items()):
        o, packed = _run(engine, [(a, b)], 1024, 2, k, 1, conf)
        assert int(o["n_used"][0]) == n
        _check_oracle(o, packed, [(a, b)], 1024, 2, k, 1, conf)
        _check_fixed(engine, o, packed, 1024, 2, k, 1)


@pytest.mark.parametrize("n_hyp", [944, 945, 1024, 65535])
def test_adaptive_at_the_size_limit(engine, n_hyp):
    rng = np.random.default_rng(n_hyp + 1)
    sets = [_mk(rng, MAX_KP, w) for w in ((0.99, 0.5, 0.2) if n_hyp < 65535 else (0.5,))]   # (the oracle scores all n_hyp)
    o, packed = _run(engine, sets, n_hyp, 5, 300, 1, 0.995, max_cnt=MAX_KP)
    _check_oracle(o, packed, sets, n_hyp, 5, 300, 1, 0.995)
    if n_hyp != 65535:
        _check_fixed(engine, o, packed, n_hyp, 5, 300, 1)


def test_adaptive_options_ranges_and_repeat(engine):
    rng = np.random.default_rng(11)
    sets = [_mk(rng, n, w) for w in RATIOS for n in (40, 300)]
    base, _ = _run(engine, sets, 2048, 4, 70, 1, 0.995)
    again, _ = _run(engine, sets, 2048, 4, 70, 1, 0.995)
    for k in base:
        assert np.array_equal(base[k], again[k]), k
    try:
        for opt in (OPT_EXACT, OPT_NO_PRUNE):
            engine.set_option(opt, 1)
            o, _ = _run(engine, sets, 2048, 4, 70, 1, 0.995)
            engine.set_option(opt, 0)
            for k in base:
                assert np.array_equal(base[k], o[k]), (opt, k)
    finally:
        engine.set_option(OPT_EXACT, 0)
        engine.set_option(OPT_NO_PRUNE, 0)
    # split pair ranges, seeded by explicit pair ids
    for k0 in (1, 4, 9):
        parts = []
        for lo, hi in ((0, k0), (k0, len(sets))):
            pts, off, cnt, off_h, cnt_h = _pack(sets[lo:hi], engine.device)
            st = torch.zeros(hi - lo, dtype=torch.int32, device=engine.device)
            ids = torch.arange(70 + lo, 70 + hi, dtype=torch.int64, device=engine.device)
            out = _host(engine.find_homography(pts, off, cnt, st, int(cnt_h.max()), 2048, 4, 0, 1, 3.0, 0.0, 4,
                                               pair_ids=ids, confidence=0.995))
            parts.append((out, st.cpu().numpy()))
        for k in ("n_used", "best_hyp", "best_cnt", "H", "H_best", "inl_cnt"):
            assert np.array_equal(np.concatenate([p[0][k] for p in parts]), base[k]), (k0, k)
        assert np.array_equal(np.concatenate([p[1] for p in parts]), base["status"])


def test_adaptive_skipped_pairs(engine):
    rng = np.random.default_rng(2)
    sets = [_mk(rng, 200, 0.8), _mk(rng, 3, 1.0), _mk(rng, 4, 1.0), _mk(rng, 200, 0.8), _mk(rng, 300, 0.8)]
    status0 = [0, 0, 0, 1, 0]
    o, packed = _run(engine, sets, 1024, 1, 0, 1, 0.995, max_cnt=250, status0=status0)
    assert o["n_used"].tolist()[1:] == [0, 0, 0, 0]            # m < 4, m == 4, status on entry, m > max_cnt
    assert o["n_used"][0] > 0
    assert o["status"].tolist() == [0, 3, 0, 1, 4]
    _check_fixed(engine, o, packed, 1024, 1, 0, 1, status0=status0)


def test_adaptive_argument_errors(engine):
    lib, h = engine.lib, engine.h
    rng = np.random.default_rng(0)
    pts, off, cnt, _, _ = _pack([_mk(rng, 50, 0.8)], engine.device)
    st = torch.zeros(1, dtype=torch.int32, device=engine.device)
    H = torch.zeros((1, 9), dtype=torch.float64, device=engine.device)
    nu = torch.full((1,), -7, dtype=torch.int32, device=engine.device)
    p_ = lambda t: C.c_void_p(t.data_ptr())
    fh = lambda n_hyp, conf: lib.evz_find_homography_adaptive(h, p_(pts), p_(off), p_(cnt), 1, 50, None, n_hyp, 0, 0, None,
                                                              1, 3.0, 0.0, 4, conf, p_(st), p_(H), None, None, None, None,
                                                              None, None, p_(nu), None)
    for conf in (0.0, 1.0, -0.1, float("nan")):
        assert fh(64, conf) == E_ARG
    for n in (0, 65536):
        assert fh(n, 0.995) == E_ARG
    torch.cuda.synchronize()
    assert int(nu[0]) == -7                                    # refused before anything ran
    assert fh(64, 0.995) == 0
    torch.cuda.synchronize()
    assert 1 <= int(nu[0]) <= 64 and int(st[0]) == 0


# ------------------------------------------------------------------------------------------------ public API
@pytest.fixture(scope="module")
def proc(engine):
    import evenvizion_b200
    evenvizion_b200._default_engine = engine
    import evenvizion_b200.processing as p
    return p


@pytest.fixture(scope="module")
def clip():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "clip_full.npz"))


def _clip_feats(clip, types, f0, f1):
    return {t: [(clip[f"{t.lower()}{f}_c"], clip[f"{t.lower()}{f}_d"]) for f in range(f0, f1)] for t in types}


GRID = np.c_[np.stack(np.meshgrid(np.linspace(0, 400, 9), np.linspace(0, 224, 6)), -1).reshape(-1, 2), np.ones(54)]


@pytest.mark.parametrize("mode", ["parallel", "reference"])
def test_geometry_from_features_adaptive_vs_oracle(proc, clip, mode):
    f = _clip_feats(clip, ("SIFT", "ORB"), 0, 25)
    H_list, status = proc.geometry_from_features(f, True, mode, n_hyp=1024, seed=0, confidence=0.995)
    ref = ransac_adaptive.video_chain_multi(f, n_hyp=1024, seed=0, none_h_processing=True, reference_exact=(mode == "reference"),
                                     confidence=0.995)
    assert np.array_equal(status, ref["status"])
    sup = chain.superposition_dict({k + 2: {"H": np.asarray(H).tolist()} for k, H in enumerate(H_list)})
    for k in range(len(H_list)):
        x = GRID @ np.asarray(sup[k + 2], np.float64).T
        y = GRID @ ref["S"][k + 1].T
        assert np.abs(x[:, :2] / x[:, 2:] - y[:, :2] / y[:, 2:]).max() < 1e-2, k


@pytest.mark.parametrize("mode", ["parallel", "reference"])
def test_geometry_batch_adaptive_equals_single(proc, clip, mode):
    feats = [_clip_feats(clip, ("SIFT", "ORB"), a, b) for a, b in [(0, 12), (30, 50), (60, 63)]]
    got = proc.geometry_from_features_batch(feats, True, mode, n_hyp=1024, seed=0, confidence=0.995)
    for f, g in zip(feats, got):
        s = proc.geometry_from_features(f, True, mode, n_hyp=1024, seed=0, confidence=0.995)
        assert np.array_equal(g[1], s[1])
        assert all(np.array_equal(x, y) for x, y in zip(g[0], s[0]))


def test_reference_loop_adaptive_does_not_synchronise(engine):
    rng = np.random.default_rng(4)
    sets = [_mk(rng, 120, w) for w in (0.9, 0.8, 0.95, 0.85, 0.99, 0.9, 0.8, 0.9, 0.95)]
    pts, off, cnt, _, cnt_h = _pack(sets, engine.device)
    status = torch.zeros(len(sets), dtype=torch.int32, device=engine.device)
    step_off = [0, 3, 6, 8, 9]
    engine.reference_chains(pts, off, cnt, status, int(cnt_h.max()), step_off, 128, 1, confidence=0.995)
    torch.cuda.synchronize()
    status.zero_()
    torch.cuda.set_sync_debug_mode("error")
    try:
        H = engine.reference_chains(pts, off, cnt, status, int(cnt_h.max()), step_off, 128, 1, confidence=0.995)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(H).all())


def test_homography_dicts_pass_confidence(proc, monkeypatch):
    import evenvizion_b200.processing.video_processing as vp
    seen = []
    monkeypatch.setattr(vp, "read_and_describe", lambda c, *a: ({"SIFT": []}, (10, 20)))
    monkeypatch.setattr(vp, "geometry_from_features_batch",
                        lambda feats, *a, confidence=None, **k: seen.append(confidence) or [([], np.zeros(0, np.int32))] * len(feats))
    vp.get_homography_dict(None, confidence=0.9)
    vp.get_homography_dicts([None, None], confidence=0.75)
    vp.get_homography_dict(None)
    assert seen == [0.9, 0.75, None]
