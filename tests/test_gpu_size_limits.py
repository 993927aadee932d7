"""The per-pair stages at the sizes include/evz.h accepts: EVZ_MAX_KP = 12 288 keypoints per frame and up to 65 535
RANSAC hypotheses, against the oracle.  Needs a B200.

The scoring kernel keeps four u16 lists per hypothesis in shared memory next to the points; at 12 288 points there is
room for 944 hypotheses, beyond that the lists live in handle scratch.  Both sides of that choice, and the kernel's
own loop boundaries (the 32-hypothesis leading batch and level-2 group, the 256-hypothesis pass-0 step), are held to
the oracle here, as are the filter, ingest, static-filter and de-dup kernels at 12 288 points."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import chain, matching, pipeline, ransac, static_filter

pytestmark = pytest.mark.gpu

MAX_KP = 12288
OPT_EXACT, OPT_NO_PRUNE = 1, 3


def _mk(rng, n, out_frac, noise=0.5):
    a = (rng.random((n, 2)) * [1920, 1080]).astype(np.float32)
    th = rng.normal() * 0.01
    s = 1 + rng.normal() * 0.01
    Ht = np.array([[s * np.cos(th), -s * np.sin(th), rng.normal() * 8], [s * np.sin(th), s * np.cos(th), rng.normal() * 8],
                   [rng.normal() * 1e-5, rng.normal() * 1e-5, 1]])
    p = np.c_[a, np.ones(n)] @ Ht.T
    b = (p[:, :2] / p[:, 2:] + rng.normal(size=(n, 2)) * noise).astype(np.float32)
    o = rng.random(n) < out_frac
    b[o] = (rng.random((int(o.sum()), 2)) * [1920, 1080]).astype(np.float32)
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
    """The kernel's matrix_H_prev map (utils.py:351-355): f64, this operation order, rounded to f32."""
    q = p.astype(np.float64)
    X = (T[0, 0] * q[:, 0] + T[0, 1] * q[:, 1]) + T[0, 2]
    Y = (T[1, 0] * q[:, 0] + T[1, 1] * q[:, 1]) + T[1, 2]
    W = (T[2, 0] * q[:, 0] + T[2, 1] * q[:, 1]) + T[2, 2]
    return np.stack([X / W, Y / W], 1).astype(np.float32)


def _check_ransac(engine, sets, n_hyp, seed, base, level, pre=None, max_cnt=None, refs=None):
    """One find_homography launch over `sets` against find_homography_seeded: status, winner, its count, its f64 model
    and its inlier mask bit-exact; the refined H within 1e-3 px of the oracle's on every inlier.  Returns the oracle
    results (reusable for another route through the kernel)."""
    pts, off, cnt, off_h, cnt_h = _pack(sets, engine.device)
    status = torch.zeros(len(sets), dtype=torch.int32, device=engine.device)
    pre_d = None if pre is None else torch.from_numpy(np.tile(pre.reshape(1, 9), (len(sets), 1))).to(engine.device)
    out = engine.find_homography(pts, off, cnt, status, int(cnt_h.max()) if max_cnt is None else max_cnt, n_hyp, seed, base,
                                 level, 3.0, 0.0, 4, pre_H=pre_d)
    st = status.cpu().numpy()
    if refs is None:
        refs = []
        for i, (a, b) in enumerate(sets):
            if pre is not None:
                a, b = _pre_map(pre, a), _pre_map(pre, b)
            refs.append(((a, b), ransac.find_homography_seeded(a, b, n_hyp, seed, base + i, level, 3.0)))
    for i, ((a, b), ref) in enumerate(refs):
        assert st[i] == ref["status"], (i, st[i], ref["status"])
        if ref["status"] != 0:
            continue
        o, m = off_h[i], cnt_h[i]
        if ref["hyp"] is not None:
            assert int(out["best_hyp"][i]) == ref["hyp"]["best"], i
            assert int(out["best_cnt"][i]) == ref["hyp"]["best_count"], i
            assert np.array_equal(out["H_best"][i].cpu().numpy(), ref["hyp"]["H_all"][ref["hyp"]["best"]]), i
        assert np.array_equal(out["mask_best"][o:o + m].cpu().numpy().astype(bool), ref["mask_best"]), i
        inl = ref["mask_best"]
        err = np.linalg.norm(_px(out["H"][i].cpu().numpy(), a[inl]) - _px(ref["H"], a[inl]), axis=1).max()
        assert err < 1e-3, (i, err)
    return refs


@pytest.mark.parametrize("level", [1, 2])
@pytest.mark.parametrize("n_hyp", [944, 945, 1024, 4096])
def test_ransac_at_the_shared_memory_edge(engine, n_hyp, level):
    """12 288 points: 944 hypotheses are the most whose lists fit in shared memory next to the points, 945 and more take
    the lists from handle scratch.  0 %, 30 % and 80 % outliers in one launch, without and with a pre-transform."""
    rng = np.random.default_rng(n_hyp * 10 + level)
    sets = [_mk(rng, MAX_KP, f) for f in (0.0, 0.3, 0.8)]
    _check_ransac(engine, sets, n_hyp, 5, 300, level)
    T = np.array([[1.01, 0.02, 5.0], [-0.01, 0.99, -3.0], [1e-5, -2e-5, 1.0]])
    _check_ransac(engine, sets, n_hyp, 5, 300, level, pre=T)


@pytest.mark.parametrize("level", [1, 2])
@pytest.mark.parametrize("n_hyp", [1, 2, 31, 32, 33, 255, 256, 257, 28583, 65535])
def test_ransac_hypothesis_count_boundaries(engine, n_hyp, level):
    """Hypothesis counts at the scoring kernel's boundaries (the leading batch kLead and the level-2 group kGrp are 32,
    pass 0 steps by 256) and at the top of the accepted range (from 28 583 on the lists of even a few hundred points do
    not fit in shared memory; 65 535 is the largest count accepted), by the default route, without pruning and with the
    exact formula only.  A max_cnt of EVZ_MAX_KP makes every count above 944 take the lists from scratch."""
    rng = np.random.default_rng(n_hyp + 7 * level)
    sets = [_mk(rng, 300, 0.0, noise=0.3), _mk(rng, 300, 0.3), _mk(rng, 257, 0.6), _mk(rng, 5, 0.0)]
    refs = None
    try:
        for opt in (None, OPT_NO_PRUNE, OPT_EXACT):
            if opt is not None:
                engine.set_option(opt, 1)
            for max_cnt in (None, MAX_KP):
                refs = _check_ransac(engine, sets, n_hyp, 9, 1000, level, max_cnt=max_cnt, refs=refs)
            if opt is not None:
                engine.set_option(opt, 0)
    finally:
        engine.set_option(OPT_NO_PRUNE, 0)
        engine.set_option(OPT_EXACT, 0)


def _chain_frames(n_frames, seed):
    from evenvizion_b200 import synth
    ch = synth.make_chain(n_frames, MAX_KP, seed=seed, device="cpu")
    return ch, [(ch["coords"][i].numpy(), ch["desc"][i].numpy()) for i in range(n_frames)]


def test_whole_path_at_max_kp(engine):
    """engine.process_pairs on frames of EVZ_MAX_KP keypoints at the default 1 024 hypotheses: every intermediate of
    every pair against oracle.pipeline.pair_geometry."""
    ch, frames = _chain_frames(4, 21)
    st = engine.ingest(ch["desc"].reshape(-1, 128), ch["coords"].reshape(-1, 2), [MAX_KP] * 4)
    r = engine.process_pairs(st, [1, 2, 3], [0, 1, 2], n_hyp=1024, seed=3)
    torch.cuda.synchronize()
    for p in range(3):
        ref = pipeline.pair_geometry(*frames[p + 1], *frames[p], n_hyp=1024, seed=3, pair_id=p)
        assert int(r.status[p]) == ref["status"] and "ransac2" in ref, p
        o, m = int(st.row_off_h[p + 1]), int(r.m_cnt[p])
        mk = ref["match"]
        assert int(r.n_filtered[p]) == len(mk["matches"]) and m == len(mk["pts_a"]), p
        g = r.m_pts[o:o + m].cpu().numpy()
        assert np.array_equal(g[:, :2], mk["pts_a"]) and np.array_equal(g[:, 2:], mk["pts_b"]), p
        assert np.array_equal(r.mask1_best[o:o + m].cpu().numpy().astype(bool), ref["ransac1"]["mask_best"]), p
        assert int(r.best_hyp1[p]) == ref["ransac1"]["hyp"]["best"], p
        ns = int(r.static_cnt[p])
        assert ns == len(ref["static_a"]) and int(r.static_r[p]) == ref["static_r"], p
        s = r.static_pts[o:o + ns].cpu().numpy()
        assert np.array_equal(s[:, :2], ref["static_a"]) and np.array_equal(s[:, 2:], ref["static_b"]), p
        assert np.array_equal(r.mask2_best[o:o + ns].cpu().numpy().astype(bool), ref["ransac2"]["mask_best"]), p
        assert int(r.best_hyp2[p]) == ref["ransac2"]["hyp"]["best"], p
        if ref["ransac2"]["status"] == 0:
            inl, Hr = ref["ransac2"]["mask_best"], ref["ransac2"]["H"]
            err = np.linalg.norm(_px(r.H[p].cpu().numpy(), ref["static_a"][inl]) - _px(Hr, ref["static_a"][inl]), axis=1)
            assert err.max() < 1e-3, (p, err.max())


@pytest.mark.parametrize("mode", ["reference", "parallel"])
def test_video_geometry_at_max_kp(engine, mode):
    """geometry_from_features on frames of EVZ_MAX_KP keypoints (the bound it passes to RANSAC is the largest frame):
    status identical to oracle.pipeline.video_chain, chain within 1e-2 px on a 9 x 6 grid over the frame."""
    import evenvizion_b200
    evenvizion_b200._default_engine = engine
    from evenvizion_b200.processing import video_processing
    _, frames = _chain_frames(4, 22)
    H_list, status = video_processing.geometry_from_features({"SIFT": frames}, True, mode, n_hyp=1024, seed=0)
    ref = pipeline.video_chain(frames, n_hyp=1024, seed=0, reference_exact=(mode == "reference"))
    assert np.array_equal(status, ref["status"])
    grid = np.stack(np.meshgrid(np.linspace(0, 1920, 9), np.linspace(0, 1080, 6)), -1).reshape(-1, 2)
    pg = np.c_[grid, np.ones(len(grid))]
    sup = chain.superposition_dict({k + 2: {"H": np.asarray(H).tolist()} for k, H in enumerate(H_list)})
    for k in range(len(H_list)):
        a = pg @ np.asarray(sup[k + 2], np.float64).T
        b = pg @ ref["S"][k + 1].T
        assert np.abs(a[:, :2] / a[:, 2:] - b[:, :2] / b[:, 2:]).max() < 1e-2, k


class _NoEngine:
    """An engine that fails on first use: proves that a refusal comes before any launch."""

    def __getattr__(self, name):
        raise AssertionError(f"engine.{name} used")


def test_multi_type_bound_refused_before_launch():
    """SIFT + ORB frames whose largest frames add up to more than EVZ_MAX_KP: RANSAC #2 and the de-dup would receive
    that sum as their bound, so geometry_from_features_batch refuses it with a ValueError naming the limit before it
    uses the engine.  A sum of exactly EVZ_MAX_KP passes the check (and reaches the engine)."""
    from evenvizion_b200.processing import video_processing
    rng = np.random.default_rng(3)

    def frames(counts, d):
        return [(rng.random((n, 2)).astype(np.float32), rng.integers(0, 256, (n, d), dtype=np.uint8)) for n in counts]

    video = {"SIFT": frames([100, 8000, 300], 128), "ORB": frames([4289, 200, 300], 32)}
    with pytest.raises(ValueError, match="12288"):
        video_processing.geometry_from_features_batch([{"SIFT": frames([10, 20], 128), "ORB": frames([10, 20], 32)}, video],
                                                      engine=_NoEngine())
    video["ORB"] = frames([4288, 200, 300], 32)
    with pytest.raises(AssertionError, match="engine"):
        video_processing.geometry_from_features_batch([video], engine=_NoEngine())


# ----------------------------------------------------------------------------- crafted inputs through the C ABI
def _p(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _hash64(k):
    """filter_kernels.cu hash64, restated on uint64."""
    k = np.asarray(k, np.uint64)
    with np.errstate(over="ignore"):
        k = k ^ (k >> np.uint64(33))
        k = k * np.uint64(0xff51afd7ed558ccd)
        k = k ^ (k >> np.uint64(33))
        k = k * np.uint64(0xc4ceb9fe1a85ec53)
        k = k ^ (k >> np.uint64(33))
    return k & np.uint64(0xFFFFFFFF)


def _colliding_coords(n, mask, y=7.25):
    """n distinct points (x, y) whose keys share the slot hash64(key) & mask (key = bits(x) << 32 | bits(y))."""
    yb = np.uint64(np.float32(y).view(np.uint32))
    xb0 = np.float32(1.0).view(np.uint32)
    want, found = None, []
    for c0 in range(0, 1 << 28, 1 << 23):
        xb = np.arange(xb0 + c0, xb0 + c0 + (1 << 23), dtype=np.uint64)
        s = _hash64((xb << np.uint64(32)) | yb) & np.uint64(mask)
        want = s[0] if want is None else want
        found.append(xb[s == want])
        if sum(len(f) for f in found) >= n:
            break
    xb = np.concatenate(found)[:n].astype(np.uint32)
    assert len(xb) == n
    return np.c_[xb.view(np.float32), np.full(n, y, np.float32)]


def _canon_ref(c):
    first, out = {}, np.empty(len(c), np.int32)
    for i, (x, y) in enumerate(c):
        out[i] = first.setdefault((float(x), float(y)), i)        # -0.0 == 0.0 as dict keys
    return out


def test_ingest_canon_at_max_kp(engine):
    """ingest_canon_kernel's open-addressing table at 12 288 keypoints: every coordinate identical, every coordinate twice,
    -0.0 / 0.0 mixes, and 2 048 distinct keys that all hash to one slot of the 32 768-slot table, repeated and interleaved.
    canon = the frame's first keypoint with an equal (x, y), against a Python dict."""
    rng = np.random.default_rng(4)
    n = MAX_KP
    same = np.tile(np.float32([[3.5, -2.25]]), (n, 1))
    base = (rng.random((n // 2, 2)) * 1000).astype(np.float32)
    twice = np.concatenate([base, base])[rng.permutation(n)]
    z = np.float32([0.0, -0.0, 1.0])
    zeros = np.stack([rng.choice(z, n), rng.choice(z, n)], 1).astype(np.float32)
    coll = _colliding_coords(2048, 32767)
    coll = coll[np.r_[np.arange(2048), rng.integers(0, 2048, n - 2048)]][rng.permutation(n)]
    frames = [same, twice, zeros, coll]
    desc = np.zeros((n * len(frames), 128), np.uint8)
    st = engine.ingest(desc, np.concatenate(frames), [n] * len(frames))
    canon = st.canon.cpu().numpy()
    for f, c in enumerate(frames):
        got = canon[st.row_off_h[f]:st.row_off_h[f] + n]
        assert np.array_equal(got, _canon_ref(c)), f
    assert len(set(map(tuple, coll.tolist()))) == 2048


def test_ingest_bad_count_for_float_descriptors(engine):
    """bad_count: float descriptor values that are not integers in [0, 255] (255.5, 256, -1, NaN; 255.0 and -0.0 are
    integers in range), against a NumPy count, over frames of 12 288 keypoints."""
    rng = np.random.default_rng(6)
    vals = np.float32([255.0, 255.5, 256.0, -1.0, -0.0, np.nan, 0.0, 17.0])
    desc = rng.choice(vals, (2 * MAX_KP, 128)).astype(np.float32)
    want = int((~(desc == np.rint(desc)) | (desc < 0) | (desc > 255)).sum())
    coords = (rng.random((2 * MAX_KP, 2)) * 100).astype(np.float32)
    with pytest.raises(ValueError) as e:
        engine.ingest(desc, coords, [MAX_KP, MAX_KP])
    assert int(str(e.value).split()[0]) == want


def _filter_run(engine, st, pairs, top2_idx, top2_d2, out_off, rows):
    dev = engine.device
    P = len(pairs)
    pq = torch.tensor([q for q, _ in pairs], dtype=torch.int32, device=dev)
    pt = torch.tensor([t for _, t in pairs], dtype=torch.int32, device=dev)
    oo = torch.tensor(out_off, dtype=torch.int32, device=dev)
    ti = torch.from_numpy(top2_idx).to(dev)
    td = torch.from_numpy(top2_d2).to(dev)
    surv = torch.full((rows,), 9, dtype=torch.uint8, device=dev)
    m_idx = torch.zeros((rows, 2), dtype=torch.int32, device=dev)
    m_pts = torch.zeros((rows, 4), dtype=torch.float32, device=dev)
    m_cnt, n_f, status = (torch.zeros(P, dtype=torch.int32, device=dev) for _ in range(3))
    engine._check(engine.lib.evz_filter_matches(engine.h, _p(ti), _p(td), _p(st.coords), _p(st.canon), _p(st.row_off),
                                                _p(st.n_kp), _p(pq), _p(pt), _p(oo), P, st.max_kp, 0.5, 4, _p(surv), _p(m_idx),
                                                _p(m_pts), _p(m_cnt), _p(n_f), _p(status), engine._stream()))
    torch.cuda.synchronize()
    return (surv.cpu().numpy(), m_idx.cpu().numpy(), m_pts.cpu().numpy(), m_cnt.cpu().numpy(), n_f.cpu().numpy(),
            status.cpu().numpy())


def test_filter_matches_at_max_kp(engine):
    """filter_matches_kernel on 12 288 x 12 288 pairs with crafted top-2 lists, written at odd out_off rows: ratio-test
    edges at the largest possible d2 (128 * 255^2), a train frame of one row (no second neighbour), one train index
    claimed by exactly one, by two and by all 12 288 queries, and one coordinate group of 12 288 members whose kept and
    dropped members interleave (its first kept member is not canon).  Against ratio_survivors, collision_filter and
    remove_double_matching."""
    rng = np.random.default_rng(8)
    n = MAX_KP
    dmax = 128 * 255 * 255
    grid = (rng.integers(0, 60, (n, 2)) * 0.25).astype(np.float32)                # 3 600 coordinate groups
    frames = [(rng.random((n, 2)) * 1920).astype(np.float32), grid,
              np.tile(np.float32([[12.5, 40.0]]), (n, 1)), np.float32([[5.0, 6.0]])]
    counts = [n, n, n, 1]
    st = engine.ingest(np.zeros((3 * n + 1, 128), np.uint8), np.concatenate(frames), counts)
    # pair 0: query 1 vs train 0, ratio edges at the top of the d2 range; train indices claimed once or twice
    d1 = rng.integers(dmax - 4000, dmax + 1, n)
    d0 = d1 // 4 + rng.integers(-3, 4, n)                                         # sqrt(d0) around sqrt(d1) / 2
    t_once = rng.permutation(n)
    t0 = np.where(rng.random(n) < 0.2, t_once[np.arange(n) // 2 * 2], t_once)     # ~20 % share their train with a neighbour
    p0 = (np.stack([t0, (t0 + 1) % n], 1), np.stack([d0, d1], 1))
    # pair 1: query 1 vs train 0, every query survives and claims train 7
    p1 = (np.stack([np.full(n, 7), np.full(n, 8)], 1), np.stack([np.full(n, 10), np.full(n, dmax)], 1))
    # pair 2: query 1 vs the one-row train frame 3: no second neighbour
    p2 = (np.stack([np.zeros(n, int), np.full(n, -1)], 1), np.stack([rng.integers(0, dmax, n), np.full(n, -1)], 1))
    # pair 3: query 2 (one coordinate) vs train 0: even queries fail the ratio test, odd ones survive with their own train
    ok = np.arange(n) % 2 == 1
    p3 = (np.stack([rng.permutation(n), np.zeros(n, int)], 1), np.stack([np.where(ok, 100, 5000), np.full(n, 10000)], 1))
    pairs = [(1, 0), (1, 0), (1, 3), (2, 0)]
    crafted = [p0, p1, p2, p3]
    out_off = [1 + k * (n + 2) for k in range(4)]                                 # odd rows
    rows = out_off[-1] + n + 1
    ti = np.full((rows, 2), -5, np.int32)
    td = np.full((rows, 2), -5, np.int32)
    for (idx, d2), o in zip(crafted, out_off):
        ti[o:o + n] = idx
        td[o:o + n] = d2
    surv, m_idx, m_pts, m_cnt, n_f, status = _filter_run(engine, st, pairs, ti, td, out_off, rows)
    for k, ((qf, tf), (idx, d2), o) in enumerate(zip(pairs, crafted, out_off)):
        s = matching.ratio_survivors(idx, d2.astype(np.int64))
        assert np.array_equal(surv[o:o + n].astype(bool), s), k
        m = matching.collision_filter(idx.astype(np.int32), s)
        assert n_f[k] == len(m), k
        assert status[k] == (0 if len(m) >= 4 else 1), k
        if status[k]:
            assert m_cnt[k] == 0, k
            continue
        pa, pb = frames[qf][m[:, 1]], frames[tf][m[:, 0]]
        na, nb, keep, val = matching.remove_double_matching(pa, pb)
        c = m_cnt[k]
        assert c == len(na), k
        assert np.array_equal(m_pts[o:o + c, :2], na) and np.array_equal(m_pts[o:o + c, 2:], nb), k
        assert np.array_equal(m_idx[o:o + c, 0], m[keep, 1]) and np.array_equal(m_idx[o:o + c, 1], m[val, 0]), k
    assert 0 < surv[out_off[0]:out_off[0] + n].sum() < n                         # the edge cuts both ways
    assert n_f[1] == 0 and n_f[2] == 0 and m_cnt[3] == 1 and m_idx[out_off[3], 0] == 1


def test_static_filter_at_max_kp(engine):
    """static_filter_kernel at 12 288 points per pair: displacements over all nine 2 048-bin windows, equal counts in
    different windows (the first inserted wins), the best bin in the last window, displacements of exactly 16 383,
    16 383.5 and just below, W = 0 and NaN points, and the overflow bin as the largest group.  best_r, out_cnt, flags,
    the kept points and r_out against oracle.static_filter."""
    rng = np.random.default_rng(9)
    n = MAX_KP

    def shifted(d):
        a = np.c_[rng.random(len(d)) * 1000, rng.random(len(d)) * 1000].astype(np.float32)
        return a, (a + np.c_[np.asarray(d, np.float64), np.zeros(len(d))]).astype(np.float32)

    # (0) spread over every window (the overflow bin is the ninth), bin 9 000 the largest
    d = np.r_[rng.integers(0, 16384, n - 310), np.full(300, 9000), np.full(10, 20000)][rng.permutation(n)].astype(np.float64)
    s0 = shifted(d)
    # (1) 40 points each in bins 15 000 (inserted first), 100 and 4 000; the rest spread with fewer per bin
    d = np.r_[15000, 100, 4000, np.tile([15000, 100, 4000], 39), rng.permutation(16000)[:n - 120] % 3000 + 5000]
    s1 = shifted(d.astype(np.float64))
    # (2) the best bin in the last window (from 2 000 on, windows start at 2 000 + 2 048 k), with values at exactly
    # 16 383, 16 383.5 and just below it
    d = np.r_[np.full(500, 16383.0), np.full(200, 16383.5), np.full(200, np.nextafter(np.float32(16383.5), 0)),
              np.full(10, 2000.0), rng.integers(2001, 14000, n - 910)][rng.permutation(n)]
    a, b = np.zeros((n, 2), np.float32), np.zeros((n, 2), np.float32)
    a[:, 1] = b[:, 1] = (rng.random(n) * 1000).astype(np.float32)
    b[:, 0] = d.astype(np.float32)                                                 # a.x = 0: the displacement is b.x exactly
    s2 = (a, b)
    # (3) the overflow bin (> 16 383) as the largest group
    d = np.r_[np.full(4000, 20000.0), rng.integers(0, 3, n - 4000)][rng.permutation(n)].astype(np.float64)
    s3 = shifted(d)
    # (4) W = 0 for the points at x = 1024 under h6 = -1/1024, and NaN coordinates
    a4, b4 = shifted(rng.integers(0, 5, n).astype(np.float64))
    a4[::97, 0] = 1024.0
    a4[5::211, 1] = np.nan
    b4[7::307, 0] = np.nan
    sets = [s0, s1, s2, s3, (a4, b4)]
    Hs = [np.eye(3).ravel()] * 4 + [np.array([1, 0, 0, 0, 1, 0, -1 / 1024, 0, 1], np.float64)]
    pts, off, cnt, off_h, cnt_h = _pack(sets, engine.device)
    status = torch.zeros(len(sets), dtype=torch.int32, device=engine.device)
    H = torch.from_numpy(np.array(Hs)).to(engine.device)
    out_pts, out_cnt, best_r, flags, r_out = engine.static_filter(pts, off, cnt, H, status, want_r=True, max_cnt=MAX_KP)
    torch.cuda.synchronize()
    want_best = [9000, 15000, 16383, 16384, None]
    for i, (a, b) in enumerate(sets):
        keep, br, bad = static_filter.static_points(Hs[i], a, b)
        r, _ = static_filter.displacement_bins(Hs[i], a, b)
        o = off_h[i]
        assert np.array_equal(r_out[o:o + n].cpu().numpy(), r), i
        assert int(best_r[i]) == br and int(out_cnt[i]) == len(keep) and int(flags[i]) == int(bad), i
        g = out_pts[o:o + len(keep)].cpu().numpy()
        assert np.array_equal(g[:, :2], a[keep], equal_nan=True) and np.array_equal(g[:, 2:], b[keep], equal_nan=True), i
        if want_best[i] is not None:
            assert br == want_best[i], (i, br)
    r0, _ = static_filter.displacement_bins(Hs[0], *s0)
    assert len(np.unique(r0 // 2048)) == 9
    assert int(flags[4]) == 1 and int(flags[1]) == 0 and int(out_cnt[2]) == 500


def test_concat_dedup_at_max_kp(engine):
    """concat_dedup_kernel at a total of exactly 12 288 points over EVZ_MAX_TYPES = 4 types: 2 048 keys that share one slot
    of the 16 384-slot table (load 0.75), every key present in all four types, and +-0.0 keys.  Against
    remove_double_matching over the concatenation (first position of a key, b-point of its last occurrence)."""
    rng = np.random.default_rng(10)
    n, T = MAX_KP, 4
    coll = _colliding_coords(2048, 16383)
    a0 = coll[np.r_[np.arange(2048), rng.integers(0, 2048, n - 2048)]][rng.permutation(n)]
    keys = (rng.random((n // T, 2)) * 1920).astype(np.float32)
    a1 = np.concatenate([keys[rng.permutation(n // T)] for _ in range(T)])
    z = np.float32([0.0, -0.0, 2.0])
    a2 = np.stack([rng.choice(z, n), rng.choice(z, n)], 1).astype(np.float32)
    pairs = []
    for a in (a0, a1, a2):
        b = (rng.random((n, 2)) * 1920).astype(np.float32)                        # distinct b: the last occurrence shows
        cuts = np.r_[0, np.sort(rng.choice(np.arange(1, n), T - 1, replace=False)), n]
        pairs.append([(a[cuts[t]:cuts[t + 1]], b[cuts[t]:cuts[t + 1]]) for t in range(T)])
    parts = []
    for t in range(T):
        sets = [pr[t] for pr in pairs]
        pts, off, cnt, _, _ = _pack(sets, engine.device)
        parts.append((pts, off, cnt))
    P = len(pairs)
    out_off = np.arange(P, dtype=np.int32) * (n + 4) + 1
    status = torch.zeros(P, dtype=torch.int32, device=engine.device)
    out_pts, out_cnt = engine.concat_dedup(parts, status, torch.from_numpy(out_off).to(engine.device), int(P * (n + 4) + 1), n)
    out_pts, out_cnt = out_pts.cpu().numpy(), out_cnt.cpu().numpy()
    for p, pr in enumerate(pairs):
        na, nb, _, _ = matching.remove_double_matching(np.concatenate([x for x, _ in pr]), np.concatenate([y for _, y in pr]))
        g = out_pts[out_off[p]:out_off[p] + out_cnt[p]]
        assert out_cnt[p] == len(na), p
        assert np.array_equal(g[:, :2].view(np.uint32), na.view(np.uint32)), p           # the sign of a zero key too
        assert np.array_equal(g[:, 2:], nb), p
    assert out_cnt[0] == 2048 and out_cnt[1] == n // T and out_cnt[2] == 4


def test_scratch_failure_reported_once(engine):
    """Lists in scratch for 2^31 - 1 pairs x 65 535 hypotheses (about 1 PB) cannot be allocated: the call returns
    EVZ_E_NOMEM before any launch, and the refused allocation is not reported again by PyTorch's next launch check or by
    the next evz call, which runs normally."""
    dev = engine.device
    pts = torch.zeros((64, 4), dtype=torch.float32, device=dev)
    i32 = lambda: torch.zeros(1, dtype=torch.int32, device=dev)
    off, cnt, st = i32(), i32() + 8, i32()
    H = torch.zeros((1, 9), dtype=torch.float64, device=dev)
    fh = lambda n_pairs: engine.lib.evz_find_homography(engine.h, _p(pts), _p(off), _p(cnt), n_pairs, MAX_KP, None, 65535, 0, 0, 1,
                                                         3.0, 0.0, 4, _p(st), _p(H), None, None, None, None, None, None,
                                                         engine._stream())
    assert fh(2 ** 31 - 1) == -3 and "scratch" in engine.lib.evz_last_error(engine.h).decode()
    x = torch.arange(1000, device=dev, dtype=torch.float32) * 2        # a PyTorch launch and its error check
    torch.cuda.synchronize()
    assert float(x.sum()) == 999000.0
    rng = np.random.default_rng(12)
    a, b = _mk(rng, 8, 0.0, noise=0.1)
    pts[:8, :2], pts[:8, 2:] = torch.from_numpy(a), torch.from_numpy(b)
    assert fh(1) == 0
    torch.cuda.synchronize()
    ref = ransac.find_homography_seeded(a, b, 65535, 0, 0, 1, 3.0)
    assert int(st[0]) == ref["status"] == 0
