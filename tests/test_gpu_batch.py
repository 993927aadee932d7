"""Many videos per call: evz_find_homography_ids, evz_chain_scan_segments, evz_chain_ref_step and
geometry_from_features_batch / get_homography_dicts against the one-video calls and, in reference mode, against a
host-loop chain.  Needs a B200."""
import ctypes as C
import os
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle import chain, pipeline

pytestmark = pytest.mark.gpu

E_ARG = -2
GRID = np.c_[np.stack(np.meshgrid(np.linspace(0, 400, 9), np.linspace(0, 224, 6)), -1).reshape(-1, 2), np.ones(54)]


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


def _fma_dot(H, S):
    """H . S with the operation order of evz_chain_ref_step, each operation rounded once (exact rationals, so the
    result does not depend on this host's BLAS)."""
    R = np.empty((3, 3))
    for i in range(3):
        for j in range(3):
            c = float(Fraction(float(H[i, 0])) * Fraction(float(S[0, j])))
            c = float(Fraction(float(H[i, 1])) * Fraction(float(S[1, j])) + Fraction(c))
            R[i, j] = float(Fraction(float(H[i, 2])) * Fraction(float(S[2, j])) + Fraction(c))
    return R


@pytest.fixture(scope="module")
def blas_is_fma_order():
    """Does this host's np.dot on 3x3 f64 round like the device chain step?  Then the reference-mode chains must match
    the host loop (`_host_reference_chain`) bit for bit; otherwise only to the tolerance of the existing tests."""
    rng = np.random.default_rng(7)
    for _ in range(300):
        H, S = rng.normal(size=(3, 3)), rng.normal(size=(3, 3)) * 100
        if not np.array_equal(np.dot(H, S), _fma_dot(H, S)):
            print("np.dot on this host does not use the fma order of evz_chain_ref_step: reference-mode H compared "
                  "within 1e-2 px instead of bit for bit")
            return False
    return True


def _chain_px(H_a, H_b):
    sa = chain.superposition_dict({k + 2: {"H": np.asarray(H).tolist()} for k, H in enumerate(H_a)})
    sb = chain.superposition_dict({k + 2: {"H": np.asarray(H).tolist()} for k, H in enumerate(H_b)})
    worst = 0.0
    for k in range(len(H_a)):
        a = GRID @ np.asarray(sa[k + 2], np.float64).T
        b = GRID @ np.asarray(sb[k + 2], np.float64).T
        worst = max(worst, np.abs(a[:, :2] / a[:, 2:] - b[:, :2] / b[:, 2:]).max())
    return worst


def _same(got, want, mode, bitwise_ref):
    (H_g, s_g), (H_w, s_w) = got, want
    assert s_g.dtype == s_w.dtype and np.array_equal(s_g, s_w)
    assert len(H_g) == len(H_w)
    if mode == "parallel" or bitwise_ref:
        assert all(np.array_equal(a, b) for a, b in zip(H_g, H_w))
    else:
        assert _chain_px(H_g, H_w) < 1e-2


def _host_reference_chain(engine, feats, policy, n_hyp, seed):
    """The reference chain of one video as a host loop (reference video_processing.py:67-105), independent of the device
    chain step: RANSAC #2 of pair k alone (sampler id k) with pre_H = the running superposition S, the None-H policy,
    then S = np.dot(H, S) / S[2][2] on the host.  The level-2 input is the driver's.  Returns (H_list, status)."""
    from evenvizion_b200 import _lib
    from evenvizion_b200.processing import video_processing as vp
    from evenvizion_b200.processing.constants import LENGTH_ACCOUNTED_POINTS, THRESHOLD_FOR_FIND_HOMOGRAPHY
    P = max(len(next(iter(feats.values()))) - 1, 0)
    if P == 0:
        return [], np.zeros(0, np.int32)
    dev = engine.device
    lay = vp.PairLayout([P], step_major=True)
    pts2, off2, cnt2, status, max_cnt = vp._level2_input(engine, [feats], lay, torch.from_numpy(lay.k).to(dev), n_hyp, seed)
    st_out = status.cpu().numpy().copy()
    H_list, S, H_prev = [], None, None
    for k in range(P):
        H = None
        if st_out[k] == 0:
            s_k = torch.zeros(1, dtype=torch.int32, device=dev)
            pre = None if S is None else torch.from_numpy(np.asarray(S, np.float64).reshape(1, 9)).to(dev)
            out = dict(H=torch.zeros((1, 9), dtype=torch.float64, device=dev), inl_cnt=torch.zeros(1, dtype=torch.int32, device=dev))
            engine.find_homography(pts2, off2[k:k + 1], cnt2[k:k + 1], s_k, max_cnt, n_hyp, seed, k, 2,
                                   THRESHOLD_FOR_FIND_HOMOGRAPHY, LENGTH_ACCOUNTED_POINTS, _lib.ST_NO_MODEL_2, pre_H=pre, out=out)
            st_out[k] = int(s_k[0])
            if st_out[k] == 0:
                H = out["H"][0].cpu().numpy().reshape(3, 3)
        if H is None:
            H = H_prev if policy else None                 # the reference reuses the previous pair's matrix (:95-96)
            if H is None:
                H = np.eye(3)                              # README.md:45: no transformation on this frame
        H_list.append(H)
        if k == 0:
            S = H
        else:
            S = np.dot(H, S)
            S = S / S[2][2]
        H_prev = H
    return H_list, st_out


# ------------------------------------------------------------------------------------------------ C ABI / engine
def _point_sets(engine, P, seed):
    rng = np.random.default_rng(seed)
    cnt = rng.integers(8, 400, P).astype(np.int32)
    cnt[:3] = (4, 5, 3)
    off = np.zeros(P, np.int32)
    off[1:] = np.cumsum(cnt + 3)[:-1]
    pts = np.zeros((int(off[-1] + cnt[-1] + 3), 4), np.float32)
    for p in range(P):
        m = int(cnt[p])
        a = rng.random((m, 2)) * [400, 224]
        H = np.eye(3) + rng.normal(size=(3, 3)) * [[2e-3, 2e-3, 2], [2e-3, 2e-3, 2], [1e-6, 1e-6, 0]]
        q = np.c_[a, np.ones(m)] @ H.T
        b = q[:, :2] / q[:, 2:] + rng.normal(size=(m, 2)) * 0.3
        out = rng.random(m) < 0.3
        b[out] = rng.random((int(out.sum()), 2)) * [400, 224]
        pts[off[p]:off[p] + m] = np.c_[a, b]
    pre = np.tile(np.eye(3).reshape(1, 9), (P, 1)) + rng.normal(size=(P, 9)) * [1e-3, 1e-3, 1, 1e-3, 1e-3, 1, 1e-7, 1e-7, 0]
    d = lambda x: torch.from_numpy(x).to(engine.device)
    return d(pts), d(off), d(cnt), d(pre), int(cnt.max())


_FH_KEYS = ("H", "mask", "inl_cnt", "best_hyp", "best_cnt", "mask_best", "H_best")


@pytest.mark.parametrize("level", [1, 2])
@pytest.mark.parametrize("with_pre", [False, True])
def test_find_homography_ids_equals_base(engine, level, with_pre):
    P, base = 40, 1234
    pts, off, cnt, pre, mx = _point_sets(engine, P, 3 + level)
    pre_H = pre if with_pre else None
    frac, fail = (0.7, 5) if level == 2 else (0.0, 4)
    st_a = torch.zeros(P, dtype=torch.int32, device=engine.device)
    st_b = st_a.clone()
    a = engine.find_homography(pts, off, cnt, st_a, mx, 256, 9, base, level, 3.0, frac, fail, pre_H=pre_H)
    ids = torch.arange(base, base + P, dtype=torch.int64, device=engine.device)
    b = engine.find_homography(pts, off, cnt, st_b, mx, 256, 9, 0, level, 3.0, frac, fail, pre_H=pre_H, pair_ids=ids)
    torch.cuda.synchronize()
    assert torch.equal(st_a, st_b) and int((st_a == 0).sum()) > P // 2
    for k in _FH_KEYS:
        assert torch.equal(a[k], b[k]), k
    # permuted and repeated ids: every pair equals a one-pair call at pair_id_base = its id
    rng = np.random.default_rng(level)
    idv = rng.permutation(np.arange(P) * 7 + 3)
    idv[5] = idv[6] = idv[7]
    st_c = torch.zeros(P, dtype=torch.int32, device=engine.device)
    c = engine.find_homography(pts, off, cnt, st_c, mx, 256, 9, 0, level, 3.0, frac, fail, pre_H=pre_H,
                               pair_ids=torch.from_numpy(idv).to(engine.device))
    for p in range(P):
        s1 = torch.zeros(1, dtype=torch.int32, device=engine.device)
        one = engine.find_homography(pts, off[p:p + 1], cnt[p:p + 1], s1, mx, 256, 9, int(idv[p]), level, 3.0, frac, fail,
                                     pre_H=None if pre_H is None else pre_H[p:p + 1])
        assert int(s1[0]) == int(st_c[p]), p
        o, m = int(off[p]), int(cnt[p])
        for k in ("H", "inl_cnt", "best_hyp", "best_cnt", "H_best"):
            assert torch.equal(one[k][0], c[k][p]), (p, k)
        for k in ("mask", "mask_best"):
            assert torch.equal(one[k][o:o + m], c[k][o:o + m]), (p, k)


def _random_steps(P, rng, fail_frac):
    G = np.tile(np.eye(3), (P, 1, 1))
    G[:, :2, :] += rng.normal(size=(P, 2, 3)) * [0.002, 0.002, 2.0]
    G[:, 2, :2] += rng.normal(size=(P, 2)) * 1e-6
    return G, rng.random(P) >= fail_frac


@pytest.mark.parametrize("policy", [True, False])
def test_chain_scan_segments_bit_identical_per_segment(engine, policy):
    rng = np.random.default_rng(11)
    lens = [0, 1, 2, 255, 256, 257, 1000, 3000, 0, 300, 257]
    seg_off = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=seg_off[1:])
    P = int(seg_off[-1])
    G, valid = _random_steps(P, rng, 0.03)
    for s in (3, 4, 5, 6, 7):                                 # failures on the first and the last pair of a segment
        valid[seg_off[s]] = False
        valid[seg_off[s + 1] - 1] = False
    valid[seg_off[9]:seg_off[10]] = False                     # a segment where every pair fails
    dev = engine.device
    Gd = torch.from_numpy(G.reshape(-1, 9)).to(dev)
    st = torch.from_numpy(np.where(valid, 0, 5).astype(np.int32)).to(dev)
    S, Hf = engine.chain_scan_segments(Gd, st, torch.from_numpy(seg_off.astype(np.int32)).to(dev), policy)
    S, Hf = S.cpu().numpy(), Hf.cpu().numpy()
    for s in range(len(lens)):
        a, b = int(seg_off[s]), int(seg_off[s + 1])
        if a == b:
            continue
        S1, Hf1, _ = engine.chain_scan(Gd[a:b], st[a:b], policy)
        assert np.array_equal(S[a:b], S1.cpu().numpy()), s
        assert np.array_equal(Hf[a:b], Hf1.cpu().numpy()), s
        ref = chain.chain_products(chain.fill_none(G[a:b], valid[a:b], policy))
        assert np.abs(S[a:b].reshape(-1, 3, 3) - ref[1:]).max() <= 1e-9 * np.abs(ref).max(), s
        assert np.abs(Hf[a:b].reshape(-1, 3, 3) - chain.fixed_plane_H(ref)).max() <= 1e-9 * np.abs(ref).max(), s


def _ref_step_host(H2, ok, sizes, policy):
    """The reference's host loop body (video_processing.py:84-105) restated per chain, with the product in the stated fma
    order."""
    out = np.empty_like(H2)
    S, Hp = [None] * sizes[0], [None] * sizes[0]
    p = 0
    for k, n in enumerate(sizes):
        for c in range(n):
            H = H2[p] if ok[p] else (Hp[c] if policy and Hp[c] is not None else np.eye(3))
            out[p] = H
            if k == 0:
                S[c] = H
            else:
                T = _fma_dot(H, S[c])
                S[c] = T / T[2][2]
            Hp[c] = H
            p += 1
    return out, S


@pytest.mark.parametrize("policy,sizes", [
    pytest.param(True, [9, 9, 7, 7, 7, 4, 2, 2, 1, 1, 1, 1], id="True"),
    pytest.param(False, [9, 9, 7, 7, 7, 4, 2, 2, 1, 1, 1, 1], id="False"),
    pytest.param(True, [1000, 1000, 999, 700, 257, 256, 1], id="1000-chains-True"),      # four CTAs
    pytest.param(False, [1000, 1000, 999, 700, 257, 256, 1], id="1000-chains-False"),
])
def test_chain_ref_step_against_host_loop(engine, policy, sizes):
    rng = np.random.default_rng(5)
    P = sum(sizes)
    H2, ok = _random_steps(P, rng, 0.15)
    ok[:2] = False                                             # first pairs that fail: identity
    ok[9:18] = False                                           # a whole step fails
    dev = engine.device
    H2d = torch.from_numpy(H2.reshape(-1, 9)).to(dev)
    st = torch.from_numpy(np.where(ok, 0, 6).astype(np.int32)).to(dev)
    H_out = torch.full((P, 9), np.nan, dtype=torch.float64, device=dev)
    S_state = torch.full((sizes[0], 9), np.nan, dtype=torch.float64, device=dev)
    a, prev = 0, None
    for k, n in enumerate(sizes):
        engine.chain_ref_step(H2d[a:a + n], st[a:a + n], k == 0, policy, S_state, None if prev is None else H_out[prev:prev + n],
                              H_out[a:a + n])
        prev, a = a, a + n
    want_H, want_S = _ref_step_host(H2, ok, sizes, policy)
    assert np.array_equal(H_out.cpu().numpy().reshape(-1, 3, 3), want_H)
    got_S = S_state.cpu().numpy().reshape(-1, 3, 3)
    for c in range(sizes[0]):
        assert np.array_equal(got_S[c], want_S[c]), c


def test_new_entry_points_error_codes(engine):
    lib, h, s, dev = engine.lib, engine.h, engine._stream(), engine.device
    p_ = lambda t: C.c_void_p(t.data_ptr())
    i32 = lambda n: torch.zeros(n, dtype=torch.int32, device=dev)
    f64 = lambda n: torch.zeros((n, 9), dtype=torch.float64, device=dev)
    pts = torch.zeros((64, 4), dtype=torch.float32, device=dev)
    ids = torch.zeros(1, dtype=torch.int64, device=dev)
    fh = lambda pid, n: lib.evz_find_homography_ids(h, p_(pts), p_(i32(1)), p_(i32(1) + 8), n, 16, None, 64, 0, pid, 1, 3.0, 0.0,
                                                     4, p_(i32(1)), p_(f64(1)), None, None, None, None, None, None, s)
    assert fh(None, 1) == E_ARG and "null" in lib.evz_last_error(h).decode()
    assert fh(p_(ids), 0) == 0
    G, st, so = f64(4), i32(4), torch.tensor([0, 4], dtype=torch.int32, device=dev)
    S = f64(4).fill_(7.0)
    assert lib.evz_chain_scan_segments(h, p_(G), p_(st), 4, None, 1, 1, p_(S), None, s) == E_ARG
    assert lib.evz_chain_scan_segments(h, p_(G), p_(st), 4, p_(so), 1, 1, None, None, s) == E_ARG
    assert lib.evz_chain_scan_segments(h, p_(G), p_(st), 0, p_(so), 1, 1, p_(S), None, s) == 0
    assert lib.evz_chain_ref_step(h, None, p_(st), 4, 1, 1, p_(S), None, p_(G), s) == E_ARG
    assert lib.evz_chain_ref_step(h, p_(G), p_(st), 4, 0, 1, p_(S), None, p_(G), s) == E_ARG      # H_prev needed
    assert lib.evz_chain_ref_step(h, p_(G), p_(st), 0, 1, 1, p_(S), None, p_(G), s) == 0
    torch.cuda.synchronize()
    assert bool((S == 7.0).all())                             # the no-ops wrote nothing
    r = engine.match(engine.ingest(np.zeros((8, 128), np.uint8), np.zeros((8, 2), np.float32), [4, 4]), [1], [0])
    torch.cuda.synchronize()
    assert int(r.status[0]) in (0, 1)


def test_reference_loop_does_not_synchronise(engine):
    pts, off, cnt, pre, mx = _point_sets(engine, 21, 9)
    status = torch.zeros(21, dtype=torch.int32, device=engine.device)
    step_off = [0, 6, 12, 16, 19, 21]
    torch.cuda.synchronize()
    engine.reference_chains(pts, off, cnt, status, mx, step_off, 128, 1)          # grows the handle's scratch once
    status.zero_()
    torch.cuda.set_sync_debug_mode("error")
    try:
        H = engine.reference_chains(pts, off, cnt, status, mx, step_off, 128, 1)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(H).all())


# ------------------------------------------------------------------------------------------------ public API
SPLITS = [(0, 1), (0, 2), (0, 40), (35, 121), (60, 121), (0, 121)]
_oracle_cache = {}


def _oracle(clip, types, f0, f1, policy):
    key = (types, f0, f1, policy)
    if key not in _oracle_cache:
        _oracle_cache[key] = pipeline.video_chain_multi(_clip_feats(clip, types, f0, f1), n_hyp=1024, seed=0,
                                                        none_h_processing=policy, reference_exact=True)
    return _oracle_cache[key]


@pytest.mark.parametrize("types", [("SIFT", "ORB"), ("SIFT",)])
def test_batch_parallel_bit_identical_to_single(proc, clip, types):
    feats = [_clip_feats(clip, types, a, b) for a, b in SPLITS]
    for policy in (True, False):
        got = proc.geometry_from_features_batch(feats, policy, "parallel", n_hyp=1024, seed=0)
        assert len(got) == len(SPLITS)
        for f, g in zip(feats, got):
            _same(g, proc.geometry_from_features(f, policy, "parallel", n_hyp=1024, seed=0), "parallel", True)


@pytest.mark.parametrize("types", [("SIFT", "ORB"), ("SIFT",)])
@pytest.mark.parametrize("policy", [True, False])
def test_batch_reference_matches_single_and_oracle(engine, proc, clip, types, policy, blas_is_fma_order):
    feats = [_clip_feats(clip, types, a, b) for a, b in SPLITS]
    got = proc.geometry_from_features_batch(feats, policy, "reference", n_hyp=1024, seed=0)
    for (a, b), f, g in zip(SPLITS, feats, got):
        single = proc.geometry_from_features(f, policy, "reference", n_hyp=1024, seed=0)
        _same(g, single, "reference", True)                   # a batch of one: batching changes nothing
        _same(g, _host_reference_chain(engine, f, policy, 1024, 0), "reference", blas_is_fma_order)
        if b - a < 2:
            continue
        ref = _oracle(clip, types, a, b, policy)
        assert np.array_equal(g[1], ref["status"])
        sup = chain.superposition_dict({k + 2: {"H": np.asarray(H).tolist()} for k, H in enumerate(g[0])})
        for k in range(b - a - 1):
            x = GRID @ np.asarray(sup[k + 2], np.float64).T
            y = GRID @ ref["S"][k + 1].T
            assert np.abs(x[:, :2] / x[:, 2:] - y[:, :2] / y[:, 2:]).max() < 1e-2, (a, b, k)


@pytest.mark.parametrize("mode", ["parallel", "reference"])
def test_batch_duplicates_and_order(proc, clip, mode):
    v = [_clip_feats(clip, ("SIFT", "ORB"), a, b) for a, b in [(0, 30), (50, 61), (70, 72)]]
    one = proc.geometry_from_features_batch([v[0], v[1], v[0], v[2]], True, mode, n_hyp=1024, seed=0)
    two = proc.geometry_from_features_batch([v[2], v[0], v[1]], True, mode, n_hyp=1024, seed=0)
    for (x, y) in [(one[0], one[2]), (one[0], two[1]), (one[1], two[2]), (one[3], two[0])]:
        _same(x, y, "parallel", True)                          # same video, same bits, wherever it sits in the batch


def _synth_feats(n_frames, n_kp, seed, unmatched_frac=0.0):
    from evenvizion_b200 import synth
    ch = synth.make_chain(n_frames, n_kp, seed=seed, device="cuda", unmatched_frac=unmatched_frac)
    d, c = ch["desc"].cpu().numpy(), ch["coords"].cpu().numpy()
    return {"SIFT": [(c[f], d[f]) for f in range(n_frames)]}


@pytest.mark.parametrize("mode", ["parallel", "reference"])
def test_batch_failures_stay_inside_their_video(engine, proc, clip, mode, blas_is_fma_order):
    a = _clip_feats(clip, ("SIFT", "ORB"), 0, 12)
    a["ORB"][5] = (a["ORB"][5][0], None)                      # a frame without descriptors
    b = _synth_feats(25, 600, 3, unmatched_frac=0.3)          # pairs without any correspondence
    c = _clip_feats(clip, ("SIFT", "ORB"), 20, 30)
    for t in c:                                               # the first pair fails: frame 0 is unrelated to frame 1
        c[t][0] = a[t][0] if t == "SIFT" else (a[t][0][0], None)
    b2 = {"SIFT": b["SIFT"]}
    for policy in (True, False):
        got = proc.geometry_from_features_batch([a, c, a], policy, mode, n_hyp=512, seed=2)
        gb = proc.geometry_from_features_batch([b2, b2], policy, mode, n_hyp=512, seed=2)
        for f, g in [(a, got[0]), (c, got[1]), (a, got[2]), (b2, gb[0])]:
            single = proc.geometry_from_features(f, policy, mode, n_hyp=512, seed=2)
            _same(g, single, mode, True)
            if mode == "reference":
                _same(g, _host_reference_chain(engine, f, policy, 512, 2), mode, blas_is_fma_order)
        assert got[1][1][0] != 0 and (gb[0][1] != 0).any()
        assert np.array_equal(got[1][0][0], np.eye(3))         # a failed first pair is an identity step


@pytest.mark.parametrize("mode", ["parallel", "reference"])
def test_batch_scale_64_videos(engine, proc, mode, blas_is_fma_order):
    from evenvizion_b200 import synth
    ch = synth.make_chain(64 * 30, 2048, seed=21, device="cuda", unmatched_frac=0.02)
    d, c = ch["desc"].cpu().numpy(), ch["coords"].cpu().numpy()
    feats = [{"SIFT": [(c[f], d[f]) for f in range(30 * v, 30 * v + 30)]} for v in range(64)]
    got = proc.geometry_from_features_batch(feats, True, mode, n_hyp=256, seed=4)
    assert len(got) == 64 and all(len(g[0]) == 29 for g in got)
    for v in (0, 17, 40, 63):
        _same(got[v], proc.geometry_from_features(feats[v], True, mode, n_hyp=256, seed=4), mode, True)
        if mode == "reference":
            _same(got[v], _host_reference_chain(engine, feats[v], True, 256, 4), mode, blas_is_fma_order)


class _FakeCapture:
    def __init__(self, frames):
        self.frames, self.i = frames, 0

    def read(self):
        if self.i >= len(self.frames):
            return False, None
        self.i += 1
        return True, self.frames[self.i - 1].copy()


def test_get_homography_dicts_equals_per_capture(engine, proc, clip, blas_is_fma_order):
    pytest.importorskip("cv2")
    fr = [[clip[f"frame{f}"] for f in range(6)], [clip[f"frame{f}"] for f in range(2, 5)]]
    got = proc.get_homography_dicts([_FakeCapture(x) for x in fr], n_hyp=1024, seed=0)
    assert len(got) == 2
    for x, g in zip(fr, got):
        want = proc.get_homography_dict(_FakeCapture(x), n_hyp=1024, seed=0)
        assert list(g) == list(want) and g["resize_info"] == want["resize_info"]
        Hg = [g[k]["H"] for k in g if k != "resize_info"]
        assert Hg == [want[k]["H"] for k in want if k != "resize_info"]
        feats, _ = proc.read_and_describe(_FakeCapture(x))
        Hh = [np.asarray(H, np.float64).tolist() for H in _host_reference_chain(engine, feats, True, 1024, 0)[0]]
        if blas_is_fma_order:
            assert Hg == Hh
        else:
            assert _chain_px(Hg, Hh) < 1e-2
