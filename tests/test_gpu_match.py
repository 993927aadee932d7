"""K1 / K1b / K2 parity: CUDA path (through the C ABI) vs the oracle.  Needs a B200."""
import numpy as np
import pytest
import torch

from oracle import matching

pytestmark = pytest.mark.gpu


def _ragged_frames(counts, d=128, seed=0, dup_coords=False):
    rng = np.random.default_rng(seed)
    frames = []
    base = rng.integers(0, 256, (max(counts) + 8, d)).astype(np.uint8)
    for i, n in enumerate(counts):
        desc = rng.integers(0, 120, (n, d)).astype(np.uint8)
        k = min(n, len(base)) * 2 // 3                      # shared structure so that the ratio test has survivors
        if k:
            sel = rng.permutation(len(base))[:k]
            desc[:k] = np.clip(base[sel].astype(np.int32) + rng.integers(-3, 4, (k, d)), 0, 255).astype(np.uint8)
        coords = (rng.random((n, 2)) * [400, 224]).astype(np.float32)
        if dup_coords and n > 30:
            coords[10:20] = coords[0:10]
            coords[25] = coords[3]
        frames.append((coords, desc))
    return frames


def _ingest(engine, frames):
    desc = np.concatenate([f[1] for f in frames]) if frames else np.zeros((0, 128), np.uint8)
    coords = np.concatenate([f[0] for f in frames])
    return engine.ingest(desc, coords, [len(f[1]) for f in frames])


def _check_pair(engine, st, r, p, frames, qf, tf):
    o = int(st.row_off_h[qf])
    nq = len(frames[qf][1])
    idx, d2 = matching.knn_top2(frames[qf][1], frames[tf][1])
    g_idx = r.top2_idx[o:o + nq].cpu().numpy()
    g_d2 = r.top2_d2[o:o + nq].cpu().numpy().astype(np.int64)
    assert np.array_equal(g_idx, idx), f"pair {p}: top-2 indices differ"
    assert np.array_equal(g_d2, d2), f"pair {p}: squared distances differ"
    surv = matching.ratio_survivors(idx, d2)
    assert np.array_equal(r.surv[o:o + nq].cpu().numpy().astype(bool), surv), f"pair {p}: ratio survivors differ"
    mk = matching.match_kps(frames[qf][0], frames[qf][1], frames[tf][0], frames[tf][1])
    assert int(r.n_filtered[p]) == len(mk["matches"])
    assert int(r.status[p]) == mk["status"]
    m = int(r.m_cnt[p])
    assert m == len(mk["pts_a"])
    if m:
        pts = r.m_pts[o:o + m].cpu().numpy()
        assert np.array_equal(pts[:, :2], mk["pts_a"]) and np.array_equal(pts[:, 2:], mk["pts_b"])
        gi = r.m_idx[o:o + m].cpu().numpy()
        assert np.array_equal(gi[:, 0], mk["matches"][mk["keep"], 1])
        assert np.array_equal(gi[:, 1], mk["matches"][mk["val"], 0])


def test_ingest_layout(engine):
    frames = _ragged_frames([300, 1, 257, 0, 512], seed=3, dup_coords=True)
    st = _ingest(engine, frames)
    assert st.rows % 256 == 0 and (st.row_off_h % 256 == 0).all()
    desc = st.desc.cpu().numpy(); ckey = st.ckey.cpu().numpy(); canon = st.canon.cpu().numpy(); co = st.coords.cpu().numpy()
    for f, (c, d) in enumerate(frames):
        o = st.row_off_h[f]; n = len(d); e = st.row_off_h[f + 1]
        assert np.array_equal(desc[o:o + n], d)
        assert (desc[o + n:e] == 0).all() and (ckey[o + n:e] == 2 ** 31 - 1).all()
        norm = (d.astype(np.int64) ** 2).sum(1)
        assert np.array_equal(ckey[o:o + n], (norm << 8) | (np.arange(o, o + n) & 255))
        assert np.array_equal(co[o:o + n], c)
        first = {}
        exp = np.array([first.setdefault((float(x), float(y)), i) for i, (x, y) in enumerate(c)], np.int32).reshape(-1)
        assert np.array_equal(canon[o:o + n], exp)


@pytest.mark.parametrize("d,counts", [
    (128, [300, 333, 257, 1, 0, 600, 128, 129]),
    (32, [300, 2600, 257, 1, 0, 600, 2048, 129]),          # ORB width: one data K block is multiplied, several train tiles
    (64, [513, 1, 1030, 255]),                             # two data K blocks
])
def test_match_ragged_pairs(engine, d, counts):
    frames = _ragged_frames(counts, d=d, seed=1, dup_coords=True)
    st = _ingest(engine, frames)
    pq = list(range(1, len(counts)))
    pt = list(range(0, len(counts) - 1))
    r = engine.match(st, pq, pt)
    torch.cuda.synchronize()
    for p, (qf, tf) in enumerate(zip(pq, pt)):
        _check_pair(engine, st, r, p, frames, qf, tf)


def test_match_compact_output_rows_through_the_c_abi(engine):
    """include/evz.h: out_off[p] is any row of the per-row output arrays with room for n_kp[pair_q[p]] rows.  The engine
    always passes row_off[pair_q[p]] (a multiple of 256); here the pairs are packed back to back at odd offsets, the same
    query frame is listed twice, and the arrays end exactly behind the last pair (the filter kernel reads its queries four
    at a time and must not look past the pair's rows)."""
    import ctypes as C
    counts = [301, 257, 4, 7, 130, 513]
    frames = _ragged_frames(counts, seed=5, dup_coords=True)
    st = _ingest(engine, frames)
    pairs = [(1, 0), (2, 1), (3, 2), (4, 0), (5, 4), (1, 5)]
    dev = engine.device
    pq = torch.tensor([q for q, _ in pairs], dtype=torch.int32, device=dev)
    pt = torch.tensor([t for _, t in pairs], dtype=torch.int32, device=dev)
    offs, o = [], 1
    for q, _ in pairs:
        offs.append(o)
        o += counts[q]
    rows = o
    out_off = torch.tensor(offs, dtype=torch.int32, device=dev)
    P = len(pairs)
    p_ = lambda t: C.c_void_p(t.data_ptr())
    top2_idx = torch.full((rows, 2), -7, dtype=torch.int32, device=dev); top2_d2 = torch.full((rows, 2), -7, dtype=torch.int32, device=dev)
    engine._check(engine.lib.evz_match_top2(engine.h, p_(st.desc), p_(st.ckey), st.rows, p_(st.row_off), p_(st.n_kp), p_(pq), p_(pt),
                                            p_(out_off), P, p_(top2_idx), p_(top2_d2), engine._stream()))
    surv = torch.full((rows,), 9, dtype=torch.uint8, device=dev)
    m_idx = torch.empty((rows, 2), dtype=torch.int32, device=dev); m_pts = torch.empty((rows, 4), dtype=torch.float32, device=dev)
    m_cnt = torch.empty(P, dtype=torch.int32, device=dev); n_f = torch.empty(P, dtype=torch.int32, device=dev)
    status = torch.empty(P, dtype=torch.int32, device=dev)
    engine._check(engine.lib.evz_filter_matches(engine.h, p_(top2_idx), p_(top2_d2), p_(st.coords), p_(st.canon), p_(st.row_off),
                                                p_(st.n_kp), p_(pq), p_(pt), p_(out_off), P, st.max_kp, 0.5, 4, p_(surv), p_(m_idx),
                                                p_(m_pts), p_(m_cnt), p_(n_f), p_(status), engine._stream()))
    torch.cuda.synchronize()
    assert int(top2_idx[0, 0]) == -7 and int(surv[0]) == 9                      # row 0 belongs to nobody
    for p, ((qf, tf), o) in enumerate(zip(pairs, offs)):
        nq = counts[qf]
        idx, d2 = matching.knn_top2(frames[qf][1], frames[tf][1])
        assert np.array_equal(top2_idx[o:o + nq].cpu().numpy(), idx), p
        assert np.array_equal(top2_d2[o:o + nq].cpu().numpy().astype(np.int64), d2), p
        assert np.array_equal(surv[o:o + nq].cpu().numpy().astype(bool), matching.ratio_survivors(idx, d2)), p
        mk = matching.match_kps(frames[qf][0], frames[qf][1], frames[tf][0], frames[tf][1])
        assert int(n_f[p]) == len(mk["matches"]) and int(status[p]) == mk["status"], p
        m = int(m_cnt[p])
        assert m == len(mk["pts_a"]), p
        if m:
            pts = m_pts[o:o + m].cpu().numpy()
            assert np.array_equal(pts[:, :2], mk["pts_a"]) and np.array_equal(pts[:, 2:], mk["pts_b"]), p


@pytest.mark.parametrize("ratio,min_pts", [(0.8, 4), (0.3, 4), (0.5, 100000), (1.0, 1), (0.7071067811865476, 4)])
def test_match_ratio_and_minimum_parameters(engine, ratio, min_pts):
    """KeyPoints.match_kps(ratio=..., min_matching_pts=...) (matching.py:75, 113-116, 190): the f32-sqrt / f64-compare ratio
    test at other ratios (1.0 keeps a query only when its two distances differ; sqrt(1/2) puts d0^2 * 2 == d1^2 on the edge),
    and the minimum that turns a pair into NoMatchesException."""
    counts = [700, 650, 129]
    frames = _ragged_frames(counts, seed=9, dup_coords=True)
    # query row 5 of frame 1 against train rows 0 / 1 of frame 0: d^2 = 50 and 100 (exactly 2 x: the sqrt(1/2) ratio edge)
    frames[0][1][0] = 0; frames[0][1][1] = 0; frames[0][1][1][:2] = [15, 5]
    frames[1][1][5] = 0; frames[1][1][5][:2] = [5, 5]
    idx, d2 = matching.knn_top2(frames[1][1][5:6], frames[0][1])
    assert idx[0].tolist() == [0, 1] and d2[0].tolist() == [50, 100]
    st = _ingest(engine, frames)
    pairs = [(1, 0), (2, 1)]
    r = engine.match(st, [q for q, _ in pairs], [t for _, t in pairs], ratio, min_pts)
    torch.cuda.synchronize()
    for p, (qf, tf) in enumerate(pairs):
        o = int(st.row_off_h[qf]); nq = counts[qf]
        mk = matching.match_kps(frames[qf][0], frames[qf][1], frames[tf][0], frames[tf][1], ratio, min_pts)
        assert np.array_equal(r.surv[o:o + nq].cpu().numpy().astype(bool), mk["surv"]), (ratio, p)
        assert int(r.n_filtered[p]) == len(mk["matches"]) and int(r.status[p]) == mk["status"], (ratio, p)
        m = int(r.m_cnt[p])
        assert m == len(mk["pts_a"])
        if m:
            pts = r.m_pts[o:o + m].cpu().numpy()
            assert np.array_equal(pts[:, :2], mk["pts_a"]) and np.array_equal(pts[:, 2:], mk["pts_b"])
    if min_pts == 100000:
        assert int(r.status[0]) == 1 and int(r.m_cnt[0]) == 0
    if ratio == 1.0:
        assert int(r.surv[int(st.row_off_h[1]) + 5]) == 1                # 50 < 100


def test_match_golden_sets(engine, golden):
    for i in range(int(golden["knn_n"])):
        q, t = golden[f"knn{i}_q"], golden[f"knn{i}_t"]
        frames = [(np.zeros((len(t), 2), np.float32) + np.arange(len(t))[:, None].astype(np.float32), t),
                  (np.zeros((len(q), 2), np.float32) + np.arange(len(q))[:, None].astype(np.float32), q)]
        if q.shape[1] != t.shape[1]:
            continue
        st = _ingest(engine, frames)
        r = engine.match(st, [1], [0])
        nq = len(q)
        idx = r.top2_idx[st.row_off_h[1]:st.row_off_h[1] + nq].cpu().numpy()
        d2 = r.top2_d2[st.row_off_h[1]:st.row_off_h[1] + nq].cpu().numpy()
        assert np.array_equal(idx, golden[f"knn{i}_idx"]), i
        dist = np.where(idx >= 0, np.sqrt(np.maximum(d2, 0).astype(np.float32)), np.float32(-1))
        assert np.array_equal(dist, golden[f"knn{i}_dist"]), i      # == cv2 DMatch.distance bit for bit
        m = int(r.n_filtered[0])
        assert m == len(golden[f"knn{i}_lowe"]), i


def test_match_reference_pairs(engine, golden):
    """match_kps outputs of the reference itself (synthetic pairs and the bundled clip)."""
    for i in range(int(golden["mk_n"])):
        frames = [(golden[f"mk{i}_tc"], golden[f"mk{i}_td"]), (golden[f"mk{i}_qc"], golden[f"mk{i}_qd"])]
        st = _ingest(engine, frames)
        r = engine.match(st, [1], [0])
        m = int(r.m_cnt[0]); o = int(st.row_off_h[1])
        pts = r.m_pts[o:o + m].cpu().numpy()
        assert np.array_equal(pts[:, :2], golden[f"mk{i}_pts_a"]) and np.array_equal(pts[:, 2:], golden[f"mk{i}_pts_b"])
    n = int(golden["clip_n"])
    frames = [(golden[f"clip{f}_c"], golden[f"clip{f}_d"]) for f in range(n)]
    st = _ingest(engine, frames)
    r = engine.match(st, list(range(1, n)), list(range(0, n - 1)))
    for p in range(n - 1):
        m = int(r.m_cnt[p]); o = int(st.row_off_h[p + 1])
        pts = r.m_pts[o:o + m].cpu().numpy()
        assert np.array_equal(pts[:, :2], golden[f"clip{p}_pts_a"]), p
        assert np.array_equal(pts[:, 2:], golden[f"clip{p}_pts_b"]), p


def test_match_full_size_properties(engine):
    """BASELINE shape (2048 kp/frame): exactness against an independent on-device computation
    (f32 GEMM of u8 values is exact below 2^24) and size-independent properties."""
    from evenvizion_b200 import synth
    ch = synth.make_chain(9, 2048, seed=5, device="cuda")
    st = engine.ingest(ch["desc"], ch["coords"])
    r = engine.match(st, list(range(1, 9)), list(range(0, 8)))
    d = ch["desc"].float()
    for p in range(8):
        q, t = d[p + 1], d[p]
        d2 = (q * q).sum(1)[:, None] + (t * t).sum(1)[None, :] - 2 * (q @ t.T)
        key = d2.double() * 4096 + torch.arange(2048, device="cuda", dtype=torch.float64)[None, :]
        top = torch.topk(key, 2, dim=1, largest=False).values
        idx = (top % 4096).long(); val = torch.div(top, 4096, rounding_mode="floor").long()
        o = int(st.row_off_h[p + 1])
        assert torch.equal(r.top2_idx[o:o + 2048].long(), idx)
        assert torch.equal(r.top2_d2[o:o + 2048].long(), val)
    # idempotence / determinism: a second run is bit-identical
    r2 = engine.match(st, list(range(1, 9)), list(range(0, 8)))
    q0 = int(st.row_off_h[1])            # rows of frame 0 are never a query: not written
    assert torch.equal(r.top2_idx[q0:], r2.top2_idx[q0:]) and torch.equal(r.top2_d2[q0:], r2.top2_d2[q0:])
    # self-match: every descriptor's nearest neighbour in its own frame is at distance 0
    rs = engine.match(st, [3], [3])
    o = int(st.row_off_h[3])
    assert (rs.top2_d2[o:o + 2048, 0] == 0).all()


def test_match_epilogue_variants_agree(engine):
    """Default route (V-space kernel) vs the key-space kernel for every pair (EVZ_OPT_MATCH_VARIANT = 5) on tie-heavy
    data, and both against the oracle."""
    from evenvizion_b200 import synth
    ch = synth.make_chain(6, 2048, seed=8, device="cuda")
    d = ch["desc"].clone()
    d[2, 100:140] = d[2, 60:100]          # exact duplicate train rows: ties inside and across chunks
    d[3, 8:16] = d[3, 0:8]
    d[4, :] = d[4, 0:1]                   # a whole frame of identical descriptors
    st = engine.ingest(d, ch["coords"])
    outs = {}
    for v in (0, 5):
        engine.set_option(2, v)
        outs[v] = engine.match(st, list(range(1, 6)), list(range(0, 5)))
    engine.set_option(2, 0)
    q0 = int(st.row_off_h[1])
    assert torch.equal(outs[0].top2_idx[q0:], outs[5].top2_idx[q0:])
    assert torch.equal(outs[0].top2_d2[q0:], outs[5].top2_d2[q0:])
    # and both equal the oracle on the tie-heavy pairs
    dn = d.cpu().numpy()
    for p in (2, 3, 4):
        idx, d2 = matching.knn_top2(dn[p + 1], dn[p])
        o = int(st.row_off_h[p + 1])
        assert np.array_equal(outs[0].top2_idx[o:o + 2048].cpu().numpy(), idx)
        assert np.array_equal(outs[0].top2_d2[o:o + 2048].cpu().numpy().astype(np.int64), d2)


def test_match_options_reject_unknown_routes(engine):
    """EVZ_OPT_MATCH_VARIANT takes 0 or 5 only and option 5 does not exist: both are EVZ_E_ARG, and the rejected
    values leave the default route in place."""
    from evenvizion_b200 import EvzError
    for v in (1, 2, 7, 8, 9):
        with pytest.raises(EvzError):
            engine.set_option(2, v)
    with pytest.raises(EvzError):
        engine.set_option(5, 1)
    frames = _ragged_frames([300, 520], seed=4)
    st = _ingest(engine, frames)
    r = engine.match(st, [1], [0])
    torch.cuda.synchronize()
    _check_pair(engine, st, r, 0, frames, 1, 0)


def _check_launch_against_gemm(engine, st, pq, pt, counts, dd, offs):
    outs = {}
    for v in (0, 5):
        engine.set_option(2, v)
        outs[v] = [engine.match(st, pq, pt) for _ in range(2 if v == 0 else 1)]
    engine.set_option(2, 0)
    torch.cuda.synchronize()
    for p, (q, t) in enumerate(zip(pq, pt)):
        nq, nt = counts[q], counts[t]
        ro = int(st.row_off_h[q])
        if nq == 0:
            continue
        Q, T = dd[offs[q]:offs[q] + nq], dd[offs[t]:offs[t] + nt]
        if nt >= 1:
            d2 = (Q * Q).sum(1)[:, None] + (T * T).sum(1)[None, :] - 2 * (Q @ T.T)
            key = d2.double() * 4096 + torch.arange(nt, device="cuda", dtype=torch.float64)[None, :]
            k = min(2, nt)
            top = torch.topk(key, k, dim=1, largest=False).values
            idx = (top % 4096).long(); val = torch.div(top, 4096, rounding_mode="floor").long()
            if k == 1:
                idx = torch.cat([idx, torch.full_like(idx, -1)], 1); val = torch.cat([val, torch.full_like(val, -1)], 1)
        else:
            idx = torch.full((nq, 2), -1, dtype=torch.long, device="cuda"); val = idx.clone()
        for v, runs in outs.items():
            for r in runs:
                assert torch.equal(r.top2_idx[ro:ro + nq].long(), idx), (v, p, nq, nt)
                assert torch.equal(r.top2_d2[ro:ro + nq].long(), val), (v, p, nq, nt)


def test_match_ragged_stress_against_device_reference(engine):
    """Many ragged items through the persistent kernel (item ring, merge double-buffering, sentinel across
    tiles, ckey ring wrap-around): every pair against an exact f32 GEMM on the device, for both match routes
    (EVZ_OPT_MATCH_VARIANT 0 and 5), and bit-identical across repeated runs."""
    rng = np.random.default_rng(123)
    sizes = [0, 1, 2, 7, 8, 9, 127, 128, 129, 255, 256, 257, 511, 512, 513, 700, 1023, 1024, 1025, 1500, 2047, 2048, 2049, 2600]
    counts = [int(rng.choice(sizes)) for _ in range(90)]
    counts[5], counts[17] = 127, 2049
    tot = sum(counts)
    base = rng.integers(0, 256, (3000, 128)).astype(np.uint8)
    desc = np.empty((tot, 128), np.uint8)
    o = 0
    for n in counts:                          # rows drawn from a shared pool (+ small noise): near-ties and exact ties
        sel = rng.integers(0, len(base), n)
        d = base[sel].astype(np.int32) + (rng.integers(-1, 2, (n, 128)) * (rng.random((n, 1)) < 0.5))
        desc[o:o + n] = np.clip(d, 0, 255).astype(np.uint8)
        o += n
    coords = rng.random((tot, 2)).astype(np.float32)
    st = engine.ingest(desc, coords, counts)
    F = len(counts)
    dd = torch.from_numpy(desc).cuda().float()
    offs = np.r_[0, np.cumsum(counts)]
    # per-row outputs are addressed by the query frame, so one launch holds each query frame once: the chain
    # pairs first, then self-matches and non-adjacent pairs
    _check_launch_against_gemm(engine, st, list(range(1, F)), list(range(0, F - 1)), counts, dd, offs)
    _check_launch_against_gemm(engine, st, [5, 0, 17, 33, 60], [5, 40, 17, 2, 88], counts, dd, offs)


def test_match_wide_norm_range_falls_back(engine):
    """A train frame whose norm range exceeds what the fifth K block of the V-space kernel can encode
    (hmax - hmin >= 1 951 004) goes through the key-space kernel, in the same launch as ordinary pairs."""
    frames = _ragged_frames([300, 280, 310, 290, 520], seed=11)
    frames[1][1][3] = 0
    frames[1][1][7] = 255            # ||t||^2 from 0 to 8 323 200 inside frame 1
    frames[3][1][5] = 255            # wide as a query frame only... and as the train frame of pair 3
    st = _ingest(engine, frames)
    pq, pt = [1, 2, 3, 4], [0, 1, 2, 3]
    r = engine.match(st, pq, pt)
    for p, (q, t) in enumerate(zip(pq, pt)):
        _check_pair(engine, st, r, p, frames, q, t)


def test_match_largest_frames(engine):
    """Frames of EVZ_MAX_KP = 12 288 keypoints (48 tiles per item: the parity bitmap buffers of the V-space kernel
    are exactly full) next to a small frame, against an exact f32 GEMM on the device."""
    rng = np.random.default_rng(77)
    counts = [12288, 12288, 300, 4100]
    tot = sum(counts)
    base = rng.integers(0, 256, (6000, 128)).astype(np.uint8)
    sel = rng.integers(0, len(base), tot)
    desc = np.clip(base[sel].astype(np.int32) + rng.integers(-2, 3, (tot, 128)), 0, 255).astype(np.uint8)
    coords = rng.random((tot, 2)).astype(np.float32)
    st = engine.ingest(desc, coords, counts)
    dd = torch.from_numpy(desc).cuda().float()
    offs = np.r_[0, np.cumsum(counts)]
    outs = {}
    pq, pt = [1, 2, 3], [0, 1, 2]
    for v in (0, 5):
        engine.set_option(2, v)
        outs[v] = engine.match(st, pq, pt)
    engine.set_option(2, 0)
    torch.cuda.synchronize()
    for p, (q, t) in enumerate(zip(pq, pt)):
        nq, nt = counts[q], counts[t]
        ro = int(st.row_off_h[q])
        Q, T = dd[offs[q]:offs[q] + nq], dd[offs[t]:offs[t] + nt]
        d2 = (Q * Q).sum(1)[:, None] + (T * T).sum(1)[None, :] - 2 * (Q @ T.T)
        key = d2.double() * 16384 + torch.arange(nt, device="cuda", dtype=torch.float64)[None, :]
        top = torch.topk(key, 2, dim=1, largest=False).values
        idx = (top % 16384).long(); val = torch.div(top, 16384, rounding_mode="floor").long()
        for v in (0, 5):
            assert torch.equal(outs[v].top2_idx[ro:ro + nq].long(), idx), (v, p)
            assert torch.equal(outs[v].top2_d2[ro:ro + nq].long(), val), (v, p)
