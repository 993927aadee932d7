"""K6 scan (evz_chain_scan, evz_chain_scan_segments, evz_chain_seed_apply, evz_chain_ref_step) and K7 (evz_remap,
evz_max_movement) at BASELINE config-5 lengths, against the extended-precision references of oracle/chain.py: the long
double fold, the exact remap and the exact corner maximum.  Needs a B200."""
import numpy as np
import pytest
import torch

from oracle import chain

pytestmark = pytest.mark.gpu

# pixel error of a 3x3 matrix: its action on a 9 x 6 grid over a 400 x 224 frame, evaluated in long double
GRID = np.c_[np.stack(np.meshgrid(np.linspace(0, 400, 9), np.linspace(0, 224, 6)), -1).reshape(-1, 2),
             np.ones(54)].astype(np.longdouble)
# Threshold of the scan against the long double fold, for S and H_fixed at every pair (see test_long_chain).
PX_TOL = 1e-7
SX, SY = 400 / 1170, 224 / 658             # the bundled clip's resize: 1170 x 658 -> 400 x 224


def _px(A, B):
    """max over matrices and grid points of the pixel distance between A and B (both [..., 9] or [..., 3, 3])"""
    A = np.asarray(A).reshape(-1, 3, 3)
    B = np.asarray(B).reshape(-1, 3, 3)
    worst = 0.0
    for i in range(0, len(A), 20000):
        a = A[i:i + 20000].astype(np.longdouble) @ GRID.T
        b = B[i:i + 20000].astype(np.longdouble) @ GRID.T
        worst = max(worst, float(np.abs(a[:, :2] / a[:, 2:] - b[:, :2] / b[:, 2:]).max()))
    return worst


def _steps(P, seed):
    """frame-plane steps as scripts/bench_chain.py: translation sigma 2 px, rotation 1e-3, perspective 1e-7"""
    rng = np.random.default_rng(seed)
    G = np.tile(np.eye(3), (P, 1, 1))
    G[:, 0, 2] = rng.normal(0, 2, P); G[:, 1, 2] = rng.normal(0, 2, P)
    G[:, 0, 1] = rng.normal(0, 1e-3, P); G[:, 1, 0] = -G[:, 0, 1]; G[:, 2, 0] = rng.normal(0, 1e-7, P)
    return G


def _failures(P, seed):
    rng = np.random.default_rng(seed)
    valid = rng.random(P) >= 0.02
    valid[:300] = False                                  # a leading run longer than one 256-pair block
    for a in (254, 510, 65533, 65789):                   # runs across 256-pair block boundaries and across pair 65 536,
        valid[a:a + 4] = False                           # where prod_carry_kernel's second chunk of 256 blocks starts
    valid[1024:1280] = False                             # a whole block
    valid[-1] = False
    return valid


def _dev(engine, x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(engine.device)


def _status(valid):
    return np.where(valid, 0, 5).astype(np.int32)


_cache = {}


def _long(engine, P, policy):
    """(G, valid, long double S [P+1] and H_fixed [P], device S and H_fixed [P,9]) of the P-pair test chain"""
    key = (P, policy)
    if key not in _cache:
        G, valid = _steps(P, P), _failures(P, P + 1)
        ref = chain.chain_products(chain.fill_none(G, valid, policy), np.longdouble)
        S, Hf, _ = engine.chain_scan(_dev(engine, G.reshape(-1, 9)), _dev(engine, _status(valid)), policy)
        _cache[key] = (G, valid, ref, chain.fixed_plane_H(ref), S.cpu().numpy(), Hf.cpu().numpy())
    return _cache[key]


# ------------------------------------------------------------------------------------------------ K6 scan
@pytest.mark.parametrize("policy", [True, False])
@pytest.mark.parametrize("P", [65535, 65536, 65537, 100000])
def test_long_chain(engine, P, policy):
    """One chain of up to 100 000 pairs (config 5), across prod_carry_kernel's 65 536-pair chunk hand-off, against the
    long double fold, S and H_fixed at every pair.

    Threshold 1e-7 px.  The scan associates the products differently from the fold, so it is not bit-exact.  An f64
    NumPy emulation of the kernels' order (Hillis-Steele in the warp, warps combined serially, block totals scanned in
    256-wide chunks, (a0 b0 + a1 b3) + a2 b6 with the power-of-two rescale) on these inputs is at most 3.3e-11 px from
    the long double fold for S and 5.1e-12 px for H_fixed; the same emulation with f32 intermediates is at least
    2.4e-2 px off for S and 8.1e-4 px for H_fixed.  1e-7 px is 3 000x above the first and 8 000x below the second."""
    G, valid, ref, Href, S, Hf = _long(engine, P, policy)
    assert np.isfinite(S).all() and np.isfinite(Hf).all()
    es, eh = _px(S, ref[1:]), _px(Hf, Href)
    print(f"scan P={P} policy={policy}: worst {es:.3g} px (S), {eh:.3g} px (H_fixed)")
    assert es < PX_TOL and eh < PX_TOL


@pytest.mark.parametrize("policy", [True, False])
@pytest.mark.parametrize("n_segs", [257, 600])
def test_segments_past_256_segments_and_256_blocks(engine, n_segs, policy):
    """More than 256 segments (seg_blocks_kernel's chunk loop), empty segments at 0, 255, 256 and last, and one segment
    of 70 000 pairs (more than 256 blocks in one segment's prod_carry_kernel): every segment against the long double
    fold and bit-identical to evz_chain_scan on that segment alone."""
    rng = np.random.default_rng(n_segs)
    lens = rng.integers(1, 300, n_segs)
    lens[[0, 255, 256, n_segs - 1]] = 0
    lens[100] = 70000
    seg_off = np.zeros(n_segs + 1, np.int64)
    np.cumsum(lens, out=seg_off[1:])
    P = int(seg_off[-1])
    G = _steps(P, n_segs + 7)
    valid = rng.random(P) >= 0.03
    for s in range(1, n_segs, 5):
        if lens[s]:
            valid[seg_off[s]] = False                    # the first pair of a segment fails
    valid[seg_off[100]:seg_off[100] + 300] = False
    Gd, st = _dev(engine, G.reshape(-1, 9)), _dev(engine, _status(valid))
    S, Hf = engine.chain_scan_segments(Gd, st, _dev(engine, seg_off.astype(np.int32)), policy)
    S, Hf = S.cpu().numpy(), Hf.cpu().numpy()
    ref_S, ref_H = np.empty((P, 3, 3), np.longdouble), np.empty((P, 3, 3), np.longdouble)
    for s in range(n_segs):
        a, b = int(seg_off[s]), int(seg_off[s + 1])
        if a == b:
            continue
        r = chain.chain_products(chain.fill_none(G[a:b], valid[a:b], policy), np.longdouble)
        ref_S[a:b], ref_H[a:b] = r[1:], chain.fixed_plane_H(r)
        S1, Hf1, _ = engine.chain_scan(Gd[a:b], st[a:b], policy)
        assert np.array_equal(S[a:b], S1.cpu().numpy()), s
        assert np.array_equal(Hf[a:b], Hf1.cpu().numpy()), s
    es, eh = _px(S, ref_S), _px(Hf, ref_H)
    print(f"segments n_segs={n_segs} policy={policy}: worst {es:.3g} px (S), {eh:.3g} px (H_fixed)")
    assert es < PX_TOL and eh < PX_TOL


@pytest.mark.parametrize("policy", [True, False])
def test_seeded_shards_at_length(engine, policy):
    """A 100 000-pair chain cut into shards at 0, 65 536, 65 537 and 80 000, where the shard at 80 000 starts with 300
    failing pairs (seed_kernel writes more than one block of leading rows), seeded on the host (seeds_from_summaries ->
    seeded evz_chain_scan) and on the device (evz_chain_seed_apply): S and H_fixed of every shard against the long
    double fold of the whole chain."""
    from evenvizion_b200.distributed import seeds_from_summaries
    P = 100000
    G, valid = _steps(P, 5), _failures(P, 6)
    valid[80000:80300] = False
    ref = chain.chain_products(chain.fill_none(G, valid, policy), np.longdouble)
    Href = chain.fixed_plane_H(ref)
    Gd, st = _dev(engine, G.reshape(-1, 9)), _dev(engine, _status(valid))
    bounds = [0, 65536, 65537, 80000, P]
    shards = list(zip(bounds[:-1], bounds[1:]))
    locals_, sums = [], []
    for a, b in shards:
        Sl, _, sm = engine.chain_scan(Gd[a:b], st[a:b], policy, want_fixed=False, want_summary=True)
        locals_.append(Sl); sums.append(sm)
    summaries = [s.cpu().numpy() for s in sums]
    assert int(round(summaries[3][18])) == 300
    gathered = torch.stack(sums)
    worst = 0.0
    for r, (a, b) in enumerate(shards):
        seed_S, seed_G = seeds_from_summaries(summaries, r, policy)
        Sh, Hh, _ = engine.chain_scan(Gd[a:b], st[a:b], policy, seed_S=_dev(engine, seed_S.reshape(9)),
                                      seed_G=None if seed_G is None else _dev(engine, seed_G.reshape(9)))
        Sd, Hd, _ = engine.chain_seed_apply(gathered, r, locals_[r], policy)
        for S_, H_ in ((Sh, Hh), (Sd, Hd)):
            es, eh = _px(S_.cpu().numpy(), ref[a + 1:b + 1]), _px(H_.cpu().numpy(), Href[a:b])
            worst = max(worst, es, eh)
            assert es < PX_TOL and eh < PX_TOL, (r, es, eh)
    print(f"seeded shards policy={policy}: worst {worst:.3g} px")


def _pow2_scale(rng, n):
    return (rng.choice([-1.0, 1.0], n) * np.ldexp(1.0, rng.integers(-200, 201, n)))[:, None, None]


@pytest.mark.parametrize("policy", [True, False])
def test_power_of_two_scaling_keeps_the_bits(engine, policy):
    """A homography is defined up to scale.  The scan's products are exact under a power-of-two scale and a sign, and
    only stored matrices are divided, so scaling every step G_k by its own +-2^e_k (|e_k| <= 200) must leave S and H_fixed
    bit for bit unchanged (np.array_equal: +0 == -0); so must it for evz_chain_scan_segments, and for S_state of
    evz_chain_ref_step after its first step."""
    rng = np.random.default_rng(8)
    P = 100000
    G, valid = _steps(P, 9), _failures(P, 10)
    Gs = G * _pow2_scale(rng, P)
    st = _dev(engine, _status(valid))
    a = engine.chain_scan(_dev(engine, G.reshape(-1, 9)), st, policy)
    b = engine.chain_scan(_dev(engine, Gs.reshape(-1, 9)), st, policy)
    assert np.array_equal(a[0].cpu().numpy(), b[0].cpu().numpy())
    assert np.array_equal(a[1].cpu().numpy(), b[1].cpu().numpy())
    seg_off = _dev(engine, np.array([0, 0, 300, 70300, 70301, 70557, 70814, P], np.int32))
    a = engine.chain_scan_segments(_dev(engine, G.reshape(-1, 9)), st, seg_off, policy)
    b = engine.chain_scan_segments(_dev(engine, Gs.reshape(-1, 9)), st, seg_off, policy)
    assert np.array_equal(a[0].cpu().numpy(), b[0].cpu().numpy())
    assert np.array_equal(a[1].cpu().numpy(), b[1].cpu().numpy())
    # the reference-exact chain step: 300 chains, 6 steps
    n, K = 300, 6
    H2 = _steps(n * K, 11)
    ok = rng.random(n * K) >= 0.15
    H2s = H2 * _pow2_scale(rng, n * K)
    runs = []
    for H in (H2, H2s):
        Hd, std = _dev(engine, H.reshape(-1, 9)), _dev(engine, _status(ok))
        S_state = torch.full((n, 9), np.nan, dtype=torch.float64, device=engine.device)
        H_out = torch.full((n * K, 9), np.nan, dtype=torch.float64, device=engine.device)
        states = []
        for k in range(K):
            sl = slice(k * n, (k + 1) * n)
            engine.chain_ref_step(Hd[sl], std[sl], k == 0, policy, S_state,
                                  None if k == 0 else H_out[(k - 1) * n:k * n], H_out[sl])
            states.append(S_state.cpu().numpy().copy())
        runs.append(states)
    for k in range(1, K):
        assert np.isfinite(runs[0][k]).all() and np.array_equal(runs[0][k], runs[1][k]), k


_A = np.array([[1.0, 0, 0], [0, 1, 0], [-2.0 ** -10, 0, 1]])
_B = np.array([[1.0, 0, 1024], [0, 1, 0], [0, 0, 1]])          # (A . B)[2][2] == 0 exactly
_E = np.array([[1.0, 0, 0], [0, 1, 0], [2.0 ** -12, 0, 1]])     # (E . A . B)[2][2] == 0.25


@pytest.mark.parametrize("e,a,b", [
    (1000, 2050, 2051),                                          # A . B formed by the first shuffle (lanes 2j, 2j + 1)
    (1800, 2085, 2100),                                          # ... as a warp total (warp 1 of block 8)
    (1800, 2088, 2248),                                          # ... as a 256-pair block total (block 8)
    (1000, 258 * 256 + 100, 259 * 256 + 50),                     # ... as a product of two block totals in the second
], ids=["first-shuffle", "warp-total", "block-total", "chunk-scan"])   # 65 536-pair chunk of prod_carry_kernel
def test_partial_product_with_zero_22(engine, e, a, b):
    """A partial product of the tree whose [2][2] is exactly 0 while every true prefix is well defined: E before A
    and B makes the prefix's [2][2] 0.25.  The tree divides only stored matrices, so every S must be finite and equal
    the long double fold (relative 1e-12: every product here is exact)."""
    P = 70000
    G = np.tile(np.eye(3), (P, 1, 1))
    G[e], G[a], G[b] = _E, _A, _B
    assert (_A @ _B)[2, 2] == 0 and (_E @ _A @ _B)[2, 2] == 0.25
    ref = chain.chain_products(G, np.longdouble)
    for policy in (True, False):
        S, Hf, _ = engine.chain_scan(_dev(engine, G.reshape(-1, 9)), _dev(engine, np.zeros(P, np.int32)), policy)
        S, Hf = S.cpu().numpy().reshape(-1, 3, 3), Hf.cpu().numpy().reshape(-1, 3, 3)
        assert np.isfinite(S).all() and np.isfinite(Hf).all()
        assert float(np.abs(S - ref[1:]).max()) <= 1e-12 * float(np.abs(ref).max())
        Href = chain.fixed_plane_H(ref)
        assert float(np.abs(Hf - Href).max()) <= 1e-12 * float(np.abs(Href).max())


# ------------------------------------------------------------------------------------------------ K7 remap
def test_remap_bundled_exact(engine, bundled):
    """Every one of the 3 664 bundled output coordinates (fixed_coordinates, and back_to_original from them) equals the
    exact remap; none lies in the tie window."""
    sup = {int(k): np.asarray(v, np.float64) for k, v in bundled["superposition"].items()}
    keys = sorted(sup)
    S = np.array([sup[k] for k in keys])
    pts, fidx, fixed, back = [], [], [], []
    for k, rects in bundled["original_coordinates"].items():
        for r, e, bk in zip(rects, bundled["fixed_coordinates"][k], bundled["back_to_original"][k]):
            pts.append([r["x1"], r["y1"]]); fidx.append(keys.index(int(k)))
            fixed.append([e["x1"], e["y1"]]); back.append([bk["x1"], bk["y1"]])
    pts, fidx = np.array(pts), np.array(fidx, np.int32)
    oh, ow = bundled["original_shape"]; ri = bundled["resize_info"]
    sx, sy = int(ri["w"]) / ow, int(ri["h"]) / oh
    Sd, Fi = _dev(engine, S.reshape(-1, 9)), _dev(engine, fidx)
    out = engine.remap(_dev(engine, pts), Fi, Sd, sx, sy, False).cpu().numpy()
    want, tie = chain.remap_exact(pts, fidx, S, sx, sy, False, exact=True)
    assert not tie.any() and np.array_equal(want, np.array(fixed)) and np.array_equal(out, want)
    out2 = engine.remap(_dev(engine, out), Fi, Sd, ow / ri["w"], oh / ri["h"], True).cpu().numpy()
    want2, tie2 = chain.remap_exact(out, fidx, S, ow / ri["w"], oh / ri["h"], True, exact=True)
    assert not tie2.any() and np.array_equal(want2, np.array(back)) and np.array_equal(out2, want2)


def _near_half_cent(S, fidx, rng, n):
    """n points whose forward transform lands within ~1e-13 of a half-cent in x (x solved in long double)"""
    pts = rng.random((n, 2)) * [1170, 658]
    for i in range(n):
        T = S[fidx[i]].reshape(3, 3).astype(np.longdouble)
        y = np.longdouble(np.float64(SY) * pts[i, 1])
        t = (np.floor(np.longdouble(rng.random() * 40000)) + np.longdouble(0.5)) / 100
        x = (t * (T[2, 1] * y + T[2, 2]) - T[0, 1] * y - T[0, 2]) / (T[0, 0] - t * T[2, 0])
        pts[i, 0] = float(x / np.longdouble(SX))
    return pts


def test_remap_config5_against_exact(engine):
    """Config 5: 8 points per frame over the 100 001 frames of the 100 000-pair chain (S from test_long_chain's scan), in
    both directions, with the bundled clip's resize.  Every output outside the tie window (100 e within 1e-6 of a
    half-integer, where the f64 evaluation order may decide the rounding) equals the long double reference, and the
    window holds fewer than 1e-4 of the points.  A sample of 2 000 points is checked against the Fraction-exact remap,
    100 of them built to land on a half-cent: the window flags those, and the kernel rounds them to either neighbour."""
    _, _, _, _, S, _ = _long(engine, 100000, True)
    Sall = np.concatenate([np.eye(3).reshape(1, 9), S])
    F = len(Sall)
    rng = np.random.default_rng(12)
    fidx = np.repeat(np.arange(F, dtype=np.int32), 8)
    pts = rng.random((len(fidx), 2)) * [1170, 658]
    Sd, Fi = _dev(engine, Sall), _dev(engine, fidx)
    fwd = engine.remap(_dev(engine, pts), Fi, Sd, SX, SY, False).cpu().numpy()
    back = engine.remap(_dev(engine, fwd), Fi, Sd, 1 / SX, 1 / SY, True).cpu().numpy()
    sample = rng.choice(len(fidx), 950, replace=False)
    # the chain's 300 leading failures make frames 0 .. 300 exact identities; there a two-decimal input times 1170 / 400
    # (or 658 / 224) lies on a half-cent for about one value in 40: true ties, left out of the window's share
    generic = ~np.all(Sall == np.eye(3).reshape(9), axis=1)[fidx]
    for inp, out, inv, scl in ((pts, fwd, False, (SX, SY)), (fwd, back, True, (1 / SX, 1 / SY))):
        want, tie = chain.remap_exact(inp, fidx, Sall, *scl, inv)
        print(f"remap inverse={inv}: {int(tie.sum())} of {len(tie)} points in the tie window, "
              f"{int((tie & generic).sum())} of {int(generic.sum())} outside the identity frames")
        assert (tie & generic).sum() < 1e-4 * generic.sum()
        assert np.array_equal(out[~tie], want[~tie])
        assert np.abs(out[tie] - want[tie]).max(initial=0.0) <= 0.0100001
        ex, tie_ex = chain.remap_exact(inp[sample], fidx[sample], Sall, *scl, inv, exact=True)
        assert np.array_equal(tie_ex, tie[sample]) and np.array_equal(ex[~tie_ex], out[sample][~tie_ex])
    bf = rng.integers(0, F, 100).astype(np.int32)
    bp = _near_half_cent(Sall, bf, rng, 100)
    got = engine.remap(_dev(engine, bp), _dev(engine, bf), Sd, SX, SY, False).cpu().numpy()
    want, tie = chain.remap_exact(bp, bf, Sall, SX, SY, False, exact=True)
    assert tie.all()
    # x: one of the two cents around the half-cent; y was not built and is decided
    assert np.abs(got[:, 0] - want[:, 0]).max() <= 0.0100001 and np.array_equal(got[:, 1], want[:, 1])
    print(f"remap: {int((got[:, 0] != want[:, 0]).sum())} of 100 points built on a half-cent rounded the other way")


# ------------------------------------------------------------------------------------------------ K7 max-movement
def _max_movement_host(S, n_frames, h, w):
    """evz_max_movement in the kernel's operation order, in f64 (the kernel is built with --fmad=false and divides
    with IEEE f64 '/'), so the result must be bit-identical"""
    S = np.asarray(S, np.float64).reshape(-1, 9)
    i = np.arange(h * w)
    x, y = (i % w).astype(np.float64), (i // w).astype(np.float64)
    best = -np.inf
    for f in range(n_frames):
        T = S[f]
        X = (T[0] * x + T[1] * y) + T[2]
        Y = (T[3] * x + T[4] * y) + T[5]
        W = (T[6] * x + T[7] * y) + T[8]
        best = np.fmax(best, np.fmax.reduce(np.fmax(X / W, Y / W)))
    return float(best)


@pytest.mark.parametrize("h,w", [(1, 1), (1, 37), (29, 1), (45, 61), (400, 400)])
def test_max_movement_bits_small_grids(engine, h, w):
    """1 x 1, one row, one column, H.W not a multiple of 2 048, and H.W > 64 . 2 048 so the grid-stride loop wraps."""
    rng = np.random.default_rng(h * 1000 + w)
    F = 5
    S = np.tile(np.eye(3), (F, 1, 1)) + rng.normal(size=(F, 3, 3)) * [[2e-2, 2e-2, 30], [2e-2, 2e-2, 30], [1e-4, 1e-4, 0]]
    got = float(engine.max_movement(_dev(engine, S.reshape(-1, 9)), F, h, w).item())
    assert got == _max_movement_host(S, F, h, w)


def test_max_movement_excludes_frame_n_frames(engine):
    """Frames [0, n_frames) only: a larger value planted in frame n_frames must not count."""
    rng = np.random.default_rng(3)
    S = np.tile(np.eye(3), (4, 1, 1)) + rng.normal(size=(4, 3, 3)) * [[1e-2, 1e-2, 10], [1e-2, 1e-2, 10], [1e-5, 1e-5, 0]]
    S[3, 0, 2] = 5000.0
    Sd = _dev(engine, S.reshape(-1, 9))
    got = float(engine.max_movement(Sd, 3, 224, 400).item())
    assert got == _max_movement_host(S, 3, 224, 400) and got < 1000
    assert float(engine.max_movement(Sd, 4, 224, 400).item()) == _max_movement_host(S, 4, 224, 400) > 5000


def test_max_movement_past_65535_frames(engine):
    """70 000 frames of 224 x 400, the unique maximum in frame 65 600 and a larger value planted in frame 70 000, against
    the exact corner maximum.  The kernel's value is an f64 evaluation of the same corner (three roundings for X, three
    for W, one division, no cancellation here): within 8 ulp.

    Before evz_max_movement looped over frames, it launched one y-block per frame; gridDim.y is limited to 65 535, so
    this call failed at launch with cudaErrorInvalidConfiguration, which the library returns as EVZ_E_CUDA and Python
    raises as EvzError.  That is a launch-configuration error the runtime returns before anything runs, not a fault on
    the device."""
    rng = np.random.default_rng(65600)
    F = 70000
    S = np.tile(np.eye(3), (F + 1, 1, 1))
    S[:, :2, 2] = rng.normal(0, 5, (F + 1, 2))
    S[:, 2, :2] = rng.normal(0, 1e-6, (F + 1, 2))
    S[65600, 0, 2] = 300.0
    S[F, 0, 2] = 600.0
    Sd = _dev(engine, S.reshape(-1, 9))
    want, frame, w_min = chain.max_movement_corners(S, F, 224, 400)
    assert frame == 65600 and w_min > 0.99
    got = float(engine.max_movement(Sd, F, 224, 400).item())
    assert abs(got - want) <= 8 * np.spacing(want), (got, want)
    want1, frame1, _ = chain.max_movement_corners(S, F + 1, 224, 400)
    got1 = float(engine.max_movement(Sd, F + 1, 224, 400).item())
    assert frame1 == F and abs(got1 - want1) <= 8 * np.spacing(want1) and got1 > got + 200
