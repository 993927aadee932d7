"""GeometryEngine: batched frame-to-frame geometry on one B200 through libevz.so.

PyTorch is used for device memory, streams and (in distributed.py) NCCL; every kernel is
hand-written CUDA behind the C ABI of include/evz.h.  All heavy results stay on the device
as torch tensors; `video_geometry` is the host-arrays-in / host-arrays-out call.
"""
import ctypes as C
from dataclasses import dataclass, field, fields
from typing import Optional

import numpy as np
import torch

from . import _lib
from ._lib import EVZ_ROW_ALIGN, EVZ_DESC_BYTES, EVZ_MAX_KP


def _ptr(t: Optional[torch.Tensor]):
    return C.c_void_p(0 if t is None else t.data_ptr())


@dataclass
class FrameStore:
    """Device-resident frame store in the layout of include/evz.h."""
    desc: torch.Tensor        # u8  [rows,128]
    ckey: torch.Tensor        # i32 [rows]
    coords: torch.Tensor      # f32 [rows,2]
    canon: torch.Tensor       # i32 [rows]
    row_off: torch.Tensor     # i32 [F+1] (device)
    n_kp: torch.Tensor        # i32 [F]   (device)
    row_off_h: np.ndarray     # host copies
    n_kp_h: np.ndarray
    d: int = 128
    keep: tuple = ()          # staging buffers kept alive until the stream has consumed them

    @property
    def n_frames(self):
        return len(self.n_kp_h)

    @property
    def rows(self):
        return int(self.row_off_h[-1])

    @property
    def max_kp(self):
        return int(self.n_kp_h.max()) if len(self.n_kp_h) else 0


@dataclass
class PairResults:
    """Everything the per-pair pipeline produces (device tensors; per-row arrays are indexed
    from out_off[p])."""
    pair_q: torch.Tensor
    pair_t: torch.Tensor
    out_off: torch.Tensor
    top2_idx: torch.Tensor
    top2_d2: torch.Tensor
    surv: torch.Tensor
    m_idx: torch.Tensor
    m_pts: torch.Tensor
    m_cnt: torch.Tensor
    n_filtered: torch.Tensor
    status: torch.Tensor
    H1: Optional[torch.Tensor] = None
    mask1: Optional[torch.Tensor] = None
    mask1_best: Optional[torch.Tensor] = None
    best_hyp1: Optional[torch.Tensor] = None
    best_cnt1: Optional[torch.Tensor] = None
    inl1: Optional[torch.Tensor] = None
    static_pts: Optional[torch.Tensor] = None
    static_cnt: Optional[torch.Tensor] = None
    static_r: Optional[torch.Tensor] = None
    flags: Optional[torch.Tensor] = None
    H: Optional[torch.Tensor] = None         # RANSAC #2 result = compute_homography's matrix
    mask2: Optional[torch.Tensor] = None
    mask2_best: Optional[torch.Tensor] = None
    best_hyp2: Optional[torch.Tensor] = None
    best_cnt2: Optional[torch.Tensor] = None
    inl2: Optional[torch.Tensor] = None
    extra: dict = field(default_factory=dict)

    _PER_ROW = ("top2_idx", "top2_d2", "surv", "m_idx", "m_pts", "mask1", "mask1_best", "static_pts", "mask2", "mask2_best")

    def pairs(self, p0, p1) -> "PairResults":
        """Pairs [p0, p1) as views into this workspace: per-pair tensors (and `extra`) sliced, per-row tensors shared
        (they are addressed through out_off), so engine calls given the view write into this workspace."""
        v = {f.name: getattr(self, f.name) for f in fields(self)}
        for k, t in v.items():
            if k not in self._PER_ROW and isinstance(t, torch.Tensor):
                v[k] = t[p0:p1]
        v["extra"] = {k: t[p0:p1] for k, t in self.extra.items()}
        return PairResults(**v)


class GeometryEngine:
    def __init__(self, device: int = 0):
        if not torch.cuda.is_available():
            raise RuntimeError("evenvizion_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device("cuda", device)
        torch.cuda.set_device(self.device)
        torch.zeros(1, device=self.device)           # make sure the primary context exists
        h = C.c_void_p()
        rc = self.lib.evz_create(device, C.byref(h))
        if rc != 0:
            raise _lib.EvzError(self.lib.evz_last_error(None).decode())
        self.h = h
        self.sm_count = self.lib.evz_sm_count(self.h)

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.evz_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def set_option(self, option: int, value: int):
        """EVZ_OPT_* switches of include/evz.h (A/B routes with identical results)."""
        self._check(self.lib.evz_set_option(self.h, int(option), int(value)))

    def match_kernel_ms(self, k=0):
        """CUDA-event time of the main match kernel of the k-th most recent `match` call (EVZ_OPT_TIME_MATCH = option 4
        must be on; synchronise the stream first)."""
        ms = C.c_float(0.0)
        self._check(self.lib.evz_match_kernel_ms(self.h, int(k), C.byref(ms)))
        return float(ms.value)

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, rc):
        _lib.check(self.h, rc)

    def _empty(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    @staticmethod
    def layout(n_kp):
        """row_off (int32 [F+1]) for per-frame keypoint counts: every frame starts at a multiple of 256."""
        n_kp = np.asarray(n_kp, np.int64)
        padded = (n_kp + EVZ_ROW_ALIGN - 1) // EVZ_ROW_ALIGN * EVZ_ROW_ALIGN
        padded = np.maximum(padded, EVZ_ROW_ALIGN)
        row_off = np.zeros(len(n_kp) + 1, np.int64)
        np.cumsum(padded, out=row_off[1:])
        if row_off[-1] >= 2 ** 31:
            raise ValueError("frame store exceeds 2^31 rows; shard the video")
        return row_off.astype(np.int32)

    # ------------------------------------------------------------------ ingest
    @staticmethod
    def _frames_input(desc, coords, n_kp):
        """The frame input of `ingest` / `video_geometry`, normalised and checked: returns (desc [rows, d],
        coords [rows, 2], n_kp int64 [F], d, is_f32), desc and coords as torch tensors where they were given."""
        desc_t = torch.as_tensor(desc)
        coords_t = torch.as_tensor(coords)
        if desc_t.dim() == 3:
            f, n, d = desc_t.shape
            if n_kp is None:
                n_kp = np.full(f, n, np.int64)
            desc_t = desc_t.reshape(f * n, d)
            coords_t = coords_t.reshape(f * n, 2)
        if n_kp is None:
            raise ValueError("n_kp is required for concatenated input")
        n_kp_h = np.asarray(n_kp, np.int64)
        if int(n_kp_h.sum()) != desc_t.shape[0] or coords_t.shape[0] != desc_t.shape[0]:
            raise ValueError("n_kp does not add up to the number of descriptor rows")
        if len(n_kp_h) and int(n_kp_h.max()) > EVZ_MAX_KP:
            raise ValueError(f"at most {EVZ_MAX_KP} keypoints per frame are supported")
        d = int(desc_t.shape[1]) if desc_t.dim() == 2 and desc_t.shape[0] else 128
        if d > EVZ_DESC_BYTES or d % 4:
            raise ValueError("descriptor width must be a multiple of 4 and at most 128")
        if desc_t.dtype == torch.uint8:
            is_f32 = 0
        elif desc_t.dtype == torch.float32:
            is_f32 = 1
        else:
            raise TypeError("descriptors must be uint8 or float32 (SIFT/ORB); SURF's non-integer floats are not supported")
        return desc_t, coords_t, n_kp_h, d, is_f32

    def _new_store(self, n_kp_h, d):
        """An unfilled FrameStore for frames of n_kp_h keypoints.  Returns (store, raw_off_h, raw_off, bad): the host and
        device offsets of every frame's first input row and the device count of non-integer descriptor values, which
        `_ingest_frames` takes.  store.keep holds the device tensors until the stream has consumed them."""
        dev = self.device
        row_off_h = self.layout(n_kp_h)
        raw_off_h = np.zeros(len(n_kp_h) + 1, np.int64)
        np.cumsum(n_kp_h, out=raw_off_h[1:])
        rows = int(row_off_h[-1])
        raw_off = torch.from_numpy(raw_off_h).to(dev, non_blocking=True)
        row_off = torch.from_numpy(row_off_h).to(dev, non_blocking=True)
        n_kp_d = torch.from_numpy(n_kp_h.astype(np.int32)).to(dev, non_blocking=True)
        bad = torch.zeros(1, dtype=torch.int32, device=dev)
        st = FrameStore(desc=self._empty((rows, EVZ_DESC_BYTES), torch.uint8), ckey=self._empty((rows,), torch.int32),
                        coords=self._empty((rows, 2), torch.float32), canon=self._empty((rows,), torch.int32),
                        row_off=row_off, n_kp=n_kp_d, row_off_h=row_off_h, n_kp_h=n_kp_h.astype(np.int32), d=d,
                        keep=(raw_off, bad))
        return st, raw_off_h, raw_off, bad

    def _ingest_frames(self, st, desc, coords, raw_off, is_f32, bad, f0, f1):
        """Frames [f0, f1) of st from the device input rows desc / coords (frame f starts at row raw_off[f])."""
        self._check(self.lib.evz_ingest(self.h, _ptr(desc), is_f32, st.d, _ptr(coords), _ptr(raw_off[f0:]),
                                        _ptr(st.row_off[f0:]), f1 - f0, _ptr(st.desc), _ptr(st.ckey), _ptr(st.coords),
                                        _ptr(st.canon), _ptr(bad), self._stream()))

    @staticmethod
    def _check_integer_descriptors(bad):
        n = int(bad.item())
        if n:
            raise ValueError(f"{n} descriptor values are not integers in [0,255]; "
                             "the int8 tensor-core matcher is exact only for SIFT/ORB-style descriptors")

    def ingest(self, desc, coords, n_kp=None, check=True) -> FrameStore:
        """desc: [sum n_kp, d] uint8 or float32 (integer-valued, <= 255), frames concatenated (a
        uniform [F, N, d] array is accepted too); coords: matching [.., 2] float32; n_kp: per-frame
        counts.  Arrays may be numpy, pinned/CPU torch or CUDA torch tensors."""
        desc_t, coords_t, n_kp_h, d, is_f32 = self._frames_input(desc, coords, n_kp)
        desc_d = desc_t.to(self.device, non_blocking=True).contiguous()
        coords_d = coords_t.to(torch.float32).to(self.device, non_blocking=True).contiguous()
        st, _, raw_off, bad = self._new_store(n_kp_h, d)
        st.keep += (desc_d, coords_d)
        if st.rows and desc_d.shape[0]:
            self._ingest_frames(st, desc_d, coords_d, raw_off, is_f32, bad, 0, st.n_frames)
        elif st.rows:
            st.desc.zero_(); st.ckey.fill_(2 ** 31 - 1); st.coords.zero_(); st.canon.fill_(-1)
        if is_f32 and check:
            self._check_integer_descriptors(bad)
        return st

    # ------------------------------------------------------------------ K1 / K1b / K2
    def _match_results(self, st: FrameStore, pair_q, pair_t) -> PairResults:
        """The outputs of `match` for the pairs (pair_q[p], pair_t[p]), allocated."""
        pq = torch.as_tensor(pair_q, dtype=torch.int32).to(self.device)
        pt = torch.as_tensor(pair_t, dtype=torch.int32).to(self.device)
        P, rows, e, i32 = int(pq.numel()), st.rows, self._empty, torch.int32
        return PairResults(pair_q=pq, pair_t=pt, out_off=st.row_off[:-1][pq.long()].contiguous(),
                           top2_idx=e((rows, 2), i32), top2_d2=e((rows, 2), i32), surv=e((rows,), torch.uint8),
                           m_idx=e((rows, 2), i32), m_pts=e((rows, 4), torch.float32), m_cnt=e((P,), i32),
                           n_filtered=e((P,), i32), status=e((P,), i32))

    def match(self, st: FrameStore, pair_q=None, pair_t=None, ratio=0.5, min_matching_pts=4, out=None) -> PairResults:
        """K1 + K1b/K2 for the pairs (pair_q[p], pair_t[p]).  Per-row outputs of pair p start at
        out_off[p] = row_off[pair_q[p]], so one call must not list the same query frame twice (the C ABI
        takes out_off as an argument and has no such restriction).
        out: a PairResults to write into instead of allocating (from `alloc_results`, or a `pairs` view of one); the pairs
        and out_off are then its own, and pair_q / pair_t are not used."""
        r = self._match_results(st, pair_q, pair_t) if out is None else out
        P = int(r.pair_q.numel())
        self._check(self.lib.evz_match_top2_d(self.h, _ptr(st.desc), int(st.d), _ptr(st.ckey), st.rows, _ptr(st.row_off),
                                              _ptr(st.n_kp), _ptr(r.pair_q), _ptr(r.pair_t), _ptr(r.out_off), P,
                                              _ptr(r.top2_idx), _ptr(r.top2_d2), self._stream()))
        self._check(self.lib.evz_filter_matches(self.h, _ptr(r.top2_idx), _ptr(r.top2_d2), _ptr(st.coords), _ptr(st.canon),
                                                _ptr(st.row_off), _ptr(st.n_kp), _ptr(r.pair_q), _ptr(r.pair_t), _ptr(r.out_off),
                                                P, st.max_kp, float(ratio), int(min_matching_pts),
                                                _ptr(r.surv), _ptr(r.m_idx), _ptr(r.m_pts), _ptr(r.m_cnt), _ptr(r.n_filtered),
                                                _ptr(r.status), self._stream()))
        return r

    # ------------------------------------------------------------------ K3 / K4
    def find_homography(self, pts, off, cnt, status, max_cnt, n_hyp=1024, seed=0, pair_id_base=0, level=1,
                        thresh=3.0, min_inlier_frac=0.0, fail_status=_lib.ST_NO_MODEL_1, pre_H=None, pair_ids=None,
                        out=None):
        """Batched seeded RANSAC + LM refit over the point lists pts[off[p]:off[p]+cnt[p]].
        status is updated in place.  Returns dict(H, mask, inl_cnt, best_hyp, best_cnt, mask_best, H_best).
        pair_ids: int64 [P] device tensor of sampler ids (pair p is seeded with pair_ids[p] instead of pair_id_base + p).
        out: a dict of those tensors to write instead of allocating them; H and inl_cnt are required, an output left
        out is not computed."""
        P = int(cnt.numel())
        if out is None:
            rows = int(pts.shape[0])
            z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=self.device)
            out = dict(H=z((P, 9), torch.float64), inl_cnt=z((P,), torch.int32), mask=z((rows,), torch.uint8),
                       best_hyp=torch.full((P,), -1, dtype=torch.int32, device=self.device), best_cnt=z((P,), torch.int32),
                       mask_best=z((rows,), torch.uint8), H_best=z((P, 9), torch.float64))
        if pair_ids is not None:
            fn, ids = self.lib.evz_find_homography_ids, _ptr(pair_ids)
        else:
            fn, ids = self.lib.evz_find_homography, int(pair_id_base)
        self._check(fn(self.h, _ptr(pts), _ptr(off), _ptr(cnt), P, int(max_cnt), _ptr(pre_H),
                       int(n_hyp), int(seed) & 0xFFFFFFFF, ids, int(level),
                       float(thresh), float(min_inlier_frac), int(fail_status),
                       _ptr(status), _ptr(out["H"]), _ptr(out.get("mask")), _ptr(out["inl_cnt"]),
                       _ptr(out.get("best_hyp")), _ptr(out.get("best_cnt")), _ptr(out.get("mask_best")),
                       _ptr(out.get("H_best")), self._stream()))
        return out

    # ------------------------------------------------------------------ K5
    def static_filter(self, pts, off, cnt, H, status, want_r=False, max_cnt=None, out=None):
        """K5.  max_cnt: host-known upper bound of cnt (read back from the device when omitted).
        out: (out_pts, out_cnt, best_r, flags) to write instead of allocating them."""
        P = int(cnt.numel())
        if max_cnt is None:
            max_cnt = int(cnt.max().item()) if P else 0
        r_out = self._empty((int(pts.shape[0]),), torch.int32) if want_r else None
        if out is None:
            out = (self._empty(tuple(pts.shape), torch.float32), self._empty((P,), torch.int32),
                   self._empty((P,), torch.int32), self._empty((P,), torch.int32))
        out_pts, out_cnt, best_r, flags = out
        self._check(self.lib.evz_static_filter(self.h, _ptr(pts), _ptr(off), _ptr(cnt), P, int(max_cnt), _ptr(H), _ptr(status),
                                               _ptr(out_pts), _ptr(out_cnt), _ptr(best_r), _ptr(flags), _ptr(r_out),
                                               self._stream()))
        if want_r:
            return out_pts, out_cnt, best_r, flags, r_out
        return out_pts, out_cnt, best_r, flags

    def concat_dedup(self, parts, status, out_off, out_rows, max_total):
        """K5b: per-pair concatenation of the point lists `parts` = [(pts, off, cnt), ...] (one entry per feature type)
        followed by remove_double_matching.  Returns (out_pts [out_rows, 4], out_cnt [P])."""
        n = len(parts)
        P = int(status.numel())
        arr = C.c_void_p * n
        pts = arr(*[p[0].data_ptr() for p in parts])
        off = arr(*[p[1].data_ptr() for p in parts])
        cnt = arr(*[p[2].data_ptr() for p in parts])
        out_pts = self._empty((int(out_rows), 4), torch.float32)
        out_cnt = self._empty((P,), torch.int32)
        self._check(self.lib.evz_concat_dedup(self.h, n, pts, off, cnt, P, _ptr(status), int(max_total), _ptr(out_off),
                                              _ptr(out_pts), _ptr(out_cnt), self._stream()))
        return out_pts, out_cnt

    # ------------------------------------------------------------------ whole per-pair path
    def process_pairs(self, st: FrameStore, pair_q, pair_t, n_hyp=1024, seed=0, pair_id_base=0,
                      ratio=0.5, thresh=3.0, min_matching_pts=4) -> PairResults:
        """match_static_kps + compute_homography for every pair (reference matching.py:131-163,
        utils.py:328-363), all on the device."""
        r = self.alloc_results(st, pair_q, pair_t)
        self._pairs_range(st, r, 0, int(r.pair_q.numel()), n_hyp, seed, pair_id_base, ratio, thresh, min_matching_pts)
        return r

    # ------------------------------------------------------------------ K6 / K7
    def chain_scan(self, G, status, policy=True, seed_S=None, seed_G=None, want_fixed=True, want_summary=False,
                   want_S=True):
        """None-H fallback + cumulative superposition.  G: [P,9] or [P,3,3] f64 device tensor."""
        G = G.reshape(-1, 9).contiguous()
        P = G.shape[0]
        S = self._empty((P, 9), torch.float64) if want_S else None
        Hf = self._empty((P, 9), torch.float64) if (want_fixed and want_S) else None
        summ = self._empty((20,), torch.float64) if want_summary else None
        if P:
            self._check(self.lib.evz_chain_scan(self.h, _ptr(G), _ptr(status), P, 1 if policy else 0, _ptr(seed_S), _ptr(seed_G),
                                                _ptr(S), _ptr(Hf), _ptr(summ), self._stream()))
        elif summ is not None:       # an empty shard: identity product, no valid pair
            summ.copy_(torch.tensor([1, 0, 0, 0, 1, 0, 0, 0, 1] * 2 + [0, 0], dtype=torch.float64))
        return S, Hf, summ

    def chain_scan_segments(self, G, status, seg_off, policy=True):
        """`chain_scan` (no seeds) restarted at every segment: segment s = pairs [seg_off[s], seg_off[s+1]) of G / status,
        seg_off an int32 [n_segs+1] device tensor.  Returns (S, H_fixed), both [P,9]."""
        G = G.reshape(-1, 9).contiguous()
        P = G.shape[0]
        S = self._empty((P, 9), torch.float64)
        Hf = self._empty((P, 9), torch.float64)
        self._check(self.lib.evz_chain_scan_segments(self.h, _ptr(G), _ptr(status), P, _ptr(seg_off), int(seg_off.numel()) - 1,
                                                     1 if policy else 0, _ptr(S), _ptr(Hf), self._stream()))
        return S, Hf

    def chain_ref_step(self, H2, status, first, policy, S_state, H_prev, H_out):
        """One reference-exact chain step for the first n = len(status) chains (include/evz.h, evz_chain_ref_step):
        writes H_out[:n] and advances S_state[:n] in place.  H_prev: the previous step's H_out (None on the first step)."""
        self._check(self.lib.evz_chain_ref_step(self.h, _ptr(H2), _ptr(status), int(status.numel()), 1 if first else 0,
                                                1 if policy else 0, _ptr(S_state), _ptr(H_prev), _ptr(H_out), self._stream()))

    def reference_chains(self, pts, off, cnt, status, max_cnt, step_off, n_hyp=1024, seed=0, policy=True, thresh=3.0,
                         min_inlier_frac=0.7, fail_status=_lib.ST_NO_MODEL_2):
        """RANSAC #2 of the reference-exact chain (video_processing.py:67-105) for several videos in lockstep.

        The pairs are in step-major order: step k is pairs [step_off[k], step_off[k+1]) = pair k of chains 0 .. n_k - 1,
        with n_0 >= n_1 >= ... (chains ordered by length, longest first), so the chains still running are a prefix.
        Step k is one RANSAC launch over its pairs, seeded with id k and pre-transformed by every chain's running
        superposition, then one evz_chain_ref_step.  The outputs are allocated before the loop and the loop neither
        allocates nor synchronises with the host.  status is updated in place; returns H_out [P,9]: the matrix the
        reference stores for every pair, after the None-H policy."""
        step_off = np.asarray(step_off, np.int64)
        K = len(step_off) - 1
        P = int(cnt.numel())
        H2 = torch.zeros((P, 9), dtype=torch.float64, device=self.device)
        H_out = self._empty((P, 9), torch.float64)
        inl = torch.zeros((P,), dtype=torch.int32, device=self.device)
        S_state = self._empty((int(step_off[1] - step_off[0]) if K else 0, 9), torch.float64)
        # pinned + non_blocking: the set-up does not synchronise with the host either
        ids = torch.from_numpy(np.repeat(np.arange(K, dtype=np.int64), np.diff(step_off))).pin_memory()
        ids = ids.to(self.device, non_blocking=True)
        for k in range(K):
            a, b = int(step_off[k]), int(step_off[k + 1])
            H2_k, status_k, prev = H2[a:b], status[a:b], int(step_off[k - 1]) if k else 0
            self.find_homography(pts, off[a:b], cnt[a:b], status_k, max_cnt, n_hyp, seed, 0, 2, thresh, min_inlier_frac,
                                 fail_status, pre_H=S_state if k else None, pair_ids=ids[a:b],
                                 out=dict(H=H2_k, inl_cnt=inl[a:b]))
            self.chain_ref_step(H2_k, status_k, k == 0, policy, S_state, H_out[prev:prev + b - a] if k else None, H_out[a:b])
        return H_out

    def chain_seed_apply(self, summaries, rank, S, policy=True, want_fixed=True):
        """Turn this rank's unseeded local scan S ([P,9], in place) into its slice of the global scan, given the
        all-gathered shard summaries ([world,20] device tensor).  Returns (S, H_fixed or None, seeds [27])."""
        world = int(summaries.shape[0])
        P = int(S.shape[0])
        Hf = self._empty((P, 9), torch.float64) if want_fixed else None
        seeds = self._empty((27,), torch.float64)
        if P:
            self._check(self.lib.evz_chain_seed_apply(self.h, _ptr(summaries), world, int(rank), 1 if policy else 0, P,
                                                      _ptr(S), _ptr(Hf), _ptr(seeds), self._stream()))
        return S, Hf, seeds

    def remap(self, pts, frame_idx, S, sx, sy, inverse=False):
        pts = pts.reshape(-1, 2).contiguous()
        out = torch.empty_like(pts)
        S = S.reshape(-1, 9).contiguous()
        if pts.shape[0]:
            self._check(self.lib.evz_remap(self.h, _ptr(pts), _ptr(frame_idx), pts.shape[0], _ptr(S), S.shape[0],
                                           float(sx), float(sy), 1 if inverse else 0, _ptr(out), self._stream()))
        return out

    def max_movement(self, S, n_frames, height, width):
        out = self._empty((1,), torch.float64)
        S = S.reshape(-1, 9).contiguous()
        self._check(self.lib.evz_max_movement(self.h, _ptr(S), int(n_frames), int(height), int(width), _ptr(out), self._stream()))
        return out

    # ------------------------------------------------------------------ video-level driver
    def _pairs_range(self, st: FrameStore, r: PairResults, p0: int, p1: int, n_hyp, seed, pair_id_base, ratio, thresh,
                     min_matching_pts=4, after_match=None):
        """match_static_kps + compute_homography for pairs [p0, p1) of an already allocated PairResults, written through a
        `pairs` view of it."""
        if p1 <= p0:
            return
        v, mk = r.pairs(p0, p1), st.max_kp
        self.match(st, ratio=ratio, min_matching_pts=min_matching_pts, out=v)
        if after_match is not None:
            after_match()
        self.find_homography(v.m_pts, v.out_off, v.m_cnt, v.status, mk, n_hyp, seed, int(pair_id_base) + p0, 1, thresh, 0.0,
                             _lib.ST_NO_MODEL_1, out=dict(H=v.H1, mask=v.mask1, inl_cnt=v.inl1, best_hyp=v.best_hyp1,
                                                          best_cnt=v.best_cnt1, mask_best=v.mask1_best, H_best=v.extra["H1_best"]))
        self.static_filter(v.m_pts, v.out_off, v.m_cnt, v.H1, v.status, max_cnt=mk, out=(v.static_pts, v.static_cnt, v.static_r, v.flags))
        self.find_homography(v.static_pts, v.out_off, v.static_cnt, v.status, mk, n_hyp, seed, int(pair_id_base) + p0, 2, thresh,
                             0.7, _lib.ST_NO_MODEL_2, out=dict(H=v.H, mask=v.mask2, inl_cnt=v.inl2, best_hyp=v.best_hyp2,
                                                               best_cnt=v.best_cnt2, mask_best=v.mask2_best, H_best=v.extra["H2_best"]))

    def alloc_results(self, st: FrameStore, pair_q, pair_t) -> PairResults:
        """Workspace for `process_pairs_into`: every per-pair / per-row output of the path, allocated once."""
        r = self._match_results(st, pair_q, pair_t)
        P, rows = int(r.pair_q.numel()), st.rows
        e, z = self._empty, lambda shape, dt: torch.zeros(shape, dtype=dt, device=self.device)
        i32, u8, f64 = torch.int32, torch.uint8, torch.float64
        r.H1, r.H = z((P, 9), f64), z((P, 9), f64)
        r.mask1, r.mask1_best, r.mask2, r.mask2_best = z((rows,), u8), z((rows,), u8), z((rows,), u8), z((rows,), u8)
        r.inl1, r.inl2, r.best_cnt1, r.best_cnt2 = z((P,), i32), z((P,), i32), z((P,), i32), z((P,), i32)
        r.best_hyp1 = torch.full((P,), -1, dtype=i32, device=self.device)
        r.best_hyp2 = torch.full((P,), -1, dtype=i32, device=self.device)
        r.extra["H1_best"], r.extra["H2_best"] = z((P, 9), f64), z((P, 9), f64)
        r.static_pts, r.static_cnt = e((rows, 4), torch.float32), e((P,), i32)
        r.static_r, r.flags = e((P,), i32), e((P,), i32)
        return r

    def process_pairs_into(self, st: FrameStore, r: PairResults, n_hyp=1024, seed=0, pair_id_base=0, ratio=0.5, thresh=3.0,
                           after_match=None) -> PairResults:
        """`process_pairs` into a workspace from `alloc_results`: no allocation, no memset, nothing but the kernels of the
        path on the current stream (what a steady-state caller -- and bench.py's timed region -- runs per batch).
        after_match: optional callable invoked between the match stage and the first RANSAC (event recording)."""
        self._pairs_range(st, r, 0, int(r.pair_q.numel()), n_hyp, seed, pair_id_base, ratio, thresh, after_match=after_match)
        return r

    def video_geometry(self, desc, coords, n_kp=None, n_hyp=1024, seed=0, none_h_processing=True,
                       ratio=0.5, thresh=3.0, pair_id_base=0, chunk_frames=None):
        """Frame chain -> per-pair G, status, cumulative S and fixed-plane H (parallel formulation).
        Host arrays in, host arrays out: this is the call bench.py times end to end.

        Host input is streamed: frames are copied to the device in chunks on a copy stream while the
        compute stream ingests and processes the pairs of the chunks that have already landed, so the
        PCIe transfer (the end-to-end bound: 136 bytes per keypoint) overlaps the kernels."""
        desc_t, coords_t, n_kp_h, d, is_f32 = self._frames_input(desc, coords, n_kp)
        F = len(n_kp_h)
        if chunk_frames is None:
            chunk_frames = max(64, -(-F // 16))
        if desc_t.is_cuda or F <= chunk_frames:
            # small or device-resident input: one ingest, one batch
            st = self.ingest(desc_t, coords_t, n_kp_h)
            r = self.process_pairs(st, torch.arange(1, F, dtype=torch.int32), torch.arange(0, F - 1, dtype=torch.int32),
                                   n_hyp, seed, pair_id_base, ratio, thresh)
        else:
            st, r = self._video_streamed(desc_t, coords_t, n_kp_h, d, is_f32, chunk_frames, n_hyp, seed, pair_id_base,
                                         ratio, thresh)
        S, Hf, _ = self.chain_scan(r.H, r.status, none_h_processing)
        return dict(G=r.H.cpu().numpy().reshape(-1, 3, 3), status=r.status.cpu().numpy(),
                    S=S.cpu().numpy().reshape(-1, 3, 3), H_fixed=Hf.cpu().numpy().reshape(-1, 3, 3), results=r, store=st)

    def _video_streamed(self, desc_t, coords_t, n_kp_h, d, is_f32, chunk_frames, n_hyp, seed, pair_id_base, ratio, thresh):
        coords_t = coords_t.to(torch.float32)
        F = len(n_kp_h)
        dev = self.device
        compute = torch.cuda.current_stream(dev)
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(dev)
        copy = self._copy_stream
        st, raw_off_h, raw_off, bad = self._new_store(n_kp_h, d)
        desc_raw = torch.empty(desc_t.shape, dtype=desc_t.dtype, device=dev)
        coords_raw = torch.empty(coords_t.shape, dtype=torch.float32, device=dev)
        st.keep += (desc_raw, coords_raw)
        r = self.alloc_results(st, torch.arange(1, F, dtype=torch.int32, device=dev),
                               torch.arange(0, F - 1, dtype=torch.int32, device=dev))
        copy.wait_stream(compute)            # the staging buffers were allocated on the compute stream
        for f0 in range(0, F, chunk_frames):
            f1 = min(F, f0 + chunk_frames)
            a, b = int(raw_off_h[f0]), int(raw_off_h[f1])
            with torch.cuda.stream(copy):
                if b > a:
                    desc_raw[a:b].copy_(desc_t[a:b], non_blocking=True)
                    coords_raw[a:b].copy_(coords_t[a:b], non_blocking=True)
                landed = copy.record_event()
            compute.wait_event(landed)
            self._ingest_frames(st, desc_raw, coords_raw, raw_off, is_f32, bad, f0, f1)
            # pairs whose query frame is in this chunk (their train frame landed with this or an earlier chunk)
            self._pairs_range(st, r, max(f0, 1) - 1, f1 - 1, n_hyp, seed, pair_id_base, ratio, thresh)
        desc_raw.record_stream(copy); coords_raw.record_stream(copy)
        st.keep = (bad,)                     # every consumer of the raw staging copies is enqueued: let them go
        if is_f32:
            self._check_integer_descriptors(bad)
        return st, r
