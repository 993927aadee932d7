#!/usr/bin/env python
"""bench.py -- frame-pairs/s of the geometry hot path (match + RANSAC H + scan) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5] [--dump-outputs DIR]

A step is one pass of the hot path over one batch of synthetic input:
  config 2 (default, BASELINE.json configs[1]): 2048 SIFT-like keypoints/frame x 10 000 frame
  pairs per GPU, 1024 RANSAC hypotheses per RANSAC level.
`value`  = pairs/s with the frame store resident in HBM (CUDA events on the launching stream,
           max over ranks); `e2e` = the same through GeometryEngine.video_geometry with pinned HOST
           buffers in and host arrays out (H2D + ingest + path + D2H inside the timed region).
Inputs are 2.6 GB per step (> 126 MB L2), so no explicit L2 flush is needed between steps.
Multi-GPU: one process per GPU (torchrun), pairs sharded by contiguous range, weak scaling,
one NCCL all-gather of the 160-byte shard summaries per step.
The inputs are generated from fixed seeds, so a run with the same arguments sees the same inputs; --dump-outputs DIR
writes what the last timed step computed (see dump_outputs) for comparing two builds output for output.
Nothing is written into the tree the benchmark runs from (it may be read-only), not even bytecode caches.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    2: dict(name="synthetic 2k SIFT keypoints/frame x 10k frame pairs, 1024 RANSAC hypotheses", n_kp=2048, pairs=10000,
            n_hyp=1024, outlier_frac=0.2, unmatched_frac=0.0),
    3: dict(name="synthetic 8k keypoints/frame x 10k pairs (match-GEMM-bound)", n_kp=8192, pairs=10000, n_hyp=1024,
            outlier_frac=0.2, unmatched_frac=0.0),
    4: dict(name="sharp motion: 20% inlier ratio, 4096 hypotheses/pair, none_H_processing=True", n_kp=2048, pairs=10000,
            n_hyp=4096, outlier_frac=0.8, unmatched_frac=0.02),
    # strong scaling: the 100 000 pairs are split over the ranks; the step also remaps 8 object points per frame
    # through the cumulative superposition.  The chain is a 10 000-frame synthetic chain repeated (the seam pairs
    # have no correspondences and exercise the None-H forward fill).
    5: dict(name="long video 100k frame pairs sharded over the GPUs + cumulative H scan + object-coord remap", n_kp=2048,
            pairs=100000, n_hyp=1024, outlier_frac=0.2, unmatched_frac=0.0, strong=True, remap_points=8, tile=10),
}
# match (prepare, build_items x2, V-space kernel, fix-up, key-space kernel for the pairs the V-space kernel cannot take),
# filter, score+refit, static, score+refit, scan (fill x3, prod x3, fixed plane)
KERNELS_PER_STEP = 6 + 1 + 2 + 1 + 2 + 7
# sharded scan: fill x3, prod x3, summary | NCCL all-gather (not ours) | seed, apply, fixed plane
KERNELS_PER_STEP_MULTI = 6 + 1 + 2 + 1 + 2 + 10
# dram__bytes_read.sum + dram__bytes_write.sum of one match_top2_vkernel<0> launch (the kernel as it ships) at config 2 x
# 10 000 pairs: ncu --set full capture of round 2, profiles/r02_prof_vkernel_raw.csv
MATCH_TRAFFIC_BYTES = {(2, 10000): 3449581000 + 324503808}
# ncu --set full of the RANSAC kernels as they ship (profiles/r02b_prof_{score,refit}_raw.csv; 2000 pairs of config 2:
# 1229 matches at level 1, 584 static points at level 2, 1024 hypotheses)
RANSAC_NCU = {
    "source": "profiles/r02b_prof_score_raw.csv, profiles/r02b_prof_refit_raw.csv (2000 pairs of config 2)",
    "score_level1": {"us": 564.7, "issue_slots_pct": 73.3, "sm_throughput_pct": 68.4, "fma_pipe_pct": 35.2, "alu_pipe_pct": 44.4,
                     "dram_pct": 1.5, "warp_instr_per_nominal_eval": 434.9e6 / (2000 * 1024 * 1229.0)},
    "score_level2": {"us": 101.9, "issue_slots_pct": 61.1, "sm_throughput_pct": 44.9, "dram_pct": 2.3,
                     "warp_instr_per_nominal_eval": 53.0e6 / (2000 * 1024 * 584.0)},
    "refit_level1": {"us": 101.5, "issue_slots_pct": 43.6, "fp64_pipe_pct": 41.0, "dram_pct": 4.8},
    "refit_level2": {"us": 67.6, "issue_slots_pct": 44.5, "fp64_pipe_pct": 41.4, "dram_pct": 3.4},
}

def config_dict(cfg, args, world):
    """The `config` object of the JSON line: the same for both arms (--impl ours / reference), so that the driver can tell
    that they ran the same workload; what a run measured about its data goes to `run_stats`."""
    P = args.pairs if args.pairs else cfg["pairs"]
    if cfg.get("strong"):
        P = P // world
    return {"workload": cfg["name"], "n_kp": cfg["n_kp"], "pairs_per_gpu": P, "n_hyp": cfg["n_hyp"], "parallelism": f"pair-range x{world}",
            "l2": f"inputs {(P + 1) * cfg['n_kp'] * 136 / 1e9:.1f} GB per step > 126 MB L2, no flush"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d.get("hbm_gbs", 6650.0), bf16_burst=d.get("bf16_tflops", 1590.0),
                    bf16_sustained=d.get("bf16_tflops_sustained", 1400.0), source="MEASURED_PEAKS.json")
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons; started before warm-up, samples filtered to the timed window."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, bufsize=1)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self, t_begin, t_end):
        """t_begin / t_end: time.time() around the timed region."""
        import datetime
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, sm_all, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                c, m = float(f[1]), float(f[2])
            except ValueError:
                continue
            sm_all.append(c); mx.append(m)
            if t_begin - 0.02 <= ts <= t_end + 0.02:
                sm.append(c)
                for n, v in zip(names, f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        use = sm if sm else sm_all[-5:]
        return dict(sm_mhz=float(np.median(use)) if use else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm), samples_total=len(sm_all))


def cpu_arm():
    """The CPU arm: the UNMODIFIED reference from oracle/_ref (oracle/build_ref.py) when it travelled with the
    snapshot, else the call-for-call port oracle/cpu_reference.py (pinned bit-exactly to the reference's H by
    tests/test_oracle_golden.py)."""
    from oracle import ref_runner
    if ref_runner.available():
        return ref_runner.time_pairs, "reference", ("unmodified reference (oracle/_ref: evenvizion.processing KeyPoints.match_static_kps "
                                                    "+ compute_homography)")
    from oracle import cpu_reference
    return cpu_reference.time_pairs, "port", "reference path restated in oracle/cpu_reference.py"


def cpu_reference_run(frames, cores, steps, warmup):
    time_pairs, kind, what = cpu_arm()
    times = []
    n = ok = 0
    for i in range(warmup + steps):
        dt, n, ok = time_pairs(frames, cores)
        if i >= warmup:
            times.append(dt)
    return float(np.mean(times)), n, ok, kind, what


def run_reference(args, cfg):
    """--impl reference: the reference's CPU path (OpenCV + its Python glue) on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from evenvizion_b200 import synth
    cores = os.cpu_count() or 1
    sample_pairs = min(48 * cores, 1024)
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    ch = synth.make_chain(sample_pairs + 1, cfg["n_kp"], seed=0, device=dev, outlier_frac=cfg["outlier_frac"],
                          unmatched_frac=cfg["unmatched_frac"])
    desc = ch["desc"].cpu().numpy(); coords = ch["coords"].cpu().numpy()
    frames = [(coords[i], desc[i]) for i in range(sample_pairs + 1)]
    sec, n, ok, kind, what = cpu_reference_run(frames, cores, args.steps, min(args.warmup, 1))
    v = n / sec
    sample = f"{n} consecutive pairs of the same synthetic chain per step ({ok} with a valid H), {cores} single-threaded OpenCV workers, {what}"
    print(json.dumps({
        "impl": "reference", "metric": "frame-pairs/sec (match+RANSAC H)", "value": v, "unit": "pairs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (OpenCV CPU)", "data": "synthetic",
        "config": config_dict(cfg, args, args.gpus), "run_stats": {"sample_pairs": n, "pairs_with_valid_H": ok},
        "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def flann_agreement(desc_h, gpu_idx, gpu_surv, ratio=0.5):
    """Reported only (north_star: "agreement with its FLANN path is reported as a rate"): the reference itself uses the
    exact "BruteForce" matcher (matching.py:102-103), so the comparison is against stock cv2.FlannBasedMatcher
    (KD-tree, trees=5, checks=50) followed by the same ratio test, on the first pairs of the benchmark chain.
    top1 = share of query keypoints whose nearest neighbour agrees with the (exact) GPU result;
    survivors_jaccard = |F and G| / |F or G| of the ratio-test survivor sets."""
    try:
        import cv2
        fl = cv2.FlannBasedMatcher(dict(algorithm=1, trees=5), dict(checks=50))
        same = tot = inter = union = 0
        for k, (gi, gs) in enumerate(zip(gpu_idx, gpu_surv)):
            q = desc_h[k + 1].numpy().astype(np.float32)
            t = desc_h[k].numpy().astype(np.float32)
            raw = fl.knnMatch(q, t, 2)
            fi = np.array([m[0].trainIdx if len(m) else -1 for m in raw])
            fs = np.array([len(m) == 2 and m[0].distance < m[1].distance * ratio for m in raw])
            same += int((fi == gi[:len(fi)]).sum()); tot += len(fi)
            inter += int((fs & gs[:len(fs)]).sum()); union += int((fs | gs[:len(fs)]).sum())
        return {"top1": same / max(tot, 1), "survivors_jaccard": inter / max(union, 1), "pairs": len(gpu_idx),
                "flann": "cv2.FlannBasedMatcher KD-tree trees=5 checks=50"}
    except Exception as exc:                    # reported-only extra: never fail the benchmark line
        return {"unavailable": repr(exc)[:200]}


def int8_ceiling(torch, dev):
    """On-box dense int8 GEMM ceiling (cuBLASLt through torch._int_mm, 8192^3), TOP/s."""
    try:
        a = torch.randint(-8, 8, (8192, 8192), dtype=torch.int8, device=dev)
        b = torch.randint(-8, 8, (8192, 8192), dtype=torch.int8, device=dev).t().contiguous().t()
        for _ in range(3):
            torch._int_mm(a, b)
        best = 1e9
        for _ in range(5):
            e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
            e0.record(); torch._int_mm(a, b); e1.record(); e1.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2 * 8192 ** 3 / (best * 1e-3) / 1e12
    except Exception:
        return None


def parity_check(eng, st, keep, coords_h, desc_h, n_hyp, pair_base, n_pairs):
    """Pairs 0 .. n_pairs-1 of the LAST timed step against the oracle (oracle/pipeline.pair_geometry) on the same
    inputs: match list and both inlier masks bit-exact, static set bit-exact, H within 1e-3 px."""
    from oracle import pipeline
    r, h1, sp, sc, h2 = keep
    bad = []
    for p in range(n_pairs):
        ref = pipeline.pair_geometry(coords_h[p + 1].numpy(), desc_h[p + 1].numpy(), coords_h[p].numpy(), desc_h[p].numpy(),
                                     n_hyp=n_hyp, seed=0, pair_id=pair_base + p)
        o = int(st.row_off_h[p + 1])
        if int(r.status[p]) != ref["status"]:
            bad.append((p, "status")); continue
        if ref["status"] != 0:
            continue
        m = int(r.m_cnt[p])
        g = r.m_pts[o:o + m].cpu().numpy()
        if not (np.array_equal(g[:, :2], ref["match"]["pts_a"]) and np.array_equal(g[:, 2:], ref["match"]["pts_b"])):
            bad.append((p, "match list")); continue
        if not np.array_equal(h1["mask_best"][o:o + m].cpu().numpy().astype(bool), ref["ransac1"]["mask_best"]):
            bad.append((p, "inlier mask 1")); continue
        ms = int(sc[p])
        gs = sp[o:o + ms].cpu().numpy()
        if not (np.array_equal(gs[:, :2], ref["static_a"]) and np.array_equal(gs[:, 2:], ref["static_b"])):
            bad.append((p, "static set")); continue
        if not np.array_equal(h2["mask_best"][o:o + ms].cpu().numpy().astype(bool), ref["ransac2"]["mask_best"]):
            bad.append((p, "inlier mask 2")); continue
        q = np.c_[ref["static_a"].astype(np.float64), np.ones(ms)]
        u = q @ h2["H"][p].cpu().numpy().reshape(3, 3).T; v = q @ ref["H"].T
        if not np.abs(u[:, :2] / u[:, 2:] - v[:, :2] / v[:, 2:]).mean() < 1e-3:
            bad.append((p, "H"))
    return {"pairs": n_pairs, "ok": not bad, "against": "oracle/pipeline.pair_geometry (match list, inlier masks, static set "
            "bit-exact; H within 1e-3 px)", "failures": bad}


# --dump-outputs: per-pair outputs of up to DUMP_PAIRS pairs, per-row outputs of the pairs that hold about DUMP_ROWS query
# keypoints (both seeded samples of the step's pairs, the second inside the first), DUMP_MAX_BYTES in all
DUMP_PAIRS = 16384
DUMP_ROWS = 1 << 18
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, st, r, S, Hf, moved, K):
    """Writes what the last timed step returned to its caller as out_dir/<name>.npy, float32 or float64 (integer outputs
    as float64, which holds them exactly), so that two builds can be compared output for output on the same inputs.
    Outputs past the stage that failed a pair are not defined by the path: they are NaN (per pair) or left out (per row)
    wherever the pair's final status is not 0.

    per pair, for the pairs in `pair` (indices into the step's pairs): status, n_filtered, m_cnt, S and H_fixed [n,3,3],
    remap [n*K,2] (the K object points of each pair's frame, configs with remap points); where status is 0: H (the
    homography compute_homography returns), H1, H1_best, H2_best [n,3,3], best_hyp1/2, best_cnt1/2, inl1/2, static_cnt,
    static_r, flags.
    per row, concatenated over the pairs in `row_pair`: top2_idx, top2_d2 [.,2] and surv over the query keypoints;
    m_idx [.,2] and m_pts [.,4] over the matches, with mask1 and mask1_best (NaN where status is not 0); static_pts [.,4],
    mask2 and mask2_best over the static points of the pairs whose status is 0."""
    import torch
    P = int(r.status.numel())
    perm = np.random.default_rng(0).permutation(P)
    pairs = np.sort(perm[:DUMP_PAIRS])
    row_pairs = np.sort(perm[:max(1, DUMP_ROWS // max(st.max_kp, 1))])

    def take(t, idx):
        v = t[torch.from_numpy(np.asarray(idx, np.int64)).to(t.device)].cpu().numpy()
        return v if v.dtype in (np.float32, np.float64) else v.astype(np.float64)

    status = take(r.status, pairs)
    out = {"pair": pairs.astype(np.float64), "status": status, "n_filtered": take(r.n_filtered, pairs),
           "m_cnt": take(r.m_cnt, pairs), "S": take(S, pairs).reshape(-1, 3, 3), "H_fixed": take(Hf, pairs).reshape(-1, 3, 3)}
    if moved is not None:
        out["remap"] = take(moved, (pairs[:, None] * K + np.arange(K)).ravel())
    late = {"H": r.H, "H1": r.H1, "H1_best": r.extra["H1_best"], "H2_best": r.extra["H2_best"], "best_hyp1": r.best_hyp1,
            "best_hyp2": r.best_hyp2, "best_cnt1": r.best_cnt1, "best_cnt2": r.best_cnt2, "inl1": r.inl1, "inl2": r.inl2,
            "static_cnt": r.static_cnt, "static_r": r.static_r, "flags": r.flags}
    for name, t in late.items():
        v = take(t, pairs)
        v[status != 0] = np.nan
        out[name] = v.reshape(-1, 3, 3) if v.ndim == 2 else v

    off = take(r.out_off, row_pairs).astype(np.int64)
    n_q = st.n_kp_h[take(r.pair_q, row_pairs).astype(np.int64)]
    ok = take(r.status, row_pairs) == 0
    m_cnt = take(r.m_cnt, row_pairs).astype(np.int64)
    s_cnt = np.where(ok, take(r.static_cnt, row_pairs), 0).astype(np.int64)
    span = lambda cnt: np.concatenate([np.arange(o, o + c) for o, c in zip(off, cnt)])
    q_rows, m_rows, s_rows = span(n_q), span(m_cnt), span(s_cnt)
    out["row_pair"] = row_pairs.astype(np.float64)
    for name in ("top2_idx", "top2_d2", "surv"):
        out[name] = take(getattr(r, name), q_rows)
    out["m_idx"], out["m_pts"] = take(r.m_idx, m_rows), take(r.m_pts, m_rows)
    for name in ("mask1", "mask1_best"):
        v = take(getattr(r, name), m_rows)
        v[np.repeat(~ok, m_cnt)] = np.nan
        out[name] = v
    out["static_pts"] = take(r.static_pts, s_rows)
    for name in ("mask2", "mask2_best"):
        out[name] = take(getattr(r, name), s_rows)

    total = sum(v.nbytes for v in out.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes, more than {DUMP_MAX_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)
    print(f"bench.py: {len(out)} arrays of the last timed step ({total / 1e6:.1f} MB) written to {out_dir}", file=sys.stderr)


def run_ours(args, cfg):
    import torch
    import torch.distributed as dist
    import evenvizion_b200 as evz
    from evenvizion_b200 import synth
    from evenvizion_b200.distributed import scan_sharded

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; evenvizion_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    eng = evz.GeometryEngine(local)
    P, N, n_hyp = cfg["pairs"], cfg["n_kp"], cfg["n_hyp"]
    if args.pairs:
        P = args.pairs
    strong = bool(cfg.get("strong"))
    if strong:
        P = P // world                      # strong scaling: the job's pairs are split over the ranks
    K = int(cfg.get("remap_points", 0))
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def make_store(P, tile, shared_chain, want_host=True):
        """Synthetic shard of this rank.  weak scaling: every rank its own chain (seed = rank).  shared_chain: ONE
        video for the whole job -- every rank builds the same base chain (seed 0), repeats it `tile` times and keeps
        its contiguous frame range [rank * P, rank * P + P] (one-frame halo: the last frame of a rank is the first of
        the next)."""
        if tile > 1:
            total = P * world if shared_chain else P
            base_f = -(-(total + 1) // tile)
            ch = synth.make_chain(base_f, N, seed=0 if shared_chain else rank, device=dev, outlier_frac=cfg["outlier_frac"],
                                  unmatched_frac=cfg["unmatched_frac"])
            f0 = rank * P if shared_chain else 0
            idx = (torch.arange(f0, f0 + P + 1, device=dev) % base_f)
            ch = dict(desc=ch["desc"].index_select(0, idx), coords=ch["coords"].index_select(0, idx))
        else:
            ch = synth.make_chain(P + 1, N, seed=rank, device=dev, outlier_frac=cfg["outlier_frac"],
                                  unmatched_frac=cfg["unmatched_frac"])
        desc_h = coords_h = None
        if want_host:
            desc_h = torch.empty(ch["desc"].shape, dtype=torch.uint8).pin_memory()
            coords_h = torch.empty(ch["coords"].shape, dtype=torch.float32).pin_memory()
            desc_h.copy_(ch["desc"]); coords_h.copy_(ch["coords"])
        torch.cuda.synchronize()
        st = eng.ingest(ch["desc"], ch["coords"])
        torch.cuda.synchronize()
        st.keep = ()                        # the raw staging copies are consumed: free them (26 GB at config 5)
        return st, desc_h, coords_h

    def make_step(st, P, pair_base, K, n_hyp):
        pq = torch.arange(1, P + 1, dtype=torch.int32, device=dev)
        pt = torch.arange(0, P, dtype=torch.int32, device=dev)
        obj = None
        if K:
            g = torch.Generator(device=dev); g.manual_seed(99 + rank)
            obj_pts = torch.rand((P * K, 2), generator=g, device=dev, dtype=torch.float64) * torch.tensor([1920.0, 1080.0], device=dev, dtype=torch.float64)
            obj = (obj_pts, torch.arange(P, dtype=torch.int32, device=dev).repeat_interleave(K).contiguous())

        work = eng.alloc_results(st, pq, pt)       # every output buffer of the path, allocated once: the timed step only launches kernels

        def step(timed):
            e = [ev() for _ in range(5)] if timed else None
            if timed: e[0].record()
            r = eng.process_pairs_into(st, work, n_hyp=n_hyp, seed=0, pair_id_base=pair_base,
                                       after_match=(e[1].record if timed else None))
            if timed: e[2].record()
            S, Hf = scan_sharded(eng, r.H, r.status, True)     # one all-gather of 160 B per rank when world > 1
            if timed: e[3].record()
            moved = None
            if obj is not None:
                moved = eng.remap(obj[0], obj[1], S, 400.0 / 1920.0, 224.0 / 1080.0, False)     # frames 2.. of the shard
            if timed: e[4].record()
            h1 = dict(mask_best=r.mask1_best)
            h2 = dict(mask_best=r.mask2_best, H=r.H)
            return (r, h1, r.static_pts, r.static_cnt, h2), (S, Hf, moved), e
        return step

    def timed_run(step, steps, warmup):
        for _ in range(warmup):
            step(False)
        sync_all()
        t0, t1 = ev(), ev()
        evs = []
        w_begin = time.time()
        t0.record()
        for _ in range(steps):
            keep, scan, e = step(True)
            evs.append(e)
        t1.record()
        sync_all()
        w_end = time.time()
        total_ms = t0.elapsed_time(t1)
        per_step = np.array([[e[i].elapsed_time(e[i + 1]) for i in range(4)] for e in evs])
        if os.environ.get("EVZ_BENCH_DEBUG"):
            print(f"[rank {rank}] per-step stage ms:\n{np.round(per_step, 3)}", file=sys.stderr, flush=True)
        stage = per_step.mean(0)
        return total_ms, stage, keep, scan, (w_begin, w_end)

    tile = int(cfg.get("tile", 1))
    st, desc_h, coords_h = make_store(P, tile if P + 1 >= 2 * tile else 1, strong)
    pair_base = rank * P
    eng.set_option(4, 1)      # EVZ_OPT_TIME_MATCH: CUDA events around the main match kernel, read back after the timed region
    step = make_step(st, P, pair_base, K, n_hyp)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    total_ms, stage, keep, scan, (w_begin, w_end) = timed_run(step, args.steps, max(args.warmup, 3))
    if os.environ.get("EVZ_BENCH_DEBUG"):
        print(f"[rank {rank}] total {total_ms / args.steps:.3f} ms/step, stages {[round(float(x), 3) for x in stage]}", file=sys.stderr, flush=True)
    clocks = sampler.stop(w_begin, w_end) if rank == 0 else None
    # per-launch duration of the dominant kernel (the last min(steps, 16) launches, all inside the timed region)
    kern_ms = [eng.match_kernel_ms(k) for k in range(min(args.steps, 16))]
    r = keep[0]
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, st, r, *scan, K)
    n_ok = int((r.status == 0).sum().item())
    mean_matches = float(r.m_cnt.float().mean().item())
    mean_static = float(keep[3].float().mean().item())
    # the timed result is checked, not just timed: first pairs of the last step against the oracle (rank 0)
    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_check(eng, st, keep, coords_h, desc_h, n_hyp, pair_base, min(P, 8 if N <= 4096 else 3))
    # first pairs of the last step, kept for the reported-only FLANN agreement rate (rank 0, below)
    flann_pairs = min(8, P)
    flann_rows = [(int(st.row_off_h[q]), int(st.n_kp_h[q])) for q in range(1, flann_pairs + 1)]
    flann_idx = [r.top2_idx[o:o + n, 0].cpu().numpy() for o, n in flann_rows]
    flann_surv = [r.surv[o:o + n].cpu().numpy().astype(bool) for o, n in flann_rows]
    del r, keep, scan

    # ---- end to end through the public host API (pinned host buffers in, host arrays out)
    out = None
    for _ in range(2):
        out = None
        out = eng.video_geometry(desc_h, coords_h, n_hyp=n_hyp, seed=0, pair_id_base=pair_base)
    sync_all()
    w0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, 3))
    for _ in range(e2e_steps):
        out = None
        out = eng.video_geometry(desc_h, coords_h, n_hyp=n_hyp, seed=0, pair_id_base=pair_base)
    sync_all()
    e2e_ms = (time.perf_counter() - w0) * 1e3 / e2e_steps
    h2d = desc_h.numel() + coords_h.numel() * 4
    d2h = sum(out[k].nbytes for k in ("G", "status", "S", "H_fixed"))
    del out
    # the ceiling of the host-buffer path: the same pinned buffers copied to the device and nothing else, all ranks
    # at the same time (one cudaMemcpyAsync per buffer); e2e cannot be faster than this
    dd = torch.empty(desc_h.shape, dtype=torch.uint8, device=dev); dc = torch.empty(coords_h.shape, dtype=torch.float32, device=dev)
    for _ in range(2):
        dd.copy_(desc_h, non_blocking=True); dc.copy_(coords_h, non_blocking=True)
    sync_all()
    w0 = time.perf_counter()
    for _ in range(3):
        dd.copy_(desc_h, non_blocking=True); dc.copy_(coords_h, non_blocking=True)
    sync_all()
    h2d_ms = (time.perf_counter() - w0) * 1e3 / 3
    del dd, dc

    if world > 1:
        t = torch.tensor([total_ms, e2e_ms, h2d_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_ms, h2d_ms = float(t[0]), float(t[1]), float(t[2])
    ms_per_step = total_ms / args.steps

    # ---- N > 1: BASELINE config 5 (one 100 000-pair video sharded over the ranks with a one-frame halo, cumulative scan
    # across the shards, remap of 8 object points per frame), and the sharded scan checked against the single-GPU scan
    c5 = None
    if world > 1 and args.config == 2 and not args.no_c5:
        del st, step
        torch.cuda.empty_cache()
        c5cfg = CONFIGS[5]
        P5 = (args.pairs * 10 if args.pairs else c5cfg["pairs"]) // world
        st5, _, _ = make_store(P5, c5cfg["tile"], True, want_host=False)
        step5 = make_step(st5, P5, rank * P5, c5cfg["remap_points"], c5cfg["n_hyp"])
        t5, stage5, keep5, (S5, _, _), _ = timed_run(step5, 2, 2)
        # scan check: every rank gathers all G / status / S; the single-GPU scan over the whole video must reproduce
        # the sharded one
        G5, s5 = keep5[4]["H"].contiguous(), keep5[0].status.contiguous()
        Gall = torch.empty((world * P5, 9), dtype=torch.float64, device=dev)
        sall = torch.empty((world * P5,), dtype=torch.int32, device=dev)
        Sall = torch.empty((world * P5, 9), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(Gall, G5); dist.all_gather_into_tensor(sall, s5); dist.all_gather_into_tensor(Sall, S5.contiguous())
        S1, _, _ = eng.chain_scan(Gall, sall, True, want_fixed=False)
        err = float(((S1 - Sall).abs().max() / Sall.abs().max()).item())
        n_fail = int((sall != 0).sum().item())
        tt = torch.tensor([t5] + list(stage5), dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t5ms = float(tt[0]) / 2
        c5 = {"workload": c5cfg["name"], "pairs_total": world * P5, "pairs_per_gpu": P5, "scaling": "strong",
              "pairs_s": world * P5 / (t5ms * 1e-3), "ms_per_step": t5ms, "match_ms": float(tt[1]), "ransac_ms": float(tt[2]),
              "scan_ms": float(tt[3]), "remap_ms": float(tt[4]), "remap_points": world * P5 * c5cfg["remap_points"],
              "failed_pairs_forward_filled": n_fail,
              "scan_check": {"max_rel_diff_sharded_vs_single_gpu_scan": err, "tolerance": 1e-9, "ok": err <= 1e-9}}
        if err > 1e-9:
            raise SystemExit(f"bench.py: sharded scan differs from the single-GPU scan by {err:.3e} (relative)")
        del st5, step5, keep5, S5, Gall, sall, Sall, S1

    if rank == 0:
        pk = peaks()
        m_ms, r_ms, s_ms, rm_ms = (float(x) for x in stage)
        k_ms = float(np.mean(kern_ms))
        ops = 2.0 * N * N * 128 * P
        achieved = ops / (k_ms * 1e-3) / 1e12
        i8 = int8_ceiling(torch, dev)
        peak2 = 2.0 * pk["bf16_burst"]
        cores = os.cpu_count() or 1
        # bounded CPU baseline on the same workload (first pairs of this rank's chain)
        cpu = None
        if world == 1 and not args.no_cpu:
            sp_pairs = min(128 * cores, 2048, P)      # about 10 s of CPU work on the box's cores
            frames = [(coords_h[i].numpy(), desc_h[i].numpy()) for i in range(sp_pairs + 1)]
            sec, n, ok, kind, what = cpu_reference_run(frames, cores, 1, 0)
            cpu = {"value": n / sec, "unit": "pairs/s", "cores": cores, "kind": kind,
                   "sample": f"first {n} pairs of the same chain, one pass ({sec:.1f} s), {cores} single-threaded OpenCV workers, "
                             f"{what} ({ok} pairs with a valid H)"}
        flann = None
        if world == 1 and not args.no_cpu:
            flann = flann_agreement(desc_h, flann_idx, flann_surv)
        if parity is not None and not parity["ok"]:
            print(json.dumps({"error": "parity check against the oracle failed", "parity_check": parity}))
            raise SystemExit(1)
        alg_bytes = (P + 1) * N * (128 + 4) + P * N * 16          # SURVEY 8(d): descriptors + norms once per frame, top-2 out per pair
        traffic = MATCH_TRAFFIC_BYTES.get((args.config, P))
        evals1 = float(n_hyp) * mean_matches * P                  # nominal hypothesis x match evaluations, level 1
        evals2 = float(n_hyp) * mean_static * P
        scan_bytes = P * (72 + 4 + 72 + 72)                       # G + status in, S + H_fixed out
        print(json.dumps({
            "metric": "frame-pairs/sec (match+RANSAC H)", "value": world * P / (ms_per_step * 1e-3), "unit": "pairs/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "u8 (s32 accumulate) match; f32/f64 RANSAC", "data": "synthetic",
            "config": config_dict(cfg, args, world),
            "run_stats": {"valid_pairs_last_step": n_ok, "mean_matches_per_pair": mean_matches, "mean_static_points_per_pair": mean_static},
            "stage_ms": {"match": m_ms, "ransac_static_ransac": r_ms, "scan": s_ms, "remap": rm_ms},
            "parity_check": parity,
            "roofline": {"kernel": "match_top2_vkernel", "bound": "tensor", "unit": "TFLOP/s",
                         "achieved": achieved, "peak": peak2, "frac": achieved / peak2,
                         "peak_source": "2 x bf16_tflops of MEASURED_PEAKS.json (dense int8 = 2 x bf16 on tcgen05; the file has no int8 entry)"
                                        if pk["source"] == "MEASURED_PEAKS.json" else "2 x fallback bf16 peak (B200_PROFILING.md)",
                         "peak_nominal_int8": 4500.0, "frac_of_nominal": achieved / 4500.0,
                         "peak_int_mm_this_run": i8, "frac_of_int_mm_this_run": (achieved / i8) if i8 else None,
                         "kernel_ms": k_ms, "ops_per_launch": ops,
                         "achieved_whole_match_stage": ops / (m_ms * 1e-3) / 1e12,
                         "traffic": traffic, "algorithmic_bytes": alg_bytes,
                         "traffic_over_algorithmic": (traffic / alg_bytes) if traffic else None,
                         "note": "ops = 2*Nq*Nt*128 per pair (int8 MAC = 2 ops); the fifth K block that carries the train norms "
                                 "(+25 % tensor work) and its 32 B/row of code bytes are implementation cost, not counted as work"},
            "ransac": {"stage_ms": r_ms, "nominal_evals_level1": evals1, "nominal_evals_level2": evals2,
                       "nominal_evals_per_s": (evals1 + evals2) / (r_ms * 1e-3),
                       "bound": "SM issue (fp32)", "ncu": RANSAC_NCU,
                       "note": "evaluations = n_hyp x points per level; exact pruning (DESIGN.md K3) executes a fraction of them"},
            "scan": {"ms": s_ms, "bytes": scan_bytes, "gbs": scan_bytes / (s_ms * 1e-3) / 1e9, "peak_gbs": pk["hbm_gbs"],
                     "frac": scan_bytes / (s_ms * 1e-3) / 1e9 / pk["hbm_gbs"], "bound": "launch latency at this size (7 launches, 2 MB)"},
            "remap": ({"ms": rm_ms, "points": P * K, "bytes": P * K * 36, "gbs": P * K * 36 / (rm_ms * 1e-3) / 1e9,
                       "frac": P * K * 36 / (rm_ms * 1e-3) / 1e9 / pk["hbm_gbs"]} if K else None),
            "cpu_baseline": cpu,
            "flann_agreement": flann,
            "e2e": {"value": world * P / (e2e_ms * 1e-3), "unit": "pairs/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms,
                    "h2d_only_ms": h2d_ms, "h2d_only_gbs_per_gpu": h2d / (h2d_ms * 1e-3) / 1e9,
                    "frac_of_h2d_ceiling": h2d_ms / e2e_ms,
                    "note": "h2d_only = the same pinned buffers copied to the device and nothing else, all ranks at once: the ceiling of the host-buffer path"},
            "config5_strong": c5,
            "gpu_launches": ((KERNELS_PER_STEP_MULTI if world > 1 else KERNELS_PER_STEP) + (1 if K else 0)) * args.steps,
            "clocks": clocks, "peaks": pk,
        }))
    if world > 1:
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True
    os.environ["PYTHONDONTWRITEBYTECODE"] = "1"         # and in the CPU arm's worker processes
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--pairs", type=int, default=0, help="override pairs per GPU (debugging only)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the bounded CPU baseline")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of the last timed step")
    ap.add_argument("--no-c5", action="store_true", help="N > 1: skip the sharded 100k-pair video (config 5) and its scan check")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--impl ours: write the outputs of the last timed step to DIR/<name>.npy (rank 0's pairs when N > 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, cfg)
    else:
        run_ours(args, cfg)


if __name__ == "__main__":
    main()
