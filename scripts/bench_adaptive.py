"""The confidence-bounded RANSAC stop (evz_find_homography_adaptive) against the fixed hypothesis count, on the config-2
and config-4 shapes of bench.py (synth.make_chain: 2 048 keypoints per frame, 10 000 pairs; config 2: 20 % outliers,
1 024 hypotheses; config 4: 80 % outliers, 2 % unmatched, 4 096 hypotheses).

Per config, in one run and alternating fixed / adaptive (confidence --conf):
  step   a full per-pair step (process_pairs_into: match, RANSAC #1, static filter, RANSAC #2), CUDA events, --steps each;
  ransac RANSAC #1 alone on the step's match lists, CUDA events, --steps each;
  n_used percentiles per level, status agreement, and the distance between the adaptive and the fixed H over a 9 x 6
  grid of the frame (median / max over the pairs where both found one).
The card's name and power limit are read in the same run.  Prints one JSON line.

    python scripts/bench_adaptive.py [--steps 20] [--warmup 2] [--conf 0.995] [--configs 2,4]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import evenvizion_b200 as evz  # noqa: E402
from evenvizion_b200 import _lib, synth  # noqa: E402

SHAPES = {2: dict(n_kp=2048, pairs=10000, n_hyp=1024, outlier_frac=0.2, unmatched_frac=0.0),
          4: dict(n_kp=2048, pairs=10000, n_hyp=4096, outlier_frac=0.8, unmatched_frac=0.02)}


def _events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def _stats(ms):
    return dict(median=float(np.median(ms)), min=float(np.min(ms)), max=float(np.max(ms)))


def run_config(eng, cfg, args):
    dev = eng.device
    P = cfg["pairs"]
    ch = synth.make_chain(P + 1, cfg["n_kp"], seed=0, device=dev, outlier_frac=cfg["outlier_frac"],
                          unmatched_frac=cfg["unmatched_frac"])
    st = eng.ingest(ch["desc"], ch["coords"])
    pq = torch.arange(1, P + 1, dtype=torch.int32, device=dev)
    pt = torch.arange(0, P, dtype=torch.int32, device=dev)
    r_fix = eng.alloc_results(st, pq, pt)
    r_ad = eng.alloc_results(st, pq, pt, confidence=args.conf)
    n_hyp = cfg["n_hyp"]
    step = {"fixed": lambda: eng.process_pairs_into(st, r_fix, n_hyp, 0),
            "adaptive": lambda: eng.process_pairs_into(st, r_ad, n_hyp, 0, confidence=args.conf)}
    times = {"fixed": [], "adaptive": []}
    for i in range(args.warmup + args.steps):
        for name in ("fixed", "adaptive"):
            e0, e1 = _events()
            e0.record()
            step[name]()
            e1.record()
            torch.cuda.synchronize()
            if i >= args.warmup:
                times[name].append(e0.elapsed_time(e1))
    # RANSAC #1 alone, on the match lists of the last step (status as the match stage left it)
    v = eng.match(st, pq, pt)
    status0 = v.status.clone()
    status = torch.empty_like(status0)
    outs = {k: dict(H=torch.zeros((P, 9), dtype=torch.float64, device=dev), inl_cnt=torch.zeros(P, dtype=torch.int32, device=dev),
                    mask_best=torch.zeros(st.rows, dtype=torch.uint8, device=dev)) for k in times}
    outs["adaptive"]["n_used"] = torch.zeros(P, dtype=torch.int32, device=dev)
    rtimes = {"fixed": [], "adaptive": []}
    for i in range(args.warmup + args.steps):
        for name in ("fixed", "adaptive"):
            status.copy_(status0)
            e0, e1 = _events()
            e0.record()
            eng.find_homography(v.m_pts, v.out_off, v.m_cnt, status, st.max_kp, n_hyp, 0, 0, 1, 3.0, 0.0, _lib.ST_NO_MODEL_1,
                                out=outs[name], confidence=args.conf if name == "adaptive" else None)
            e1.record()
            torch.cuda.synchronize()
            if i >= args.warmup:
                rtimes[name].append(e0.elapsed_time(e1))
    # outputs of the last full steps
    sf, sa = r_fix.status.cpu().numpy(), r_ad.status.cpu().numpy()
    both = (sf == 0) & (sa == 0)
    W, H = float(ch["coords"][..., 0].max()), float(ch["coords"][..., 1].max())
    g = np.stack(np.meshgrid(np.linspace(0, W, 9), np.linspace(0, H, 6)), -1).reshape(-1, 2)
    g = np.c_[g, np.ones(len(g))]
    Hf = r_fix.H.cpu().numpy().reshape(-1, 3, 3)[both]
    Ha = r_ad.H.cpu().numpy().reshape(-1, 3, 3)[both]
    xf, xa = np.einsum("pij,kj->pki", Hf, g), np.einsum("pij,kj->pki", Ha, g)
    d = np.linalg.norm(xf[..., :2] / xf[..., 2:] - xa[..., :2] / xa[..., 2:], axis=-1).max(1) if len(Hf) else np.zeros(1)
    pct = lambda x: {str(q): int(np.percentile(x, q)) for q in (5, 25, 50, 75, 95, 100)}
    nu1 = r_ad.extra["n_used1"].cpu().numpy()
    nu2 = r_ad.extra["n_used2"].cpu().numpy()
    tf, ta = np.median(times["fixed"]), np.median(times["adaptive"])
    rf, ra = np.median(rtimes["fixed"]), np.median(rtimes["adaptive"])
    return dict(pairs=P, n_kp=cfg["n_kp"], n_hyp=n_hyp, outlier_frac=cfg["outlier_frac"],
                step_ms=dict(fixed=_stats(times["fixed"]), adaptive=_stats(times["adaptive"]), adaptive_over_fixed=float(ta / tf)),
                ransac1_ms=dict(fixed=_stats(rtimes["fixed"]), adaptive=_stats(rtimes["adaptive"]), adaptive_over_fixed=float(ra / rf)),
                n_used_level1=pct(nu1[nu1 > 0]) if (nu1 > 0).any() else {},
                n_used_level2=pct(nu2[nu2 > 0]) if (nu2 > 0).any() else {},
                pairs_ok=dict(fixed=int((sf == 0).sum()), adaptive=int((sa == 0).sum())),
                status_equal=int((sf == sa).sum()),
                H_grid_px=dict(pairs=int(both.sum()), median=float(np.median(d)), max=float(np.max(d))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--conf", type=float, default=0.995)
    ap.add_argument("--configs", default="2,4")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_adaptive.py needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    eng = evz.GeometryEngine(0)
    res = {f"config{c}": run_config(eng, SHAPES[int(c)], args) for c in args.configs.split(",")}
    print(json.dumps(dict(gpu=smi[0] if smi else "unknown", confidence=args.conf, steps=args.steps, results=res)))


if __name__ == "__main__":
    main()
