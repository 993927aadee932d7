"""RANSAC on both sides of the scoring kernel's shared-memory choice.  At 12 288 points per pair (EVZ_MAX_KP) the four
u16 lists of a hypothesis (8 bytes each) fit in shared memory next to the points for up to 944 hypotheses; from 945 on
they live in handle scratch.  bench.py config 2 times the shared-memory side at its own sizes; this script times the
global side at the reference's default of 1 024 hypotheses, with 944 hypotheses (shared memory, same points) beside it.

Workload: --pairs pairs of 12 288 point pairs (_mk of tests/test_gpu_size_limits.py: a near-identity homography,
0.5 px noise, --outliers outliers), one evz_find_homography call per repetition (level 1, threshold 3).  Times are CUDA
events around the call, after two warm-up calls, median of --reps.  Prints one JSON line.

    python scripts/bench_ransac_lists.py [--pairs 1000] [--reps 5] [--outliers 0.3] [--level 1]
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

N = 12288


def point_sets(n_pairs, out_frac, seed):
    rng = np.random.default_rng(seed)
    pts = np.zeros((n_pairs * N, 4), np.float32)
    for p in range(n_pairs):
        a = (rng.random((N, 2)) * [1920, 1080]).astype(np.float32)
        th, s = rng.normal() * 0.01, 1 + rng.normal() * 0.01
        Ht = np.array([[s * np.cos(th), -s * np.sin(th), rng.normal() * 8], [s * np.sin(th), s * np.cos(th), rng.normal() * 8],
                       [rng.normal() * 1e-5, rng.normal() * 1e-5, 1]])
        q = np.c_[a, np.ones(N)] @ Ht.T
        b = (q[:, :2] / q[:, 2:] + rng.normal(size=(N, 2)) * 0.5).astype(np.float32)
        o = rng.random(N) < out_frac
        b[o] = (rng.random((int(o.sum()), 2)) * [1920, 1080]).astype(np.float32)
        pts[p * N:(p + 1) * N, :2], pts[p * N:(p + 1) * N, 2:] = a, b
    return pts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--outliers", type=float, default=0.3)
    ap.add_argument("--level", type=int, default=1)
    args = ap.parse_args()
    eng = evz.GeometryEngine(0)
    dev = eng.device
    P = args.pairs
    pts = torch.from_numpy(point_sets(P, args.outliers, 1)).to(dev)
    off = torch.arange(P, dtype=torch.int32, device=dev) * N
    cnt = torch.full((P,), N, dtype=torch.int32, device=dev)
    status = torch.zeros(P, dtype=torch.int32, device=dev)
    res = {}
    for n_hyp in (944, 1024):
        out = dict(H=torch.zeros((P, 9), dtype=torch.float64, device=dev), inl_cnt=torch.zeros(P, dtype=torch.int32, device=dev),
                   best_cnt=torch.zeros(P, dtype=torch.int32, device=dev))
        ms = []
        for r in range(args.reps + 2):
            status.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            eng.find_homography(pts, off, cnt, status, N, n_hyp, 0, 0, args.level, 3.0, 0.0, 4, out=out)
            e1.record()
            torch.cuda.synchronize()
            if r >= 2:
                ms.append(e0.elapsed_time(e1))
        ok = int((status == 0).sum())
        res[str(n_hyp)] = dict(lists="shared" if n_hyp == 944 else "global", ms_median=float(np.median(ms)),
                               ms_min=float(np.min(ms)), ms_max=float(np.max(ms)), us_per_pair=float(np.median(ms)) * 1e3 / P,
                               pairs_ok=ok, mean_best_cnt=float(out["best_cnt"].double().mean()))
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps(dict(pairs=P, points=N, outliers=args.outliers, level=args.level, reps=args.reps,
                          gpu=smi[0] if smi else "unknown", results=res)))


if __name__ == "__main__":
    main()
