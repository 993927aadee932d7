"""Many videos per call: a loop of geometry_from_features (one video per call) against one geometry_from_features_batch
call, in both modes, on three workloads:

  clip16   the bundled clip's SIFT + ORB features (tests/golden/clip_full.npz, 121 frames of 400x224) as 16 videos
  synth64  64 synthetic videos x 121 frames x 512 keypoints (evenvizion_b200.synth.make_chain), SIFT only
  long1    one synthetic video of 2 001 frames (2 000 pairs) x 2 048 keypoints: one long reference chain

Features are extracted beforehand; detection is not timed.  Times are host time ending in torch.cuda.synchronize(),
after one warm-up call of each variant on every workload, median of --reps runs.  Agreement: both arms must give the
same status and the same bits in both modes.

    python scripts/bench_batch.py [--reps 3] [--n-hyp 1024] [--only clip16,synth64,long1]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import evenvizion_b200  # noqa: E402
from evenvizion_b200 import synth  # noqa: E402
from evenvizion_b200.processing import geometry_from_features, geometry_from_features_batch  # noqa: E402


def clip16():
    z = np.load(os.path.join(ROOT, "tests", "golden", "clip_full.npz"))
    n = int(z["n_frames"])
    v = {t: [(z[f"{t.lower()}{f}_c"], z[f"{t.lower()}{f}_d"]) for f in range(n)] for t in ("SIFT", "ORB")}
    return [v] * 16


def synth_videos(n_videos, n_frames, n_kp, seed):
    out = []
    for i in range(n_videos):
        ch = synth.make_chain(n_frames, n_kp, seed=seed + i, device="cuda")
        d, c = ch["desc"].cpu().numpy(), ch["coords"].cpu().numpy()
        out.append({"SIFT": [(c[f], d[f]) for f in range(n_frames)]})
    return out


def agree(loop, batch):
    status = all(np.array_equal(a[1], b[1]) for a, b in zip(loop, batch))
    bits = all(len(a[0]) == len(b[0]) and all(np.array_equal(x, y) for x, y in zip(a[0], b[0])) for a, b in zip(loop, batch))
    return dict(ok=bool(status and bits), status_equal=bool(status), bits_equal=bool(bits))


def timed(fn, reps):
    ts, out = [], None
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--n-hyp", type=int, default=1024)
    ap.add_argument("--only", default="clip16,synth64,long1")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_batch.py needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps({"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None}))
    eng = evenvizion_b200.default_engine()
    makers = {"clip16": clip16, "synth64": lambda: synth_videos(64, 121, 512, 100), "long1": lambda: synth_videos(1, 2001, 2048, 7)}
    for name in args.only.split(","):
        videos = makers[name]()
        n_pairs = sum(len(next(iter(v.values()))) - 1 for v in videos)
        for mode in ("parallel", "reference"):
            loop_fn = lambda: [geometry_from_features(v, True, mode, args.n_hyp, 0, eng) for v in videos]
            batch_fn = lambda: geometry_from_features_batch(videos, True, mode, args.n_hyp, 0, eng)
            loop_fn(); batch_fn()                                  # warm-up of every shape
            t_loop, r_loop = timed(loop_fn, args.reps)
            t_batch, r_batch = timed(batch_fn, args.reps)
            print(json.dumps(dict(workload=name, mode=mode, videos=len(videos), pairs=n_pairs,
                                  loop_s=round(t_loop, 4), batch_s=round(t_batch, 4),
                                  loop_videos_per_s=round(len(videos) / t_loop, 2), batch_videos_per_s=round(len(videos) / t_batch, 2),
                                  loop_pairs_per_s=round(n_pairs / t_loop, 1), batch_pairs_per_s=round(n_pairs / t_batch, 1),
                                  speedup=round(t_loop / t_batch, 3), agree=agree(r_loop, r_batch))), flush=True)


if __name__ == "__main__":
    main()
