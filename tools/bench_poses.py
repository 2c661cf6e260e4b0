"""Device time of sod_final_poses (Main.post_process on the device) for V bins per frame and B frames, plus the
worst cases of its walks, and the host time of post_process_arrays on the same inputs.

    python tools/bench_poses.py --out profiles/r11_poses_bench.json
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "sift-based-od_b200"))

from sod_b200 import engine as E  # noqa: E402
from sod_b200 import postprocess as P  # noqa: E402


def _frames(rng, v, b):
    """b frames of v bins each, as the affine stage leaves them: a few objects per frame, bins near each other."""
    n = v * b
    cx = rng.uniform(0, 1200, n) + rng.integers(0, 4, n) * 2000.0
    cy = rng.uniform(0, 900, n)
    scale = rng.uniform(0.3, 1.5, n)
    angle = rng.uniform(-np.pi, np.pi, n)
    w, h = np.full(n, 640.0), np.full(n, 480.0)
    return np.stack([cx, cy, angle, scale, w, h], 1), np.repeat(np.arange(b, dtype=np.int32), v)


def _device_ms(mean, seg, reps):
    n = mean.shape[0]
    fp = E.FinalPoses(n, "cuda")
    md, sd = torch.from_numpy(mean).cuda(), torch.from_numpy(seg).cuda()
    fp.run(md, sd, n)
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fp.run(md, sd, n)
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times))


def _host_ms(mean, seg, reps):
    import time
    args = (mean[:, 0], mean[:, 1], mean[:, 3], mean[:, 2], mean[:, 4], mean[:, 5])
    P.post_process_arrays(*args, segment=seg)
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        P.post_process_arrays(*args, segment=seg)
        times.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rng = np.random.default_rng(0)
    rows = []
    for v in (10, 100, 1000, 4096):
        for b in (1, 16, 256):
            if v * b > 65536:
                rows.append(dict(v=v, b=b, note="not measured: more than 65,536 bins in one call"))
                continue
            mean, seg = _frames(rng, v, b)
            rows.append(dict(v=v, b=b, device_ms=_device_ms(mean, seg, args.reps),
                             post_process_arrays_ms=_host_ms(mean, seg, min(args.reps, 5))))
            print(rows[-1], flush=True)
    n = 4096                                     # one cluster, all within 1 degree
    one = np.stack([rng.uniform(0, 50, n), rng.uniform(0, 50, n), 0.3 + rng.uniform(0, np.radians(0.9), n),
                    rng.uniform(1.0, 2.0, n), np.full(n, 1000.0), np.full(n, 800.0)], 1)
    worst = {"one_cluster_4096_within_1_degree": _device_ms(one, np.zeros(n, np.int32), args.reps)}
    r = np.random.default_rng(8)                 # test_cluster_past_the_recursion_limit_equals_oracle's chain
    n = 2200
    cx = np.concatenate([np.arange(1500) * 100.0 + r.uniform(-20, 20, 1500), r.uniform(0, 150000, n - 1500)])
    cy = np.concatenate([r.uniform(-30, 30, 1500), r.uniform(2000, 50000, n - 1500)])
    scale = r.choice([0.5, 1.0, 2.0], n)
    angle = r.choice([0.1, 0.11, 0.125, 0.5, 2.0], n) + r.uniform(-0.004, 0.004, n)
    perm = r.permutation(n)
    chain = np.stack([cx[perm], cy[perm], angle[perm], scale[perm], np.full(n, 1500.0), np.full(n, 1000.0)], 1)
    worst["chain_2200"] = _device_ms(chain, np.zeros(n, np.int32), args.reps)
    print(worst, flush=True)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    result = dict(card=card[0] if card else torch.cuda.get_device_name(),
                  what="sod_final_poses device time (CUDA events around the call, median) and post_process_arrays "
                       "host time (upload, call, read-back, Python lists)",
                  sizes=rows, worst_ms=worst)
    if args.out:
        Path(args.out).write_text(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
