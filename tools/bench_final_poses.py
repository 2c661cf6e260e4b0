"""What the final poses cost on the host, for a before / after comparison of two checkouts of this library.

For the 3-object database of tools/bench_live.py (its objects planted twice in every frame, so poses are found),
per frame size:
  live     host wall time of LiveDetector.detect([frame]), and the part of it spent in DetectionPipeline.final_poses
           (a checkout whose replay ends with the poses never calls it: reported as null)
  stream   DetectionPipeline.final_poses on the fetched result of a 16-frame FrameStream batch (host wall time of the
           call, every batch)
Median, p99 and the count of each.  --tree selects the checkout whose sod_b200 (and tools / tests helpers) are
imported; run the two checkouts in alternating processes:

    python tools/bench_final_poses.py --tree <checkout> --out result.json
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch


def stats(ms):
    if not ms:
        return None
    a = np.asarray(ms)
    return dict(median_ms=float(np.median(a)), p99_ms=float(np.percentile(a, 99)), n=len(a))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", default=str(Path(__file__).resolve().parent.parent))
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--batches", type=int, default=12)
    ap.add_argument("--max-keypoints", type=int, default=4000)
    ap.add_argument("--sizes", default="640x480,1200x900,2000x1500")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    tree = Path(args.tree).resolve()
    sys.path.insert(0, str(tree / "tools"))
    import bench_live as BL          # puts the checkout's package and test helpers on sys.path
    from sod_b200.live import LiveDetector
    from sod_b200.pipeline import DetectionPipeline
    from sod_b200.sift import GpuSift
    from sod_b200.stream import FrameStream
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    sizes = [tuple(int(v) for v in s.split("x")) for s in args.sizes.split(",")]
    rng = np.random.default_rng(11)
    mdb, objs = BL.small_database(rng)
    R, B = args.max_keypoints, 16
    pipe = DetectionPipeline(mdb, max_queries=B * R, frame_wh=np.zeros((B, 2), np.int32))
    sift = GpuSift(max_keypoints=R)
    inner: list[float] = []
    final_poses = pipe.final_poses

    def timed(out):
        t0 = time.perf_counter()
        r = final_poses(out)
        inner.append((time.perf_counter() - t0) * 1e3)
        return r

    pipe.final_poses = timed
    result = dict(card=card[0] if card else None, frames=args.frames, warmup=args.warmup,
                  batches=args.batches, max_keypoints=R, sizes={})
    for (w, h) in sizes:
        pool = BL.scene_frames(rng, objs, w, h, 8)
        live = LiveDetector(pipe, sift, (w, h))
        host, inside, found = [], [], 0
        for i in range(args.warmup + args.frames):
            del inner[:]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            (res,) = live.detect([pool[i % len(pool)]])
            t1 = time.perf_counter()
            if i >= args.warmup:
                host.append((t1 - t0) * 1e3)
                inside.extend(inner)
                found += len(res["final_pose"])
        stream = FrameStream(pipe, sift, batch_frames=B, workers=1)
        del inner[:]
        batch_ms = []
        for b in range(args.batches + 1):
            frames = [pool[(b + k) % len(pool)] for k in range(B)]
            del inner[:]
            list(stream.run(frames))
            if b > 0:
                batch_ms.extend(inner)
        rec = dict(live_detect=stats(host), final_poses_inside_detect=stats(inside), poses_per_frame=found / args.frames,
                   stream_16_frames_final_poses=stats(batch_ms))
        result["sizes"][f"{w}x{h}"] = rec
        print(f"{w}x{h}", json.dumps({k: (round(v["median_ms"], 3) if isinstance(v, dict) else v)
                                       for k, v in rec.items()}), flush=True)
    if args.out:
        Path(args.out).write_text(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
