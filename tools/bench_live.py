"""Latency of one camera frame to its final poses: LiveDetector's graph replay against the two eager routes.

For every frame size and database, three routes run on the same frames, alternated frame by frame in one process:
  live    LiveDetector(pipeline, GpuSift(max_keypoints=R), size).detect([frame])
  stream  FrameStream(pipeline, GpuSift(max_keypoints=R), batch_frames=1).run([frame]) (the device path)
  eager   GpuSift.extract_batch + DetectionPipeline.load_queries / detect_device / fetch / final_poses
The metric is host wall time from a host frame (a u8 gray array) to final poses on the host, median and p99 over
--frames frames after --warmup frames.  Also reported: the device time of one replay (CUDA events around the graph
over repeated replays) and the matcher's device time at the R capacity rows against the frame's true row count, which
is what padding to the capacity costs.

Databases: the benchmark's 1,000 objects x 1,000 rows (bench.make_workload, synthetic: its objects never appear in
the frames) and a 3-object database built with cv2 SIFT from textured images that are planted in the frames.

    python tools/bench_live.py --out profiles/r10_live_bench.json

--rig 1920x1080,1280x720,640x480,640x480 times a camera rig instead: one call takes one frame per camera, host frames
to the final poses of all of them, through three routes alternated call by call:
  rig         one LiveDetector over the rig's sizes: one replay
  per_camera  one LiveDetector per size, called camera after camera (one replay and one synchronise each)
  eager       GpuSift.extract_mixed + DetectionPipeline.load_queries / detect_device / fetch / final_poses
Reported with the host times: the device time of the rig's replay and the sum of the per-camera replays.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import cv2
import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "sift-based-od_b200"))
sys.path.insert(0, str(ROOT / "tests"))
import imaging  # noqa: E402
from sod_b200.live import LiveDetector  # noqa: E402
from sod_b200.pipeline import DetectionPipeline  # noqa: E402
from sod_b200.sift import GpuSift  # noqa: E402
from sod_b200.stream import FrameStream  # noqa: E402


def small_database(rng, n_objects=3):
    """Three textured 600x400 objects through cv2 SIFT, as the reference's GenerateDatabaseInfo stores them."""
    from SiftHelperFunctions import get_centroid, make_temp_kp
    from sod_b200.database import PackedDatabase
    rows, objs = [], []
    for i in range(n_objects):
        obj = imaging.textured(rng, 600, 400)
        kp, des = cv2.SIFT_create().detectAndCompute(obj, None)
        rows.append([make_temp_kp(kp), des, (600, 400), get_centroid(kp), f"obj{i}.png"])
        objs.append(obj)
    mdb = PackedDatabase.from_reference_rows(rows).to_model_database()
    mdb.object_of_image = np.arange(n_objects, dtype=np.int32)
    return mdb, objs


def big_database():
    import bench
    args = type("A", (), dict(objects=1000, kp_per_object=1000, frames=1, per_frame=64, instances=1,
                              inlier_frac=0.2, false_frac=0.02))()
    return bench.make_database(bench.make_workload(args, torch.device("cuda")))


def scene_frames(rng, objs, w, h, n):
    frames = []
    for _ in range(n):
        fr = imaging.textured(rng, w, h, shapes=200)
        for _ in range(2):
            o = int(rng.integers(0, len(objs)))
            fr, _ = imaging.place(rng, fr, objs[o], w / 1200.0 * float(rng.uniform(0.6, 1.1)),
                                  float(rng.uniform(-90, 90)), w * float(rng.uniform(0.3, 0.7)),
                                  h * float(rng.uniform(0.3, 0.7)))
        frames.append(fr)
    return frames


def eager_route(pipe, sift, frame, w, h):
    sb = sift.extract_batch([frame])
    if sb.rows == 0:
        return {}
    pipe.scene.frame_wh[:, 0].fill_(w)
    pipe.scene.frame_wh[:, 1].fill_(h)
    pipe.load_queries(sb.des, sb.xy, sb.angle, sb.octave, sb.frame)
    return pipe.final_poses(pipe.fetch(pipe.detect_device(sb.rows)))


def stats(ms):
    a = np.asarray(ms)
    return dict(median_ms=float(np.median(a)), p99_ms=float(np.percentile(a, 99)), mean_ms=float(a.mean()), n=len(a))


def device_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def run(db_name, mdb, sizes, frames_by_size, args):
    out = {}
    R = args.max_keypoints
    pipe = DetectionPipeline(mdb, max_queries=R, frame_wh=np.zeros((1, 2), np.int32))
    sift = GpuSift(max_keypoints=R)
    for (w, h) in sizes:
        pool = frames_by_size[(w, h)]
        live = LiveDetector(pipe, sift, (w, h))
        stream = FrameStream(pipe, sift, batch_frames=1, workers=1)
        routes = {
            "live": lambda f: live.detect([f])[0]["final_pose"],
            "stream": lambda f: next(iter(stream.run([f])))[1]["final_pose"],
            "eager": lambda f: eager_route(pipe, sift, f, w, h),
        }
        times = {k: [] for k in routes}
        for i in range(args.warmup + args.frames):
            f = pool[i % len(pool)]
            for name in (list(routes) if i % 2 == 0 else list(routes)[::-1]):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                routes[name](f)
                t1 = time.perf_counter()
                if i >= args.warmup:
                    times[name].append((t1 - t0) * 1e3)
        # rows per frame, replay device time, matcher at the capacity against the true rows
        counts = [int(sift.extract_batch([f]).count[0]) for f in pool]
        live.detect([pool[0]])
        graph = live._graph(True)[0]
        replay = device_ms(graph.replay, 50)
        q = pipe.q_des
        n_true = int(np.median(counts))
        m_cap = device_ms(lambda: pipe.matcher.top2(q[:R]), 50)
        m_true = device_ms(lambda: pipe.matcher.top2(q[:max(n_true, 1)]), 50)
        rec = dict(size=[w, h], rows_per_frame=counts, capacity_rows=R,
                   host_ms={k: stats(v) for k, v in times.items()}, replay_device_ms=replay,
                   matcher_device_ms={"capacity_rows": m_cap, "true_rows_median": m_true, "true_rows": n_true})
        print(db_name, f"{w}x{h}", json.dumps({k: round(v["median_ms"], 3) for k, v in rec["host_ms"].items()}),
              f"replay {replay:.3f} ms, matcher {m_cap:.3f} ms at {R} rows / {m_true:.3f} ms at {n_true}", flush=True)
        out[f"{w}x{h}"] = rec
    return out


def run_rig(db_name, mdb, sizes, pool, args):
    R, B = args.max_keypoints, len(sizes)
    pipe = DetectionPipeline(mdb, max_queries=B * R, frame_wh=np.zeros((B, 2), np.int32))
    sift = GpuSift(max_keypoints=R)
    rig = LiveDetector(pipe, sift, sizes)
    cams = {s: LiveDetector(pipe, sift, s) for s in sizes}

    def eager(frames):
        sb = sift.extract_mixed(frames)
        if sb.rows == 0:
            return {}
        pipe.scene.frame_wh[:B].copy_(torch.from_numpy(sb.frame_sizes.astype(np.int32)))
        pipe.load_queries(sb.des, sb.xy, sb.angle, sb.octave, sb.frame)
        return pipe.final_poses(pipe.fetch(pipe.detect_device(sb.rows)))

    routes = {
        "rig": lambda fr: [r["final_pose"] for r in rig.detect(fr)],
        "per_camera": lambda fr: [cams[s].detect([f])[0]["final_pose"] for s, f in zip(sizes, fr)],
        "eager": eager,
    }
    times = {k: [] for k in routes}
    for i in range(args.warmup + args.frames):
        fr = pool[i % len(pool)]
        for name in (list(routes) if i % 2 == 0 else list(routes)[::-1]):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            routes[name](fr)
            t1 = time.perf_counter()
            if i >= args.warmup:
                times[name].append((t1 - t0) * 1e3)
    rig_replay = device_ms(rig._graph(True)[0].replay, 50)
    cam_replay = {f"{w}x{h}": device_ms(cams[(w, h)]._graph(True)[0].replay, 50) for w, h in cams}
    per_camera = sum(cam_replay[f"{w}x{h}"] for w, h in sizes)
    rows = [int(c) for c in sift.extract_mixed(pool[0]).count]
    rec = dict(sizes=[list(s) for s in sizes], capacity_rows_per_frame=R, rows_first_call=rows,
               host_ms={k: stats(v) for k, v in times.items()},
               replay_device_ms=dict(rig=rig_replay, per_camera_sum=per_camera, per_size=cam_replay))
    print(db_name, "rig", json.dumps({k: round(v["median_ms"], 3) for k, v in rec["host_ms"].items()}),
          f"replay {rig_replay:.3f} ms, per-camera replays {per_camera:.3f} ms", flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--max-keypoints", type=int, default=4000)
    ap.add_argument("--pool", type=int, default=8, help="distinct frames per size, cycled")
    ap.add_argument("--sizes", default="640x480,1200x900,2000x1500")
    ap.add_argument("--rig", default=None, help="camera sizes of a rig, e.g. 1920x1080,1280x720,640x480,640x480")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_live needs a CUDA device")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    print("card:", card[0] if card else "unknown", flush=True)
    sizes = [tuple(int(v) for v in s.split("x")) for s in args.sizes.split(",")]
    rng = np.random.default_rng(11)
    small, objs = small_database(rng)
    if args.rig:
        rig = [tuple(int(v) for v in s.split("x")) for s in args.rig.split(",")]
        by_size = {s: scene_frames(rng, objs, *s, args.pool) for s in set(rig)}
        pool = [[by_size[s][(i + k) % args.pool] for k, s in enumerate(rig)] for i in range(args.pool)]
        result = dict(card=card[0] if card else None, frames=args.frames, warmup=args.warmup,
                      max_keypoints=args.max_keypoints, rig={})
        result["rig"]["3 objects"] = run_rig("3 objects", small, rig, pool, args)
        result["rig"]["1000 objects x 1000 rows"] = run_rig("1000 x 1000", big_database(), rig, pool, args)
        if args.out:
            Path(args.out).parent.mkdir(parents=True, exist_ok=True)
            Path(args.out).write_text(json.dumps(result, indent=1))
        return
    frames = {s: scene_frames(rng, objs, *s, args.pool) for s in sizes}
    result = dict(card=card[0] if card else None, frames=args.frames, warmup=args.warmup,
                  max_keypoints=args.max_keypoints, databases={})
    result["databases"]["3 objects"] = run("3 objects", small, sizes, frames, args)
    result["databases"]["1000 objects x 1000 rows"] = run("1000 x 1000", big_database(), sizes, frames, args)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
