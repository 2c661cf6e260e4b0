"""GPU SIFT (sod_b200.sift.GpuSift) against host cv2.SIFT, per frame and through FrameStream, in one run.

    python tools/bench_sift.py --out profiles/sift_bench.json

Per size (640x480, 1200x900, 2000x1500 synthetic frames): device time of sod_sift_extract (CUDA events on the
extractor's stream), wall time of a whole GpuSift call (upload, kernels, read-back), device time of the pyramid
alone (sod_sift_describe of one keypoint: the descriptor costs one block) with its bytes computed from the
shapes, and host cv2.SIFT_create().detectAndCompute.  Then FrameStream frames/s on a 3-object cv2 database with
each extractor.  Every timed pass is preceded by warm-up passes of the same shape; the pyramid of a 1200x900
frame (144 MB) does not fit the 126 MB L2, smaller ones mostly do (stated per size in the record).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import cv2
import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "sift-based-od_b200"))
sys.path.insert(0, str(ROOT / "tests"))
import imaging  # noqa: E402
from sod_b200 import _capi  # noqa: E402
from sod_b200.sift import GpuSift  # noqa: E402

L2_BYTES = 126 * 2 ** 20


def pyramid_bytes(w, h):
    """Minimum DRAM traffic of the pyramid: u8 in, the doubled image written and read once, and per octave five
    blurs that each read their source level and write their level, plus the halving (read a quarter, write)."""
    lib = _capi.lib
    n_oct, total, wh = 0, w * h + 3 * (4 * w * h * 4), (C.c_int32 * 2)()
    while lib.sod_sift_level_offset(w, h, n_oct - 1, 0, C.cast(wh, C.c_void_p)) >= 0:
        px = wh[0] * wh[1]
        total += 5 * 2 * 4 * px + (2 * 4 * px if n_oct else 0)
        n_oct += 1
    return total, n_oct


def device_ms(stream, fn, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record(stream)
    for _ in range(reps):
        fn()
    end.record(stream)
    end.synchronize()
    return start.elapsed_time(end) / reps


def per_frame(gpu, w, h, reps, host_reps):
    gray = imaging.textured(np.random.default_rng(w), w, h, shapes=200)
    for _ in range(3):
        r = gpu.extract(gray)
    lib, st = _capi.lib, gpu._stream
    b = gpu._upload(gray)
    one = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in
           (r["xy"][:1], r["size"][:1], r["angle"][:1], r["octave"][:1])]
    des = torch.empty((1, 128), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def extract():
        _capi.check(lib.sod_sift_extract(b.img.data_ptr(), w, h, w, C.byref(b.out), b.ws.data_ptr(), b.bytes,
                                         st.cuda_stream), "sod_sift_extract")

    def pyramid():
        _capi.check(lib.sod_sift_describe(b.img.data_ptr(), w, h, w, *(t.data_ptr() for t in one), 1, des.data_ptr(),
                                          None, b.ws.data_ptr(), b.bytes, st.cuda_stream), "sod_sift_describe")

    device_ms(st, extract, 3)
    dev = device_ms(st, extract, reps)
    device_ms(st, pyramid, 3)
    pyr = device_ms(st, pyramid, reps)
    t = time.perf_counter()
    for _ in range(reps):
        gpu.extract(gray)
    wall = (time.perf_counter() - t) / reps * 1e3
    sift = cv2.SIFT_create()
    sift.detectAndCompute(gray, None)
    t = time.perf_counter()
    for _ in range(host_reps):
        kp, _ = sift.detectAndCompute(gray, None)
    host = (time.perf_counter() - t) / host_reps * 1e3
    nbytes, n_oct = pyramid_bytes(w, h)
    ws_pyr = int(lib.sod_sift_workspace_bytes(w, h, 0))
    return dict(width=w, height=h, keypoints_gpu=len(r["xy"]), keypoints_cv2=len(kp), gpu_extract_device_ms=dev,
                gpu_call_wall_ms=wall, cv2_host_ms=host, speedup_device_vs_cv2=host / dev,
                speedup_call_vs_cv2=host / wall, pyramid_device_ms=pyr, pyramid_octaves=n_oct,
                pyramid_min_bytes=nbytes, pyramid_gbps=nbytes / (pyr * 1e-3) / 1e9, pyramid_workspace_bytes=ws_pyr,
                pyramid_fits_l2=ws_pyr <= L2_BYTES)


def stream_fps(n_frames, workers):
    from SiftHelperFunctions import get_centroid, make_temp_kp
    from sod_b200.database import PackedDatabase
    from sod_b200.pipeline import DetectionPipeline
    from sod_b200.stream import FrameStream, sift_features
    rng = np.random.default_rng(7)
    rows, objs = [], []
    for i in range(3):
        obj = imaging.textured(rng, 600, 400)
        kp, des = cv2.SIFT_create().detectAndCompute(obj, None)
        rows.append([make_temp_kp(kp), des, (600, 400), get_centroid(kp), f"obj{i}.png"])
        objs.append(obj)
    db = PackedDatabase.from_reference_rows(rows)
    frames = []
    for i in range(n_frames):
        fr = imaging.textured(rng, 1200, 900, shapes=200)
        fr, _ = imaging.place(rng, fr, objs[i % 3], 0.8, 20 * i, 600, 450)
        frames.append(fr)
    out = {}
    for name, ex in (("cv2", sift_features), ("gpu", GpuSift())):
        pipe = DetectionPipeline(db.to_model_database(), max_queries=40000, frame_wh=np.zeros((4, 2), np.int32),
                                 per_object_spaces=False)
        fs = FrameStream(pipe, extractor=ex, batch_frames=4, workers=workers)
        for _ in fs.run(frames[:8]):
            pass
        t = time.perf_counter()
        found = sum(len(r["final_pose"]) > 0 for _, r in fs.run(frames))
        dt = time.perf_counter() - t
        out[name] = dict(frames=n_frames, seconds=dt, frames_per_s=n_frames / dt, frames_with_a_pose=found)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--stream-frames", type=int, default=32)
    ap.add_argument("--workers", type=int, default=8)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sift.py needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    rec = dict(device=torch.cuda.get_device_name(0), nvidia_smi=q[0] if q else None, host_cpus=os.cpu_count(),
               cv2_version=cv2.__version__, cv2_threads=cv2.getNumThreads(), frames=[])
    gpu = GpuSift()
    for (w, h) in ((640, 480), (1200, 900), (2000, 1500)):
        rec["frames"].append(per_frame(gpu, w, h, a.reps, a.host_reps))
        print(json.dumps(rec["frames"][-1]), flush=True)
    rec["frame_stream_1200x900"] = stream_fps(a.stream_frames, a.workers)
    print(json.dumps(rec["frame_stream_1200x900"]), flush=True)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
