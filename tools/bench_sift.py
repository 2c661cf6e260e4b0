"""GPU SIFT (sod_b200.sift.GpuSift) against host cv2.SIFT, per frame and through FrameStream, in one run.

    python tools/bench_sift.py --out profiles/sift_bench.json [--parent-lib path/to/other/libsod_b200.so]

Per size (640x480, 1200x900, 2000x1500 synthetic frames): device time of sod_sift_extract (CUDA events on the
extractor's stream), wall time of a whole GpuSift call (upload, kernels, read-back), device time of the pyramid
alone (sod_sift_describe of one keypoint: the descriptor costs one block) with its bytes computed from the
shapes, and host cv2.SIFT_create().detectAndCompute.  Then FrameStream frames/s on a 3-object cv2 database with
each extractor.  Every timed pass is preceded by warm-up passes of the same shape; the pyramid of a 1200x900
frame (144 MB) does not fit the 126 MB L2, smaller ones mostly do (stated per size in the record).

Batch leg: device time per frame of sod_sift_extract_batch at B = 1, 4 and 16 distinct frames per size (input
already on the device), and FrameStream frames/s through the batched device path.  With --parent-lib, the device
time of sod_sift_extract of that library and of this tree's, each in its own process, alternated --ab-rounds
times.
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
SIZES = ((640, 480), (1200, 900), (2000, 1500))


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


def batch_per_frame(w, h, batches, reps):
    """Device ms per frame of sod_sift_extract_batch for each batch size, frames distinct and on the device."""
    gpu = GpuSift()
    rng = np.random.default_rng(w + 1)
    frames = [imaging.textured(rng, w, h, shapes=200) for _ in range(max(batches))]
    out = {}
    for n in batches:
        sb = gpu.extract_batch(frames[:n])
        b = gpu._batch_buffers[(w, h, n)]
        _, st_out = b.out(0)
        st = gpu._stream

        def run():
            _capi.check(_capi.lib.sod_sift_extract_batch(b.img.data_ptr(), w, h, w, w * h, n, 0, C.byref(st_out),
                                                         b.ws.data_ptr(), b.bytes, st.cuda_stream),
                        "sod_sift_extract_batch")

        device_ms(st, run, 3)
        ms = device_ms(st, run, max(3, reps // n))
        out[str(n)] = dict(frames=n, keypoints=int(sb.rows), device_ms_per_batch=ms, device_ms_per_frame=ms / n,
                           workspace_bytes=b.bytes)
    del gpu
    torch.cuda.empty_cache()
    return out


def single_extract_ms(lib_path, reps):
    """Device ms of sod_sift_extract per size with the library at lib_path, bound here to the two entry points
    every version of it has (the A/B leg: one process per run)."""
    lib = C.CDLL(lib_path)
    lib.sod_sift_workspace_bytes.restype = C.c_size_t
    lib.sod_sift_workspace_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int64]
    lib.sod_sift_extract.restype = C.c_int
    lib.sod_sift_extract.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.POINTER(_capi.SiftOut),
                                     C.c_void_p, C.c_size_t, C.c_void_p]
    st, cap, out = torch.cuda.Stream(), 1 << 16, {}
    for (w, h) in SIZES:
        gray = imaging.textured(np.random.default_rng(w), w, h, shapes=200)
        nbytes = int(lib.sod_sift_workspace_bytes(w, h, cap))
        ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        img = torch.from_numpy(gray).cuda()
        arrays = [torch.empty(s, dtype=dt, device="cuda") for s, dt in
                  (((cap, 2), torch.float32), (cap, torch.float32), (cap, torch.float32), (cap, torch.float32),
                   (cap, torch.int32), ((cap, 128), torch.uint8), (2, torch.int32))]
        so = _capi.SiftOut(*(t.data_ptr() for t in arrays), cap)
        torch.cuda.synchronize()

        def extract():
            if lib.sod_sift_extract(img.data_ptr(), w, h, w, C.byref(so), ws.data_ptr(), nbytes, st.cuda_stream):
                raise RuntimeError(f"sod_sift_extract failed in {lib_path}")

        device_ms(st, extract, 3)
        out[f"{w}x{h}"] = device_ms(st, extract, reps)
        n, overflow = (int(v) for v in arrays[-1].cpu())
        out[f"{w}x{h}_keypoints"] = n
        assert not overflow
    return out


def ab_single(parent_lib, rounds, reps):
    """sod_sift_extract of the parent library and of this tree, alternated, each in a fresh process."""
    runs = {"parent": [], "this_tree": []}
    for _ in range(rounds):
        for name, lib in (("parent", parent_lib), ("this_tree", str(_capi._LIB_PATH))):
            r = subprocess.run([sys.executable, __file__, "--out", "-", "--single-lib", lib, "--reps", str(reps)],
                               capture_output=True, text=True)
            if r.returncode:
                raise RuntimeError(f"single-frame run of {lib} failed:\n{r.stderr}")
            runs[name].append(json.loads(r.stdout.strip().splitlines()[-1]))
    med = {name: {k: float(np.median([r[k] for r in v])) for k in v[0]} for name, v in runs.items()}
    return dict(rounds=runs, median_ms=med)


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
    per_frame_gpu = GpuSift()
    # "gpu": GpuSift per frame on the host path (a plain callable); "gpu_batch": the device path, 16-frame SIFT
    # batches, each detection pass as many frames as fit max_queries
    for name, ex, bf in (("cv2", sift_features, 4), ("gpu", lambda fr: per_frame_gpu(fr), 4),
                         ("gpu_batch", GpuSift(), 16)):
        pipe = DetectionPipeline(db.to_model_database(), max_queries=40000, frame_wh=np.zeros((bf, 2), np.int32),
                                 per_object_spaces=False)
        fs = FrameStream(pipe, extractor=ex, batch_frames=bf, workers=workers)
        for _ in fs.run(frames[:2 * bf]):
            pass
        t = time.perf_counter()
        found = sum(len(r["final_pose"]) > 0 for _, r in fs.run(frames))
        dt = time.perf_counter() - t
        out[name] = dict(frames=n_frames, batch_frames=bf, seconds=dt, frames_per_s=n_frames / dt,
                         frames_with_a_pose=found)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--stream-frames", type=int, default=256)
    ap.add_argument("--workers", type=int, default=8)
    ap.add_argument("--parent-lib", default=None, help="another build of libsod_b200.so to compare sod_sift_extract with")
    ap.add_argument("--ab-rounds", type=int, default=3)
    ap.add_argument("--single-lib", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sift.py needs a CUDA device")
    if a.single_lib:
        print(json.dumps(single_extract_ms(a.single_lib, a.reps)))
        return
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    rec = dict(device=torch.cuda.get_device_name(0), nvidia_smi=q[0] if q else None, host_cpus=os.cpu_count(),
               cv2_version=cv2.__version__, cv2_threads=cv2.getNumThreads(), frames=[])
    gpu = GpuSift()
    for (w, h) in SIZES:
        rec["frames"].append(per_frame(gpu, w, h, a.reps, a.host_reps))
        print(json.dumps(rec["frames"][-1]), flush=True)
    del gpu
    torch.cuda.empty_cache()
    rec["batch"] = {}
    for (w, h) in SIZES:
        rec["batch"][f"{w}x{h}"] = batch_per_frame(w, h, (1, 4, 16), 16 * a.reps)
        print(json.dumps({f"{w}x{h}": rec["batch"][f"{w}x{h}"]}), flush=True)
    if a.parent_lib:
        rec["single_frame_ab"] = ab_single(a.parent_lib, a.ab_rounds, a.reps)
        print(json.dumps(rec["single_frame_ab"]["median_ms"]), flush=True)
    rec["frame_stream_1200x900"] = stream_fps(a.stream_frames, a.workers)
    print(json.dumps(rec["frame_stream_1200x900"]), flush=True)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
