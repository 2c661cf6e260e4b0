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
time of sod_sift_extract and of sod_sift_extract_batch (16 frames) of that library and of this tree's, each in its
own process, alternated --ab-rounds times.

--mixed runs only the mixed-size legs (and the A/B with --parent-lib): device time per frame of 16 distinct frames
of assorted sizes through sod_sift_extract_mixed, through sod_sift_extract one frame at a time and through
sod_sift_extract_batch grouped by size; the same for a skewed mix (one 2000x1500 frame and fifteen 64x48 ones,
where a launch sized for the largest frame would leave most blocks empty); and GenerateDatabaseInfo.build_database
images/s on a folder of synthetic PNGs of distinct heights, GPU against cv2.  With --parent-lib, both mixes also run
through that library and through this tree's, each in its own process (SOD_B200_LIB), alternated --ab-rounds times.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
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
    lib.sod_sift_batch_workspace_bytes.restype = C.c_size_t
    lib.sod_sift_batch_workspace_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int64]
    lib.sod_sift_extract_batch.restype = C.c_int
    lib.sod_sift_extract_batch.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int32,
                                           C.c_int64, C.POINTER(_capi.SiftBatchOut), C.c_void_p, C.c_size_t,
                                           C.c_void_p]
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
        del ws, arrays
        # sod_sift_extract_batch of 16 distinct frames of this size, per frame
        B, bcap = 16, 1 << 15
        rng = np.random.default_rng(w + 1)
        imgs = torch.from_numpy(np.stack([imaging.textured(rng, w, h, shapes=200) for _ in range(B)])).cuda()
        nbytes = int(lib.sod_sift_batch_workspace_bytes(w, h, B, bcap))
        ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        rows = B * bcap
        t = [torch.empty(s, dtype=dt, device="cuda") for s, dt in
             (((rows, 2), torch.float32), (rows, torch.float32), (rows, torch.float32), (rows, torch.float32),
              (rows, torch.int32), ((rows, 128), torch.uint8), (rows, torch.int32), (3 * B + 1, torch.int32))]
        fl = t[-1]
        bo = _capi.SiftBatchOut(*(x.data_ptr() for x in t[:7]), fl[:B].data_ptr(), fl[B:2 * B].data_ptr(),
                                fl[2 * B:3 * B].data_ptr(), fl[3 * B:].data_ptr(), rows, bcap)
        torch.cuda.synchronize()

        def batch():
            if lib.sod_sift_extract_batch(imgs.data_ptr(), w, h, w, w * h, B, 0, C.byref(bo), ws.data_ptr(), nbytes,
                                          st.cuda_stream):
                raise RuntimeError(f"sod_sift_extract_batch failed in {lib_path}")

        device_ms(st, batch, 2)
        out[f"batch16_{w}x{h}_per_frame"] = device_ms(st, batch, max(3, reps // 4)) / B
        f = fl.cpu().numpy()
        assert not f[2 * B:].any()
        out[f"batch16_{w}x{h}_keypoints"] = int(f[:B].sum())
        del ws, t, imgs
        torch.cuda.empty_cache()
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


MIXED_SIZES = ((640, 480), (640, 480), (640, 480), (640, 480), (800, 600), (800, 600), (800, 600), (1200, 900),
               (1200, 900), (1200, 900), (480, 640), (480, 640), (1600, 1200), (1600, 1200), (2000, 1500),
               (2000, 1500))
SKEWED_SIZES = ((2000, 1500),) + ((64, 48),) * 15


def mixed_per_frame(sizes, reps, seed):
    """Device ms per frame of one mixed batch of these (distinct) frames: sod_sift_extract_mixed, sod_sift_extract
    of each frame in turn, and sod_sift_extract_batch of the frames grouped by size.  Inputs on the device."""
    lib = _capi.lib
    rng = np.random.default_rng(seed)
    frames = [imaging.textured(rng, w, h, shapes=200) for w, h in sizes]
    dev = [torch.from_numpy(f).cuda() for f in frames]
    n = len(frames)
    gpu = GpuSift()
    mb = gpu.extract_mixed(dev)
    b = gpu._mixed[0]
    st = gpu._stream
    wh = (C.c_int32 * (2 * n))(*[v for s in sizes for v in s])
    ptrs = (C.c_void_p * n)(*[d.data_ptr() for d in dev])
    pitch = (C.c_int64 * n)(*[w for w, _ in sizes])

    def mixed():
        _capi.check(lib.sod_sift_extract_mixed(C.cast(ptrs, C.c_void_p), C.cast(wh, C.c_void_p),
                                               C.cast(pitch, C.c_void_p), n, 0, C.byref(b.out), b.ws.data_ptr(),
                                               b.ws.numel(), st.cuda_stream), "sod_sift_extract_mixed")

    singles = []
    for f in frames:
        gpu.extract(f)
    for d, (w, h) in zip(dev, sizes):
        sb = gpu._buffers[(w, h)]
        singles.append((d, w, h, sb))

    def one_by_one():
        for d, w, h, sb in singles:
            _capi.check(lib.sod_sift_extract(d.data_ptr(), w, h, w, C.byref(sb.out), sb.ws.data_ptr(), sb.bytes,
                                             st.cuda_stream), "sod_sift_extract")

    groups = {}
    for k, s in enumerate(sizes):
        groups.setdefault(s, []).append(k)
    grouped = []
    for (w, h), ks in groups.items():
        stacked = torch.stack([dev[k] for k in ks]).contiguous()
        gpu.extract_batch(stacked)
        bb = gpu._batch_buffers[(w, h, len(ks))]
        grouped.append((stacked, w, h, len(ks), bb, bb.out(0)[1]))

    def by_size():
        for x, w, h, m, bb, so in grouped:
            _capi.check(lib.sod_sift_extract_batch(x.data_ptr(), w, h, w, w * h, m, 0, C.byref(so), bb.ws.data_ptr(),
                                                   bb.bytes, st.cuda_stream), "sod_sift_extract_batch")

    torch.cuda.synchronize()
    out = dict(frames=n, sizes=[list(s) for s in sizes], keypoints=int(mb.rows), size_groups=len(groups),
               mixed_workspace_bytes=int(b.ws.numel()))
    for name, fn in (("mixed", mixed), ("single_each", one_by_one), ("batch_by_size", by_size)):
        device_ms(st, fn, 2)
        out[f"{name}_device_ms_per_frame"] = device_ms(st, fn, reps) / n
    out["mixed_speedup_vs_single_each"] = out["single_each_device_ms_per_frame"] / out["mixed_device_ms_per_frame"]
    out["mixed_speedup_vs_batch_by_size"] = out["batch_by_size_device_ms_per_frame"] / out["mixed_device_ms_per_frame"]
    del gpu
    torch.cuda.empty_cache()
    return out


def mixed_legs():
    return dict(assorted=mixed_per_frame(MIXED_SIZES, 20, 31), skewed=mixed_per_frame(SKEWED_SIZES, 20, 32))


def ab_mixed(parent_lib, rounds):
    """Both mixes with the parent library and with this tree's, alternated, each run in a fresh process."""
    runs = {"parent": [], "this_tree": []}
    for _ in range(rounds):
        for name, lib in (("parent", parent_lib), ("this_tree", str(_capi._LIB_PATH))):
            r = subprocess.run([sys.executable, __file__, "--out", "-", "--mixed-legs"],
                               env=dict(os.environ, SOD_B200_LIB=lib), capture_output=True, text=True)
            if r.returncode:
                raise RuntimeError(f"mixed run of {lib} failed:\n{r.stderr}")
            runs[name].append(json.loads(r.stdout.strip().splitlines()[-1]))
    keys = ("mixed_device_ms_per_frame", "single_each_device_ms_per_frame", "batch_by_size_device_ms_per_frame")
    med = {name: {f"{mix}.{k}": float(np.median([r[mix][k] for r in v])) for mix in ("assorted", "skewed")
                  for k in keys} for name, v in runs.items()}
    spread = {name: {f"{mix}.mixed": [min(r[mix]["mixed_device_ms_per_frame"] for r in v),
                                      max(r[mix]["mixed_device_ms_per_frame"] for r in v)]
                     for mix in ("assorted", "skewed")} for name, v in runs.items()}
    return dict(rounds=runs, median_ms_per_frame=med, min_max_mixed_ms_per_frame=spread)


def builder_fps(n_images):
    """GenerateDatabaseInfo.build_database images/s, GPU (GpuSift) against cv2, on PNGs of distinct heights."""
    import GenerateDatabaseInfo as G
    rng = np.random.default_rng(9)
    out = {}
    with tempfile.TemporaryDirectory() as d:
        for i in range(n_images):
            img = imaging.textured(rng, 600, 300 + 5 * i, shapes=150)
            cv2.imwrite(os.path.join(d, f"img_{i:04d}.png"), cv2.cvtColor(img, cv2.COLOR_GRAY2BGR))
        warm = os.path.join(d, "warm")
        os.mkdir(warm)
        for i in range(3):
            cv2.imwrite(os.path.join(warm, f"w{i}.png"), cv2.imread(os.path.join(d, f"img_{i:04d}.png")))
        gpu = GpuSift()
        G.build_database(warm, os.path.join(d, "w.pkl"), extractor=gpu)
        G.build_database(warm, os.path.join(d, "w.pkl"))
        for name, ex in (("gpu", gpu), ("cv2", None)):
            t = time.perf_counter()
            rows = G.build_database(d, os.path.join(d, f"{name}.pkl"), extractor=ex)
            dt = time.perf_counter() - t
            out[name] = dict(images=len(rows), seconds=dt, images_per_s=len(rows) / dt,
                             keypoints=int(sum(len(r[0]) for r in rows)))
    out["heights_after_resize"] = [int(1500 * (300 + 5 * i) / 600) for i in (0, n_images - 1)]
    out["gpu_speedup_vs_cv2"] = out["gpu"]["images_per_s"] / out["cv2"]["images_per_s"]
    return out


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
    ap.add_argument("--mixed-legs", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--mixed", action="store_true", help="only the mixed-size legs (and the A/B with --parent-lib)")
    ap.add_argument("--builder-images", type=int, default=64)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sift.py needs a CUDA device")
    if a.single_lib:
        print(json.dumps(single_extract_ms(a.single_lib, a.reps)))
        return
    if a.mixed_legs:
        print(json.dumps(mixed_legs()))
        return
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    rec = dict(device=torch.cuda.get_device_name(0), nvidia_smi=q[0] if q else None, host_cpus=os.cpu_count(),
               cv2_version=cv2.__version__, cv2_threads=cv2.getNumThreads(), frames=[])
    if a.mixed:
        del rec["frames"]
        rec["mixed_assorted"] = mixed_per_frame(MIXED_SIZES, a.reps, 31)
        print(json.dumps(rec["mixed_assorted"]), flush=True)
        rec["mixed_skewed"] = mixed_per_frame(SKEWED_SIZES, a.reps, 32)
        print(json.dumps(rec["mixed_skewed"]), flush=True)
        rec["build_database"] = builder_fps(a.builder_images)
        print(json.dumps(rec["build_database"]), flush=True)
        if a.parent_lib:
            rec["mixed_ab"] = ab_mixed(a.parent_lib, a.ab_rounds)
            print(json.dumps(rec["mixed_ab"]["median_ms_per_frame"]), flush=True)
            rec["single_frame_ab"] = ab_single(a.parent_lib, a.ab_rounds, a.reps)
            print(json.dumps(rec["single_frame_ab"]["median_ms"]), flush=True)
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(rec, indent=1) + "\n")
        return
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
