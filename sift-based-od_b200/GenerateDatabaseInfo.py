"""Model-database builder, drop-in for GenerateDatabaseInfo.py:1-37.

`save_object` and the pickle row layout [temp_kp, des, img_size, centroid, path] are unchanged, so
main.Main.get_query_features reads databases written by either implementation.  Unlike the
reference, importing this module does nothing; run it as a script or call build_database().
OpenCV SIFT stays the default feature extractor; build_database(..., extractor=GpuSift()) runs the
SIFT of many training images at once on the GPU (GpuSift.extract_mixed) and writes the same rows.
"""
import os
import pickle
import sys
from collections import namedtuple
from concurrent.futures import ThreadPoolExecutor
from functools import lru_cache

import cv2
import numpy as np

from SiftHelperFunctions import get_centroid, make_temp_kp

MAX_DIM = 1500  # reference :23
# GPU path: at most this many images per extract_mixed call, and at most this many bytes of SIFT workspace
# (pyramids and keypoint slabs, as sod_sift_mixed_workspace_bytes counts them) per call.  A 1500x1000 image's
# pyramid is about 190 MB, so a chunk of 1500-wide images is bounded by the budget long before 64 frames.
GPU_CHUNK_FRAMES = 64
GPU_CHUNK_BYTES = 8 << 30
GPU_DECODE_THREADS = 8

_Kp = namedtuple("_Kp", "pt")


def save_object(obj, filename):
    with open(filename, 'wb') as outp:  # overwrites any existing file
        pickle.dump(obj, outp, pickle.HIGHEST_PROTOCOL)


def _prepare(path):
    """The reference's preprocessing: decode, resize to MAX_DIM wide, gray.  None for a file cv2 cannot read."""
    img = cv2.imread(path)
    if img is None:
        return None
    img = cv2.resize(img, (MAX_DIM, int(MAX_DIM * img.shape[0] / img.shape[1])))
    return cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)


def build_database(image_dir, out_file='training_data.pkl', packed_file=None, extractor=None):
    """Writes the reference's pickle; with packed_file also the array form that loads straight into
    HBM (sod_b200/database.py), which main.Main.load_database reads as well.

    extractor=None runs cv2.SIFT_create() one image at a time, as the reference does.  With a GpuSift,
    host threads decode and resize the images and their SIFT runs on the GPU in mixed-size batches
    (chunks of gpu_chunks, read back once per chunk); the rows are laid out as the cv2 path lays them out."""
    paths = [os.path.join(image_dir, name) for name in os.listdir(image_dir)]
    if extractor is None:
        data = _rows_cv2(paths)
    else:
        data = _rows_gpu(paths, extractor)
    save_object(data, out_file)
    if packed_file is not None:
        from sod_b200.database import PackedDatabase
        PackedDatabase.from_reference_rows(data).save(packed_file)
    return data


def _rows_cv2(paths):
    sift = cv2.SIFT_create()
    data = []
    for path in paths:
        img = cv2.imread(path)
        if img is None:
            continue
        img = cv2.resize(img, (MAX_DIM, int(MAX_DIM * img.shape[0] / img.shape[1])))
        img_size = (img.shape[1], img.shape[0])
        gray = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
        kp, des = sift.detectAndCompute(gray, None)
        data.append([make_temp_kp(kp), des, img_size, get_centroid(kp), path])
    return data


@lru_cache(maxsize=4096)
def _frame_bytes(w, h):
    """SIFT workspace of one w x h frame in a mixed batch (its pyramid): sod_sift_mixed_workspace_bytes."""
    import ctypes as C

    from sod_b200 import _capi
    wh = (C.c_int32 * 2)(w, h)
    return int(_capi.lib.sod_sift_mixed_workspace_bytes(C.cast(wh, C.c_void_p), 1, 0))


def gpu_chunks(sizes, max_frames=None, budget=None):
    """Consecutive chunks of the (w, h) list: at most max_frames images each, and pyramids within budget bytes
    (a single image larger than the budget is a chunk of its own).  Lists of indices, in input order."""
    max_frames = GPU_CHUNK_FRAMES if max_frames is None else max_frames
    budget = GPU_CHUNK_BYTES if budget is None else budget
    chunks, cur, used = [], [], 0
    for i, (w, h) in enumerate(sizes):
        b = _frame_bytes(w, h)
        if cur and (len(cur) == max_frames or used + b > budget):
            chunks.append(cur)
            cur, used = [], 0
        cur.append(i)
        used += b
    if cur:
        chunks.append(cur)
    return chunks


def _rows_from_batch(batch, k, path):
    """Row k of a SiftBatch whose arrays were read back to the host, in the cv2 path's layout."""
    lo, hi = int(batch.offset[k]), int(batch.offset[k] + batch.count[k])
    pts = [tuple(p) for p in batch.xy[lo:hi].tolist()]
    temp_kp = list(zip(pts, batch.size[lo:hi].tolist(), batch.angle[lo:hi].tolist(),
                       batch.response[lo:hi].tolist(), batch.octave[lo:hi].tolist(), [-1] * (hi - lo)))
    des = batch.des[lo:hi].astype(np.float32) if hi > lo else None
    centroid = get_centroid([_Kp(p) for p in pts])        # same sums, and the same error for no keypoints
    return [temp_kp, des, batch.size_of(k), centroid, path]


def _decoded(paths, window):
    """(path, gray) of every readable image in input order, decoded by host threads `window` paths ahead."""
    with ThreadPoolExecutor(GPU_DECODE_THREADS) as pool:
        ahead = [pool.submit(_prepare, p) for p in paths[:window]]
        for i, path in enumerate(paths):
            if i + window < len(paths):
                ahead.append(pool.submit(_prepare, paths[i + window]))
            gray = ahead[i].result()
            ahead[i] = None
            if gray is not None:
                yield path, gray


def _rows_gpu(paths, extractor):
    data, pending = [], []

    def run(chunk):
        batch = extractor.extract_mixed([g for _, g in chunk])
        host = _HostBatch(batch)                     # one read-back per chunk
        for k, (path, _) in enumerate(chunk):
            data.append(_rows_from_batch(host, k, path))

    for item in _decoded(paths, 2 * GPU_CHUNK_FRAMES):
        pending.append(item)
        chunks = gpu_chunks([(g.shape[1], g.shape[0]) for _, g in pending])
        if len(chunks) > 1:                          # the first chunk is closed: nothing later joins it
            run(pending[:len(chunks[0])])
            pending = pending[len(chunks[0]):]
    for chunk in gpu_chunks([(g.shape[1], g.shape[0]) for _, g in pending]):
        run([pending[i] for i in chunk])
    return data


class _HostBatch:
    """A SiftBatch's rows copied to host numpy arrays in one pass."""

    def __init__(self, batch):
        for name in ("des", "xy", "size", "angle", "response", "octave"):
            v = getattr(batch, name)
            setattr(self, name, v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v))
        self.count, self.offset, self.size_of = batch.count, batch.offset, batch.size_of


if __name__ == "__main__":
    build_database(sys.argv[1], sys.argv[2] if len(sys.argv) > 2 else 'training_data.pkl',
                   sys.argv[3] if len(sys.argv) > 3 else None)
