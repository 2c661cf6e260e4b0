"""Batched multi-frame front end (SURVEY.md §8f N3): the caller side of the path.

The reference handles one image per process run: Main.get_query_features (main.py:36-46) reads it,
runs OpenCV SIFT, and the matcher starts when that is done.  For a stream of frames the host-side
SIFT is the slow stage, so FrameStream extracts features of upcoming frames on a pool of host
threads (OpenCV releases the GIL) while the GPU runs match -> ratio -> Hough -> affine on the
previous batch; batches are packed into pinned, double-buffered staging while the GPU is busy, their
host->device copies run on the pipeline's copy stream under the previous batch's kernels, and
results are handed to the caller while the next batch runs.  OpenCV SIFT itself stays the default extractor.

With an extractor that has extract_batch (sod_b200.sift.GpuSift) the stream runs on the device instead: worker
threads only decode and convert frames, runs of same-size frames are extracted in one SIFT pass, and the rows go
from the SIFT output to the pipeline's query buffers by device-to-device copies.
"""
from __future__ import annotations

from collections import deque
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass
from typing import Callable, Iterable, Iterator

import numpy as np


@dataclass
class FrameFeatures:
    """What the path reads from one query image (main.py:43-46): descriptors + keypoint fields."""
    des: np.ndarray      # u8 [n,128]
    xy: np.ndarray       # f32 [n,2]
    angle: np.ndarray    # f32 [n]
    octave: np.ndarray   # i32 [n]
    size: tuple          # (width, height) of the frame

    def __len__(self) -> int:
        return int(self.des.shape[0])


def sift_features(image, max_keypoints: int | None = None) -> FrameFeatures:
    """cv2.SIFT on one BGR / gray image or file path, as get_query_features does (main.py:40-46).
    A SIFT object is created per call: cv2.SIFT is not safe to share between threads."""
    import cv2
    if isinstance(image, (str, bytes)) or hasattr(image, "__fspath__"):
        img = cv2.imread(str(image))
        if img is None:
            raise FileNotFoundError(str(image))
    else:
        img = np.asarray(image)
    gray = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY) if img.ndim == 3 else img
    kp, des = cv2.SIFT_create().detectAndCompute(gray, None)
    n = len(kp)
    if n == 0:
        des = np.zeros((0, 128), np.float32)
    if max_keypoints is not None and n > max_keypoints:
        kp, des, n = kp[:max_keypoints], des[:max_keypoints], max_keypoints
    if n and not (np.all(des == np.rint(des)) and des.min() >= 0 and des.max() <= 255):
        raise ValueError("SIFT descriptors are not integer-valued 0..255")
    return FrameFeatures(des.astype(np.uint8), np.array([k.pt for k in kp], np.float32).reshape(-1, 2),
                         np.array([k.angle for k in kp], np.float32), np.array([k.octave for k in kp], np.int32),
                         (int(gray.shape[1]), int(gray.shape[0])))


def plan_batches(counts: Iterable[int], max_frames: int, max_rows: int) -> list[list[int]]:
    """Greedy in-order packing of frames (by descriptor count) into batches of at most max_frames
    frames and max_rows descriptor rows; a frame never straddles batches."""
    batches, cur, rows = [], [], 0
    for i, c in enumerate(counts):
        if c > max_rows:
            raise ValueError(f"frame {i} has {c} descriptors, more than the pipeline's max_queries {max_rows}")
        if cur and (len(cur) == max_frames or rows + c > max_rows):
            batches.append(cur)
            cur, rows = [], 0
        cur.append(i)
        rows += c
    if cur:
        batches.append(cur)
    return batches


def split_frame(out: dict, poses: dict, spaces_per_frame: int, slot: int, lo: int, hi: int, **extra) -> dict:
    """The part of a fetched batch result that belongs to frame `slot`, whose query rows are [lo, hi): match pairs
    as (query keypoint index within the frame, database row), verified bins, final poses; `extra` (such as the
    frame's FrameFeatures) is added as it is."""
    ok = out["ok"][lo:hi].astype(bool)
    gpf = spaces_per_frame
    mine = (out["valid_group"] // gpf) == slot
    return dict(match_q=np.nonzero(ok)[0].astype(np.int32), match_t=out["idx"][lo:hi, 0][ok],
                n_descriptors=hi - lo, valid_group=out["valid_group"][mine] % gpf, valid_code=out["valid_code"][mine],
                votes=out["votes"][mine], live=(out["status"][mine] & 1).astype(bool), params=out["params"][mine],
                final_pose=poses.get(slot, []), **extra)


def one_rank_error(who: str) -> str:
    """Why a device-side SIFT path refuses a database-sharded pipeline of several ranks."""
    return (f"{who} needs the whole batch on one rank: every rank of a database-sharded pipeline would need the "
            "same query rows, and GPU SIFT descriptors may differ by 1 between runs; use "
            "DetectionPipeline(shard='frames')")


class _Staging:
    """One set of pinned host buffers for a batch (allocated lazily; torch only needed on the GPU side)."""

    def __init__(self, max_rows: int, max_frames: int, pin: bool):
        import torch
        mk = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=pin)  # noqa: E731
        self.des = mk((max_rows, 128), torch.uint8)
        self.xy = mk((max_rows, 2), torch.float32)
        self.angle = mk(max_rows, torch.float32)
        self.octave = mk(max_rows, torch.int32)
        self.frame = mk(max_rows, torch.int32)
        self.frame_wh = mk((max_frames, 2), torch.int32)

    def fill(self, feats: list[FrameFeatures]) -> int:
        off = 0
        self.frame_wh.zero_()
        for slot, f in enumerate(feats):
            n = len(f)
            self.des[off:off + n] = _t(f.des)
            self.xy[off:off + n] = _t(f.xy)
            self.angle[off:off + n] = _t(f.angle)
            self.octave[off:off + n] = _t(f.octave)
            self.frame[off:off + n] = slot
            self.frame_wh[slot, 0], self.frame_wh[slot, 1] = f.size
            off += n
        return off


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a))


class FrameStream:
    """Runs a DetectionPipeline over a sequence of frames.

    pipeline      a DetectionPipeline built with max_queries >= the rows of one batch and
                  frame_wh of shape [batch_frames, 2] (its values are overwritten per batch)
    extractor     image -> FrameFeatures (default: sift_features)
    batch_frames  frames per GPU pass
    workers       host threads running the extractor
    prefetch      frames whose extraction may be in flight ahead of the GPU
    features      add each frame's FrameFeatures to its result (result["features"])

    run(frames) yields (frame_index, result) in input order; result holds the frame's matches and
    verified bins (see _split) and, with poses=True, the final poses of the frame.

    An extractor with extract_batch and prepare (GpuSift) selects the device path: workers run prepare (decode,
    colour conversion; CUDA tensors pass as they are), consecutive frames of one size form a SIFT batch of up to
    batch_frames frames, and each detection pass takes the longest prefix of a batch's frames whose rows fit
    max_queries.  The SIFT of the next batch is enqueued before the host waits for the current pass.  The device
    path needs a pipeline whose ranks do not share one batch (shard="frames" or one rank)."""

    def __init__(self, pipeline, extractor: Callable[[object], FrameFeatures] = sift_features, batch_frames: int = 8,
                 workers: int = 8, prefetch: int | None = None, poses: bool = True, features: bool = False):
        self.pipeline, self.extractor = pipeline, extractor
        self.batch_frames = int(batch_frames)
        if pipeline.scene.n_frames < self.batch_frames:
            raise ValueError("pipeline.frame_wh must have one row per frame of a batch")
        self.workers = int(workers)
        self.prefetch = int(prefetch) if prefetch is not None else 2 * self.batch_frames + self.workers
        self.poses, self.features = poses, bool(features)
        self._staging: list[_Staging] = []

    # -------------------------------------------------------------------------------- GPU side
    def _stage(self, feats: list[FrameFeatures], slot: int) -> int:
        """Pack one batch into the pinned staging set `slot` (host work; the GPU may be busy)."""
        p = self.pipeline
        if not self._staging:
            self._on_gpu = p.device.type == "cuda"
            self._staging = [_Staging(p.max_queries, self.batch_frames, self._on_gpu) for _ in range(2)]
            self._copied = [None, None]
        if self._copied[slot] is not None:
            self._copied[slot].synchronize()      # the copies that read this staging set have finished
        return self._staging[slot].fill(feats)

    def _enqueue(self, slot: int, n: int):
        """Host->device copies (on the pipeline's copy stream, so they overlap the kernels of the
        previous batch) and the kernels of one staged batch, all asynchronous."""
        p, st = self.pipeline, self._staging[slot]
        p.scene.frame_wh[:self.batch_frames].copy_(st.frame_wh, non_blocking=True)
        p.load_queries(st.des[:n], st.xy[:n], st.angle[:n], st.octave[:n], st.frame[:n], slot=slot,
                       overlap=self._on_gpu)
        self._copied[slot] = getattr(p, "_loaded", [None, None])[slot]
        return p.detect_device(n, slot)

    def _fetch(self, r):
        """Device->host read of a pass (synchronises) + final poses."""
        if r is None:                                # no descriptors in the whole pass
            z = np.zeros(0, np.int32)
            return dict(ok=np.zeros(0, np.uint8), idx=np.zeros((0, 2), np.int32), valid_group=z, valid_code=z, votes=z,
                        status=z, params=np.zeros((0, 6))), {}
        out = self.pipeline.fetch(r)
        return out, (self.pipeline.final_poses(out) if self.poses else {})

    def _finish(self, r, feats: list[FrameFeatures], first_index: int):
        """Device->host read of a batch + final poses, split per frame."""
        out, poses = self._fetch(r)
        starts = np.cumsum([0] + [len(f) for f in feats])
        return [(first_index + k, self._split(out, poses, k, starts[k], starts[k + 1], feats[k]))
                for k in range(len(feats))]

    def _split(self, out: dict, poses: dict, slot: int, lo: int, hi: int, feats: FrameFeatures | None) -> dict:
        return split_frame(out, poses, self.pipeline.spaces_per_frame, slot, lo, hi,
                           **({"features": feats} if self.features else {}))

    # -------------------------------------------------------------------------------- driver
    def run(self, frames: Iterable) -> Iterator[tuple[int, dict]]:
        if hasattr(self.extractor, "extract_batch"):
            return self._run_device(frames)
        return self._run_host(frames)

    def _run_host(self, frames: Iterable) -> Iterator[tuple[int, dict]]:
        p = self.pipeline
        with ThreadPoolExecutor(self.workers) as pool:
            pending: deque = deque()          # futures of extracted frames, input order
            it = iter(frames)
            exhausted = False

            def top_up():
                nonlocal exhausted
                while not exhausted and len(pending) < self.prefetch:
                    try:
                        pending.append(pool.submit(self.extractor, next(it)))
                    except StopIteration:
                        exhausted = True

            def next_batch():
                """Longest in-order prefix of extracted frames that fits one GPU pass."""
                feats, rows = [], 0
                while pending and len(feats) < self.batch_frames:
                    f = pending[0].result()
                    if len(f) > p.max_queries:
                        raise ValueError(f"a frame has {len(f)} descriptors, more than max_queries {p.max_queries}")
                    if feats and rows + len(f) > p.max_queries:
                        break
                    pending.popleft()
                    feats.append(f)
                    rows += len(f)
                    top_up()
                return feats

            top_up()
            # Per iteration: stage batch i on the host while the GPU runs batch i-1, read back i-1
            # (the pipeline's result buffers are single: they must be consumed before the next
            # launch), enqueue i, then hand i-1's frames to the caller while i runs.
            index, slot, prev = 0, 0, None
            while True:
                feats = next_batch()
                n = self._stage(feats, slot) if feats else 0
                results = self._finish(*prev) if prev is not None else []
                prev = (self._enqueue(slot, n) if n else None, feats, index) if feats else None
                yield from results
                if prev is None:
                    break
                index += len(feats)
                slot ^= 1

    # -------------------------------------------------------------------------------- device path
    def _prepared(self, pool, frames: Iterable) -> Iterator[list]:
        """Runs of consecutive same-size prepared frames, at most batch_frames long, in input order; preparation
        runs up to `prefetch` frames ahead on the worker threads."""
        pending: deque = deque()
        it = iter(frames)
        exhausted = False
        while True:
            while not exhausted and len(pending) < self.prefetch:
                try:
                    pending.append(pool.submit(self.extractor.prepare, next(it)))
                except StopIteration:
                    exhausted = True
            if not pending:
                return
            run = [pending.popleft().result()]
            shape = tuple(run[0].shape[-2:])
            while len(run) < self.batch_frames:
                if not pending:
                    if exhausted:
                        break
                    try:
                        pending.append(pool.submit(self.extractor.prepare, next(it)))
                    except StopIteration:
                        exhausted = True
                        break
                if tuple(pending[0].result().shape[-2:]) != shape:
                    break
                run.append(pending.popleft().result())
            yield run

    def _passes(self, pool, frames: Iterable) -> Iterator[tuple]:
        """(SIFT batch, first frame, end frame, input index of the batch's frame 0, host features or None) per
        detection pass: the longest prefix of the batch's remaining frames whose rows fit max_queries.  SIFT
        batches alternate between the extractor's two output sets."""
        index, slot = 0, 0
        for run in self._prepared(pool, frames):
            sb = self.extractor.extract_batch(run, slot=slot)
            feats = [sb.features(k) for k in range(len(sb))] if self.features else None
            count, a = np.asarray(sb.count), 0
            while a < len(count):
                b, rows = a, 0
                while b < len(count) and rows + count[b] <= self.pipeline.max_queries:
                    rows += count[b]
                    b += 1
                if b == a:
                    raise ValueError(f"a frame has {int(count[a])} descriptors, more than max_queries "
                                     f"{self.pipeline.max_queries}")
                yield sb, a, b, index, feats
                a = b
            index += len(count)
            slot ^= 1

    def _enqueue_device(self, sb, a: int, b: int, slot: int):
        """Frame size, device-to-device copies of frames [a, b) of SIFT batch sb into query-buffer set `slot`,
        and the pass's kernels.  The pass keeps the frames' indices within the SIFT batch, so frame k's Hough
        spaces are k * spaces_per_frame + object."""
        p = self.pipeline
        lo, hi = int(sb.offset[a]), int(sb.offset[b - 1] + sb.count[b - 1])
        if hi == lo:
            return None
        p.scene.frame_wh[:, 0].fill_(sb.frame_size[0])
        p.scene.frame_wh[:, 1].fill_(sb.frame_size[1])
        p.load_queries(sb.des[lo:hi], sb.xy[lo:hi], sb.angle[lo:hi], sb.octave[lo:hi], sb.frame[lo:hi], slot=slot,
                       overlap=p.device.type == "cuda")
        return p.detect_device(hi - lo, slot)

    def _finish_device(self, r, sb, a: int, b: int, index: int, feats) -> list:
        out, poses = self._fetch(r)
        base = int(sb.offset[a])
        return [(index + k, self._split(out, poses, k, int(sb.offset[k]) - base,
                                        int(sb.offset[k] + sb.count[k]) - base, feats[k] if feats else None))
                for k in range(a, b)]

    def _run_device(self, frames: Iterable) -> Iterator[tuple[int, dict]]:
        p = self.pipeline
        if getattr(p, "world", 1) > 1 and getattr(p, "shard_mode", "db") == "db":
            raise ValueError(one_rank_error("FrameStream's device path"))
        with ThreadPoolExecutor(self.workers) as pool:
            # Per pass: take the next pass (which may run the next SIFT batch, while the GPU still runs the
            # previous pass), read back the previous pass, enqueue this one, hand the previous frames over.
            prev, slot = None, 0
            for sb, a, b, index, feats in self._passes(pool, frames):
                results = self._finish_device(*prev) if prev is not None else []
                prev = (self._enqueue_device(sb, a, b, slot), sb, a, b, index, feats)
                yield from results
                slot ^= 1
            if prev is not None:
                yield from self._finish_device(*prev)
