"""One camera frame (or a batch of B same-size frames) to detections in one CUDA-graph replay.

A single frame is launch-bound end to end: GPU SIFT is about 60 pyramid launches plus its sort and scan passes, and
the detection pass about 18 more.  LiveDetector captures all of it once per frame size and replays it for every later
frame, with one host synchronise per call:

    live = LiveDetector(pipeline, GpuSift(max_keypoints=R), (640, 480))
    for frame in camera:
        (result,) = live.detect([frame])

The graph holds the upload from pinned staging, the SIFT batch (GpuSift.enqueue_batch), the copies of its packed rows
into the pipeline's query buffers (a fixed B x R rows), the true row total offset[B-1] + count[B-1] on the device, the
detection pass on that capacity with the row count read by the compaction only (DetectionPipeline.detect_device's
n_dev), the final poses of the verified bins (DetectionPipeline.final_poses_device: Main.post_process on the device),
and the device-to-host copies of the counters, the SIFT flags, idx / ok of the capacity rows, the records of up to
max_bins verified bins and the poses.  The rows past the true count hold the previous frame's rows: they are matched
and their matches are dropped by the compaction.  After the replay's one synchronise, detect only reads pinned
memory.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _capi
from .sift import SiftBatch, _gray, _is_cuda
from .stream import one_rank_error, split_frame

# the verified-bin fields read back per call, as DetectionPipeline.fetch reads them
_BIN_FIELDS = ("valid_bin", "params", "votes", "status", "valid_group", "valid_code", "valid_order", "valid_mean")


class LiveDetector:
    """Detections of B same-size frames per call, the whole path replayed as one CUDA graph.

    pipeline    a single-rank (or shard="frames") DetectionPipeline on u8 descriptors, with
                max_queries >= frames x sift.max_keypoints and frame_wh of at least `frames` rows (its values are
                overwritten by every call)
    sift        a GpuSift with max_keypoints set: a frame keeps cv2's first max_keypoints keypoints
    frame_size  (width, height) of every frame
    frames      B, frames per call
    max_bins    verified bins read back per call (at most 65,536, the limit of the pose clustering); a call that
                verifies more raises
    features    add each frame's FrameFeatures (its SIFT rows, read back from the device) to its result

    detect(frames) returns one dict per frame with the fields of a FrameStream frame result.  The graph is captured
    on the first call, after warm-up runs, once for host inputs and once for CUDA inputs if both occur; several
    LiveDetectors (one per frame size) may share a pipeline and a GpuSift when their calls do not overlap."""

    def __init__(self, pipeline, sift, frame_size, frames: int = 1, max_bins: int = 4096, features: bool = False):
        p = pipeline
        if getattr(p, "world", 1) > 1 and getattr(p, "shard_mode", "db") == "db":
            raise ValueError(one_rank_error("LiveDetector"))
        if getattr(p, "float_path", False):
            raise ValueError("LiveDetector needs a pipeline on u8 descriptors: GPU SIFT gives u8 rows, and this "
                             "pipeline's database is float32 (the bf16 path)")
        self.frames = int(frames)
        if self.frames < 1:
            raise ValueError("frames must be >= 1")
        if getattr(sift, "max_keypoints", None) is None:
            raise ValueError("LiveDetector needs GpuSift(max_keypoints=R): it bounds a frame's rows at R")
        self.per_frame = min(int(sift.capacity), max(1, int(sift.max_keypoints)))
        self.rows = self.frames * self.per_frame
        if self.rows > p.max_queries:
            raise ValueError(f"{self.frames} frames x max_keypoints {self.per_frame} = {self.rows} rows, more than the "
                             f"pipeline's max_queries {p.max_queries}")
        if p.scene.n_frames < self.frames:
            raise ValueError("pipeline.frame_wh must have one row per frame of a call")
        w, h = (int(v) for v in frame_size)
        if w < 1 or h < 1:
            raise ValueError(f"frame_size {frame_size} out of range")
        self.pipeline, self.sift, self.frame_size = p, sift, (w, h)
        self.max_bins, self.features = int(max_bins), bool(features)
        self._img = self._host = None
        self._graphs: dict[bool, tuple] = {}      # host upload in the graph? -> (graph, what it reads and writes)

    # ------------------------------------------------------------------------------------------------ inputs
    def _frames(self, frames) -> bool:
        """Stage one call's frames: host ones in the pinned staging (uploaded by the graph), CUDA ones straight
        into the device image buffer.  -> True when the graph's upload is wanted (all frames on the host)."""
        w, h = self.frame_size
        frames = list(frames.unbind(0)) if _is_cuda(frames) and frames.dim() == 3 else list(frames)
        if len(frames) != self.frames:
            raise ValueError(f"LiveDetector takes {self.frames} frames per call, got {len(frames)}")
        frames = [f if _is_cuda(f) else _gray(f) for f in frames]
        for k, f in enumerate(frames):
            if tuple(f.shape) != (h, w) or (_is_cuda(f) and f.dtype != torch.uint8):
                raise ValueError(f"frame {k}: expected a {w}x{h} u8 image, got {f.dtype} {tuple(f.shape)}")
        if self._img is None:
            dev = self.pipeline.device
            self._img = torch.empty((self.frames, h, w), dtype=torch.uint8, device=dev)
            self._host = torch.empty((self.frames, h, w), dtype=torch.uint8, pin_memory=True)
        upload = not any(_is_cuda(f) for f in frames)
        for k, f in enumerate(frames):
            if upload:
                self._host[k].copy_(torch.from_numpy(f))
            else:
                self._img[k].copy_(f if _is_cuda(f) else torch.from_numpy(f))
        return upload

    # ------------------------------------------------------------------------------------------------ the graph
    def _pinned(self, src: torch.Tensor) -> torch.Tensor:
        return torch.empty(src.shape, dtype=src.dtype, pin_memory=True)

    def _body(self, upload: bool, host: dict | None) -> dict:
        """The whole path, enqueued on the current stream (warm-up runs and the captured one alike)."""
        p, B, R = self.pipeline, self.frames, self.rows
        w, h = self.frame_size
        if upload:
            self._img.copy_(self._host, non_blocking=True)
        t = self.sift.enqueue_batch(self._img, slot=0)
        p.scene.frame_wh[:, 0].fill_(w)
        p.scene.frame_wh[:, 1].fill_(h)
        p.load_queries(t["des"][:R], t["xy"][:R], t["angle"][:R], t["octave"][:R], t["frame"][:R], slot=0)
        fl = t["flags"]
        n_dev = fl[B - 1:B] + fl[2 * B - 1:2 * B]            # offset[B-1] + count[B-1]: the rows of this call
        r = p.detect_device(R, 0, _events=False, n_dev=n_dev)
        a = r["affine"]
        k = min(self.max_bins, a.cap_valid, _capi.MAX_CLUSTER_BINS)    # the poses are clustered on the device
        g, code, order, mean = r["records"]
        dev = dict(counters=r["counters"], flags=fl, idx=r["idx"][:R], ok=r["ok"][:R], valid_bin=a.valid_bin[:k],
                   params=a.params[:k], votes=a.votes[:k], status=a.status[:k], valid_group=g[:k], valid_code=code[:k],
                   valid_order=order[:k], valid_mean=mean[:k])
        fp = p.final_poses_device(r, k)
        dev.update(pose=fp["pose"], pose_frame=fp["frame"], pose_shape=fp["shape_bin"], pose_counters=fp["counters"])
        if host is None:
            host = {name: self._pinned(v) for name, v in dev.items()}
        for name, v in dev.items():
            host[name].copy_(v, non_blocking=True)
        return dict(host=host, sift=t, n_dev=n_dev, k=k, poses=fp["poses"])

    def _graph(self, upload: bool):
        entry = self._graphs.get(upload)
        if entry is not None:
            return entry
        p = self.pipeline
        cur = torch.cuda.current_stream(p.device)
        side = torch.cuda.Stream(p.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            host = None
            for _ in range(2):
                host = self._body(upload, host)["host"]
        cur.wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            state = self._body(upload, host)
        # The workspaces the graph was captured with (allocated during the warm-up, outside its pool) stay alive
        # with it, even if another caller of the pipeline later grows them.
        state["keep"] = (p.matcher._ws, p.matcher._qn, p.voter._ws, p._hough[0], p._aff[0], p.scene.frame_wh,
                         p._qset(0), self.sift._batch_buffers[(*self.frame_size, self.frames)], state["poses"])
        entry = self._graphs[upload] = (graph, state)
        return entry

    # ------------------------------------------------------------------------------------------------ host side
    def detect(self, frames) -> list[dict]:
        """One call: B frames (host gray / BGR images, CUDA u8 [H, W] tensors, or a CUDA u8 [B, H, W] tensor) ->
        one result per frame (match_q, match_t, n_descriptors, valid_group, valid_code, votes, live, params,
        final_pose, and features if asked for).  Raises SodError naming a frame with more keypoints than the SIFT
        capacity, RuntimeError on a Hough / affine output overflow or on more verified bins than max_bins."""
        p, B = self.pipeline, self.frames
        w, h = self.frame_size
        upload = self._frames(frames)
        with torch.cuda.device(p.device):
            graph, state = self._graph(upload)
            graph.replay()
            torch.cuda.current_stream(p.device).synchronize()
        hv = {name: v.numpy() for name, v in state["host"].items()}
        fl = hv["flags"]
        count, offset, overflow = fl[:B].astype(np.int64), fl[B:2 * B].astype(np.int64), fl[2 * B:3 * B]
        bad = np.nonzero(overflow)[0]
        if len(bad):
            raise _capi.SodError(f"sod_sift_extract_batch: more than capacity={self.sift.capacity} keypoints in frame "
                                 f"{int(bad[0])} ({w}x{h}) of the batch; use a larger GpuSift(capacity=...)")
        if fl[3 * B]:
            raise _capi.SodError("sod_sift_extract_batch: the packed rows exceed the output buffers")
        c = hv["counters"]
        n_m, n_bins, n_votes, n_edge, ovf, n_open = (int(v) for v in c[:6])
        n_valid, ovf2, n_singular, n_res_edge = (int(v) for v in c[9:13])
        if ovf or ovf2:
            raise RuntimeError("output capacity exceeded")
        if n_valid > state["k"]:
            raise RuntimeError(f"{n_valid} verified bins, more than the {state['k']} this LiveDetector reads back; "
                               "use a larger LiveDetector(max_bins=...)")
        rows = int(count.sum())
        out = {name: hv[name][:rows].copy() for name in ("idx", "ok")}
        out.update({name: hv[name][:n_valid].copy() for name in _BIN_FIELDS})
        out.update(row_lo=0, n_matches=n_m, n_bins=n_bins, n_votes=n_votes, n_near_edge=n_edge,
                   n_unresolved_edge=n_open, n_valid=n_valid, n_singular=n_singular, n_residual_edge=n_res_edge)
        n_clusters = int(hv["pose_counters"][0])
        poses: dict[int, list] = {}
        for pose, frame, shape in zip(hv["pose"][:n_clusters], hv["pose_frame"][:n_clusters].tolist(),
                                      hv["pose_shape"][:n_clusters].tolist()):
            cx, cy, ori, scale = pose[:4].tolist()
            poses.setdefault(frame, []).append(((cx, cy), ori, scale, (pose[4], pose[5]) if shape >= 0 else (0, 0)))
        sb = None
        if self.features:
            t = state["sift"]
            sb = SiftBatch(t["des"][:rows], t["xy"][:rows], t["angle"][:rows], t["octave"][:rows], t["size"][:rows],
                           t["response"][:rows], t["frame"][:rows], count, offset, (w, h))
        return [split_frame(out, poses, p.spaces_per_frame, k, int(offset[k]), int(offset[k] + count[k]),
                            **({"features": sb.features(k)} if sb is not None else {}))
                for k in range(B)]
