"""One camera frame (or a batch of B frames, of one size or of a camera rig's sizes) to detections in one CUDA-graph
replay.

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

A rig of cameras of different resolutions is one LiveDetector over a list of sizes, frame k of a call of size k:

    rig = LiveDetector(pipeline, GpuSift(max_keypoints=R), [(1920, 1080), (1280, 720), (640, 480)])
    wide, left, right = rig.detect([f0, f1, f2])

Its graph uploads the host frames from one pinned arena into one device arena, runs them through one mixed-size SIFT
pass (GpuSift.enqueue_mixed, over the detector's own SIFT buffers), copies each frame's (w, h) into the pipeline's
frame_wh on the device, and continues as above with B x R rows.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _capi
from .sift import SiftBatch, _align256, _gray, _is_cuda, _MixedBuffers, mixed_workspace_bytes
from .stream import one_rank_error, split_frame

# the verified-bin fields read back per call, as DetectionPipeline.fetch reads them
_BIN_FIELDS = ("valid_bin", "params", "votes", "status", "valid_group", "valid_code", "valid_order", "valid_mean")


class LiveDetector:
    """Detections of B frames per call, the whole path replayed as one CUDA graph.

    pipeline    a single-rank (or shard="frames") DetectionPipeline on u8 descriptors, with
                max_queries >= frames x sift.max_keypoints and frame_wh of at least `frames` rows (its values are
                overwritten by every call)
    sift        a GpuSift with max_keypoints set: a frame keeps cv2's first max_keypoints keypoints
    frame_size  (width, height) of every frame, or a list of B (width, height), one per frame of a call (a camera
                rig, at most 64 frames); a list of equal sizes is B frames of that size
    frames      B, frames per call (default: 1, or the length of the list, which it must then equal)
    max_bins    verified bins read back per call (at most 65,536, the limit of the pose clustering); a call that
                verifies more raises
    features    add each frame's FrameFeatures (its SIFT rows, read back from the device) to its result

    detect(frames) returns one dict per frame with the fields of a FrameStream frame result.  The graph is captured
    on the first call, after warm-up runs, once for host inputs and once for CUDA inputs if both occur; several
    LiveDetectors (of one size, or rigs) may share a pipeline and a GpuSift when their calls do not overlap.  A rig
    owns the SIFT buffers its graph writes, so no other call of the GpuSift can move them."""

    def __init__(self, pipeline, sift, frame_size, frames: int | None = None, max_bins: int = 4096,
                 features: bool = False):
        p = pipeline
        if getattr(p, "world", 1) > 1 and getattr(p, "shard_mode", "db") == "db":
            raise ValueError(one_rank_error("LiveDetector"))
        if getattr(p, "float_path", False):
            raise ValueError("LiveDetector needs a pipeline on u8 descriptors: GPU SIFT gives u8 rows, and this "
                             "pipeline's database is float32 (the bf16 path)")
        sizes = np.asarray(frame_size, dtype=np.int64)
        if sizes.ndim == 2 and sizes.shape[1] == 2 and len(sizes) >= 1:
            if frames is not None and int(frames) != len(sizes):
                raise ValueError(f"frames={frames}, but frame_size lists {len(sizes)} sizes")
            frames = len(sizes)
            if (sizes == sizes[0]).all():
                sizes = sizes[0]                    # one size: the uniform path
            elif frames > _capi.SIFT_MAX_MIXED_FRAMES:
                raise ValueError(f"a rig of {frames} frames of different sizes; at most "
                                 f"{_capi.SIFT_MAX_MIXED_FRAMES}")
        elif sizes.shape != (2,):
            raise ValueError(f"frame_size {frame_size}: expected (width, height) or a list of them")
        if (sizes < 1).any():
            raise ValueError(f"frame_size {frame_size} out of range")
        self.frames = 1 if frames is None else int(frames)
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
        self.pipeline, self.sift = p, sift
        self.max_bins, self.features = int(max_bins), bool(features)
        # a rig: frame_sizes int [B, 2] and frame_size None; one size: frame_size (w, h) and frame_sizes None
        self.mixed = sizes.ndim == 2
        self.frame_size = None if self.mixed else (int(sizes[0]), int(sizes[1]))
        self.frame_sizes = sizes if self.mixed else None
        # a rig the mixed pass would refuse (a side above 32768, too many keypoint slots) is refused here
        self._ws_bytes = mixed_workspace_bytes(sizes, sift.capacity) if self.mixed else 0
        self._img = self._host = None
        self._graphs: dict[bool, tuple] = {}      # host upload in the graph? -> (graph, what it reads and writes)

    def _size(self, k: int) -> tuple:
        """Frame k's (w, h)."""
        return self.frame_size if not self.mixed else (int(self.frame_sizes[k][0]), int(self.frame_sizes[k][1]))

    # ------------------------------------------------------------------------------------------------ inputs
    def _frames(self, frames) -> bool:
        """Stage one call's frames: host ones in the pinned staging (uploaded by the graph), CUDA ones straight
        into the device image buffer.  -> True when the graph's upload is wanted (all frames on the host)."""
        frames = list(frames.unbind(0)) if _is_cuda(frames) and frames.dim() == 3 else list(frames)
        if len(frames) != self.frames:
            raise ValueError(f"LiveDetector takes {self.frames} frames per call, got {len(frames)}")
        frames = [f if _is_cuda(f) else _gray(f) for f in frames]
        for k, f in enumerate(frames):
            w, h = self._size(k)
            if tuple(f.shape) != (h, w) or (_is_cuda(f) and f.dtype != torch.uint8):
                raise ValueError(f"frame {k}: expected a {w}x{h} u8 image, got {f.dtype} {tuple(f.shape)}")
        if self._img is None:
            self._alloc()
        upload = not any(_is_cuda(f) for f in frames)
        for k, f in enumerate(frames):
            if upload:
                self._host[k].copy_(torch.from_numpy(f))
            else:
                self._img[k].copy_(f if _is_cuda(f) else torch.from_numpy(f))
        return upload

    def _alloc(self) -> None:
        """The device image buffer and its pinned staging: [B, h, w] for one size; for a rig, one arena of the
        frames at 256-byte aligned offsets (self._img holds their [h, w] views), and the rig's own SIFT buffers."""
        dev = self.pipeline.device
        if not self.mixed:
            w, h = self.frame_size
            self._img = torch.empty((self.frames, h, w), dtype=torch.uint8, device=dev)
            self._host = torch.empty((self.frames, h, w), dtype=torch.uint8, pin_memory=True)
            return
        off = np.cumsum([0] + [_align256(int(w) * int(h)) for w, h in self.frame_sizes]).tolist()
        self._arena = torch.empty(off[-1], dtype=torch.uint8, device=dev)
        self._host_arena = torch.empty(off[-1], dtype=torch.uint8, pin_memory=True)

        def views(arena):
            return [arena[off[k]:off[k] + int(w) * int(h)].view(int(h), int(w))
                    for k, (w, h) in enumerate(self.frame_sizes)]

        img = views(self._arena)
        self._layout = self.sift._mixed_layout(img, "LiveDetector")
        self._sb = _MixedBuffers(dev)
        self._sb.fit(self._ws_bytes, 0, self.frames, self.sift.capacity, self.sift.max_keypoints)
        self._wh = torch.from_numpy(self.frame_sizes.astype(np.int32)).to(dev)
        self._img, self._host = img, views(self._host_arena)        # last: a failed allocation above is retried

    # ------------------------------------------------------------------------------------------------ the graph
    def _pinned(self, src: torch.Tensor) -> torch.Tensor:
        return torch.empty(src.shape, dtype=src.dtype, pin_memory=True)

    def _sift(self, upload: bool) -> tuple:
        """Upload (if wanted) and SIFT of the call's frames and their sizes in frame_wh, enqueued on the current
        stream.  -> (the SIFT output tensors, the rows of this call on the device: offset[B-1] + count[B-1])."""
        p, B = self.pipeline, self.frames
        if not self.mixed:
            w, h = self.frame_size
            if upload:
                self._img.copy_(self._host, non_blocking=True)
            t = self.sift.enqueue_batch(self._img, slot=0)
            p.scene.frame_wh[:, 0].fill_(w)
            p.scene.frame_wh[:, 1].fill_(h)
            F = B
        else:
            if upload:
                self._arena.copy_(self._host_arena, non_blocking=True)
            t = self.sift._enqueue_mixed(self._sb, self._img, self._layout)
            p.scene.frame_wh[:B].copy_(self._wh)
            F = self._sb.frames
        fl = t["flags"]
        return t, fl[B - 1:B] + fl[F + B - 1:F + B]

    def _body(self, upload: bool, host: dict | None) -> dict:
        """The whole path, enqueued on the current stream (warm-up runs and the captured one alike)."""
        p, R = self.pipeline, self.rows
        t, n_dev = self._sift(upload)
        p.load_queries(t["des"][:R], t["xy"][:R], t["angle"][:R], t["octave"][:R], t["frame"][:R], slot=0)
        fl = t["flags"]
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
        sift = self.sift._batch_buffers[(*self.frame_size, self.frames)] if not self.mixed else self._sb
        state["keep"] = (p.matcher._ws, p.matcher._qn, p.voter._ws, p._hough[0], p._aff[0], p.scene.frame_wh,
                         p._qset(0), sift, state["poses"])
        entry = self._graphs[upload] = (graph, state)
        return entry

    # ------------------------------------------------------------------------------------------------ host side
    def detect(self, frames) -> list[dict]:
        """One call: B frames, frame k of the detector's size k (host gray / BGR images, CUDA u8 [H, W] tensors, which
        may be pitched, or, for one size, a CUDA u8 [B, H, W] tensor) ->
        one result per frame (match_q, match_t, n_descriptors, valid_group, valid_code, votes, live, params,
        final_pose, and features if asked for).  Raises SodError naming a frame with more keypoints than the SIFT
        capacity, RuntimeError on a Hough / affine output overflow or on more verified bins than max_bins."""
        p, B = self.pipeline, self.frames
        upload = self._frames(frames)
        with torch.cuda.device(p.device):
            graph, state = self._graph(upload)
            graph.replay()
            torch.cuda.current_stream(p.device).synchronize()
        hv = {name: v.numpy() for name, v in state["host"].items()}
        fl = hv["flags"]
        F = (len(fl) - 1) // 3
        count, offset, overflow = fl[:B].astype(np.int64), fl[F:F + B].astype(np.int64), fl[2 * F:2 * F + B]
        fn = "sod_sift_extract_mixed" if self.mixed else "sod_sift_extract_batch"
        bad = np.nonzero(overflow)[0]
        if len(bad):
            w, h = self._size(int(bad[0]))
            raise _capi.SodError(f"{fn}: more than capacity={self.sift.capacity} keypoints in frame {int(bad[0])} "
                                 f"({w}x{h}) of the batch; use a larger GpuSift(capacity=...)")
        if fl[3 * F]:
            raise _capi.SodError(f"{fn}: the packed rows exceed the output buffers")
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
                           t["response"][:rows], t["frame"][:rows], count, offset, self.frame_size,
                           frame_sizes=self.frame_sizes)
        return [split_frame(out, poses, p.spaces_per_frame, k, int(offset[k]), int(offset[k] + count[k]),
                            **({"features": sb.features(k)} if sb is not None else {}))
                for k in range(B)]
