"""SIFT on the GPU (sod_sift_extract / sod_sift_describe): cv2.SIFT_create() with its default parameters, with
keypoints and descriptors in OpenCV's conventions, so everything downstream (unpack_sift_octave, the Hough
pose, the u8 matcher, the drop-in Main) reads them unchanged.  Opt-in: OpenCV SIFT stays the default extractor
and the reference; DESIGN.md 2 states how closely this one agrees with it.

    stream = FrameStream(pipeline, extractor=GpuSift())

GpuSift.extract_batch runs many same-size frames in one pass (sod_sift_extract_batch) and leaves the result on the
device, in the layout DetectionPipeline.load_queries takes; FrameStream uses it when the extractor has it.
GpuSift.extract_mixed does the same for frames of different sizes (sod_sift_extract_mixed), such as the training
images GenerateDatabaseInfo.build_database resizes to one width.
"""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass, field

import numpy as np

from . import _capi
from .stream import FrameFeatures


def _gray(image) -> np.ndarray:
    """A path, a BGR image or a gray image -> contiguous u8 gray, decoded and converted on the host exactly as
    stream.sift_features does."""
    import cv2
    if isinstance(image, (str, bytes)) or hasattr(image, "__fspath__"):
        img = cv2.imread(str(image))
        if img is None:
            raise FileNotFoundError(str(image))
    else:
        img = np.asarray(image)
    gray = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY) if img.ndim == 3 else img
    if gray.dtype != np.uint8 or gray.ndim != 2:
        raise ValueError(f"expected an 8-bit gray or BGR image, got {gray.dtype} {gray.shape}")
    return np.ascontiguousarray(gray)


def _is_cuda(x) -> bool:
    return getattr(x, "is_cuda", False)


@dataclass
class SiftBatch:
    """The keypoints of a batch of frames, packed frame after frame on the device.

    des u8 [rows, 128], xy f32 [rows, 2], angle, size, response f32 [rows], octave, frame i32 [rows]: frame k's
    keypoints are rows offset[k]:offset[k] + count[k] (host arrays), in the order GpuSift.extract gives for that
    frame alone.  frame_size is the (w, h) of a same-size batch (None for a mixed one); frame_sizes (int [B, 2], None for a same-size
    batch) gives each frame's own (w, h).  The tensors are GpuSift's buffers: the next extract_batch of the same
    size, batch and slot, or the next extract_mixed of the same slot, overwrites them."""
    des: object
    xy: object
    angle: object
    octave: object
    size: object
    response: object
    frame: object
    count: np.ndarray
    offset: np.ndarray
    frame_size: tuple
    frame_sizes: np.ndarray | None = field(default=None)

    def __len__(self) -> int:
        return len(self.count)

    @property
    def rows(self) -> int:
        return int(self.count.sum())

    def arrays(self, k: int) -> dict:
        """Frame k's keypoints as host arrays, in the format of GpuSift.extract."""
        lo, hi = int(self.offset[k]), int(self.offset[k] + self.count[k])
        out = {name: getattr(self, name)[lo:hi].cpu().numpy()
               for name in ("xy", "size", "angle", "response", "octave", "des")}
        out["frame_size"] = self.size_of(k)
        return out

    def size_of(self, k: int) -> tuple:
        """Frame k's (w, h)."""
        if self.frame_sizes is None:
            return self.frame_size
        return int(self.frame_sizes[k][0]), int(self.frame_sizes[k][1])

    def features(self, k: int) -> FrameFeatures:
        r = self.arrays(k)
        return FrameFeatures(r["des"], r["xy"], r["angle"], r["octave"], r["frame_size"])


class _BatchBuffers:
    """Device workspace, pinned host staging, device input and packed output rows for one (size, frames)."""

    def __init__(self, width: int, height: int, frames: int, capacity: int, max_keypoints: int | None, device):
        import torch
        self.bytes = int(_capi.lib.sod_sift_batch_workspace_bytes(width, height, frames, capacity))
        if self.bytes == 0:
            raise ValueError(f"sod_sift: {frames} frames of {width}x{height} with capacity {capacity} out of range")
        rows = frames * (capacity if max_keypoints is None else min(capacity, max(1, int(max_keypoints))))
        mk = lambda shape, dt: torch.empty(shape, dtype=dt, device=device)  # noqa: E731
        self.ws = mk(self.bytes, torch.uint8)
        self.img = mk((frames, height, width), torch.uint8)
        self.host = None                       # pinned [frames, h, w], made on the first host upload
        self.outs = [None, None]               # output rows per slot, made on first use
        self.frames, self.rows, self.capacity, self.device = frames, rows, capacity, device
        self.flags = torch.empty((3 * frames + 1,), dtype=torch.int32, pin_memory=True)

    def out(self, slot: int):
        import torch
        if self.outs[slot] is None:
            f, r = self.frames, self.rows
            mk = lambda shape, dt: torch.empty(shape, dtype=dt, device=self.device)  # noqa: E731
            t = dict(xy=mk((r, 2), torch.float32), size=mk(r, torch.float32), angle=mk(r, torch.float32),
                     response=mk(r, torch.float32), octave=mk(r, torch.int32), des=mk((r, 128), torch.uint8),
                     frame=mk(r, torch.int32), flags=mk(3 * f + 1, torch.int32))
            fl = t["flags"]
            st = _capi.SiftBatchOut(*(t[k].data_ptr() for k in ("xy", "size", "angle", "response", "octave", "des",
                                                                  "frame")),
                                    fl[:f].data_ptr(), fl[f:2 * f].data_ptr(), fl[2 * f:3 * f].data_ptr(),
                                    fl[3 * f:].data_ptr(), r, self.capacity)
            self.outs[slot] = (t, st)
        return self.outs[slot]


class _MixedBuffers:
    """One output slot of extract_mixed: device workspace, device input arena, pinned staging and packed output
    rows, each grown to the largest batch seen and reused for any mix that fits, whatever its sizes."""

    def __init__(self, device):
        self.device = device
        self.ws = self.arena = self.host = self.t = self.out = self.flags = None
        self.frames = 0

    def _mk(self, shape, dt):
        import torch
        return torch.empty(shape, dtype=dt, device=self.device)

    def fit(self, ws_bytes: int, arena_bytes: int, frames: int, capacity: int, max_keypoints: int | None) -> None:
        import torch
        if self.ws is None or self.ws.numel() < ws_bytes:
            self.ws = None                    # release before allocating the larger one
            self.ws = self._mk(ws_bytes, torch.uint8)
        if arena_bytes and (self.arena is None or self.arena.numel() < arena_bytes):
            self.arena = self.host = None
            self.arena = self._mk(arena_bytes, torch.uint8)
            self.host = torch.empty(arena_bytes, dtype=torch.uint8, pin_memory=True)
        if frames > self.frames:
            self.t = self.out = None
            f, r = frames, frames * (capacity if max_keypoints is None else min(capacity, max(1, int(max_keypoints))))
            mk = self._mk
            t = dict(xy=mk((r, 2), torch.float32), size=mk(r, torch.float32), angle=mk(r, torch.float32),
                     response=mk(r, torch.float32), octave=mk(r, torch.int32), des=mk((r, 128), torch.uint8),
                     frame=mk(r, torch.int32), flags=mk(3 * f + 1, torch.int32))
            fl = t["flags"]
            self.out = _capi.SiftBatchOut(*(t[k].data_ptr() for k in ("xy", "size", "angle", "response", "octave",
                                                                       "des", "frame")),
                                          fl[:f].data_ptr(), fl[f:2 * f].data_ptr(), fl[2 * f:3 * f].data_ptr(),
                                          fl[3 * f:].data_ptr(), r, capacity)
            self.t, self.frames = t, frames
            self.flags = torch.empty((3 * f + 1,), dtype=torch.int32, pin_memory=True)


def _align256(n: int) -> int:
    return (n + 255) & ~255


class _Buffers:
    """Device workspace, input image and output arrays for one image size."""

    def __init__(self, width: int, height: int, capacity: int, device):
        import torch
        self.bytes = int(_capi.lib.sod_sift_workspace_bytes(width, height, capacity))
        if self.bytes == 0:
            raise ValueError(f"sod_sift: image size {width}x{height} or capacity {capacity} out of range")
        mk = lambda shape, dt: torch.empty(shape, dtype=dt, device=device)  # noqa: E731
        self.ws = mk(self.bytes, torch.uint8)
        self.img = mk((height, width), torch.uint8)
        self.xy = mk((capacity, 2), torch.float32)
        self.size = mk(capacity, torch.float32)
        self.angle = mk(capacity, torch.float32)
        self.response = mk(capacity, torch.float32)
        self.octave = mk(capacity, torch.int32)
        self.des = mk((capacity, 128), torch.uint8)
        self.counters = mk(2, torch.int32)
        self.out = _capi.SiftOut(*(t.data_ptr() for t in (self.xy, self.size, self.angle, self.response, self.octave,
                                                           self.des, self.counters)), capacity)


class GpuSift:
    """Callable image -> FrameFeatures, a drop-in for stream.sift_features on the GPU.

    max_keypoints  keep the first n keypoints in cv2's sorted order (None = all), as sift_features does
    capacity       keypoints one frame may produce before duplicate removal; a frame with more raises
                   (the output is never truncated silently)
    device         CUDA device (default: the current one)

    One instance may be shared by FrameStream's worker threads: decoding and colour conversion run in the
    calling thread, the device part holds a lock and runs on the instance's own stream.  Buffers are cached per
    image size."""

    def __init__(self, max_keypoints: int | None = None, capacity: int = 1 << 16, device=None):
        self.max_keypoints = max_keypoints
        self.capacity = int(capacity)
        if not 1 <= self.capacity <= (1 << 24):
            raise ValueError(f"capacity {capacity} out of range (1..2^24)")
        self._device = device
        self._lock = threading.Lock()
        self._stream = None
        self._buffers: dict[tuple[int, int], _Buffers] = {}
        self._batch_buffers: dict[tuple[int, int, int], _BatchBuffers] = {}
        self._mixed: list[_MixedBuffers | None] = [None, None]

    def _setup_stream(self) -> None:
        import torch
        if self._stream is None:
            self._device = torch.device("cuda", torch.cuda.current_device()) if self._device is None \
                else torch.device(self._device)
            self._stream = torch.cuda.Stream(self._device)

    def _setup(self, width: int, height: int) -> _Buffers:
        self._setup_stream()
        b = self._buffers.get((width, height))
        if b is None:
            b = self._buffers[(width, height)] = _Buffers(width, height, self.capacity, self._device)
        return b

    def _upload(self, gray: np.ndarray) -> _Buffers:
        import torch
        h, w = gray.shape
        b = self._setup(w, h)
        with torch.cuda.stream(self._stream):
            b.img.copy_(torch.from_numpy(gray))
        return b

    def extract(self, image) -> dict:
        """All keypoint fields as numpy arrays: xy, size, angle, response, octave, des, and the frame's (w, h)."""
        import torch
        gray = _gray(image)
        h, w = gray.shape
        with self._lock, torch.cuda.device(self._device or torch.cuda.current_device()):
            b = self._upload(gray)
            _capi.check(_capi.lib.sod_sift_extract(b.img.data_ptr(), w, h, w, C.byref(b.out), b.ws.data_ptr(),
                                                   b.bytes, self._stream.cuda_stream), "sod_sift_extract")
            with torch.cuda.stream(self._stream):
                n, overflow = (int(v) for v in b.counters.cpu())
                if overflow:
                    raise _capi.SodError(f"sod_sift_extract: more than capacity={self.capacity} keypoints in a "
                                         f"{w}x{h} frame; use a larger GpuSift(capacity=...)")
                if self.max_keypoints is not None:
                    n = min(n, int(self.max_keypoints))
                out = {k: getattr(b, k)[:n].cpu().numpy()
                       for k in ("xy", "size", "angle", "response", "octave", "des")}
        out["frame_size"] = (w, h)
        return out

    @staticmethod
    def prepare(image):
        """What extract_batch takes of one frame: a CUDA u8 [H, W] tensor as it is, anything else as _gray makes
        it (decoded and converted on the host).  FrameStream's worker threads call this."""
        return image if _is_cuda(image) else _gray(image)

    def extract_batch(self, images, slot: int = 0) -> SiftBatch:
        """SIFT of a batch of same-size frames in one pass, the result left on the device.

        images  a CUDA u8 tensor [B, H, W], or a list of CUDA u8 [H, W] tensors and / or host images / paths
                (decoded and converted as extract does; an all-host list is uploaded as one pinned [B, H, W] copy)
        slot    0 or 1: which of two output sets to fill, so that a caller can read one batch while the next is
                extracted

        Waits for the batch (counts are read on the host); a frame with more than `capacity` keypoints raises
        SodError naming it."""
        import torch
        if slot not in (0, 1):
            raise ValueError("slot must be 0 or 1")
        dev_in = _is_cuda(images)
        frames = images if dev_in else [self.prepare(im) for im in images]
        if len(frames) == 0:
            raise ValueError("extract_batch needs at least one frame")
        shapes = {tuple(f.shape[-2:]) for f in frames} if not dev_in else {tuple(images.shape[-2:])}
        if len(shapes) != 1:
            raise ValueError(f"extract_batch needs frames of one size, got {sorted(shapes)}")
        (h, w), n = shapes.pop(), len(frames)
        if dev_in and (images.dim() != 3 or images.dtype != torch.uint8):
            raise ValueError(f"expected a u8 [B, H, W] tensor, got {images.dtype} {tuple(images.shape)}")
        with self._lock, torch.cuda.device(self._device or torch.cuda.current_device()):
            self._setup_stream()
            b = self._batch_buffers.get((w, h, n))
            if b is None:
                b = self._batch_buffers[(w, h, n)] = _BatchBuffers(w, h, n, self.capacity, self.max_keypoints,
                                                                   self._device)
            t, out = b.out(slot)
            src, pitch, fstride = b.img, w, w * h
            if dev_in or any(_is_cuda(f) for f in frames):
                # CUDA inputs come from the caller's current stream; host inputs need no wait, so the SIFT can
                # run beside the caller's other work (FrameStream's previous detection pass)
                self._stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(self._stream):
                if dev_in:
                    if images.device != b.img.device:
                        raise ValueError(f"images are on {images.device}, GpuSift on {b.img.device}")
                    if images.stride(2) == 1 and images.stride(1) >= w and images.stride(0) >= images.stride(1) * h:
                        src, pitch, fstride = images, images.stride(1), images.stride(0)
                    else:
                        b.img.copy_(images)
                else:
                    on_host = [k for k, f in enumerate(frames) if not _is_cuda(f)]
                    if on_host and b.host is None:
                        b.host = torch.empty((n, h, w), dtype=torch.uint8, pin_memory=True)
                    for k in on_host:
                        b.host[k].copy_(torch.from_numpy(frames[k]))
                    if len(on_host) == n:
                        b.img.copy_(b.host, non_blocking=True)
                    else:
                        for k, f in enumerate(frames):
                            b.img[k].copy_(f if _is_cuda(f) else b.host[k], non_blocking=True)
                mk = 0 if self.max_keypoints is None else max(1, int(self.max_keypoints))
                _capi.check(_capi.lib.sod_sift_extract_batch(src.data_ptr(), w, h, pitch, fstride, n, mk,
                                                             C.byref(out), b.ws.data_ptr(), b.bytes,
                                                             self._stream.cuda_stream), "sod_sift_extract_batch")
                b.flags.copy_(t["flags"], non_blocking=True)
            # the whole batch is done once this returns: its rows may be read on any stream, and the pinned
            # staging and the workspace are free for the next call
            self._stream.synchronize()
            fl = b.flags.numpy()
            count, offset, overflow = fl[:n].astype(np.int64), fl[n:2 * n].astype(np.int64), fl[2 * n:3 * n]
        bad = np.nonzero(overflow)[0]
        if len(bad):
            raise _capi.SodError(f"sod_sift_extract_batch: more than capacity={self.capacity} keypoints in frame "
                                 f"{int(bad[0])} ({w}x{h}) of the batch; use a larger GpuSift(capacity=...)")
        if fl[3 * n]:
            raise _capi.SodError("sod_sift_extract_batch: the packed rows exceed the output buffers")
        rows = int(count.sum())
        return SiftBatch(t["des"][:rows], t["xy"][:rows], t["angle"][:rows], t["octave"][:rows], t["size"][:rows],
                         t["response"][:rows], t["frame"][:rows], count, offset, (w, h))

    def extract_mixed(self, images, slot: int = 0) -> SiftBatch:
        """SIFT of a batch of frames of any sizes in one pass (sod_sift_extract_mixed), the result left on the device.

        images  a list of up to 64 frames, each a CUDA u8 [H, W] tensor (pitched or not) or a host image / path
                (decoded and converted as extract does)
        slot    0 or 1: which of two output sets to fill

        Frame k's rows are those extract gives for it alone, in the same order; SiftBatch.frame_sizes holds each
        frame's (w, h).  The buffers of a slot are grown to the largest batch seen, not kept per size.  Waits for
        the batch; a frame with more than `capacity` keypoints raises SodError naming it."""
        import torch
        if slot not in (0, 1):
            raise ValueError("slot must be 0 or 1")
        frames = [self.prepare(im) for im in images]
        n = len(frames)
        if not 1 <= n <= _capi.SIFT_MAX_MIXED_FRAMES:
            raise ValueError(f"extract_mixed takes 1..{_capi.SIFT_MAX_MIXED_FRAMES} frames, got {n}")
        for k, f in enumerate(frames):
            if f.ndim != 2 or (f.dtype != torch.uint8 if _is_cuda(f) else f.dtype != np.uint8):
                raise ValueError(f"frame {k}: expected a u8 [H, W] image, got {f.dtype} {tuple(f.shape)}")
        sizes = np.array([(f.shape[1], f.shape[0]) for f in frames], np.int32)
        wh = (C.c_int32 * (2 * n))(*sizes.reshape(-1).tolist())
        need = int(_capi.lib.sod_sift_mixed_workspace_bytes(C.cast(wh, C.c_void_p), n, self.capacity))
        if need == 0:
            raise ValueError(f"sod_sift: {n} frames of sizes {sizes.tolist()} with capacity {self.capacity} out of "
                             "range")
        # frames that need a copy (host images, CUDA tensors whose rows are not unit-stride) go to the arena,
        # each at a 256-byte aligned offset with pitch = width
        in_place = [_is_cuda(f) and f.stride(1) == 1 and f.stride(0) >= f.shape[1] for f in frames]
        at, arena_off = 0, []
        for f, keep in zip(frames, in_place):
            arena_off.append(at)
            if not keep:
                at += _align256(f.shape[0] * f.shape[1])
        with self._lock, torch.cuda.device(self._device or torch.cuda.current_device()):
            self._setup_stream()
            b = self._mixed[slot]
            if b is None:
                b = self._mixed[slot] = _MixedBuffers(self._device)
            b.fit(need, at, n, self.capacity, self.max_keypoints)
            if any(_is_cuda(f) for f in frames):
                self._stream.wait_stream(torch.cuda.current_stream())
            ptrs, pitches = [], []
            try:
                with torch.cuda.stream(self._stream):
                    host = [k for k, f in enumerate(frames) if not _is_cuda(f)]
                    for k in host:
                        h, w = frames[k].shape
                        b.host[arena_off[k]:arena_off[k] + h * w].copy_(torch.from_numpy(frames[k]).reshape(-1))
                    if host:
                        b.arena[:at].copy_(b.host[:at], non_blocking=True)
                    for k, f in enumerate(frames):
                        h, w = f.shape
                        if _is_cuda(f) and f.device != b.ws.device:
                            raise ValueError(f"frame {k} is on {f.device}, GpuSift on {b.ws.device}")
                        if in_place[k]:
                            ptrs.append(f.data_ptr())
                            pitches.append(f.stride(0))
                            continue
                        if _is_cuda(f):
                            b.arena[arena_off[k]:arena_off[k] + h * w].view(h, w).copy_(f)
                        ptrs.append(b.arena[arena_off[k]:].data_ptr())
                        pitches.append(w)
                    mk = 0 if self.max_keypoints is None else max(1, int(self.max_keypoints))
                    _capi.check(_capi.lib.sod_sift_extract_mixed(
                        C.cast((C.c_void_p * n)(*ptrs), C.c_void_p), C.cast(wh, C.c_void_p),
                        C.cast((C.c_int64 * n)(*pitches), C.c_void_p), n, mk, C.byref(b.out), b.ws.data_ptr(),
                        b.ws.numel(), self._stream.cuda_stream), "sod_sift_extract_mixed")
                    b.flags.copy_(b.t["flags"], non_blocking=True)
            finally:
                # as in extract_batch: once this returns the rows may be read on any stream and the buffers are
                # free; also when a step above raised, since the pinned staging may still be in a copy
                self._stream.synchronize()
            fl, F = b.flags.numpy(), b.frames
            count, offset = fl[:n].astype(np.int64), fl[F:F + n].astype(np.int64)
            overflow, rows_overflow = fl[2 * F:2 * F + n].copy(), int(fl[3 * F])
            t = b.t
        bad = np.nonzero(overflow)[0]
        if len(bad):
            k = int(bad[0])
            raise _capi.SodError(f"sod_sift_extract_mixed: more than capacity={self.capacity} keypoints in frame {k} "
                                 f"({sizes[k][0]}x{sizes[k][1]}) of the batch; use a larger GpuSift(capacity=...)")
        if rows_overflow:
            raise _capi.SodError("sod_sift_extract_mixed: the packed rows exceed the output buffers")
        rows = int(count.sum())
        return SiftBatch(t["des"][:rows], t["xy"][:rows], t["angle"][:rows], t["octave"][:rows], t["size"][:rows],
                         t["response"][:rows], t["frame"][:rows], count, offset, None,
                         frame_sizes=sizes.astype(np.int64))

    def __call__(self, image) -> FrameFeatures:
        r = self.extract(image)
        return FrameFeatures(r["des"], r["xy"], r["angle"], r["octave"], r["frame_size"])

    def describe(self, image, xy, size, angle, octave) -> np.ndarray:
        """cv2.SIFT.compute(gray, keypoints) for keypoints given as arrays (pt [n, 2], size, angle, octave as
        cv2 packs it): u8 descriptors [n, 128].  Raises if an octave / layer names no level of the pyramid."""
        import torch
        gray = _gray(image)
        h, w = gray.shape
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        n = xy.shape[0]
        arrays = [np.ascontiguousarray(a, dt).reshape(n) for a, dt in
                  ((size, np.float32), (angle, np.float32), (octave, np.int32))]
        with self._lock, torch.cuda.device(self._device or torch.cuda.current_device()):
            b = self._upload(gray)
            with torch.cuda.stream(self._stream):
                dev = [torch.from_numpy(a).to(self._device) for a in [xy] + arrays]
                des = torch.empty((n, 128), dtype=torch.uint8, device=self._device)
                n_invalid = torch.zeros(1, dtype=torch.int32, device=self._device)
                _capi.check(_capi.lib.sod_sift_describe(b.img.data_ptr(), w, h, w, *(t.data_ptr() for t in dev), n,
                                                        des.data_ptr(), n_invalid.data_ptr(), b.ws.data_ptr(),
                                                        b.bytes, self._stream.cuda_stream), "sod_sift_describe")
                bad = int(n_invalid.cpu()[0])
                if bad:
                    raise ValueError(f"{bad} keypoints name no octave / layer of the {w}x{h} image's pyramid")
                return des.cpu().numpy()

    def gaussian_level(self, frame_size: tuple[int, int], octave: int, level: int,
                       batch: tuple[int, int] | None = None) -> np.ndarray:
        """Gaussian level `level` (0..5) of `octave` (-1 = the doubled image) of the last frame of this size
        extracted or described, f32 [h, w].  batch = (frames, k): frame k of the last extract_batch of `frames`
        frames of this size."""
        import torch
        w, h = frame_size
        wh = (C.c_int32 * 2)()
        off = int(_capi.lib.sod_sift_level_offset(w, h, octave, level, C.cast(wh, C.c_void_p)))
        if off < 0:
            _capi.check(-1, "sod_sift_level_offset")
        with self._lock:
            if batch is None:
                ws = self._buffers[(w, h)].ws
            else:
                ws = self._batch_buffers[(w, h, batch[0])].ws
                off += batch[1] * int(_capi.lib.sod_sift_batch_workspace_bytes(w, h, 1, 0))
            self._stream.synchronize()
            n = wh[0] * wh[1]
            return ws[off:off + 4 * n].view(torch.float32).reshape(wh[1], wh[0]).cpu().numpy()
