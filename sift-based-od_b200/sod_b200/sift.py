"""SIFT on the GPU (sod_sift_extract / sod_sift_describe): cv2.SIFT_create() with its default parameters, with
keypoints and descriptors in OpenCV's conventions, so everything downstream (unpack_sift_octave, the Hough
pose, the u8 matcher, the drop-in Main) reads them unchanged.  Opt-in: OpenCV SIFT stays the default extractor
and the reference; DESIGN.md 2 states how closely this one agrees with it.

    stream = FrameStream(pipeline, extractor=GpuSift())
"""
from __future__ import annotations

import ctypes as C
import threading

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

    def _setup(self, width: int, height: int) -> _Buffers:
        import torch
        if self._stream is None:
            self._device = torch.device("cuda", torch.cuda.current_device()) if self._device is None \
                else torch.device(self._device)
            self._stream = torch.cuda.Stream(self._device)
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

    def gaussian_level(self, frame_size: tuple[int, int], octave: int, level: int) -> np.ndarray:
        """Gaussian level `level` (0..5) of `octave` (-1 = the doubled image) of the last frame of this size
        extracted or described, f32 [h, w]."""
        import torch
        w, h = frame_size
        wh = (C.c_int32 * 2)()
        off = int(_capi.lib.sod_sift_level_offset(w, h, octave, level, C.cast(wh, C.c_void_p)))
        if off < 0:
            _capi.check(-1, "sod_sift_level_offset")
        with self._lock:
            b = self._buffers[(w, h)]
            self._stream.synchronize()
            n = wh[0] * wh[1]
            return b.ws[off:off + 4 * n].view(torch.float32).reshape(wh[1], wh[0]).cpu().numpy()
