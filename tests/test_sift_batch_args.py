"""CPU-side checks of batched SIFT: workspace sizes and argument errors of sod_sift_extract_batch before any CUDA
call, GpuSift.extract_batch's input checks, and FrameStream's device path with a stand-in batch extractor and
pipeline (batches split at size changes, passes split at max_queries, input order, empty frames)."""
import ctypes as C

import numpy as np
import pytest
import torch

from sod_b200.stream import FrameStream
from test_stream import _EchoPipeline


def test_batch_workspace_bytes():
    from sod_b200._capi import lib
    one = lib.sod_sift_workspace_bytes(640, 480, 1000)
    assert lib.sod_sift_batch_workspace_bytes(640, 480, 1, 1000) == one
    pyramid = lib.sod_sift_batch_workspace_bytes(640, 480, 1, 0)
    assert pyramid == lib.sod_sift_workspace_bytes(640, 480, 0) and pyramid % 256 == 0
    for frames in (2, 5, 16):
        ws = lib.sod_sift_batch_workspace_bytes(640, 480, frames, 1000)
        assert ws >= frames * pyramid + frames * 1000 * (40 + 24 + 8 * 4)
        assert lib.sod_sift_batch_workspace_bytes(640, 480, frames, 0) == frames * pyramid
    assert lib.sod_sift_batch_workspace_bytes(0, 480, 1, 10) == 0
    assert lib.sod_sift_batch_workspace_bytes(640, 32769, 1, 10) == 0
    assert lib.sod_sift_batch_workspace_bytes(640, 480, 0, 10) == 0
    assert lib.sod_sift_batch_workspace_bytes(640, 480, 4097, 10) == 0
    assert lib.sod_sift_batch_workspace_bytes(640, 480, 2, -1) == 0
    assert lib.sod_sift_batch_workspace_bytes(640, 480, 2, (1 << 24) + 1) == 0
    assert lib.sod_sift_batch_workspace_bytes(640, 480, 256, 1 << 16) > 0            # frames x cap = 2^24
    assert lib.sod_sift_batch_workspace_bytes(640, 480, 257, 1 << 16) == 0


def test_extract_batch_rejects_bad_arguments_without_gpu():
    from sod_b200._capi import SiftBatchOut, lib
    fake = 1 << 20                         # never dereferenced: validation fails first
    f = lib.sod_sift_extract_batch

    def err(*args):
        assert f(*args) == -1
        return lib.sod_last_error()

    out = SiftBatchOut(*([fake] * 11), 400, 100)
    need = lib.sod_sift_batch_workspace_bytes(10, 10, 4, 100)
    ok = (fake, 10, 10, 10, 100, 4, 0, C.byref(out), fake, need, None)

    def with_(**kw):
        names = ("gray", "w", "h", "pitch", "stride", "frames", "max", "out", "ws", "bytes", "stream")
        a = dict(zip(names, ok))
        a.update(kw)
        return tuple(a[n] for n in names)

    assert b"null image" in err(*with_(gray=None))
    assert b"out of range" in err(*with_(w=0))
    assert b"out of range" in err(*with_(h=32769))
    assert b"pitch" in err(*with_(pitch=9))
    assert b"frames 0" in err(*with_(frames=0))
    assert b"frames 4097" in err(*with_(frames=4097))
    assert b"frame_stride" in err(*with_(stride=99))
    assert b"max_per_frame" in err(*with_(max=-1))
    assert b"null out" in err(*with_(out=None))
    for field, value, what in (("cap_per_frame", 0, b"cap_per_frame"), ("cap_per_frame", (1 << 22) + 1, b"cap_per_frame"),
                               ("cap_rows", 0, b"cap_rows"), ("cap_rows", (1 << 24) + 1, b"cap_rows")):
        bad = SiftBatchOut(*([fake] * 11), 400, 100)
        setattr(bad, field, value)
        assert what in err(*with_(out=C.byref(bad)))
    for i, name in enumerate(("xy", "size", "angle", "response", "octave", "des", "frame", "count", "offset",
                              "overflow", "rows_overflow")):
        bad = SiftBatchOut(*([fake] * 11), 400, 100)
        setattr(bad, name, None)
        assert b"null output" in err(*with_(out=C.byref(bad))), name
    assert b"workspace" in err(*with_(ws=None))
    assert b"workspace" in err(*with_(bytes=need - 1))
    assert b"workspace" in err(*with_(ws=fake + 16))                         # misaligned
    # the stride may exceed pitch x height (frames with gaps between them), and frames = 1 is allowed
    one = SiftBatchOut(*([fake] * 11), 100, 100)
    assert b"workspace" in err(fake, 10, 10, 10, 100, 1, 0, C.byref(one), fake, 0, None)


def test_extract_batch_rejects_mixed_sizes_before_any_device_work():
    from sod_b200.sift import GpuSift
    g = GpuSift()
    with pytest.raises(ValueError, match="one size"):
        g.extract_batch([np.zeros((10, 12), np.uint8), np.zeros((10, 13), np.uint8)])
    with pytest.raises(ValueError, match="at least one"):
        g.extract_batch([])
    with pytest.raises(ValueError, match="slot"):
        g.extract_batch([np.zeros((10, 12), np.uint8)], slot=2)


# ------------------------------------------------------------------------------- FrameStream's device path
class _FakeBatchSift:
    """Stands in for GpuSift on the CPU: frame i is an image filled with i whose size is sizes[i]; it has
    counts[i] keypoints, descriptor bytes 0 and 1 = (row within the frame) % 256 and i."""

    def __init__(self, counts):
        self.counts, self.calls = counts, []

    @staticmethod
    def prepare(image):
        return image

    def extract_batch(self, images, slot=0):
        from sod_b200.sift import SiftBatch
        ids = [int(im[0, 0]) for im in images]
        self.calls.append((ids, slot))
        count = np.array([self.counts[i] for i in ids], np.int64)
        offset = np.concatenate([[0], np.cumsum(count)[:-1]]).astype(np.int64)
        rows = int(count.sum())
        des = torch.zeros((rows, 128), dtype=torch.uint8)
        frame = torch.zeros(rows, dtype=torch.int32)
        for k, i in enumerate(ids):
            lo, n = int(offset[k]), int(count[k])
            des[lo:lo + n, 0] = torch.arange(n) % 256
            des[lo:lo + n, 1] = i
            frame[lo:lo + n] = k
        h, w = images[0].shape
        z = torch.zeros(rows, dtype=torch.float32)
        return SiftBatch(des, torch.zeros((rows, 2)), z, torch.zeros(rows, dtype=torch.int32), z, z, frame, count,
                         offset, (w, h))


def _frames(sizes):
    return [np.full(s, i, np.uint8) for i, s in enumerate(sizes)]


def test_device_path_batches_passes_and_order():
    A, B = (48, 64), (30, 40)
    sizes = [A, A, A, A, B, B, A, A, A, B]
    counts = [7, 0, 30, 12, 0, 0, 25, 3, 9, 0]
    ex = _FakeBatchSift(counts)
    pipe = _EchoPipeline(max_queries=40, n_frames=3)
    got = list(FrameStream(pipe, ex, batch_frames=3, workers=3, features=True).run(_frames(sizes)))
    # SIFT batches: at most batch_frames consecutive frames of one size, output sets alternating
    assert ex.calls == [([0, 1, 2], 0), ([3], 1), ([4, 5], 0), ([6, 7, 8], 1), ([9], 0)]
    # passes: longest prefix of a batch that fits max_queries; frame ids are the slots within the SIFT batch
    assert [n for n, _ in pipe.calls] == [37, 12, 37]           # [7,0,30] [12] ([0,0] has no rows) [25,3,9]
    assert pipe.calls[0][1].tolist() == [[64, 48]] * 3
    assert [i for i, _ in got] == list(range(len(sizes)))
    for i, r in got:
        assert r["n_descriptors"] == counts[i]
        np.testing.assert_array_equal(r["match_q"], np.arange(counts[i])[np.arange(counts[i]) % 2 == 1])
        assert (r["match_t"] == i).all()
        assert len(r["features"]) == counts[i] and r["features"].size == sizes[i][::-1]
        if counts[i]:
            assert r["final_pose"] and r["votes"].tolist() == [5] and r["live"].tolist() == [True]
        else:
            assert r["final_pose"] == [] and len(r["votes"]) == 0


def test_device_path_splits_a_batch_at_max_queries():
    counts = [15, 15, 15, 15, 0, 15]
    ex = _FakeBatchSift(counts)
    pipe = _EchoPipeline(max_queries=30, n_frames=6)
    got = dict(FrameStream(pipe, ex, batch_frames=6, workers=2).run(_frames([(20, 20)] * 6)))
    assert [ids for ids, _ in ex.calls] == [[0, 1, 2, 3, 4, 5]]
    assert [n for n, _ in pipe.calls] == [30, 30, 15]            # [0,1] [2,3,4] [5]
    assert sorted(got) == list(range(6))
    for i, r in got.items():
        assert r["n_descriptors"] == counts[i] and (r["match_t"] == i).all()
        assert bool(r["final_pose"]) == bool(counts[i])


def test_device_path_errors():
    with pytest.raises(ValueError, match="max_queries"):
        list(FrameStream(_EchoPipeline(10, 2), _FakeBatchSift([5, 11]), batch_frames=2, workers=1)
             .run(_frames([(8, 8)] * 2)))

    class Sharded(_EchoPipeline):
        world, shard_mode = 2, "db"

    with pytest.raises(ValueError, match="shard='frames'"):
        list(FrameStream(Sharded(10, 2), _FakeBatchSift([1]), batch_frames=2, workers=1).run(_frames([(8, 8)])))
    assert list(FrameStream(_EchoPipeline(10, 2), _FakeBatchSift([]), batch_frames=2, workers=1).run([])) == []
