"""CPU-side checks of the live path: argument errors of sod_compact_matches_dev before any CUDA call, LiveDetector's
refusals with a stand-in pipeline and GPU SIFT, and the per-frame split helper against FrameStream's results."""
import numpy as np
import pytest
import torch

from sod_b200.live import LiveDetector
from sod_b200.stream import FrameStream, split_frame
from test_stream import _EchoPipeline, _frame


def test_compact_matches_dev_rejects_bad_arguments_without_gpu():
    from sod_b200._capi import lib
    fake = 1 << 20                         # never dereferenced: validation fails first
    f = lib.sod_compact_matches_dev
    names = ("idx", "pass_", "cap", "n_dev", "lo", "hi", "mq", "mt", "n_out", "scratch", "stream")
    ok = dict(zip(names, (fake, fake, 100, fake, 0, 2 ** 31 - 1, fake, fake, fake, fake, None)))

    def err(**kw):
        a = dict(ok, **kw)
        assert f(*(a[n] for n in names)) == -1
        return lib.sod_last_error()

    assert b"n_query_cap < 0" in err(cap=-1)
    for name in ("idx", "pass_", "n_dev", "mq", "mt", "n_out", "scratch"):
        assert b"null pointer" in err(**{name: None}), name
        assert b"null pointer" in err(cap=0, **{name: None}), name       # checked before n_out is zeroed
    assert lib.sod_compact_scratch_bytes(100) == lib.sod_compact_scratch_bytes(1) == 16


class _Sift:
    def __init__(self, max_keypoints, capacity=1 << 16):
        self.max_keypoints, self.capacity = max_keypoints, capacity


def test_live_detector_refusals():
    pipe = _EchoPipeline(max_queries=1000, n_frames=2)
    with pytest.raises(ValueError, match="max_keypoints"):
        LiveDetector(pipe, _Sift(None), (64, 48))
    with pytest.raises(ValueError, match="max_queries 1000"):
        LiveDetector(pipe, _Sift(501), (64, 48), frames=2)
    LiveDetector(pipe, _Sift(500), (64, 48), frames=2)
    LiveDetector(pipe, _Sift(5000, capacity=500), (64, 48), frames=2)      # rows bounded by the SIFT capacity
    with pytest.raises(ValueError, match="one row per frame"):
        LiveDetector(pipe, _Sift(100), (64, 48), frames=3)
    with pytest.raises(ValueError, match="frames must be"):
        LiveDetector(pipe, _Sift(100), (64, 48), frames=0)

    class Sharded(_EchoPipeline):
        world, shard_mode = 2, "db"

    with pytest.raises(ValueError, match="LiveDetector needs the whole batch on one rank.*shard='frames'"):
        LiveDetector(Sharded(1000, 2), _Sift(100), (64, 48))

    class Frames(_EchoPipeline):
        world, shard_mode = 2, "frames"

    LiveDetector(Frames(1000, 2), _Sift(100), (64, 48))

    class Float(_EchoPipeline):
        float_path = True

    with pytest.raises(ValueError, match="bf16"):
        LiveDetector(Float(1000, 2), _Sift(100), (64, 48))


def test_live_detector_refuses_frames_of_another_size_or_count():
    live = LiveDetector(_EchoPipeline(max_queries=1000, n_frames=2), _Sift(100), (64, 48), frames=2)
    good = np.zeros((48, 64), np.uint8)
    with pytest.raises(ValueError, match="frame 1: expected a 64x48"):
        live.detect([good, np.zeros((48, 65), np.uint8)])
    with pytest.raises(ValueError, match="frame 0: expected a 64x48"):
        live.detect([np.zeros((64, 48, 3), np.uint8), good])           # BGR, but transposed
    with pytest.raises(ValueError, match="2 frames per call, got 1"):
        live.detect([good])


def test_sharded_error_wording_is_shared_with_frame_stream():
    class Sharded(_EchoPipeline):
        world, shard_mode = 2, "db"

    class _BatchSift:
        def extract_batch(self, images, slot=0):
            raise AssertionError("not reached")

        prepare = staticmethod(lambda im: im)

    with pytest.raises(ValueError) as stream_err:
        list(FrameStream(Sharded(10, 2), _BatchSift(), batch_frames=2, workers=1).run([np.zeros((8, 8), np.uint8)]))
    with pytest.raises(ValueError) as live_err:
        LiveDetector(Sharded(10, 2), _Sift(5), (8, 8))
    assert str(stream_err.value).startswith("FrameStream's device path needs the whole batch on one rank: ")
    assert str(live_err.value) == str(stream_err.value).replace("FrameStream's device path", "LiveDetector")


@pytest.mark.parametrize("features", [False, True])
def test_split_helper_gives_frame_stream_results(features):
    """FrameStream's per-frame results are split_frame of its fetched batch: the stand-in's batch results are
    rebuilt here by hand and split with the helper."""
    counts = [7, 0, 30, 12, 0]
    feats = [_frame(i, n) for i, n in enumerate(counts)]
    pipe = _EchoPipeline(max_queries=100, n_frames=5)
    got = list(FrameStream(pipe, lambda f: f, batch_frames=5, workers=2, features=features).run(feats))
    assert len(pipe.calls) == 1
    des = np.concatenate([f.des for f in feats])
    frame = np.repeat(np.arange(len(counts)), counts).astype(np.int32)
    out = pipe.fetch(dict(des=torch.from_numpy(des), frame=torch.from_numpy(frame)))
    poses = pipe.final_poses(out)
    starts = np.cumsum([0] + counts)
    for k, (i, r) in enumerate(got):
        assert i == k
        want = split_frame(out, poses, 1, k, starts[k], starts[k + 1], **({"features": feats[k]} if features else {}))
        assert sorted(r) == sorted(want)
        for key, v in want.items():
            if isinstance(v, np.ndarray):
                assert v.dtype == r[key].dtype
                np.testing.assert_array_equal(r[key], v)
            else:
                assert r[key] == v if key != "features" else r[key] is v
