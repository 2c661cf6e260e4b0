"""CPU-side checks of LiveDetector over a camera rig (a list of frame sizes): every refusal happens in the constructor,
before any CUDA call, with a stand-in pipeline and GPU SIFT; frames of the wrong size or count are refused naming
the frame and its size; a list of equal sizes is the one-size detector."""
import numpy as np
import pytest

from sod_b200.live import LiveDetector
from sod_b200.stream import FrameStream
from test_live_args import _Sift
from test_stream import _EchoPipeline

RIG = [(64, 48), (32, 40), (48, 64)]


def test_rig_refusals():
    pipe = _EchoPipeline(max_queries=1000, n_frames=3)
    with pytest.raises(ValueError, match="max_keypoints"):
        LiveDetector(pipe, _Sift(None), RIG)
    with pytest.raises(ValueError, match="max_queries 1000"):
        LiveDetector(pipe, _Sift(334), RIG)
    rig = LiveDetector(pipe, _Sift(333), RIG)
    assert rig.frames == 3 and rig.mixed and rig.frame_size is None
    assert rig.frame_sizes.tolist() == [list(s) for s in RIG]
    LiveDetector(pipe, _Sift(5000, capacity=333), RIG)                   # rows bounded by the SIFT capacity
    LiveDetector(pipe, _Sift(100), RIG, frames=3)
    with pytest.raises(ValueError, match="frames=2, but frame_size lists 3 sizes"):
        LiveDetector(pipe, _Sift(100), RIG, frames=2)
    with pytest.raises(ValueError, match="one row per frame"):
        LiveDetector(pipe, _Sift(100), RIG + [(16, 16)])
    with pytest.raises(ValueError, match="out of range"):
        LiveDetector(pipe, _Sift(100), [(64, 48), (0, 48)])
    # sizes or keypoint slots the mixed-size SIFT pass refuses: refused here, not on the first call
    with pytest.raises(ValueError, match="sod_sift: 2 frames of sizes \\[\\[64, 48\\], \\[32769, 48\\]\\]"):
        LiveDetector(pipe, _Sift(100), [(64, 48), (32769, 48)])
    with pytest.raises(ValueError, match="with capacity 16777216 out of range"):
        LiveDetector(_EchoPipeline(max_queries=1000, n_frames=3), _Sift(100, capacity=1 << 24), RIG)
    with pytest.raises(ValueError, match="expected \\(width, height\\) or a list"):
        LiveDetector(pipe, _Sift(100), [(64, 48, 1)])
    with pytest.raises(ValueError, match="expected \\(width, height\\) or a list"):
        LiveDetector(pipe, _Sift(100), [])
    big = _EchoPipeline(max_queries=10000, n_frames=65)
    sizes = [(16 + k, 16) for k in range(65)]
    with pytest.raises(ValueError, match="a rig of 65 frames of different sizes; at most 64"):
        LiveDetector(big, _Sift(10), sizes)
    assert LiveDetector(big, _Sift(10), sizes[:64]).frames == 64

    class Float(_EchoPipeline):
        float_path = True

    with pytest.raises(ValueError, match="bf16"):
        LiveDetector(Float(1000, 3), _Sift(100), RIG)


def test_equal_sizes_take_the_one_size_path():
    pipe = _EchoPipeline(max_queries=1000, n_frames=3)
    live = LiveDetector(pipe, _Sift(100), [(64, 48)] * 3)
    assert not live.mixed and live.frame_size == (64, 48) and live.frames == 3 and live.frame_sizes is None
    one = LiveDetector(pipe, _Sift(100), (64, 48))
    assert not one.mixed and one.frames == 1 and one.frame_size == (64, 48)
    assert LiveDetector(pipe, _Sift(100), [(64, 48)]).frames == 1
    with pytest.raises(ValueError, match="frames=2, but frame_size lists 3 sizes"):
        LiveDetector(pipe, _Sift(100), [(64, 48)] * 3, frames=2)


def test_rig_refuses_frames_of_another_size_or_count():
    rig = LiveDetector(_EchoPipeline(max_queries=1000, n_frames=3), _Sift(100), RIG)
    good = [np.zeros((h, w), np.uint8) for w, h in RIG]
    with pytest.raises(ValueError, match="frame 1: expected a 32x40"):
        rig.detect([good[0], np.zeros((48, 64), np.uint8), good[2]])
    with pytest.raises(ValueError, match="frame 2: expected a 48x64"):
        rig.detect(good[:2] + [np.zeros((48, 64, 3), np.uint8)])          # BGR, but transposed
    with pytest.raises(ValueError, match="expected an 8-bit gray or BGR image, got float32"):
        rig.detect([np.zeros((48, 64), np.float32)] + good[1:])
    with pytest.raises(ValueError, match="3 frames per call, got 2"):
        rig.detect(good[:2])
    with pytest.raises(ValueError, match="3 frames per call, got 4"):
        rig.detect(good + good[:1])


def test_rig_sharded_error_wording_is_shared_with_frame_stream():
    class Sharded(_EchoPipeline):
        world, shard_mode = 2, "db"

    class _BatchSift:
        def extract_batch(self, images, slot=0):
            raise AssertionError("not reached")

        prepare = staticmethod(lambda im: im)

    with pytest.raises(ValueError) as stream_err:
        list(FrameStream(Sharded(10, 2), _BatchSift(), batch_frames=2, workers=1).run([np.zeros((8, 8), np.uint8)]))
    with pytest.raises(ValueError) as live_err:
        LiveDetector(Sharded(1000, 3), _Sift(5), RIG)
    assert str(live_err.value) == str(stream_err.value).replace("FrameStream's device path", "LiveDetector")

    class Frames(_EchoPipeline):
        world, shard_mode = 2, "frames"

    assert LiveDetector(Frames(1000, 3), _Sift(100), RIG).mixed


def test_enqueue_mixed_refuses_host_frames_before_any_cuda_call():
    from sod_b200.sift import GpuSift
    g = GpuSift(max_keypoints=10)
    with pytest.raises(ValueError, match="frame 0: expected a CUDA u8 \\[H, W\\] tensor, got ndarray"):
        g.enqueue_mixed([np.zeros((8, 8), np.uint8)] * 2)
    with pytest.raises(ValueError, match="slot must be 0 or 1"):
        g.enqueue_mixed([], slot=2)
