"""Batched GPU SIFT (GpuSift.extract_batch, sod_sift_extract_batch) against GpuSift.extract of each frame alone,
and FrameStream's device path end to end against the drop-in Main on the features it extracted."""
import numpy as np
import pytest
import torch

import imaging
from test_gpu_sift import _database, _main_on

pytestmark = pytest.mark.gpu

FIELDS = ("xy", "size", "angle", "response", "octave")


@pytest.fixture(scope="module")
def gpu():
    from sod_b200.sift import GpuSift
    return GpuSift()


def _frames(seed, w, h, n, flat=None):
    rng = np.random.default_rng(seed)
    out = [imaging.textured(rng, w, h, shapes=200) if w >= 64 else rng.integers(0, 256, (h, w), dtype=np.uint8)
           for _ in range(n)]
    if flat is not None:
        out[flat] = np.full((h, w), 128, np.uint8)
    return out


def _assert_batch_equals_single(batch, singles):
    assert len(batch) == len(singles)
    np.testing.assert_array_equal(batch.count, [len(s["xy"]) for s in singles])
    np.testing.assert_array_equal(batch.offset, np.concatenate([[0], np.cumsum(batch.count)[:-1]]))
    frame = batch.frame.cpu().numpy()
    np.testing.assert_array_equal(frame, np.repeat(np.arange(len(singles)), batch.count))
    equal = total = 0
    for k, one in enumerate(singles):
        got = batch.arrays(k)
        for f in FIELDS:                                  # bit-identical, in the same order
            assert got[f].dtype == one[f].dtype and np.array_equal(got[f].view(np.uint8), one[f].view(np.uint8)), (k, f)
        d = np.abs(got["des"].astype(np.int32) - one["des"].astype(np.int32))
        assert d.size == 0 or d.max() <= 1, k           # float atomics: a byte may move by 1 between runs
        equal += int((d == 0).sum())
        total += d.size
    return equal, total


@pytest.mark.parametrize("seed,w,h,n,flat", [(41, 640, 480, 5, 3), (42, 641, 479, 3, None), (43, 47, 33, 2, None),
                                             (44, 1200, 900, 4, None)])
def test_batch_equals_single_frames(gpu, seed, w, h, n, flat):
    frames = _frames(seed, w, h, n, flat)
    singles = [gpu.extract(f) for f in frames]
    batch = gpu.extract_batch(frames)
    equal, total = _assert_batch_equals_single(batch, singles)
    if flat is not None:
        assert batch.count[flat] == 0
    print(f"batch {n} x {w}x{h}: {list(batch.count)} keypoints, descriptor bytes equal {equal}/{total}")
    assert total == 0 or equal >= 0.999 * total


def test_batch_pyramid_is_the_single_frame_pyramid(gpu):
    w, h, n = 641, 479, 3
    frames = _frames(45, w, h, n)
    gpu.extract_batch(frames)
    for k, f in enumerate(frames):
        gpu.extract(f)
        for o in range(-1, 2):
            for lv in range(6):
                one = gpu.gaussian_level((w, h), o, lv)
                got = gpu.gaussian_level((w, h), o, lv, batch=(n, k))
                assert np.array_equal(got.view(np.uint32), one.view(np.uint32)), (k, o, lv)


def test_max_keypoints_keeps_each_frames_first_n(gpu):
    from sod_b200.sift import GpuSift
    frames = _frames(46, 640, 480, 3, flat=1)
    full = gpu.extract_batch(frames)
    head = GpuSift(max_keypoints=50).extract_batch(frames)
    assert list(head.count) == [50, 0, 50]
    np.testing.assert_array_equal(head.offset, [0, 50, 50])
    for k in (0, 2):
        a, b = head.arrays(k), full.arrays(k)
        for f in FIELDS:
            np.testing.assert_array_equal(a[f], b[f][:50])


def test_overflow_names_the_frame(gpu):
    from sod_b200._capi import SodError
    from sod_b200.sift import GpuSift
    frames = _frames(47, 640, 480, 3, flat=0)
    frames[2] = np.full((480, 640), 30, np.uint8)
    n = len(gpu.extract(frames[1])["xy"])
    assert n > 200
    with pytest.raises(SodError, match="frame 1 "):
        GpuSift(capacity=200).extract_batch(frames)
    assert GpuSift(capacity=200).extract_batch([frames[0], frames[2]]).rows == 0


def test_cuda_input_equals_host_input(gpu):
    w, h, n = 640, 480, 3
    frames = _frames(48, w, h, n)
    host = gpu.extract_batch(frames)
    want = [host.arrays(k) for k in range(n)]
    stacked = torch.from_numpy(np.stack(frames)).cuda()
    padded = torch.zeros((n, h + 3, w + 40), dtype=torch.uint8, device="cuda")
    padded[:, :h, :w] = stacked
    for images in (stacked, list(stacked.unbind(0)), padded[:, :h, :w]):   # the last one: pitch and stride
        _assert_batch_equals_single(gpu.extract_batch(images), want)
    with pytest.raises(ValueError, match="one size"):
        gpu.extract_batch([stacked[0], stacked[1, :, :-1]])


def _scene(rng, objs, db, sizes, placements):
    frames, truth = [], []
    for (w, h), pl in zip(sizes, placements):
        fr = imaging.textured(rng, w, h, shapes=200)
        t = []
        for (o, s, deg, cx, cy) in pl:
            fr, m = imaging.place(rng, fr, objs[o], s, deg, cx, cy)
            c = db.img_centroid[o]
            t.append((m @ np.array([c[0], c[1], 1.0]), s, deg))
        frames.append(fr)
        truth.append(t)
    return frames, truth


def _check_against_main(db, frames, truth, results):
    kps_db = db.keypoints()
    db_index = {id(k): i for i, k in enumerate(kps_db)}
    assert sorted(results) == list(range(len(frames)))
    for i in range(len(frames)):
        r = results[i]
        feats = r["features"]
        assert feats.size == (frames[i].shape[1], frames[i].shape[0])
        assert r["n_descriptors"] == len(feats)
        m = _main_on(db, feats, kps_db)
        assert [t[1].class_id for t in m.matching_keypoints] == r["match_q"].tolist()
        assert [db_index[id(t[0])] for t in m.matching_keypoints] == r["match_t"].tolist()
        assert int(r["live"].sum()) == len(m.valid_bins)
        got = np.array([[c[0], c[1], o, s, sh[0], sh[1]] for (c, o, s, sh) in r["final_pose"]]).reshape(-1, 6)
        want = np.array([[c[0], c[1], o, s, sh[0], sh[1]] for (c, o, s, sh) in m.final_pose]).reshape(-1, 6)
        assert got.shape == want.shape
        np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-9)
        for (xy, s, deg) in truth[i]:
            d = np.hypot(got[:, 0] - xy[0], got[:, 1] - xy[1]) if len(got) else np.array([np.inf])
            j = int(d.argmin())
            assert d[j] < 40, (i, xy, got[:, :2])
            assert 0.5 * s <= got[j, 3] <= 2.0 * s
            err = (np.degrees(got[j, 2]) - deg + 180.0) % 360.0 - 180.0
            assert abs(err) < 3.0, (i, deg, np.degrees(got[j, 2]))
        if not truth[i]:
            assert len(got) == 0


def test_stream_device_path_finds_the_objects_of_a_cv2_database():
    """The scenario of test_stream_with_gpu_sift_finds_the_objects_of_a_cv2_database through the device path."""
    from sod_b200.pipeline import DetectionPipeline
    from sod_b200.sift import GpuSift
    from sod_b200.stream import FrameStream
    rng = np.random.default_rng(7)
    db, objs = _database(rng)
    placements = [[(0, 0.8, 20, 500, 400)], [(1, 1.0, -35, 700, 450), (2, 0.6, 90, 250, 250)], [],
                  [(2, 1.2, 5, 600, 500)], [(0, 0.7, 170, 800, 300)]]
    frames, truth = _scene(rng, objs, db, [(1200, 900)] * 5, placements)
    pipe = DetectionPipeline(db.to_model_database(), max_queries=20000, frame_wh=np.zeros((2, 2), np.int32),
                             per_object_spaces=False)
    results = dict(FrameStream(pipe, extractor=GpuSift(), batch_frames=2, workers=4, features=True).run(frames))
    _check_against_main(db, frames, truth, results)


def test_stream_device_path_with_two_sizes_and_passes_split_at_max_queries():
    from sod_b200.pipeline import DetectionPipeline
    from sod_b200.sift import GpuSift
    from sod_b200.stream import FrameStream
    rng = np.random.default_rng(8)
    db, objs = _database(rng)
    A, B = (1200, 900), (800, 600)
    sizes = [A, B, A, A, A, B, B]
    placements = [[(0, 0.8, 20, 500, 400)], [(1, 0.7, 30, 400, 300)], [(2, 1.0, -10, 600, 450)], [],
                  [(1, 0.9, 60, 700, 400)], [], [(0, 0.6, -80, 350, 280)]]
    frames, truth = _scene(rng, objs, db, sizes, placements)
    frames[4] = torch.from_numpy(frames[4]).cuda()            # a frame already on the device
    pipe = DetectionPipeline(db.to_model_database(), max_queries=12000, frame_wh=np.zeros((4, 2), np.int32),
                             per_object_spaces=False)
    gpu = GpuSift()
    stream = FrameStream(pipe, extractor=gpu, batch_frames=4, workers=3, features=True)
    results = dict(stream.run(frames))
    # the run of three 1200x900 frames (about 5,000 keypoints each) is one SIFT batch and two detection passes
    assert sorted(gpu._batch_buffers) == [(800, 600, 1), (800, 600, 2), (1200, 900, 1), (1200, 900, 3)]
    frames[4] = frames[4].cpu().numpy()
    _check_against_main(db, frames, truth, results)
