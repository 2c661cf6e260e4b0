"""Mixed-size GPU SIFT (GpuSift.extract_mixed, sod_sift_extract_mixed) against GpuSift.extract of each frame alone,
and GenerateDatabaseInfo.build_database on the GPU against the cv2-built database and through DetectionPipeline."""
import ctypes as C
import os

import cv2
import numpy as np
import pytest
import torch

import imaging
from test_gpu_sift import _pair
from test_gpu_sift_batch import FIELDS, _assert_batch_equals_single, _check_against_main, _scene

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    from sod_b200.sift import GpuSift
    return GpuSift()


def _frame(rng, w, h):
    return imaging.textured(rng, w, h, shapes=200) if w >= 64 and h >= 64 else \
        rng.integers(0, 256, (h, w), dtype=np.uint8)


def _mix(seed, sizes, flat=None):
    rng = np.random.default_rng(seed)
    out = [_frame(rng, w, h) for w, h in sizes]
    if flat is not None:
        out[flat] = np.full(out[flat].shape, 128, np.uint8)
    return out


# octave counts differ (47x33 has 4, 1200x900 has 9), the largest frame is not first, one frame is flat
MIX = [(640, 480), (641, 479), (480, 640), (47, 33), (1200, 900), (640, 480)]


def _check(batch, singles, sizes):
    assert batch.frame_sizes.tolist() == [list(s) for s in sizes]
    for k, s in enumerate(sizes):
        assert batch.arrays(k)["frame_size"] == tuple(s)
    equal, total = _assert_batch_equals_single(batch, singles)
    assert total == 0 or equal >= 0.999 * total
    return equal, total


@pytest.mark.parametrize("sizes,flat", [(MIX, 5), (MIX[:1], None), ([(1500, 1000), (1500, 2000)], None)])
def test_mixed_equals_single_frames(gpu, sizes, flat):
    frames = _mix(51, sizes, flat)
    singles = [gpu.extract(f) for f in frames]
    batch = gpu.extract_mixed(frames)
    equal, total = _check(batch, singles, sizes)
    if flat is not None:
        assert batch.count[flat] == 0
    if len(frames) == 1:
        same = gpu.extract_batch(frames)
        _assert_batch_equals_single(same, singles)
    print(f"mixed {sizes}: {list(batch.count)} keypoints, descriptor bytes equal {equal}/{total}")


def _levels(w, h):
    from sod_b200._capi import lib
    wh = (C.c_int32 * 2)()
    o = -1
    while lib.sod_sift_level_offset(w, h, o, 0, C.cast(wh, C.c_void_p)) >= 0:
        yield o
        o += 1


def test_mixed_pyramid_is_the_single_frame_pyramid(gpu):
    from sod_b200._capi import lib
    sizes = [(641, 479), (47, 33), (480, 640)]
    frames = _mix(52, sizes)
    gpu.extract_mixed(frames)
    ws = gpu._mixed[0].ws
    base, got = 0, []
    for (w, h) in sizes:                       # frame k's pyramid after the single-frame pyramids of 0..k-1
        lv = {}
        for o in _levels(w, h):
            for l in range(6):
                wh = (C.c_int32 * 2)()
                off = base + int(lib.sod_sift_level_offset(w, h, o, l, C.cast(wh, C.c_void_p)))
                lv[o, l] = ws[off:off + 4 * wh[0] * wh[1]].view(torch.float32).reshape(wh[1], wh[0]).cpu().numpy()
        got.append(lv)
        base += int(lib.sod_sift_batch_workspace_bytes(w, h, 1, 0))
    for k, (f, (w, h)) in enumerate(zip(frames, sizes)):
        gpu.extract(f)
        for (o, l), a in got[k].items():
            one = gpu.gaussian_level((w, h), o, l)
            assert np.array_equal(a.view(np.uint32), one.view(np.uint32)), (k, o, l)


def test_max_keypoints_keeps_each_frames_first_n(gpu):
    from sod_b200.sift import GpuSift
    sizes = [(640, 480), (300, 200), (800, 500)]
    frames = _mix(53, sizes, flat=1)
    full = gpu.extract_mixed(frames, slot=1)
    head = GpuSift(max_keypoints=50).extract_mixed(frames)
    assert list(head.count) == [50, 0, 50]
    np.testing.assert_array_equal(head.offset, [0, 50, 50])
    for k in (0, 2):
        a, b = head.arrays(k), full.arrays(k)
        for f in FIELDS:
            np.testing.assert_array_equal(a[f], b[f][:50])


def test_overflow_names_the_frame(gpu):
    from sod_b200._capi import SodError
    from sod_b200.sift import GpuSift
    frames = _mix(54, [(300, 200), (640, 480), (500, 300)])
    frames[0] = np.full((200, 300), 128, np.uint8)
    frames[2] = np.full((300, 500), 30, np.uint8)
    assert len(gpu.extract(frames[1])["xy"]) > 200
    with pytest.raises(SodError, match=r"frame 1 \(640x480\)"):
        GpuSift(capacity=200).extract_mixed(frames)
    assert GpuSift(capacity=200).extract_mixed([frames[0], frames[2]]).rows == 0


def test_cuda_inputs_equal_host_inputs(gpu):
    sizes = [(640, 480), (333, 251), (480, 640)]
    frames = _mix(55, sizes)
    want = [gpu.extract(f) for f in frames]
    dev = [torch.from_numpy(f).cuda() for f in frames]
    padded = torch.zeros((251 + 5, 333 + 60), dtype=torch.uint8, device="cuda")
    padded[:251, :333] = dev[1]
    cols = torch.from_numpy(np.ascontiguousarray(frames[2].T)).cuda().t()    # rows not unit-stride: copied
    for images in (dev, [dev[0], padded[:251, :333], cols], [frames[0], padded[:251, :333], dev[2]]):
        _check(gpu.extract_mixed(images), want, sizes)


def test_new_sizes_do_not_grow_gpu_memory():
    from sod_b200.sift import GpuSift
    g = GpuSift()
    rng = np.random.default_rng(56)
    g.extract_mixed([_frame(rng, 640, 480 + k) for k in range(8)])        # the largest mix of the run
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    for r in range(6):
        sizes = [(int(rng.integers(100, 640)), int(rng.integers(100, 480))) for _ in range(int(rng.integers(1, 9)))]
        b = g.extract_mixed([_frame(rng, w, h) for w, h in sizes])
        assert b.frame_sizes.tolist() == [list(s) for s in sizes]
        torch.cuda.synchronize()
        assert torch.cuda.memory_allocated() == before, r


# ------------------------------------------------------------------------------- the database builder on the GPU
def _training_folder(path, rng):
    """Three training images of different aspect ratios (1500x1000, 1500x750, 1500x1250 after the builder's
    resize), a file that is no image, saved as PNG so that both builders decode the same pixels."""
    for name, (w, h) in (("b_obj.png", (1200, 800)), ("a_obj.png", (1200, 600)), ("c_obj.png", (1200, 1000))):
        img = imaging.textured(rng, w, h, shapes=200)
        cv2.imwrite(os.path.join(path, name), cv2.cvtColor(img, cv2.COLOR_GRAY2BGR))
    with open(os.path.join(path, "readme.txt"), "w") as f:
        f.write("not an image")


def _arrays(row):
    t = row[0]
    return {"xy": np.array([k[0] for k in t], np.float32).reshape(-1, 2),
            "size": np.array([k[1] for k in t], np.float32), "angle": np.array([k[2] for k in t], np.float32),
            "response": np.array([k[3] for k in t], np.float32), "octave": np.array([k[4] for k in t], np.int32)}


def test_build_database_on_the_gpu(tmp_path):
    import GenerateDatabaseInfo as G
    from sod_b200.database import PackedDatabase
    from sod_b200.pipeline import DetectionPipeline
    from sod_b200.sift import GpuSift
    from sod_b200.stream import FrameStream
    rng = np.random.default_rng(57)
    _training_folder(str(tmp_path), rng)
    ref = G.build_database(str(tmp_path), str(tmp_path / "cv2.pkl"))
    gpu = GpuSift()
    got = G.build_database(str(tmp_path), str(tmp_path / "gpu.pkl"), str(tmp_path / "gpu.sodb"), extractor=gpu)
    assert [r[4] for r in got] == [r[4] for r in ref] and len(got) == 3
    assert [r[2] for r in got] == [r[2] for r in ref]
    assert sorted(r[2][1] for r in got) == [750, 1000, 1250]
    equal = total = 0
    paired = np.zeros(4, np.int64)             # cv2 keypoints paired, cv2 keypoints, gpu paired, gpu keypoints
    for g, c in zip(got, ref):
        a, b = _arrays(g), _arrays(c)
        assert g[1].dtype == np.float32 and g[1].shape == (len(g[0]), 128)
        assert all(k[5] == -1 for k in g[0])
        p_ref, p_got = _pair(b, a) >= 0, _pair(a, b) >= 0
        paired += [p_ref.sum(), len(p_ref), p_got.sum(), len(p_got)]
        print(f"{os.path.basename(g[4])} {g[2]}: cv2 {len(c[0])} gpu {len(g[0])}, paired {p_ref.mean():.5f} / "
              f"{p_got.mean():.5f}")
        # the rows are GpuSift.extract of the image the builder prepared
        one = gpu.extract(G._prepare(g[4]))
        for f in FIELDS:
            assert np.array_equal(a[f].view(np.uint8), one[f].view(np.uint8)), f
        d = np.abs(g[1].astype(np.int32) - one["des"].astype(np.int32))
        assert d.max() <= 1
        equal, total = equal + int((d == 0).sum()), total + d.size
    assert equal >= 0.999 * total
    # over the folder, as tests/test_gpu_sift.py pairs them: same octave and layer, |dpt| <= 0.1 px, angle within 1
    print(f"paired over the folder: cv2 {paired[0]}/{paired[1]}, gpu {paired[2]}/{paired[3]}")
    assert paired[0] >= 0.999 * paired[1] and paired[2] >= 0.999 * paired[3]
    # the GPU-built database finds objects placed in scenes
    db = PackedDatabase.open(tmp_path / "gpu.sodb")
    objs = [G._prepare(r[4]) for r in got]
    placements = [[(0, 0.4, 20, 500, 400)], [(1, 0.5, -35, 650, 450)], [], [(2, 0.35, 100, 600, 450)]]
    frames, truth = _scene(rng, objs, db, [(1200, 900)] * 4, placements)
    pipe = DetectionPipeline(db.to_model_database(), max_queries=20000, frame_wh=np.zeros((2, 2), np.int32),
                             per_object_spaces=False)
    results = dict(FrameStream(pipe, extractor=GpuSift(), batch_frames=2, workers=4, features=True).run(frames))
    _check_against_main(db, frames, truth, results)
