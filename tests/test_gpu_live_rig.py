"""LiveDetector over a camera rig (frames of different sizes in one CUDA-graph replay) against the eager path: every
replayed frame against DetectionPipeline.detect on the same SIFT rows with that frame's (w, h) and against
GpuSift.extract of the frame alone; host, CUDA and pitched inputs; sharing a pipeline and a GpuSift with a one-size
detector and with extract_mixed; the errors raised after the replay; and the flattened mixed-size schedule
(GpuSift.enqueue_mixed / extract_mixed) against single-frame pyramids and keypoints."""
import ctypes as C

import numpy as np
import pytest
import torch

import imaging
from test_gpu_live import _assert_same, _eager, _sequence
from test_gpu_sift import _database
from test_gpu_sift_mixed import _frame, _levels

pytestmark = pytest.mark.gpu

R = 3000
# four sizes, one portrait, 320x240 with fewer octaves than 1200x900 (8 against 10, the doubled image's octave -1
# included)
RIG = [(640, 480), (1200, 900), (480, 640), (320, 240)]
FIELDS = ("xy", "size", "angle", "response", "octave")
FEATURES = ("xy", "angle", "octave")          # the keypoint fields of a FrameFeatures


@pytest.fixture(scope="module")
def database():
    db, objs = _database(np.random.default_rng(21))
    return db, objs


def _pipelines(db, spaces, frames=len(RIG)):
    from sod_b200.pipeline import DetectionPipeline
    mdb = db.to_model_database()
    if spaces == "objects":
        mdb.object_of_image = np.arange(len(mdb.img_centroid), dtype=np.int32)
    mk = lambda: DetectionPipeline(mdb, max_queries=frames * R,  # noqa: E731
                                   frame_wh=np.zeros((frames, 2), np.int32))
    return mk(), mk()


def _eager_rig(ref, feats: list, sizes) -> list[dict]:
    """DetectionPipeline.detect + final_poses on the frames' SIFT rows, frame k with its own (w, h)."""
    if sum(len(f) for f in feats) == 0:
        return _eager(ref, feats, sizes[0])
    ref.scene.frame_wh[:len(sizes)].copy_(torch.tensor(np.asarray(sizes, np.int32)))
    cat = lambda name: np.concatenate([getattr(f, name) for f in feats])  # noqa: E731
    counts = [len(f) for f in feats]
    frame = np.repeat(np.arange(len(feats)), counts).astype(np.int32)
    out = ref.detect(cat("des"), cat("xy").reshape(-1, 2), cat("angle"), cat("octave"), frame)
    poses = ref.final_poses(out)
    starts = np.cumsum([0] + counts)
    gpf = ref.spaces_per_frame
    res = []
    for k in range(len(feats)):
        ok = out["ok"][starts[k]:starts[k + 1]].astype(bool)
        mine = out["valid_group"] // gpf == k
        res.append(dict(match_q=np.nonzero(ok)[0], match_t=out["idx"][starts[k]:starts[k + 1], 0][ok],
                        group=out["valid_group"][mine] % gpf, code=out["valid_code"][mine], votes=out["votes"][mine],
                        live=(out["status"][mine] & 1).astype(bool), params=out["params"][mine],
                        final_pose=poses.get(k, [])))
    return res


def _rows_equal_extract(feats, one, tag):
    """A frame's rows against GpuSift.extract of the frame alone: keypoints bit-identical, descriptors within 1;
    returns (equal bytes, bytes)."""
    for f in FEATURES:
        a = np.ascontiguousarray(getattr(feats, f)).reshape(-1)
        b = np.ascontiguousarray(one[f]).reshape(-1)
        assert a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8)), (tag, f)
    d = np.abs(feats.des.astype(np.int32) - one["des"].astype(np.int32))
    assert d.size == 0 or d.max() <= 1, tag
    return int((d == 0).sum()), d.size


def _check_call(got: list, ref, frames, sizes, check_sift, tag):
    """One rig call: each frame's rows against single-frame extraction, every frame against the eager path."""
    equal = total = 0
    for k, (r, fr) in enumerate(zip(got, frames)):
        assert r["features"].size == tuple(sizes[k]), (tag, k)
        e, t = _rows_equal_extract(r["features"], check_sift.extract(fr), (tag, k))
        equal, total = equal + e, total + t
        assert r["n_descriptors"] == len(r["features"])
    want = _eager_rig(ref, [r["features"] for r in got], sizes)
    for k in range(len(got)):
        _assert_same(got[k], want[k], (tag, k))
    return equal, total


@pytest.mark.parametrize("spaces", ["objects", "single"])
def test_every_rig_replay_equals_the_eager_path(database, spaces):
    from sod_b200.live import LiveDetector
    from sod_b200.sift import GpuSift
    db, objs = database
    pipe, ref = _pipelines(db, spaces)
    rng = np.random.default_rng(31)
    sift, check_sift = GpuSift(max_keypoints=R), GpuSift(max_keypoints=R)
    seqs = [_sequence(rng, objs, w, h) for w, h in RIG]         # each slot: flat frames, rich -> sparse
    rig = LiveDetector(pipe, sift, RIG, features=True)
    assert rig.mixed
    equal = total = found = 0
    counts = []
    for i in range(12):
        frames = [seq[(i + k) % 12] for k, seq in enumerate(seqs)]
        got = rig.detect(frames)
        e, t = _check_call(got, ref, frames, RIG, check_sift, (spaces, i))
        equal, total = equal + e, total + t
        counts.append([len(r["features"]) for r in got])
        found += sum(len(r["final_pose"]) for r in got)
    assert len(rig._graphs) == 1
    flat = np.array(counts).reshape(-1)
    assert 0 in flat and R in flat, counts
    assert found > 0
    print(f"{spaces}: keypoints {counts}, poses {found}, descriptor bytes equal {equal}/{total}")
    assert equal >= 0.99999 * total


def test_rig_inputs_and_sharing(database):
    from sod_b200.live import LiveDetector
    from sod_b200.sift import GpuSift
    db, objs = database
    pipe, ref = _pipelines(db, "objects")
    rng = np.random.default_rng(32)
    sift, check_sift = GpuSift(max_keypoints=R), GpuSift(max_keypoints=R)
    seqs = [_sequence(rng, objs, w, h, n=4) for w, h in RIG]
    rig = LiveDetector(pipe, sift, RIG, features=True)
    one = LiveDetector(pipe, sift, (640, 480), features=True)
    # a one-size detector and the rig share the pipeline and the GpuSift, called alternately
    for i in range(4):
        frames = [seq[i] for seq in seqs]
        _check_call(rig.detect(frames), ref, frames, RIG, check_sift, ("rig", i))
        (got,) = one.detect([seqs[0][(i + 1) % 4]])
        (want,) = _eager(ref, [got["features"]], (640, 480))
        _assert_same(got, want, ("one", i))
    # CUDA inputs, one of them pitched and one transposed (rows not unit-stride): a second graph, same rows
    frames = [seq[1] for seq in seqs]
    host = rig.detect(frames)
    dev = [torch.from_numpy(f).cuda() for f in frames]
    padded = torch.zeros((900 + 3, 1200 + 40), dtype=torch.uint8, device="cuda")
    padded[:900, :1200] = dev[1]
    dev[1] = padded[:900, :1200]
    dev[2] = torch.from_numpy(np.ascontiguousarray(frames[2].T)).cuda().t()
    cuda = rig.detect(dev)
    assert len(rig._graphs) == 2
    for k in range(len(RIG)):
        for f in FEATURES:
            np.testing.assert_array_equal(getattr(cuda[k]["features"], f), getattr(host[k]["features"], f))
    for k, r in enumerate(_eager_rig(ref, [r["features"] for r in cuda], RIG)):
        _assert_same(cuda[k], r, ("cuda", k))
    # an extract_mixed of a larger batch on the same GpuSift (its slot buffers grow) changes nothing for the rig
    before = rig.detect(frames)
    big = sift.extract_mixed([_frame(rng, 1200, 900) for _ in range(6)] + [_frame(rng, 64, 48)])
    assert big.rows > 0 and sift._mixed[0].frames == 7
    after = rig.detect(frames)
    for k in range(len(RIG)):
        for f in FEATURES:
            np.testing.assert_array_equal(getattr(after[k]["features"], f), getattr(before[k]["features"], f))
    _check_call(after, ref, frames, RIG, check_sift, "after extract_mixed")
    # a list of equal sizes is the one-size path
    two = LiveDetector(pipe, sift, [(640, 480)] * 2, features=True)
    assert not two.mixed and two.frames == 2 and two.frame_size == (640, 480)
    pair = two.detect([seqs[0][0], seqs[0][1]])
    for k, r in enumerate(_eager(ref, [r["features"] for r in pair], (640, 480))):
        _assert_same(pair[k], r, ("equal sizes", k))


def test_rig_errors_after_the_replay(database):
    from sod_b200._capi import SodError
    from sod_b200.live import LiveDetector
    from sod_b200.sift import GpuSift
    db, objs = database
    rng = np.random.default_rng(33)
    flats = [np.full((h, w), 128, np.uint8) for w, h in RIG]
    rich = imaging.textured(rng, 1200, 900, shapes=200)
    pipe, _ = _pipelines(db, "objects")
    small = LiveDetector(pipe, GpuSift(max_keypoints=R, capacity=200), RIG)
    with pytest.raises(SodError, match=r"sod_sift_extract_mixed: more than capacity=200 keypoints in frame 1 "
                                       r"\(1200x900\)"):
        small.detect([flats[0], rich, flats[2], flats[3]])
    assert [r["n_descriptors"] for r in small.detect(flats)] == [0, 0, 0, 0]
    frame, _ = imaging.place(rng, imaging.textured(rng, 640, 480, shapes=200), objs[0], 0.6, 10.0, 320.0, 240.0)
    frames = [frame] + flats[1:]
    pipe2, _ = _pipelines(db, "objects")
    pipe2._hough[0].cap_bins = 1
    with pytest.raises(RuntimeError, match="output capacity exceeded"):
        LiveDetector(pipe2, GpuSift(max_keypoints=R), RIG).detect(frames)
    pipe3, _ = _pipelines(db, "objects")
    full = LiveDetector(pipe3, GpuSift(max_keypoints=R), RIG).detect(frames)[0]
    assert len(full["valid_code"]) > 1
    with pytest.raises(RuntimeError, match="max_bins"):
        LiveDetector(pipe3, GpuSift(max_keypoints=R), RIG, max_bins=1).detect(frames)


# ------------------------------------------------------------------------------------- the flattened schedule
# 6 % of the largest frame's grid is real: every pyramid launch is flattened
SKEWED = [(2000, 1500)] + [(64, 48)] * 15
# the small frames have octaves without an interior (47x33: octave 3 is 11x8) or lack the late octaves altogether;
# about a quarter of the largest frame's grid is real, so most launches keep that grid and a few late ones are
# flattened: one pass with both forms
NO_INTERIOR = [(47, 33), (1200, 900), (23, 41), (30, 17), (641, 479)]


@pytest.mark.parametrize("sizes", [SKEWED, NO_INTERIOR], ids=["skewed", "no_interior"])
def test_flat_schedule_pyramids_and_keypoints_are_single_frame_ones(sizes):
    from sod_b200._capi import lib
    from sod_b200.sift import GpuSift
    rng = np.random.default_rng(34)
    frames = [_frame(rng, w, h) for w, h in sizes]
    gpu = GpuSift()
    dev = [torch.from_numpy(f).cuda() for f in frames]
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        t = gpu.enqueue_mixed(dev)
    st.synchronize()
    n, F = len(sizes), gpu._mixed[0].frames
    fl = t["flags"].cpu().numpy()
    count, offset = fl[:n], fl[F:F + n]
    assert not fl[2 * F:2 * F + n].any() and not fl[3 * F]
    ws = gpu._mixed[0].ws
    levels, base = [], 0
    for (w, h) in sizes:                       # frame k's pyramid after the single-frame pyramids of 0..k-1
        lv = {}
        for o in _levels(w, h):
            for lvl in range(6):
                wh = (C.c_int32 * 2)()
                off = base + int(lib.sod_sift_level_offset(w, h, o, lvl, C.cast(wh, C.c_void_p)))
                lv[o, lvl] = ws[off:off + 4 * wh[0] * wh[1]].view(torch.float32).reshape(wh[1], wh[0]).cpu().numpy()
        levels.append(lv)
        base += int(lib.sod_sift_batch_workspace_bytes(w, h, 1, 0))
    rows = {name: t[name][:int(count.sum())].cpu().numpy() for name in FIELDS}
    single = GpuSift()
    for k, (f, (w, h)) in enumerate(zip(frames, sizes)):
        one = single.extract(f)
        for (o, lvl), a in levels[k].items():
            b = single.gaussian_level((w, h), o, lvl)
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), (k, o, lvl)
        assert count[k] == len(one["xy"]), k
        for name in FIELDS:
            got = rows[name][offset[k]:offset[k] + count[k]]
            assert np.array_equal(np.ascontiguousarray(got).view(np.uint8),
                                  np.ascontiguousarray(one[name]).view(np.uint8)), (k, name)
    # extract_mixed (the same pass, then its wait and checks) agrees with the enqueued pass
    batch = gpu.extract_mixed(frames)
    np.testing.assert_array_equal(batch.count, count)
    print(f"{len(sizes)} frames: keypoints {count.tolist()}")
