"""LiveDetector (one CUDA-graph replay per call) against the eager path: sod_compact_matches_dev against
sod_compact_matches, every replayed frame against DetectionPipeline.detect on the same SIFT rows and against
GpuSift.extract_batch of the frame, batches, graph reuse and the errors raised after the replay."""
import numpy as np
import pytest
import torch

import imaging
from test_gpu_sift import _database

pytestmark = pytest.mark.gpu

R = 3000                      # max_keypoints: a textured 1200x900 frame has more, a 640x480 one about as many
SIZES = ((640, 480), (1200, 900))
FIELDS = ("xy", "angle", "octave")


# ------------------------------------------------------------------------------------------------ compaction
def test_compact_matches_dev_equals_host_count_on_the_first_k_rows():
    from sod_b200 import engine as E
    rng = np.random.default_rng(3)
    cap = 5000
    idx = torch.from_numpy(rng.integers(-1, 1 << 20, (cap, 2), dtype=np.int32)).cuda()
    ok = torch.from_numpy(rng.integers(0, 2, cap, dtype=np.uint8) * rng.integers(1, 256, cap, dtype=np.uint8)).cuda()
    for k in (0, 1, cap - 1, cap):
        for lo, hi in ((0, 2 ** 31 - 1), (1 << 18, 3 << 18)):
            n_dev = torch.tensor([k], dtype=torch.int32, device="cuda")
            mq, mt, n = E.compact_matches(idx, ok, lo, hi, n_dev=n_dev)
            wq, wt, wn = E.compact_matches(idx[:k].contiguous(), ok[:k].contiguous(), lo, hi)
            m = int(wn)
            assert int(n) == m, (k, lo)
            assert torch.equal(mq[:m], wq[:m]) and torch.equal(mt[:m], wt[:m]), (k, lo)
    # an empty capacity zeroes the count
    from sod_b200._capi import check, lib
    out = torch.full((1,), 7, dtype=torch.int32, device="cuda")
    one = torch.zeros(1, dtype=torch.int32, device="cuda")
    scratch = torch.empty(int(lib.sod_compact_scratch_bytes(0)), dtype=torch.uint8, device="cuda")
    check(lib.sod_compact_matches_dev(E._ptr(idx), E._ptr(ok), 0, E._ptr(one), 0, 2 ** 31 - 1, E._ptr(one),
                                      E._ptr(one), E._ptr(out), E._ptr(scratch), E._stream()), "compact")
    assert int(out) == 0


# ------------------------------------------------------------------------------------------------ scenes
@pytest.fixture(scope="module")
def database():
    rng = np.random.default_rng(21)
    db, objs = _database(rng)
    return db, objs


def _sequence(rng, objs, w, h, n=12):
    """n frames of one size: textured scenes with planted objects, a flat frame (no keypoints), a sparse frame
    (one object on a flat background) right after a keypoint-rich one, so stale rows lie past the count."""
    s = w / 1200.0
    frames = []
    for i in range(n):
        kind = i % 4
        if kind == 2:
            fr = np.full((h, w), 128, np.uint8)
        else:
            fr = np.full((h, w), 128, np.uint8) if kind == 3 else imaging.textured(rng, w, h, shapes=200)
            for j in range(1 if kind == 3 else 1 + i % 2):
                o = int(rng.integers(0, len(objs)))
                fr, _ = imaging.place(rng, fr, objs[o], s * float(rng.uniform(0.6, 1.1)), float(rng.uniform(-90, 90)),
                                      w * float(rng.uniform(0.3, 0.7)), h * float(rng.uniform(0.3, 0.7)))
        frames.append(fr)
    frames[2], frames[3] = frames[3], frames[2]        # rich (1), sparse (2), flat (3)
    return frames


def _pipelines(db, spaces):
    from sod_b200.pipeline import DetectionPipeline
    mdb = db.to_model_database()
    if spaces == "objects":
        mdb.object_of_image = np.arange(len(mdb.img_centroid), dtype=np.int32)
    mk = lambda: DetectionPipeline(mdb, max_queries=2 * R, frame_wh=np.zeros((2, 2), np.int32))  # noqa: E731
    return mk(), mk()


def _eager(ref, feats: list, size) -> list[dict]:
    """DetectionPipeline.detect + final_poses on the given SIFT rows, split per frame here."""
    ref.scene.frame_wh[:, 0].fill_(size[0])
    ref.scene.frame_wh[:, 1].fill_(size[1])
    cat = lambda name: np.concatenate([getattr(f, name) for f in feats])  # noqa: E731
    counts = [len(f) for f in feats]
    if sum(counts) == 0:                               # nothing to match: DetectionPipeline is not called
        z = np.zeros(0, np.int32)
        return [dict(match_q=z, match_t=z, group=z, code=z, votes=z, live=np.zeros(0, bool),
                     params=np.zeros((0, 6)), final_pose=[]) for _ in feats]
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


def _assert_same(got: dict, want: dict, tag):
    np.testing.assert_array_equal(got["match_q"], want["match_q"], err_msg=str(tag))
    np.testing.assert_array_equal(got["match_t"], want["match_t"], err_msg=str(tag))
    og, ow = np.lexsort((got["valid_code"], got["valid_group"])), np.lexsort((want["code"], want["group"]))
    np.testing.assert_array_equal(got["valid_group"][og], want["group"][ow], err_msg=str(tag))
    np.testing.assert_array_equal(got["valid_code"][og], want["code"][ow], err_msg=str(tag))
    np.testing.assert_array_equal(got["votes"][og], want["votes"][ow], err_msg=str(tag))
    np.testing.assert_array_equal(got["live"][og], want["live"][ow], err_msg=str(tag))
    assert np.array_equal(got["params"][og].view(np.uint64), want["params"][ow].view(np.uint64)), tag
    pose = lambda ps: np.array([[c[0], c[1], o, s, sh[0], sh[1]] for (c, o, s, sh) in ps]).reshape(-1, 6)  # noqa
    np.testing.assert_array_equal(pose(got["final_pose"]), pose(want["final_pose"]), err_msg=str(tag))


def _assert_rows_equal_extract_batch(feats, one, tag):
    """The live SIFT rows against GpuSift.extract_batch of the frame: keypoints bit-identical, descriptors
    within 1; returns (equal bytes, bytes)."""
    for f in FIELDS:
        a = np.ascontiguousarray(getattr(feats, f)).reshape(-1)
        b = np.ascontiguousarray(one[f]).reshape(-1)
        assert a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8)), (tag, f)
    d = np.abs(feats.des.astype(np.int32) - one["des"].astype(np.int32))
    assert d.size == 0 or d.max() <= 1, tag
    return int((d == 0).sum()), d.size


@pytest.mark.parametrize("spaces", ["objects", "single"])
def test_every_replay_equals_the_eager_path(database, spaces):
    from sod_b200.live import LiveDetector
    from sod_b200.sift import GpuSift
    db, objs = database
    pipe, ref = _pipelines(db, spaces)
    rng = np.random.default_rng(5)
    sift, check_sift = GpuSift(max_keypoints=R), GpuSift(max_keypoints=R)
    seqs = {size: _sequence(rng, objs, *size) for size in SIZES}
    lives = {size: LiveDetector(pipe, sift, size, features=True) for size in SIZES}
    equal = total = 0
    counts, found = [], 0
    for i in range(12):                       # the two sizes alternate: two graphs, one pipeline
        for size in SIZES:
            frame = seqs[size][i]
            (got,) = lives[size].detect([frame])
            feats = got["features"]
            counts.append(len(feats))
            one = check_sift.extract_batch([frame]).arrays(0)
            e, t = _assert_rows_equal_extract_batch(feats, one, (size, i))
            equal, total = equal + e, total + t
            (want,) = _eager(ref, [feats], size)
            _assert_same(got, want, (spaces, size, i))
            assert got["n_descriptors"] == len(feats)
            found += len(got["final_pose"])
    assert {size: len(lv._graphs) for size, lv in lives.items()} == {size: 1 for size in SIZES}
    assert 0 in counts and R in counts, counts
    assert found > 0
    print(f"{spaces}: keypoints {counts}, poses {found}, descriptor bytes equal {equal}/{total}")
    assert equal >= 0.999 * total


def test_batch_of_two_gives_each_frame_what_one_gives(database):
    from sod_b200.live import LiveDetector
    from sod_b200.sift import GpuSift
    db, objs = database
    pipe, ref = _pipelines(db, "objects")
    rng = np.random.default_rng(6)
    frames = _sequence(rng, objs, 640, 480, n=8)
    sift = GpuSift(max_keypoints=R)
    one = LiveDetector(pipe, sift, (640, 480), features=True)
    two = LiveDetector(pipe, sift, (640, 480), frames=2, features=True)
    for i in range(0, len(frames), 2):
        pair = two.detect(frames[i:i + 2])
        singles = [one.detect([f])[0] for f in frames[i:i + 2]]
        want = _eager(ref, [r["features"] for r in pair], (640, 480))
        for k in range(2):
            _assert_same(pair[k], want[k], (i, k))
            a, b = pair[k]["features"], singles[k]["features"]
            _assert_rows_equal_extract_batch(a, dict(xy=b.xy, angle=b.angle, octave=b.octave, des=b.des), (i, k))
            if np.array_equal(a.des, b.des):
                np.testing.assert_array_equal(pair[k]["match_q"], singles[k]["match_q"])
                np.testing.assert_array_equal(pair[k]["match_t"], singles[k]["match_t"])
                np.testing.assert_array_equal(np.sort(pair[k]["valid_code"]), np.sort(singles[k]["valid_code"]))


def test_replays_reuse_their_graph_and_memory(database):
    from sod_b200.live import LiveDetector
    from sod_b200.sift import GpuSift
    db, objs = database
    pipe, ref = _pipelines(db, "objects")
    rng = np.random.default_rng(7)
    sift = GpuSift(max_keypoints=R)
    seqs = {size: _sequence(rng, objs, *size, n=6) for size in SIZES}
    lives = {size: LiveDetector(pipe, sift, size, features=True) for size in SIZES}
    for size in SIZES:
        lives[size].detect([seqs[size][0]])
    for i in range(1, 6):
        for size in SIZES:
            torch.cuda.synchronize()
            before = torch.cuda.memory_allocated()
            (got,) = lives[size].detect([seqs[size][i]])
            torch.cuda.synchronize()
            assert torch.cuda.memory_allocated() == before, (size, i)
            (want,) = _eager(ref, [got["features"]], size)
            _assert_same(got, want, (size, i))
    # CUDA inputs: a second graph of the same size (no upload), same answers
    frame = seqs[(640, 480)][1]
    host = lives[(640, 480)].detect([frame])[0]
    dev = lives[(640, 480)].detect(torch.from_numpy(frame).cuda()[None])[0]
    assert len(lives[(640, 480)]._graphs) == 2 and len(lives[(1200, 900)]._graphs) == 1
    for key in ("n_descriptors", "valid_group", "valid_code"):
        np.testing.assert_array_equal(np.sort(np.atleast_1d(host[key])), np.sort(np.atleast_1d(dev[key])))


def test_errors_after_the_replay(database):
    from sod_b200._capi import SodError
    from sod_b200.live import LiveDetector
    from sod_b200.sift import GpuSift
    db, objs = database
    pipe, _ = _pipelines(db, "objects")
    rng = np.random.default_rng(8)
    rich = imaging.textured(rng, 640, 480, shapes=200)
    flat = np.full((480, 640), 128, np.uint8)
    live = LiveDetector(pipe, GpuSift(max_keypoints=R, capacity=200), (640, 480), frames=2)
    with pytest.raises(SodError, match="frame 1 "):
        live.detect([flat, rich])
    assert [r["n_descriptors"] for r in live.detect([flat, flat])] == [0, 0]
    # a Hough output set whose bin capacity is one: flagged on the device, raised after the replay
    pipe2, _ = _pipelines(db, "objects")
    pipe2._hough[0].cap_bins = 1
    frame, _ = imaging.place(rng, imaging.textured(rng, 640, 480, shapes=200), objs[0], 0.6, 10.0, 320.0, 240.0)
    with pytest.raises(RuntimeError, match="output capacity exceeded"):
        LiveDetector(pipe2, GpuSift(max_keypoints=R), (640, 480)).detect([frame])
    # more verified bins than the records read back
    pipe3, _ = _pipelines(db, "objects")
    few = LiveDetector(pipe3, GpuSift(max_keypoints=R), (640, 480), max_bins=1)
    full = LiveDetector(_pipelines(db, "objects")[0], GpuSift(max_keypoints=R), (640, 480)).detect([frame])[0]
    assert len(full["valid_code"]) > 1
    with pytest.raises(RuntimeError, match="max_bins"):
        few.detect([frame])
