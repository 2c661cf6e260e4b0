"""CPU-side checks of mixed-size SIFT batches: workspace sizes and argument errors of sod_sift_extract_mixed before
any CUDA call, the binding against the header, SiftBatch.frame_sizes, and GenerateDatabaseInfo.build_database's GPU
path with a stand-in extractor (chunking, input order, row layout, centroid, the empty-image error)."""
import ctypes as C
import pickle
import re
from pathlib import Path

import cv2
import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
GEOM_BYTES = 160                      # one frame's geometry record in the workspace (sod.h)


def _wh(sizes):
    flat = [v for s in sizes for v in s]
    return C.cast((C.c_int32 * len(flat))(*flat), C.c_void_p)


def _align(n):
    return (n + 255) & ~255


def test_mixed_workspace_bytes():
    from sod_b200._capi import lib
    sizes = [(640, 480), (47, 33), (480, 640), (1500, 1000), (1, 1)]
    pyr = [lib.sod_sift_batch_workspace_bytes(w, h, 1, 0) for w, h in sizes]
    n, cap = len(sizes), 1000
    # the slabs of n frames: a uniform batch's workspace less its pyramids
    slabs = lib.sod_sift_batch_workspace_bytes(640, 480, n, cap) - n * pyr[0]
    assert lib.sod_sift_mixed_workspace_bytes(_wh(sizes), n, cap) == sum(pyr) + slabs + _align(n * GEOM_BYTES)
    assert lib.sod_sift_mixed_workspace_bytes(_wh(sizes), n, 0) == sum(pyr) + _align(n * GEOM_BYTES)
    one = lib.sod_sift_mixed_workspace_bytes(_wh(sizes[:1]), 1, cap)
    assert one == lib.sod_sift_batch_workspace_bytes(640, 480, 1, cap) + 256
    for bad in ([(0, 480)], [(640, 32769)], [(640, 480), (-1, 5)]):
        assert lib.sod_sift_mixed_workspace_bytes(_wh(bad), len(bad), 10) == 0
    assert lib.sod_sift_mixed_workspace_bytes(None, 1, 10) == 0
    assert lib.sod_sift_mixed_workspace_bytes(_wh([(8, 8)]), 0, 10) == 0
    assert lib.sod_sift_mixed_workspace_bytes(_wh([(8, 8)] * 65), 65, 10) == 0
    assert lib.sod_sift_mixed_workspace_bytes(_wh([(8, 8)] * 64), 64, 10) > 0
    assert lib.sod_sift_mixed_workspace_bytes(_wh([(8, 8)]), 1, -1) == 0
    assert lib.sod_sift_mixed_workspace_bytes(_wh([(8, 8)] * 2), 2, 1 << 23) > 0      # frames x cap = 2^24
    assert lib.sod_sift_mixed_workspace_bytes(_wh([(8, 8)] * 3), 3, 1 << 23) == 0


def test_extract_mixed_rejects_bad_arguments_without_gpu():
    from sod_b200._capi import SiftBatchOut, lib
    fake = 1 << 20                         # never dereferenced: validation fails first
    f = lib.sod_sift_extract_mixed
    sizes = [(10, 10), (12, 7)]
    need = lib.sod_sift_mixed_workspace_bytes(_wh(sizes), 2, 100)

    def arr(t, vals):
        return C.cast((t * len(vals))(*vals), C.c_void_p)

    out = SiftBatchOut(*([fake] * 11), 200, 100)
    ok = dict(images=arr(C.c_void_p, [fake, fake]), wh=_wh(sizes), pitch=arr(C.c_int64, [10, 12]), frames=2, max=0,
              out=C.byref(out), ws=fake, bytes=need, stream=None)

    def err(**kw):
        a = dict(ok)
        a.update(kw)
        assert f(*a.values()) == -1
        return lib.sod_last_error()

    assert b"null image, size or pitch" in err(images=None)
    assert b"null image, size or pitch" in err(wh=None)
    assert b"null image, size or pitch" in err(pitch=None)
    assert b"frames 0" in err(frames=0)
    assert b"frames 65" in err(frames=65)
    assert b"frame 1: null image" in err(images=arr(C.c_void_p, [fake, None]))
    assert b"frame 1: image size 0x7" in err(wh=_wh([(10, 10), (0, 7)]))
    assert b"frame 0: image size 10x32769" in err(wh=_wh([(10, 32769), (12, 7)]))
    assert b"frame 1: pitch 11 < width 12" in err(pitch=arr(C.c_int64, [10, 11]))
    assert b"max_per_frame" in err(max=-1)
    assert b"null out" in err(out=None)
    for field, value, what in (("cap_per_frame", 0, b"cap_per_frame"), ("cap_per_frame", (1 << 23) + 1, b"cap_per_frame"),
                               ("cap_rows", 0, b"cap_rows"), ("cap_rows", (1 << 24) + 1, b"cap_rows")):
        bad = SiftBatchOut(*([fake] * 11), 200, 100)
        setattr(bad, field, value)
        assert what in err(out=C.byref(bad))
    for name in ("xy", "size", "angle", "response", "octave", "des", "frame", "count", "offset", "overflow",
                 "rows_overflow"):
        bad = SiftBatchOut(*([fake] * 11), 200, 100)
        setattr(bad, name, None)
        assert b"null output" in err(out=C.byref(bad)), name
    assert b"workspace" in err(ws=None)
    assert b"workspace" in err(bytes=need - 1)
    assert b"workspace" in err(ws=fake + 16)                               # misaligned


def test_protos_match_the_header():
    """The two new prototypes as sod.h declares them (argument count and the pointer / integer kinds)."""
    from sod_b200 import _capi
    text = re.sub(r"/\*.*?\*/", "", (ROOT / "include" / "sod.h").read_text(), flags=re.S)
    kinds = {"int32_t": C.c_int32, "int64_t": C.c_int64, "size_t": C.c_size_t, "sod_stream_t": C.c_void_p}
    for name in ("sod_sift_mixed_workspace_bytes", "sod_sift_extract_mixed"):
        m = re.search(r"(\w+)\s+" + name + r"\(([^)]*)\)", text)
        ret, params = m.group(1), [p.strip() for p in m.group(2).split(",")]
        res, args = _capi._PROTOS[name]
        assert res == {"size_t": C.c_size_t, "int": C.c_int}[ret]
        assert len(args) == len(params), name
        for p, a in zip(params, args):
            t = p.rsplit(" ", 1)[0].replace("const ", "").strip()
            if "*" in p:
                assert a in (C.c_void_p,) or a.__name__.startswith("LP_"), (name, p)
            else:
                assert a == kinds[t], (name, p)
    assert _capi.SIFT_MAX_MIXED_FRAMES == int(re.search(r"SOD_SIFT_MAX_MIXED_FRAMES (\d+)", text).group(1))


def test_sift_batch_frame_sizes():
    from sod_b200.sift import SiftBatch
    z = torch.zeros(5)
    xy = torch.arange(10, dtype=torch.float32).reshape(5, 2)
    des = torch.zeros((5, 128), dtype=torch.uint8)
    same = SiftBatch(des, xy, z, z.int(), z, z, z.int(), np.array([2, 3]), np.array([0, 2]), (64, 48))
    assert same.frame_sizes is None and same.arrays(1)["frame_size"] == (64, 48)
    mixed = SiftBatch(des, xy, z, z.int(), z, z, z.int(), np.array([2, 3]), np.array([0, 2]), None,
                      frame_sizes=np.array([[64, 48], [30, 70]]))
    assert mixed.arrays(0)["frame_size"] == (64, 48) and mixed.features(1).size == (30, 70)
    np.testing.assert_array_equal(mixed.arrays(1)["xy"], xy[2:].numpy())


def test_extract_mixed_rejects_bad_input_before_any_device_work():
    from sod_b200.sift import GpuSift
    g = GpuSift()
    with pytest.raises(ValueError, match="1..64 frames"):
        g.extract_mixed([])
    with pytest.raises(ValueError, match="1..64 frames"):
        g.extract_mixed([np.zeros((10, 12), np.uint8)] * 65)
    with pytest.raises(ValueError, match="slot"):
        g.extract_mixed([np.zeros((10, 12), np.uint8)], slot=2)
    with pytest.raises(ValueError, match="out of range"):
        g.extract_mixed([np.zeros((10, 12), np.uint8), np.zeros((5, 32769), np.uint8)])
    with pytest.raises(ValueError, match="8-bit"):
        g.extract_mixed([np.zeros((10, 12), np.uint8), np.zeros((5, 6), np.float32)])


# ------------------------------------------------------------------------------- build_database's GPU path
class _FakeMixedSift:
    """Stands in for GpuSift on the CPU: an image whose pixel (0, 0) is v has v % 7 keypoints at (x, y) = (v + k / 3,
    k * 1.1 + 0.2), size 2 + k, angle 10 k, response k / 100, octave 0x100 | k, descriptor bytes (v + k) % 256."""

    def __init__(self):
        self.calls = []

    def extract_mixed(self, images, slot=0):
        from sod_b200.sift import SiftBatch
        self.calls.append([(im.shape[1], im.shape[0]) for im in images])
        vals = [int(im[0, 0]) for im in images]
        count = np.array([v % 7 for v in vals], np.int64)
        offset = np.concatenate([[0], np.cumsum(count)[:-1]]).astype(np.int64)
        cols = {k: [] for k in ("xy", "size", "angle", "response", "octave", "des", "frame")}
        for f, v in enumerate(vals):
            for k in range(v % 7):
                cols["xy"].append((v + k / 3, k * 1.1 + 0.2))
                cols["size"].append(2 + k)
                cols["angle"].append(10 * k)
                cols["response"].append(k / 100)
                cols["octave"].append(0x100 | k)
                cols["des"].append([(v + k) % 256] * 128)
                cols["frame"].append(f)
        t = lambda a, dt, shape: torch.tensor(np.asarray(a, dt).reshape(shape))  # noqa: E731
        return SiftBatch(t(cols["des"], np.uint8, (-1, 128)), t(cols["xy"], np.float32, (-1, 2)),
                         t(cols["angle"], np.float32, -1), t(cols["octave"], np.int32, -1),
                         t(cols["size"], np.float32, -1), t(cols["response"], np.float32, -1),
                         t(cols["frame"], np.int32, -1), count, offset, None,
                         frame_sizes=np.array([(im.shape[1], im.shape[0]) for im in images], np.int64))


def _folder(tmp_path, values_heights):
    """PNG files named so that os.listdir's order is not the value order, plus a file that is no image."""
    for i, (v, h) in enumerate(values_heights):
        img = np.full((h, 150, 3), v, np.uint8)          # resized to 1500 wide: (1500, 10 h)
        cv2.imwrite(str(tmp_path / f"{(i * 7919) % 1000:03d}_{i}.png"), img)
    (tmp_path / "notes.txt").write_text("not an image")


def test_build_database_gpu_rows_order_and_centroid(tmp_path):
    import os

    import GenerateDatabaseInfo as G
    from SiftHelperFunctions import get_centroid
    vals = [(1 + i * 7 + (i % 6), 100 + 3 * i) for i in range(9)]
    _folder(tmp_path, vals)
    ex = _FakeMixedSift()
    data = G.build_database(str(tmp_path), str(tmp_path / "db.pkl"), str(tmp_path / "db.sodb"), extractor=ex)
    names = [n for n in os.listdir(tmp_path) if n.endswith(".png")]
    listed = [n for n in os.listdir(tmp_path) if n in names]
    assert [r[4] for r in data] == [os.path.join(str(tmp_path), n) for n in listed]
    assert sum(len(c) for c in ex.calls) == len(names)
    for row in data:
        i = int(Path(row[4]).stem.split("_")[1])
        v, h = vals[i]
        temp_kp, des, img_size, centroid, _ = row
        assert img_size == (1500, 10 * h) and all(type(x) is int for x in img_size)
        n = v % 7
        assert len(temp_kp) == n and des.dtype == np.float32 and des.shape == (n, 128)
        for k, t in enumerate(temp_kp):
            assert t == ((float(np.float32(v + k / 3)), float(np.float32(k * 1.1 + 0.2))), float(2 + k),
                         float(10 * k), float(np.float32(k / 100)), 0x100 | k, -1)
            assert all(type(x) is float for x in t[0]) and type(t[4]) is int
        np.testing.assert_array_equal(des, np.full((n, 128), (v + np.arange(n)[:, None]) % 256, np.float32))

        class K:
            def __init__(self, pt):
                self.pt = pt
        want = get_centroid([K(t[0]) for t in temp_kp])
        assert centroid == want and all(type(x) is float for x in centroid)
    with open(tmp_path / "db.pkl", "rb") as f:
        again = pickle.load(f)
    assert [r[4] for r in again] == [r[4] for r in data] and again[0][0] == data[0][0]
    assert (tmp_path / "db.sodb").exists()


def test_build_database_gpu_centroid_is_a_left_to_right_sum(tmp_path):
    """A sum where pairwise (numpy) and left-to-right summation differ: the row must hold the latter."""
    import GenerateDatabaseInfo as G
    xs = np.array([1e8, 1.0, -1e8, 1.0, 3.3, 1e-3] * 3, np.float32)

    class One:
        def extract_mixed(self, images, slot=0):
            from sod_b200.sift import SiftBatch
            n = len(xs)
            z = torch.zeros(n)
            xy = torch.tensor(np.stack([xs, xs[::-1]], 1).copy())
            return SiftBatch(torch.zeros((n, 128), dtype=torch.uint8), xy, z, torch.zeros(n, dtype=torch.int32), z,
                             z, torch.zeros(n, dtype=torch.int32), np.array([n]), np.array([0]), None,
                             frame_sizes=np.array([[1500, 1000]]))

    cv2.imwrite(str(tmp_path / "a.png"), np.full((100, 150, 3), 9, np.uint8))
    row = G.build_database(str(tmp_path), str(tmp_path / "db.pkl"), extractor=One())[0]
    sx = sy = 0
    for x, y in zip(xs.tolist(), xs[::-1].tolist()):
        sx, sy = sx + x, sy + y
    assert row[3] == (sx / len(xs), sy / len(xs))


def test_build_database_empty_image_raises_as_the_cv2_path(tmp_path):
    import GenerateDatabaseInfo as G
    cv2.imwrite(str(tmp_path / "flat.png"), np.full((100, 150, 3), 7, np.uint8))      # 7 % 7 = 0 keypoints
    with pytest.raises(ZeroDivisionError) as gpu_err:
        G.build_database(str(tmp_path), str(tmp_path / "g.pkl"), extractor=_FakeMixedSift())
    with pytest.raises(ZeroDivisionError) as cv2_err:
        G.build_database(str(tmp_path), str(tmp_path / "c.pkl"))
    assert str(gpu_err.value) == str(cv2_err.value)


def test_gpu_chunks_by_frame_count_and_budget(monkeypatch):
    import GenerateDatabaseInfo as G
    sizes = [(1500, 1000 + i) for i in range(10)]
    per = [G._frame_bytes(w, h) for w, h in sizes]
    assert G.gpu_chunks(sizes, max_frames=4, budget=1 << 62) == [[0, 1, 2, 3], [4, 5, 6, 7], [8, 9]]
    budget = per[7] + per[8] + per[9]                  # any three fit, no four
    assert G.gpu_chunks(sizes, max_frames=64, budget=budget) == [[0, 1, 2], [3, 4, 5], [6, 7, 8], [9]]
    assert G.gpu_chunks(sizes, max_frames=64, budget=per[0] + per[1]) == [[0, 1], [2], [3], [4], [5], [6], [7], [8],
                                                                          [9]]
    assert G.gpu_chunks(sizes[:2], max_frames=64, budget=1) == [[0], [1]]    # one image over budget: alone
    assert G.gpu_chunks(sizes) == [list(range(10))]                           # defaults: 10 x 190 MB < 8 GB
    assert G.gpu_chunks([(1500, 1000)] * 100, budget=1 << 62) == [list(range(64)), list(range(64, 100))]
    # build_database follows the same chunks, in input order, across its decode window
    monkeypatch.setattr(G, "GPU_CHUNK_FRAMES", 3)
    assert G.gpu_chunks(sizes[:7]) == [[0, 1, 2], [3, 4, 5], [6]]


def test_build_database_chunks_the_images(tmp_path, monkeypatch):
    import os

    import GenerateDatabaseInfo as G
    _folder(tmp_path, [(1 + i + i // 6, 100 + i) for i in range(11)])       # no value a multiple of 7
    monkeypatch.setattr(G, "GPU_CHUNK_FRAMES", 4)
    ex = _FakeMixedSift()
    data = G.build_database(str(tmp_path), str(tmp_path / "db.pkl"), extractor=ex)
    assert [len(c) for c in ex.calls] == [4, 4, 3]
    heights = [r[2][1] for r in data]
    assert [s[1] for c in ex.calls for s in c] == heights
    assert len(data) == 11 and [r[4] for r in data] == [os.path.join(str(tmp_path), n)
                                                         for n in os.listdir(tmp_path) if n.endswith(".png")]
    monkeypatch.setattr(G, "GPU_CHUNK_FRAMES", 64)
    monkeypatch.setattr(G, "GPU_CHUNK_BYTES", 2 * G._frame_bytes(1500, 1100) + 1)   # any two, never three
    ex = _FakeMixedSift()
    G.build_database(str(tmp_path), str(tmp_path / "db.pkl"), extractor=ex)
    assert [len(c) for c in ex.calls] == [2] * 5 + [1]
