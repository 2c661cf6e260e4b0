"""GPU SIFT (sod_b200.sift.GpuSift) against cv2.SIFT_create() as the reference: pyramid, descriptors at cv2's
keypoints, detection, edge cases, and FrameStream end to end with the GPU extractor."""
import cv2
import numpy as np
import pytest
from scipy.spatial import cKDTree

import imaging

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    from sod_b200.sift import GpuSift
    return GpuSift()


def _cv2_pyramid(gray, n_oct):
    """The recipe cv2's SIFT follows: resize x2, GaussianBlur chain, every other pixel of level 3."""
    h, w = gray.shape
    base = cv2.resize(gray.astype(np.float32), (2 * w, 2 * h), interpolation=cv2.INTER_LINEAR)
    s0 = float(np.sqrt(np.float32(max(np.float32(1.6) ** 2 - np.float32(1.0), np.float32(0.01)))))
    k = 2.0 ** (1 / 3)
    sig = [np.sqrt((1.6 * k ** (i - 1) * k) ** 2 - (1.6 * k ** (i - 1)) ** 2) for i in range(6)]
    levels, cur = [], cv2.GaussianBlur(base, (0, 0), s0, sigmaY=s0)
    for o in range(n_oct):
        if o:
            p = levels[-1][3]
            cur = p[:2 * (p.shape[0] // 2):2, :2 * (p.shape[1] // 2):2]
        octave = [cur]
        for i in range(1, 6):
            octave.append(cv2.GaussianBlur(octave[-1], (0, 0), sig[i], sigmaY=sig[i]))
        levels.append(octave)
    return levels


def _cv2_sift(gray):
    kp, des = cv2.SIFT_create().detectAndCompute(gray, None)
    a = {"xy": np.array([k.pt for k in kp], np.float32).reshape(-1, 2),
         "size": np.array([k.size for k in kp], np.float32), "angle": np.array([k.angle for k in kp], np.float32),
         "response": np.array([k.response for k in kp], np.float32),
         "octave": np.array([k.octave for k in kp], np.int32)}
    a["des"] = des if des is not None else np.zeros((0, 128), np.float32)
    return kp, a


@pytest.mark.parametrize("seed,w,h", [(11, 640, 480), (12, 641, 479), (13, 1200, 900)])
def test_pyramid_matches_the_cv2_recipe(gpu, seed, w, h):
    gray = imaging.textured(np.random.default_rng(seed), w, h)
    gpu.extract(gray)
    want = _cv2_pyramid(gray, 3)
    worst = 0.0
    for o in range(3):
        for lv in range(6):
            got = gpu.gaussian_level((w, h), o - 1, lv)
            assert got.shape == want[o][lv].shape, (o, lv)
            err = float(np.abs(got - want[o][lv]).max())
            assert err <= 1e-3, (o - 1, lv, err)
            worst = max(worst, err)
    print(f"pyramid {w}x{h}: max |gpu - cv2| over octaves -1..1 = {worst:.2e}")


@pytest.mark.parametrize("seed,w,h", [(21, 640, 480), (22, 1200, 900)])
def test_descriptors_at_cv2_keypoints(gpu, seed, w, h):
    gray = imaging.textured(np.random.default_rng(seed), w, h, shapes=200)
    _, ref = _cv2_sift(gray)
    got = gpu.describe(gray, ref["xy"], ref["size"], ref["angle"], ref["octave"])
    d = np.abs(got.astype(np.int32) - ref["des"].astype(np.int32))
    bytes_ok, rows_ok = float((d <= 1).mean()), float((d.max(axis=1) <= 2).mean())
    print(f"describe {w}x{h}: {len(d)} keypoints, bytes |d|<=1 {bytes_ok:.5f}, rows max|d|<=2 {rows_ok:.5f}, "
          f"max |d| {int(d.max())}")
    assert bytes_ok >= 0.99 and rows_ok >= 0.99


def _pair(a, b):
    """For every keypoint of a: is there one in b with equal octave and layer, |dpt| <= 0.1 px and angle within
    1 degree?  Returns the index of that partner or -1."""
    tree = cKDTree(b["xy"].astype(np.float64))
    out = np.full(len(a["xy"]), -1)
    for i, near in enumerate(tree.query_ball_point(a["xy"].astype(np.float64), 0.1)):
        for j in near:
            da = (float(a["angle"][i]) - float(b["angle"][j]) + 180.0) % 360.0 - 180.0
            if (a["octave"][i] & 0xFFFF) == (b["octave"][j] & 0xFFFF) and abs(da) <= 1.0:
                out[i] = j
                break
    return out


@pytest.mark.parametrize("seed,w,h", [(31, 640, 480), (32, 800, 600), (33, 1200, 900)])
def test_detection_agrees_with_cv2(gpu, seed, w, h):
    gray = imaging.textured(np.random.default_rng(seed), w, h, shapes=200)
    _, ref = _cv2_sift(gray)
    got = gpu.extract(gray)
    n_ref, n_got = len(ref["xy"]), len(got["xy"])
    r2g, g2r = _pair(ref, got), _pair(got, ref)
    f_ref, f_got = float((r2g >= 0).mean()), float((g2r >= 0).mean())
    m = r2g >= 0
    rel_size = np.abs(got["size"][r2g[m]] / ref["size"][m] - 1)
    rel_resp = np.abs(got["response"][r2g[m]] / ref["response"][m] - 1)
    print(f"detect {w}x{h}: cv2 {n_ref} gpu {n_got}, cv2 paired {f_ref:.4f}, gpu paired {f_got:.4f}, "
          f"max rel size {rel_size.max():.2e}, max rel response {rel_resp.max():.2e}, "
          f"response > 1e-3: {int((rel_resp > 1e-3).sum())}")
    assert f_ref >= 0.95 and f_got >= 0.95
    assert abs(n_got - n_ref) <= 0.03 * n_ref
    keys = list(zip(got["xy"][:, 0], got["xy"][:, 1], got["size"], got["angle"], got["response"], got["octave"]))
    assert keys == sorted(keys)
    assert len(set((k[0], k[1], k[2], k[3]) for k in keys)) == len(keys)     # duplicates removed
    assert rel_size.max() <= 1e-3 and rel_resp.max() <= 1e-3


def test_edge_cases(gpu):
    from sod_b200._capi import SodError
    from sod_b200.sift import GpuSift
    for img in (np.full((480, 640), 128, np.uint8), np.full((8, 8), 7, np.uint8),
                np.random.default_rng(1).integers(0, 256, (8, 8), dtype=np.uint8),
                np.random.default_rng(2).integers(0, 256, (16, 16), dtype=np.uint8)):
        f = gpu(img)
        assert len(f) == 0 and f.des.shape == (0, 128) and f.xy.shape == (0, 2)
    small = np.random.default_rng(0).integers(0, 256, (33, 47), dtype=np.uint8)
    _, ref = _cv2_sift(small)
    got = gpu.extract(small)
    assert len(got["xy"]) == len(ref["xy"]) == 2
    np.testing.assert_allclose(got["xy"], ref["xy"], atol=0.1)
    np.testing.assert_array_equal(got["octave"] & 0xFFFF, ref["octave"] & 0xFFFF)
    gray = imaging.textured(np.random.default_rng(5), 640, 480)
    with pytest.raises(SodError, match="capacity"):
        GpuSift(capacity=10)(gray)
    full = gpu(gray)
    head = GpuSift(max_keypoints=50)(gray)            # the first n in sorted order, as sift_features keeps them
    assert len(head) == 50
    np.testing.assert_array_equal(head.xy, full.xy[:50])
    np.testing.assert_array_equal(head.octave, full.octave[:50])
    bgr = cv2.cvtColor(gray, cv2.COLOR_GRAY2BGR)      # a BGR image goes through the same cvtColor as cv2's path
    np.testing.assert_array_equal(gpu(bgr).xy, full.xy)
    with pytest.raises(ValueError):
        gpu.describe(gray, [[10.0, 10.0]], [3.0], [0.0], [20])   # octave 20: no such level


def _database(rng, n_objects=3):
    from SiftHelperFunctions import get_centroid, make_temp_kp
    from sod_b200.database import PackedDatabase
    rows, objs = [], []
    for i in range(n_objects):
        obj = imaging.textured(rng, 600, 400)
        kp, des = cv2.SIFT_create().detectAndCompute(obj, None)
        rows.append([make_temp_kp(kp), des, (600, 400), get_centroid(kp), f"obj{i}.png"])
        objs.append(obj)
    return PackedDatabase.from_reference_rows(rows), objs


def _main_on(db, feats, kps_db):
    import main as dropin_main
    m = dropin_main.Main()
    m.kp, m.des = kps_db, db.des
    m.img_size_list, m.img_centroid_list = db.per_keypoint_lists()
    m.kp_query = [cv2.KeyPoint(float(feats.xy[i, 0]), float(feats.xy[i, 1]), 1.0, float(feats.angle[i]), 0.0,
                               int(feats.octave[i]), i) for i in range(len(feats))]
    m.des_query = feats.des
    m.rgb_query = np.zeros((feats.size[1], feats.size[0], 3), np.uint8)
    m.image_query_size = feats.size
    m.run_matcher()
    m.apply_hough_transform(15)
    m.get_valid_bins(5)
    m.apply_affine_parameters(4)
    m.post_process()
    return m


def test_stream_with_gpu_sift_finds_the_objects_of_a_cv2_database():
    """The scenario of test_gpu_stream.py (same placements and tolerances) with GpuSift as FrameStream's
    extractor, against a database built with cv2 SIFT."""
    from sod_b200.pipeline import DetectionPipeline
    from sod_b200.sift import GpuSift
    from sod_b200.stream import FrameStream
    rng = np.random.default_rng(7)
    db, objs = _database(rng)
    placements = [[(0, 0.8, 20, 500, 400)], [(1, 1.0, -35, 700, 450), (2, 0.6, 90, 250, 250)], [],
                  [(2, 1.2, 5, 600, 500)], [(0, 0.7, 170, 800, 300)]]
    frames, truth = [], []
    for pl in placements:
        fr = imaging.textured(rng, 1200, 900, shapes=200)
        t = []
        for (o, s, deg, cx, cy) in pl:
            fr, m = imaging.place(rng, fr, objs[o], s, deg, cx, cy)
            c = db.img_centroid[o]
            t.append((m @ np.array([c[0], c[1], 1.0]), s, deg))
        frames.append(fr)
        truth.append(t)

    gpu, seen = GpuSift(), {}

    def extractor(fr):                     # shared by the stream's worker threads
        f = gpu(fr)
        seen[id(fr)] = f
        return f

    pipe = DetectionPipeline(db.to_model_database(), max_queries=20000, frame_wh=np.zeros((2, 2), np.int32),
                             per_object_spaces=False)
    results = dict(FrameStream(pipe, extractor=extractor, batch_frames=2, workers=4).run(frames))
    assert sorted(results) == list(range(len(frames)))

    kps_db = db.keypoints()
    db_index = {id(k): i for i, k in enumerate(kps_db)}
    for i, fr in enumerate(frames):
        feats = seen[id(fr)]
        r = results[i]
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
