"""sod_final_poses (Main.post_process on the device) bit-exact against the oracle per segment and against the
reference's fixture: multi-segment inputs, the worst cases of the walks, the tie-breaks, the live pre-pass on
permuted records, device counts inside a captured CUDA graph, and LiveDetector with no host step after its
replay."""
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import sod_oracle as O

pytestmark = pytest.mark.gpu
GOLD = Path(__file__).resolve().parent / "golden"


def _oracle(cx, cy, scale, angle, w, h, seg=None):
    """oracle.post_process per segment, clusters mapped back to input indices and ordered by their lowest bin."""
    n = len(cx)
    seg = np.zeros(n, np.int32) if seg is None else np.asarray(seg)
    got = []
    for s in np.unique(seg):
        idx = np.nonzero(seg == s)[0]
        cl, subs, ori, fin = O.post_process(cx[idx], cy[idx], scale[idx], angle[idx], [w[i] for i in idx],
                                            [h[i] for i in idx])
        for c, sc, o, f in zip(cl, subs, ori, fin):
            got.append(([int(idx[i]) for i in c], [[int(idx[i]) for i in sub] for sub in sc], o, f))
    got.sort(key=lambda r: r[0][0])
    return [r[0] for r in got], [r[1] for r in got], [r[2] for r in got], [r[3] for r in got]


def _check(cx, cy, scale, angle, w, h, seg=None):
    from sod_b200 import postprocess as P
    want = _oracle(cx, cy, scale, angle, w, h, seg)
    clusters, subs, ori, final = P.post_process_arrays(cx, cy, scale, angle, w, h, segment=seg)
    assert clusters == want[0]
    assert subs == want[1]
    np.testing.assert_array_equal(np.array(ori), np.array(want[2]))
    got = np.array([[c[0], c[1], o, s, sh[0], sh[1]] for (c, o, s, sh) in final], np.float64).reshape(-1, 6)
    np.testing.assert_array_equal(got, np.array(want[3], np.float64).reshape(-1, 6))
    return clusters


def _random(rng, n, spread=3000.0):
    cx = rng.uniform(0, spread, n).round(1)
    cy = rng.uniform(0, spread, n).round(1)
    scale = rng.choice([0.25, 0.5, 1.0, 2.0], n) * rng.uniform(0.9, 1.1, n)
    angle = rng.choice([-1.0, 0.0, 0.5, 2.0], n) + rng.uniform(-0.03, 0.03, n)
    w = rng.integers(100, 800, n).tolist()
    h = rng.integers(100, 800, n).tolist()
    return cx, cy, scale, angle, w, h


def test_fixture():
    from sod_b200 import postprocess as P
    z = np.load(GOLD / "postprocess.npz")
    w, h = [int(v) for v in z["img_w"]], [int(v) for v in z["img_h"]]
    clusters, subs, ori, final = P.post_process_arrays(z["cx"], z["cy"], z["scale"], z["angle"], w, h)
    assert [i for c in clusters for i in c] == z["cluster_members"].tolist()
    assert [len(s) for s in subs] == z["subs_per_cluster"].tolist()
    assert [i for s in subs for sub in s for i in sub] == z["sub_members"].tolist()
    np.testing.assert_array_equal(np.array(ori), z["orientation"])
    got = np.array([[c[0], c[1], o, s, sh[0], sh[1]] for (c, o, s, sh) in final], np.float64)
    np.testing.assert_array_equal(got, z["final"])


@pytest.mark.parametrize("layout", ["interleaved", "sorted"])
@pytest.mark.parametrize("n", [1, 40, 700])
def test_random_segments_equal_oracle(layout, n):
    rng = np.random.default_rng(n + (layout == "sorted"))
    cx, cy, scale, angle, w, h = _random(rng, n, spread=100.0 * np.sqrt(n))
    seg = rng.integers(-3, 5, n).astype(np.int32)
    if layout == "sorted":
        seg = np.sort(seg)
    clusters = _check(cx, cy, scale, angle, w, h, seg)
    if n > 1:
        assert max(len(c) for c in clusters) > 1 and len(clusters) > 1


def test_more_bins_than_walk_ctas_over_thousands_of_segments():
    """9,000 bins: three large segments of clustered bins and ~5,000 small ones, interleaved.  More segments and more
    clusters than the walks have CTAs (4,096), so CTAs take several entries of the start lists."""
    rng = np.random.default_rng(14)
    big, small = 3 * 1000, 6000
    cx, cy, scale, angle, w, h = _random(rng, big + small, spread=2000.0)
    seg = np.concatenate([np.repeat([-5, 100, 7], 1000), rng.integers(1000, 20000, small)]).astype(np.int32)
    cx[:big] = rng.uniform(0, 1500, big).round(1)
    perm = rng.permutation(big + small)
    cx, cy, scale, angle, seg = cx[perm], cy[perm], scale[perm], angle[perm], seg[perm]
    w, h = [w[i] for i in perm], [h[i] for i in perm]
    clusters = _check(cx, cy, scale, angle, w, h, seg)
    assert len(set(seg.tolist())) > 4096 and len(clusters) > 4096 and max(len(c) for c in clusters) > 50


def test_one_cluster_of_4096_bins_within_one_degree():
    rng = np.random.default_rng(9)
    n = 4096
    cx, cy = rng.uniform(0, 50, n), rng.uniform(0, 50, n)
    scale = rng.uniform(1.0, 2.0, n)
    angle = 0.3 + rng.uniform(0, np.radians(0.9), n)
    clusters = _check(cx, cy, scale, angle, [1000] * n, [800] * n)
    assert len(clusters) == 1 and len(clusters[0]) == n


def test_ties_later_subcluster_and_first_smallest_area_win():
    # one position cluster; two orientation sub-clusters of 3 bins each (the later one must give the orientation)
    # and equal areas (the first bin with the smallest area must give the shape)
    cx = np.array([0.0, 1.0, 2.0, 3.0, 4.0, 5.0])
    cy = np.zeros(6)
    scale = np.array([1.0, 2.0, 1.0, 0.5, 1.0, 0.5])
    angle = np.array([0.0, 1.0, 0.001, 1.001, 0.002, 1.002])
    w, h = [400, 200, 400, 800, 400, 800], [300, 150, 300, 600, 300, 600]
    from sod_b200 import postprocess as P
    _check(cx, cy, scale, angle, w, h)
    _, subs, ori, final = P.post_process_arrays(cx, cy, scale, angle, w, h)
    assert [len(s) for s in subs[0]] == [3, 3] and subs[0][1][0] == 1
    assert ori[0] == (1.0 + 1.001 + 1.002) / 3
    assert final[0][2] == (1.0 + 2.0 + 1.0 + 0.5 + 1.0 + 0.5) / 6
    assert final[0][-1] == (400, 300)           # area 120000 at bins 0, 1 and 3: the first one met gives the shape


def test_all_bins_isolated():
    n = 3000
    cx = np.arange(n) * 1000.0
    clusters = _check(cx, np.zeros(n), np.ones(n), np.zeros(n), [100] * n, [100] * n,
                      (np.arange(n) % 7).astype(np.int32))
    assert clusters == [[i] for i in range(n)]


def _records(rng, frames, per_frame, gpf):
    """Affine records: live bins of several frames (group = frame * gpf + object) with unique insertion keys,
    non-live bins interleaved, the whole list permuted."""
    rows = []
    for f in range(frames):
        cx, cy, scale, angle, w, h = _random(rng, per_frame, spread=1500.0)
        for i in range(per_frame):
            rows.append((f * gpf + int(rng.integers(0, gpf)), cx[i], cy[i], angle[i], scale[i], w[i], h[i]))
    n = len(rows)
    perm = rng.permutation(n)
    group = np.array([rows[i][0] for i in perm], np.int32)
    mean = np.array([rows[i][1:] for i in perm], np.float64)
    order = rng.permutation(np.arange(n, dtype=np.int64) * 3 + 5)
    status = np.where(rng.random(n) < 0.7, 1, 2 + 4 * rng.integers(0, 2, n)).astype(np.int32) | (3 << 8)
    return status, group, order, mean


def _host_route(status, group, order, mean, gpf):
    """DetectionPipeline.final_poses' host route: lexsort, then post_process_arrays with the frame as segment."""
    from sod_b200 import postprocess as P
    live = (status & 1).astype(bool)
    g, o, m = group[live], order[live], mean[live]
    frame = g // gpf
    s = np.lexsort((o, g, frame))
    m, frame = m[s], frame[s].astype(np.int32)
    clusters, _, _, final = P.post_process_arrays(m[:, 0], m[:, 1], m[:, 3], m[:, 2], m[:, 4], m[:, 5],
                                                  segment=frame)
    return np.array([[c[0], c[1], o_, s_, sh[0], sh[1]] for (c, o_, s_, sh) in final]).reshape(-1, 6), \
        np.array([frame[c[0]] for c in clusters], np.int32)


def test_live_prepass_on_permuted_records_equals_host_lexsort():
    from sod_b200 import engine as E
    rng = np.random.default_rng(11)
    gpf = 3
    status, group, order, mean = _records(rng, frames=5, per_frame=60, gpf=gpf)
    want_pose, want_frame = _host_route(status, group, order, mean, gpf)
    n = len(status)
    cap = n + 17                                   # slots past the count hold garbage
    dev = lambda a, fill: torch.from_numpy(np.concatenate([a, np.full((17,) + a.shape[1:], fill, a.dtype)])).cuda()  # noqa
    fp = E.FinalPoses(cap, "cuda")
    n_dev = torch.tensor([n], dtype=torch.int32, device="cuda")
    fp.run_records(dev(status, 1), dev(group, 0), dev(order, 0), dev(mean, 7.0), cap, n_dev, gpf)
    h = fp.host(cap)
    nc = int(h["counters"][0])
    assert nc == len(want_pose) and int(h["counters"][1]) == int((status & 1).sum())
    np.testing.assert_array_equal(h["pose"][:nc], want_pose)
    np.testing.assert_array_equal(h["segment"][:nc], want_frame)


def test_graph_replay_with_device_counts_equals_eager_calls():
    from sod_b200 import engine as E
    rng = np.random.default_rng(12)
    cap = 500
    cx, cy, scale, angle, w, h = _random(rng, cap)
    mean = torch.from_numpy(np.stack([cx, cy, angle, scale, np.array(w, float), np.array(h, float)], 1)).cuda()
    seg = torch.from_numpy(rng.integers(0, 4, cap).astype(np.int32)).cuda()
    n_dev = torch.zeros(1, dtype=torch.int32, device="cuda")
    fp, ref = E.FinalPoses(cap, "cuda"), E.FinalPoses(cap, "cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fp.run(mean, seg, cap, n_dev)              # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fp.run(mean, seg, cap, n_dev)
    for count in (0, 1, 217, cap, cap + 1000):
        n_dev.fill_(count)
        g.replay()
        got = fp.host(cap)
        k = min(count, cap)
        if k:
            ref.run(mean[:k].contiguous(), seg[:k].contiguous(), k)
            want = ref.host(k)
        nc = int(got["counters"][0])
        assert int(got["counters"][1]) == k
        if k == 0:
            assert nc == 0
            continue
        assert nc == int(want["counters"][0])
        for name in ("cluster_offset",):
            np.testing.assert_array_equal(got[name][:nc + 1], want[name][:nc + 1])
        for name in ("cluster_bins", "sub_bins", "sub_first"):
            np.testing.assert_array_equal(got[name][:k], want[name][:k])
        for name in ("pose", "shape_bin", "segment"):
            np.testing.assert_array_equal(got[name][:nc], want[name][:nc])


def test_live_detector_needs_no_host_step_after_the_replay(monkeypatch):
    from test_gpu_live import R, _eager, _pipelines, _sequence
    from test_gpu_sift import _database
    from sod_b200 import postprocess as P
    from sod_b200._capi import lib
    from sod_b200.live import LiveDetector
    from sod_b200.sift import GpuSift
    rng = np.random.default_rng(21)
    db, objs = _database(rng)
    pipe, ref = _pipelines(db, "objects")
    live = LiveDetector(pipe, GpuSift(max_keypoints=R), (640, 480), features=True)
    frames = _sequence(np.random.default_rng(5), objs, 640, 480, n=4)
    live.detect([frames[0]])                       # capture the graph

    def refuse(*a, **k):
        raise AssertionError("host pose clustering after the replay")

    found = 0
    for fr in frames:
        with monkeypatch.context() as m:
            m.setattr(P, "_graph", refuse)
            m.setattr(P, "post_process_arrays", refuse)
            m.setattr(lib, "sod_pose_adjacency", refuse)
            m.setattr(lib, "sod_final_poses", refuse)
            (got,) = live.detect([fr])
        (want,) = _eager(ref, [got["features"]], (640, 480))
        pose = lambda ps: np.array([[c[0], c[1], o, s, sh[0], sh[1]] for (c, o, s, sh) in ps]).reshape(-1, 6)  # noqa
        np.testing.assert_array_equal(pose(got["final_pose"]), pose(want["final_pose"]))
        found += len(got["final_pose"])
    assert found > 0
