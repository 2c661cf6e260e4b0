"""Hough voting (K4) and affine verification (K5) at every size class they dispatch on, against the oracle.

Both stages pick their code path by data size (sod_hough.cu, sod_affine.cu):

- matches per Hough space: <= 1,024 one match per thread (vote_space_small), <= 65,535 16-bit arrival ranks
  (vote_space<false>), more 32-bit ranks (vote_space<true>);
- Hough spaces per call: 16 sub-counters per space up to 4,096 spaces, fewer above (group_sub_shift), a
  three-launch grid scan past 2 x 8,192 sub-counters (device_exclusive_scan);
- votes per bin: 1 (no sort), 2-16 (one thread, insertion sort), 17-1,024 (one warp, bitonic sort), more
  (one CTA, bitmap sort in windows of 2^20 match ids);
- detail_min_count: bins below it get no members, means or order key;
- pairs per affine bin: <= 32 one thread (16 staged in shared memory), more one warp (512 staged).

Every scene below is built so that it lands in the class it targets, and every test asserts that from its
own input.  Expected outputs come from the scalar oracle (oracle/sod_oracle.py) or from `reference_hough`,
a numpy restatement of it that scales to 10^6 matches and is pinned to the scalar oracle by a CPU test here.
"""
import math

import numpy as np
import pytest

import scenes
from oracle import sod_oracle as O

gpu = pytest.mark.gpu
BINS = 15
W, H = 4032, 3024
WINDOW = 1 << 20           # match ids per bitmap window of hough_finish_huge_kernel (kWindowBits)
FINISH_SIZES = (1, 2, 16, 17, 1024, 1025)   # both sides of every finish-kernel class boundary
LUT = O.sigma_lut(BINS)    # sigma bin of the scale ratio 2^k, k = -24..24
K_OF_SIGMA = {}            # sigma bin -> smallest k >= 0 that reaches it
for _k in range(25):
    K_OF_SIGMA.setdefault(LUT[_k + 24], _k)
SIGMAS = np.array(sorted(K_OF_SIGMA))       # at bins = 15: 0 2 4 6 9 11 13 14


# ------------------------------------------------------------------------------------------------
# reference and comparison helpers (CPU)
# ------------------------------------------------------------------------------------------------
def vote_offset(o):
    """(dx, dy, dt, ds) of vote o in the device's (dx<<3)|(dy<<2)|(dt<<1)|ds layout = the reference's loop order."""
    return np.array([(o >> 3) & 1, (o >> 2) & 1, (o >> 1) & 1, o & 1], np.int64)


def reference_hough(scene, match_q, match_t, bins=BINS, pose=None):
    """Main.apply_hough_transform as whole-array numpy, one entry per (group, code), sorted by key
    = group * bins^4 + code: vote count, members ascending (the reference's append order), insertion-order
    key min(match_id * 16 + o) and the six running means (mean * j + v) / (j + 1) in member order.
    pose: [M,4] poses to average instead of the vectorised ones (numpy's cos / sin)."""
    pose_v, base = O.hough_base_bins_vectorized(scene, match_q, match_t, bins)
    pose = pose_v if pose is None else np.asarray(pose, np.float64)
    n = len(match_q)
    img = scene.m_image[np.asarray(match_t, np.int64)]
    group = np.zeros(n, np.int64) if scene.img_group is None else scene.img_group[img].astype(np.int64)
    nb4 = bins ** 4
    assert (int(group.max()) + 1) * nb4 * n * 16 < 2 ** 62
    comp = []
    for o in range(16):
        p = base.astype(np.int64) + vote_offset(o)
        ok = np.flatnonzero((p < bins).all(1))
        code = ((p[ok, 0] * bins + p[ok, 1]) * bins + p[ok, 2]) * bins + p[ok, 3]
        comp.append(((group[ok] * nb4 + code) * n + ok) * 16 + o)
    comp = np.sort(np.concatenate(comp))          # by bin key, then match id
    off = comp % 16
    mid = comp // 16 % n
    key = comp // 16 // n
    del comp
    ukey, start, count = np.unique(key, return_index=True, return_counts=True)
    vals = np.concatenate([pose, scene.img_size[img]], 1)[mid]      # [votes, 6] in member order
    # running means, vectorised over the bins one member position at a time
    by = np.argsort(-count, kind="stable")
    c_sorted, s_sorted = count[by], start[by]
    mean = vals[s_sorted].copy()
    n_active = np.searchsorted(-c_sorted, -np.arange(int(c_sorted[0])), side="left")  # bins with count > j
    for j in range(1, int(c_sorted[0])):
        na = n_active[j]
        mean[:na] = (mean[:na] * j + vals[s_sorted[:na] + j]) / (j + 1)
    means = np.empty_like(mean)
    means[by] = mean
    return dict(base=base, pose=pose_v, group_of=group, key=ukey, group=ukey // nb4, code=ukey % nb4, count=count,
                offset=start, members=mid.astype(np.int64), order_key=mid[start] * 16 + off[start], mean=means)


def _segments(count):
    """Position of every element of consecutive segments of these lengths inside its segment."""
    count = np.asarray(count, np.int64)
    return np.arange(int(count.sum())) - np.repeat(np.cumsum(count) - count, count)


def assert_hough_equal(h, ref, bins=BINS, detail_min=1, mean_rows=None):
    """A device result (HoughResult.host()) equals the reference: the same (group, code) -> count map and,
    for every bin of at least detail_min votes, the same members, order key and means (records are
    compared by (group, code), never by record index: the kernels write them in atomic order).
    mean_rows: indices into the reference's bins whose means are compared (default: all detailed)."""
    got_key = h["group"].astype(np.int64) * bins ** 4 + h["code"].astype(np.int64)
    srt = np.argsort(got_key, kind="stable")
    np.testing.assert_array_equal(got_key[srt], ref["key"], err_msg="bin keys differ")
    np.testing.assert_array_equal(h["count"][srt], ref["count"], err_msg="vote counts differ")
    assert h["n_votes"] == int(ref["count"].sum())
    d = np.flatnonzero(ref["count"] >= detail_min)
    cnt = ref["count"][d]
    pos = _segments(cnt)
    got = h["members"][np.repeat(h["offset"][srt][d].astype(np.int64), cnt) + pos]
    want = ref["members"][np.repeat(ref["offset"][d], cnt) + pos]
    bad = np.flatnonzero(got != want)
    assert len(bad) == 0, f"members differ at {len(bad)} positions, first in bin key {ref['key'][d][np.searchsorted(np.cumsum(cnt), bad[0], side='right')]}"
    np.testing.assert_array_equal(h["order_key"][srt][d], ref["order_key"][d], err_msg="insertion-order keys differ")
    rows = d if mean_rows is None else np.asarray(mean_rows)
    np.testing.assert_allclose(h["mean"][srt][rows], ref["mean"][rows], rtol=1e-12, atol=1e-9, err_msg="means differ")


def host_view(ref, rng):
    """The reference in the layout of HoughResult.host(), records in a shuffled order (what a correct device
    result looks like); the CPU test perturbs it to show that assert_hough_equal notices."""
    p = rng.permutation(len(ref["key"]))
    return dict(group=ref["group"][p].astype(np.int32), code=ref["code"][p].astype(np.int32),
                count=ref["count"][p].astype(np.int32), offset=ref["offset"][p].astype(np.int32),
                order_key=ref["order_key"][p].copy(), mean=ref["mean"][p].copy(),
                members=ref["members"].astype(np.int32), n_votes=int(ref["count"].sum()))


def oracle_affine(scene, bins_spec, threshold=4):
    """O.affine_verify on explicit bins [(member ids, isigma)]: per bin (live, votes, keep mask, params)."""
    objs = []
    for mem, isg in bins_spec:
        b = O.Bin(0, (0, 0, 0, int(isg)), (0.0, 0.0), int(mem[0]), (0.0, 0.0, 0.0, 0.0))
        b.members = [int(m) for m in mem]
        b.votes = len(b.members)
        objs.append(b)
    live = {id(b) for b in O.affine_verify(scene, np.arange(len(scene.q_xy)), np.arange(len(scene.q_xy)), objs,
                                           threshold)}
    out = []
    for (mem, _), b in zip(bins_spec, objs):
        out.append((id(b) in live, b.votes, np.isin(mem, b.members), np.asarray(b.affine, np.float64)))
    return out


def assert_affine_equal(got, want):
    """got / want: per bin (live, votes, keep mask, params).  live, votes and the keep mask exactly, the
    parameters within 1e-9 relative to the bin's largest parameter."""
    assert len(got) == len(want)
    for i, ((gl, gv, gk, gp), (wl, wv, wk, wp)) in enumerate(zip(got, want)):
        assert (bool(gl), int(gv)) == (bool(wl), int(wv)), f"bin {i}: (live, votes) {(gl, gv)} != {(wl, wv)}"
        np.testing.assert_array_equal(np.asarray(gk, bool), wk, err_msg=f"bin {i}: member_keep differs")
        np.testing.assert_allclose(gp, wp, rtol=1e-9, atol=1e-9 * np.abs(wp).max(), err_msg=f"bin {i}: params")


# ------------------------------------------------------------------------------------------------
# scenes with controlled bin sizes
# ------------------------------------------------------------------------------------------------
def cell_scene(rng, cell, space, n_spaces=1, width=W, height=H, bins=BINS, spread=0.3):
    """Match i (query keypoint i <-> model keypoint i) gets a pose inside base bin cell[i] = (ix, iy, it, is),
    within `spread` bin widths of its middle, in Hough space space[i] (one model image per space).
    k matches of one cell vote k times into each of the cell's (up to) 16 bins; cells at least two apart in
    some dimension share no bin.  Poses stay far from every truncation edge, so numpy's cos / sin give the
    same bins as any libm."""
    cell = np.asarray(cell, np.int64)
    img = np.asarray(space, np.int32)
    n = len(cell)
    assert np.isin(cell[:, 3], SIGMAS).all()
    cent = np.stack([rng.uniform(300, 1200, n_spaces), rng.uniform(200, 800, n_spaces)], 1)
    size = np.stack([rng.integers(1000, 2000, n_spaces), rng.integers(700, 1300, n_spaces)], 1).astype(np.float64)
    m_xy = np.stack([rng.uniform(0, 1500, n), rng.uniform(0, 1000, n)], 1).astype(np.float32)
    m_ang = rng.uniform(0, 360, n).astype(np.float32)
    m_oct = rng.integers(-1, 2, n)
    k = np.array([K_OF_SIGMA[int(s)] for s in SIGMAS])[np.searchsorted(SIGMAS, cell[:, 3])]
    deg = (cell[:, 2] + 0.5 + rng.uniform(-spread, spread, n)) * (360.0 / bins)
    q_ang = np.mod(m_ang.astype(np.float64) + deg, 360.0).astype(np.float32)
    q_ang[q_ang >= 360.0] = 0.0
    s = np.exp2(k.astype(np.float64))
    tx = (cent[img, 0] - m_xy[:, 0].astype(np.float64)) * s
    ty = (cent[img, 1] - m_xy[:, 1].astype(np.float64)) * s
    a = np.mod((q_ang.astype(np.float64) - m_ang.astype(np.float64)) * (math.pi / 180.0) + 2 * math.pi, 2 * math.pi)
    x = (cell[:, 0] + 1.5 + rng.uniform(-spread, spread, n)) * width / bins     # int(x * bins / W) - 1 = ix
    y = (cell[:, 1] + 1.5 + rng.uniform(-spread, spread, n)) * height / bins
    q_xy = np.stack([x - (np.cos(a) * tx - np.sin(a) * ty), y - (np.sin(a) * tx + np.cos(a) * ty)], 1)
    one = np.ones(n, np.int64)
    sc = O.Scene(q_xy.astype(np.float32), q_ang, scenes.pack_octave(m_oct + k, one), m_xy, m_ang,
                 scenes.pack_octave(m_oct, one), img, cent, size, width, height,
                 np.arange(n_spaces, dtype=np.int32) if n_spaces > 1 else None)
    pose, base = O.hough_base_bins_vectorized(sc, np.arange(n), np.arange(n), bins)
    np.testing.assert_array_equal(base, cell)
    for f in (pose[:, 0] * bins / width, pose[:, 1] * bins / height, pose[:, 2] * bins / (2 * math.pi)):
        assert np.abs(f - np.rint(f)).min() > 0.4 - spread  # far from every truncation edge
    return sc


def lattice_cells(rng, k, sigmas=(2, 4, 6, 9, 11, 13)):
    """k distinct cells with even ix, iy, it and sigma bins two apart: no two share a bin."""
    ev = np.arange(0, BINS, 2)
    all_cells = np.stack(np.meshgrid(ev, ev, ev, np.asarray(sigmas), indexing="ij"), -1).reshape(-1, 4)
    return all_cells[rng.choice(len(all_cells), k, replace=False)]


def scattered_cells(rng, k, avoid=None):
    """k random cells; with `avoid`, none shares a bin with any of those cells."""
    out = np.empty((0, 4), np.int64)
    while len(out) < k:
        c = np.concatenate([rng.integers(0, BINS, (2 * k, 3)), rng.choice(SIGMAS, (2 * k, 1))], 1)
        if avoid is not None:
            for r in np.asarray(avoid):
                c = c[np.abs(c - r).max(1) > 1]
        out = np.concatenate([out, c])
    return out[:k]


def finish_scene(rng, n_spaces=1, spread=0.3):
    """Bins of exactly 1, 2, 16, 17, 1,024 and 1,025 votes (each size from one isolated cell, whose bins all
    hold that many votes; the first cell sits at ix = 14, where half its votes fall off the grid); match ids
    interleave the cells.  Over two spaces, sizes 1, 16, 1,024 go to space 0 and 2, 17, 1,025 to space 1, at
    the same three cells: equal bin codes in both spaces."""
    cells = lattice_cells(rng, len(FINISH_SIZES))
    cells[0, 0] = BINS - 1
    if n_spaces == 2:
        cells[1::2] = cells[0::2]
    cell = np.concatenate([np.repeat(c[None], k, 0) for c, k in zip(cells, FINISH_SIZES)])
    space = np.concatenate([np.full(k, i % n_spaces) for i, k in enumerate(FINISH_SIZES)])
    perm = rng.permutation(len(cell))
    return cell_scene(rng, cell[perm], space[perm], n_spaces, spread=spread), len(cell)


def _device(sc):
    from sod_b200 import engine as E
    n_spaces = 1 if sc.img_group is None else len(sc.img_group)
    return E.SceneArrays(sc.q_xy, sc.q_angle, sc.q_octave, sc.m_xy, sc.m_angle, sc.m_octave, sc.m_image,
                         sc.img_centroid, sc.img_size, np.array([[sc.width, sc.height]], np.int32),
                         img_group=sc.img_group, groups_per_frame=n_spaces)


def _vote(sc, ref, detail_min_count=1, voter=None):
    """Hough-vote every match of the scene on the device; checks the poses' base bins first (a mismatch there
    is a pose bug, not a voting bug)."""
    import torch
    from sod_b200 import engine as E
    n = len(sc.q_xy)
    ids = torch.arange(n, dtype=torch.int32, device="cuda")
    voter = voter or E.HoughVoter(_device(sc), BINS)
    res = voter.vote(ids, ids, detail_min_count=detail_min_count)
    bb = res.base_bin[:n].cpu().numpy().view(np.uint32)
    np.testing.assert_array_equal(np.stack([(bb >> s) & 0xFF for s in (0, 8, 16, 24)], 1), ref["base"])
    h = res.host()
    assert h["n_near_edge"] == 0 and h["n_unresolved_edge"] == 0
    return h, res, voter


def _space_sizes(ref):
    return np.bincount(ref["group_of"])


# ------------------------------------------------------------------------------------------------
# CPU: the reference and the comparison helpers
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_spaces", [1, 2])
def test_reference_hough_equals_scalar_oracle(n_spaces):
    """reference_hough against O.hough_vote (held to the real reference by test_oracle_golden.py) on bins of
    every finish class: identical keys in insertion order, counts, members, order keys and - fed the scalar
    oracle's libm poses - bit-identical means."""
    sc, n = finish_scene(np.random.default_rng(11 + n_spaces), n_spaces)
    ids = np.arange(n)
    table = O.hough_vote(sc, ids, ids, BINS)
    pose = np.array([sc.pose_of(i, i) for i in range(n)])
    ref = reference_hough(sc, ids, ids, BINS, pose=pose)
    assert sorted(set(ref["count"].tolist())) == list(FINISH_SIZES)
    order = np.argsort(ref["order_key"])
    keys = [(int(g), *(int(v) for v in np.unravel_index(int(c), (BINS,) * 4)))
            for g, c in zip(ref["group"][order], ref["code"][order])]
    assert keys == list(table.keys())
    bins = list(table.values())
    assert ref["count"][order].tolist() == [b.votes for b in bins]
    for i, b in zip(order, bins):
        assert ref["members"][ref["offset"][i]:ref["offset"][i] + ref["count"][i]].tolist() == b.members
        assert ref["order_key"][i] // 16 == b.members[0]
    want = np.array([[b.centroid[0], b.centroid[1], b.angle, b.scale, *b.img_size] for b in bins])
    np.testing.assert_array_equal(ref["mean"][order], want)


def test_comparison_helpers_catch_perturbed_results():
    """The helpers accept a correct result in any record order and reject each way a finish or affine kernel
    could plausibly go wrong: two members swapped, the ids of a second bitmap window dropped, a bin's first
    member moved, one member_keep flag flipped."""
    rng = np.random.default_rng(5)
    sc, n = finish_scene(rng)
    ids = np.arange(n)
    ref = reference_hough(sc, ids, ids)
    spread = np.arange(n) * 1000                              # the same bins with match ids spanning 2 windows
    ref["members"] = spread[ref["members"]]
    ref["order_key"] = spread[ref["order_key"] // 16] * 16 + ref["order_key"] % 16
    huge = int(np.argmax(ref["count"]))
    mem = ref["members"][ref["offset"][huge]:ref["offset"][huge] + ref["count"][huge]]
    assert ref["count"][huge] > 1024 and mem[-1] - mem[0] >= WINDOW
    assert_hough_equal(host_view(ref, rng), ref)

    def fails(h):
        with pytest.raises(AssertionError):
            assert_hough_equal(h, ref)

    h = host_view(ref, rng)                                   # swap two members of the huge bin
    o = int(ref["offset"][huge])
    h["members"][[o + 3, o + 4]] = h["members"][[o + 4, o + 3]]
    fails(h)
    h = host_view(ref, rng)                                   # move a bin's first member to its end
    small = int(np.flatnonzero((ref["count"] > 2) & (ref["count"] <= 16))[0])
    o, c = int(ref["offset"][small]), int(ref["count"][small])
    h["members"][o:o + c] = np.roll(h["members"][o:o + c], -1)
    fails(h)
    h = host_view(ref, rng)                                   # the second window of the huge bin lost
    o = int(ref["offset"][huge])
    lost = o + np.flatnonzero(mem >= mem[0] + WINDOW)
    h["members"] = np.delete(h["members"], lost)
    r = h["code"] == ref["code"][huge]
    h["count"][r] -= len(lost)
    h["offset"][h["offset"] > o] -= len(lost)
    h["n_votes"] -= len(lost)
    fails(h)

    keep = np.ones(40, bool)
    keep[[3, 17]] = False
    want = [(True, 38, keep, np.array([1.0, 0.1, -0.1, 1.0, 500.0, 300.0]))]
    assert_affine_equal([(True, 38, keep.copy(), want[0][3] * (1 + 1e-12))], want)
    flipped = keep.copy()
    flipped[25] = False
    with pytest.raises(AssertionError):
        assert_affine_equal([(True, 38, flipped, want[0][3])], want)


# ------------------------------------------------------------------------------------------------
# GPU: Hough voting by size class
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n", [1024, 1025, 65535, 65536])
def test_single_space_of_n_matches(n):
    """One Hough space on both sides of the vote-kernel boundaries (<= 1,024 matches: one match per thread;
    <= 65,535: 16-bit arrival ranks; more: 32-bit).  All but 8 matches lie in the 16 cells around one bin, so
    that bin takes n - 8 votes: arrival ranks up to n - 9, the largest the space's format must hold."""
    rng = np.random.default_rng(n)
    block = np.array([6, 6, 6, 13]) + np.stack([vote_offset(o) for o in range(16)])
    cell = np.concatenate([np.repeat(block, [n - 8 - 120] + list(range(1, 16)), 0), scattered_cells(rng, 8, block)])
    cell = cell[rng.permutation(n)]
    sc = cell_scene(rng, cell, np.zeros(n, np.int32))
    ids = np.arange(n)
    ref = reference_hough(sc, ids, ids)
    assert _space_sizes(ref).tolist() == [n] and ref["count"].max() == n - 8
    h, _, _ = _vote(sc, ref)
    assert_hough_equal(h, ref)


@gpu
@pytest.mark.parametrize("n_spaces", [1, 2])
def test_finish_classes(n_spaces):
    """Bins of exactly 1, 2, 16, 17, 1,024 and 1,025 votes in one call: every finish kernel (none / thread /
    warp / CTA) on both sides of each of its boundaries, in one space and split over two."""
    sc, n = finish_scene(np.random.default_rng(21 + n_spaces), n_spaces)
    ids = np.arange(n)
    ref = reference_hough(sc, ids, ids)
    assert sorted(set(ref["count"].tolist())) == list(FINISH_SIZES)
    assert len(_space_sizes(ref)) == n_spaces
    h, _, _ = _vote(sc, ref)
    assert_hough_equal(h, ref)


@gpu
def test_detail_min_count_skips_only_small_bins():
    """detail_min_count 1, 2, 17 and 1,025 on the finish-class scene: the (group, code) -> count map never
    changes, and every bin of at least d votes keeps the members, means and order key of the d = 1 run and
    of the reference.  At d = 17 the thread kernel only queues bins for the warp and CTA kernels; at d =
    1,025 only the CTA kernel has work."""
    sc, n = finish_scene(np.random.default_rng(31))
    ids = np.arange(n)
    ref = reference_hough(sc, ids, ids)
    first, _, voter = _vote(sc, ref, 1)
    assert_hough_equal(first, ref)
    first_key = first["group"].astype(np.int64) * BINS ** 4 + first["code"]
    for d, detailed in ((2, {2, 16, 17, 1024, 1025}), (17, {17, 1024, 1025}), (1025, {1025})):
        assert set(ref["count"][ref["count"] >= d].tolist()) == detailed
        h, _, _ = _vote(sc, ref, d, voter)
        assert_hough_equal(h, ref, detail_min=d)
        key = h["group"].astype(np.int64) * BINS ** 4 + h["code"]
        a, b = np.argsort(first_key), np.argsort(key)
        np.testing.assert_array_equal(key[b], first_key[a])
        np.testing.assert_array_equal(h["count"][b], first["count"][a])
        big = first["count"][a] >= d
        np.testing.assert_array_equal(h["order_key"][b][big], first["order_key"][a][big])
        np.testing.assert_array_equal(h["mean"][b][big], first["mean"][a][big])
        for i, j in zip(b[big], a[big]):
            np.testing.assert_array_equal(h["members"][h["offset"][i]:h["offset"][i] + h["count"][i]],
                                          first["members"][first["offset"][j]:first["offset"][j] + first["count"][j]])


@gpu
def test_huge_bins_span_two_bitmap_windows():
    """More than 2^20 + 2 matches in two spaces.  Space A: 3,000 matches of one pose, whose ids span the whole
    range and include id_lo + 2^20 - 1 and id_lo + 2^20, the two sides of the first window edge of the CTA
    finish's bitmap sort.  Space B: everything else (> 65,535 matches: 32-bit ranks), one pose of 120,000
    matches (ranks past 16 bits) among uniformly scattered ones."""
    rng = np.random.default_rng(41)
    n = WINDOW + 40_000
    lo = 7
    a_ids = np.unique(np.concatenate([[lo, lo + WINDOW - 1, lo + WINDOW, n - 1],
                                      rng.choice(np.arange(lo + 1, n - 1), 2996, replace=False)]))
    space = np.ones(n, np.int32)
    space[a_ids] = 0
    cell = scattered_cells(rng, n)
    cell[a_ids] = lattice_cells(rng, 1)[0]
    b_ids = np.flatnonzero(space == 1)
    cell[rng.choice(b_ids, 120_000, replace=False)] = lattice_cells(rng, 1)[0]
    sc = cell_scene(rng, cell, space, 2)
    ids = np.arange(n)
    ref = reference_hough(sc, ids, ids)
    assert n > WINDOW + 2 and _space_sizes(ref)[1] > 65535 and ref["count"].max() > 65536
    in_a = ref["group"] == 0
    assert (ref["count"][in_a] == len(a_ids)).all() and len(a_ids) > 1024
    assert a_ids[0] == lo and {lo + WINDOW - 1, lo + WINDOW} <= set(a_ids.tolist())
    h, _, _ = _vote(sc, ref)
    sample = np.sort(np.concatenate([np.flatnonzero(in_a | (ref["count"] > 1024)),
                                     rng.choice(len(ref["key"]), 2000, replace=False)]))
    assert_hough_equal(h, ref, mean_rows=np.unique(sample))
    # space A against the scalar oracle, mapped back to match ids
    table = O.hough_vote(sc, a_ids, a_ids, BINS)
    ga = np.flatnonzero(h["group"] == 0)                          # host order = insertion order
    assert [(0, *np.unravel_index(int(c), (BINS,) * 4)) for c in h["code"][ga]] == list(table.keys())
    for i, b in zip(ga, table.values()):
        np.testing.assert_array_equal(h["members"][h["offset"][i]:h["offset"][i] + h["count"][i]], a_ids[b.members])
        np.testing.assert_allclose(h["mean"][i], [b.centroid[0], b.centroid[1], b.angle, b.scale, *b.img_size],
                                   rtol=1e-12, atol=1e-9)


def _sub_shift(n_spaces):
    """group_sub_shift (sod_hough.cu): log2 of the sub-counters per space, up to 16, within 65,536 in all."""
    s = 0
    while s < 4 and (n_spaces << (s + 1)) <= 65536:
        s += 1
    return s


@gpu
@pytest.mark.parametrize("n_spaces, shift, grid_scan", [(1, 4, False), (1024, 4, False), (1025, 4, True),
                                                        (4096, 4, True), (4097, 3, True), (70_000, 0, True)])
def test_number_of_spaces(n_spaces, shift, grid_scan):
    """One model image per space: one-launch vs three-launch scan of the sub-counters (more than 2 x 8,192),
    16 sub-counters per space down to 8 from 4,097 spaces and 1 from 32,769.  Most spaces hold 0-5 matches,
    space 0 holds 1,100 (the general vote form next to the one-match-per-thread one); matches arrive in
    random order, so every space's matches spread over many sub-lists."""
    rng = np.random.default_rng(n_spaces)
    per = rng.choice([0, 1, 2, 3, 5], n_spaces) if n_spaces > 1 else np.array([3000])
    per[0] = max(per[0], 1100)
    space = np.repeat(np.arange(n_spaces, dtype=np.int32), per)
    space = space[rng.permutation(len(space))]
    n = len(space)
    sc = cell_scene(rng, scattered_cells(rng, n), space, n_spaces)
    ids = np.arange(n)
    ref = reference_hough(sc, ids, ids)
    assert _sub_shift(n_spaces) == shift and ((n_spaces << shift) > 2 * 8192) == grid_scan
    assert len(_space_sizes(ref)) == n_spaces and _space_sizes(ref)[0] > 1024
    keys, counts = O.vote_counts_vectorized(ref["base"], ref["group_of"], BINS)
    np.testing.assert_array_equal(keys, ref["key"])
    np.testing.assert_array_equal(counts, ref["count"])
    h, _, _ = _vote(sc, ref)
    assert_hough_equal(h, ref)


# ------------------------------------------------------------------------------------------------
# GPU: affine verification by size class
# ------------------------------------------------------------------------------------------------
AFFINE_SIZES = (5, 16, 17, 32, 33, 512, 513, 3000)   # thread kernel (16 staged) / warp kernel (512 staged)
AW, AH = 1500, 1000


def affine_scene(rng, sizes=AFFINE_SIZES):
    """Explicit bins of the given sizes: inliers under a random similarity with noise below a quarter of the
    residual limit W * isigma / 128 (H for v), in bins of more than 32 pairs 10 % outliers 12-20 limits
    off and 10 % 4-6 limits off along one axis, in smaller ones one 4-6 limits off (each bin needs a second
    pass to see that nothing more goes),
    and a last bin of 5 pairs, 2 of them far off, that ends below the affine threshold."""
    bins, m_all, q_all = [], [], []
    base = 0
    for k in list(sizes) + [5]:
        isg = int(rng.integers(3, 9))
        lim = np.array([AW, AH]) * isg / 128.0
        th, s = rng.uniform(0, 2 * math.pi), rng.uniform(0.5, 2.0)
        rot = s * np.array([[math.cos(th), -math.sin(th)], [math.sin(th), math.cos(th)]])
        m = np.stack([rng.uniform(0, 1500, k), rng.uniform(0, 1000, k)], 1)
        q = m @ rot.T + rng.uniform(200, 1200, 2) + rng.uniform(-0.24, 0.24, (k, 2)) * lim
        last = len(bins) == len(sizes)
        n_far = 2 if last else (0 if k <= 33 else k // 10)
        n_near = 0 if last else (1 if k <= 33 else k // 10)
        out = rng.choice(k, n_far + n_near, replace=False)
        axis = rng.integers(0, 2, len(out))
        mag = np.where(np.arange(len(out)) < n_far, rng.uniform(12, 20, len(out)), rng.uniform(4, 6, len(out)))
        q[out, axis] += rng.choice([-1, 1], len(out)) * mag * lim[axis]
        bins.append((np.arange(base, base + k), isg))
        m_all.append(m)
        q_all.append(q)
        base += k
    m_xy = np.concatenate(m_all).astype(np.float32)
    q_xy = np.concatenate(q_all).astype(np.float32)
    z = np.zeros(base, np.float32)
    zi = np.zeros(base, np.int32)
    scene = O.Scene(q_xy, z, zi, m_xy, z, zi, zi, np.zeros((1, 2)), np.zeros((1, 2)), AW, AH)
    return scene, bins


def test_affine_scene_lands_in_its_classes():
    """CPU: the affine scene's bins need more than one pass, the last one dies, the others survive."""
    scene, spec = affine_scene(np.random.default_rng(55))
    want = oracle_affine(scene, spec)
    assert [len(m) for m, _ in spec] == list(AFFINE_SIZES) + [5]
    assert [w[0] for w in want] == [True] * len(AFFINE_SIZES) + [False]
    assert all(w[1] < len(m) for w, (m, _) in zip(want, spec))     # every bin lost pairs


@gpu
def test_affine_by_size_class():
    """Bins of 5, 16, 17, 32, 33, 512, 513 and 3,000 pairs through dropin._PairBatch: both affine kernels on
    both sides of their stage sizes, fit / prune until nothing changes, against O.affine_verify: live, votes
    and member_keep exactly, parameters within 1e-9; no residual on the edge of its limit, no singular fit."""
    import cv2
    from PoseBin import PoseBin
    from sod_b200 import dropin, engine as E
    scene, spec = affine_scene(np.random.default_rng(55))
    want = oracle_affine(scene, spec)
    kp = lambda p: cv2.KeyPoint(float(p[0]), float(p[1]), 1.0)  # noqa: E731
    bins = [PoseBin((0, 0, 0, isg), (1500, 1000), len(mem), [(kp(scene.m_xy[i]), kp(scene.q_xy[i])) for i in mem],
                    (0.0, 0.0, 0.0, 1.0)) for mem, isg in spec]
    batch = dropin._PairBatch(bins, AW, AH)
    a = E.affine_verify(batch.scene, batch.ids, batch.ids, batch.h, vote_threshold=0, affine_threshold=4,
                        factor=128.0, factor_y=128.0).host(batch.total)
    assert a["n_residual_edge"] == 0 and a["n_singular"] == 0
    pos = np.empty(len(spec), np.int64)
    pos[a["valid_bin"]] = np.arange(len(spec))
    got = [(a["live"][p], a["votes"][p], a["member_keep"][mem], a["params"][p]) for p, (mem, _) in zip(pos, spec)]
    assert_affine_equal(got, want)
    assert (a["passes"][pos][:-1] >= 2).all()


@gpu
def test_affine_after_voting_with_bins_past_the_stage():
    """HoughVoter -> affine_verify on the finish-class scene: bins of 1,024 and 1,025 votes reach the warp
    affine kernel past its 512-pair stage in the order the finish kernels sorted them; against the scalar
    oracle's hough_vote -> valid_bins -> affine_verify."""
    from sod_b200 import engine as E
    import torch
    sc, n = finish_scene(np.random.default_rng(61), spread=0.02)
    ids = np.arange(n)
    ref = reference_hough(sc, ids, ids)
    h, res, _ = _vote(sc, ref)
    dids = torch.arange(n, dtype=torch.int32, device="cuda")
    a = E.affine_verify(_device(sc), dids, dids, res, 5, 4).host(h["n_votes"])
    assert a["n_residual_edge"] == 0 and a["n_singular"] == 0
    table = O.hough_vote(sc, ids, ids, BINS)
    valid = O.valid_bins(table, 5)
    assert max(b.votes for b in valid) > 512
    spec = [(np.array(b.members), b.pose[3]) for b in valid]
    want = oracle_affine(sc, spec)
    row = {int(r): i for i, r in enumerate(h["rec"])}
    lut = {(int(g), int(c)): i for i, (g, c) in enumerate(zip(h["group"], h["code"]))}
    assert a["n_valid"] == len(valid)
    got = [None] * len(valid)
    for v, rec in enumerate(a["valid_bin"]):
        i = row[int(rec)]
        key = (int(h["group"][i]), *np.unravel_index(int(h["code"][i]), (BINS,) * 4))
        j = [k for k, b in enumerate(valid) if (b.group, *b.pose) == key][0]
        assert lut[(key[0], int(h["code"][i]))] == i
        sl = slice(h["offset"][i], h["offset"][i] + h["count"][i])
        np.testing.assert_array_equal(h["members"][sl], spec[j][0])
        got[j] = (a["live"][v], a["votes"][v], a["member_keep"][sl], a["params"][v])
    assert_affine_equal(got, want)
