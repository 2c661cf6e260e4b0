"""GPU parity of the Hough voting and affine verification kernels against the golden fixtures (real
reference outputs) and against the oracle on larger seeded inputs."""
from pathlib import Path

import numpy as np
import pytest
import torch

import scenes
from oracle import sod_oracle as O

pytestmark = pytest.mark.gpu
GOLD = Path(__file__).resolve().parent / "golden"


def _scene_arrays(src, prefix="in_", groups=False):
    from sod_b200 import engine as E
    g = (lambda k: src[prefix + k])
    img_group = src["img_group"] if groups else None
    gpf = int(np.max(img_group)) + 1 if groups else 1
    return E.SceneArrays(g("q_xy"), g("q_angle"), g("q_octave"), g("m_xy"), g("m_angle"), g("m_octave"),
                         g("m_image"), g("img_centroid"), np.asarray(g("img_size"), np.float64),
                         np.array([[int(g("width")), int(g("height"))]], np.int32),
                         img_group=img_group, groups_per_frame=gpf)


def _decode(code, bins):
    out = np.zeros((len(code), 4), np.int64)
    c = code.astype(np.int64).copy()
    for d in (3, 2, 1, 0):
        out[:, d] = c % bins
        c //= bins
    return out


@pytest.mark.parametrize("name", ["scene_single", "scene_multi", "scene_tiny", "scene_c1"])
def test_hough_matches_reference_golden(name):
    from sod_b200 import engine as E
    z = np.load(GOLD / f"{name}.npz")
    bins = int(z["bins"])
    sc = _scene_arrays(z)
    mq = torch.from_numpy(z["match_q"]).cuda()
    mt = torch.from_numpy(z["match_t"]).cuda()
    res = E.HoughVoter(sc, bins).vote(mq, mt)
    h = res.host()
    assert h["n_near_edge"] == 0
    # bins in reference dict insertion order, votes and members bit-exact
    np.testing.assert_array_equal(_decode(h["code"], bins), z["bin_keys"])
    np.testing.assert_array_equal(h["count"], z["bin_votes"])
    goff = z["bin_mem_off"]
    for i in range(h["n_bins"]):
        mem = h["members"][h["offset"][i]:h["offset"][i] + h["count"][i]]
        pairs = z["bin_mem"][goff[i]:goff[i + 1]]
        np.testing.assert_array_equal(z["match_q"][mem], pairs[:, 0])
        np.testing.assert_array_equal(z["match_t"][mem], pairs[:, 1])
    # running means: same recurrence; cos/sin may differ from libm in the last bit
    np.testing.assert_allclose(h["mean"], z["bin_means"], rtol=1e-12, atol=1e-9)
    # poses against the oracle's libm evaluation
    scene = O.Scene(z["in_q_xy"], z["in_q_angle"], z["in_q_octave"], z["in_m_xy"], z["in_m_angle"],
                    z["in_m_octave"], z["in_m_image"], z["in_img_centroid"], z["in_img_size"],
                    int(z["in_width"]), int(z["in_height"]))
    want = np.array([scene.pose_of(int(a), int(b)) for a, b in zip(z["match_q"], z["match_t"])])
    np.testing.assert_allclose(res.pose[:len(want)].cpu().numpy(), want, rtol=1e-13, atol=1e-10)


@pytest.mark.parametrize("name", ["scene_single", "scene_multi", "scene_tiny", "scene_c1"])
def test_affine_matches_reference_golden(name):
    from sod_b200 import engine as E
    z = np.load(GOLD / f"{name}.npz")
    bins = int(z["bins"])
    sc = _scene_arrays(z)
    mq = torch.from_numpy(z["match_q"]).cuda()
    mt = torch.from_numpy(z["match_t"]).cuda()
    res = E.HoughVoter(sc, bins).vote(mq, mt)
    aff = E.affine_verify(sc, mq, mt, res, int(z["vote_thr"]), int(z["affine_thr"]))
    h = res.host()
    a = aff.host(h["n_votes"])
    # valid bins (votes >= threshold) in reference order
    rec_pos = {int(r): i for i, r in enumerate(h["rec"])}
    pos = np.array([rec_pos[int(r)] for r in a["valid_bin"]])
    order = np.argsort(pos)
    keys = _decode(h["code"][pos[order]], bins)
    np.testing.assert_array_equal(keys, z["valid_keys"])
    live = a["live"][order]
    np.testing.assert_array_equal(keys[live], z["live_keys"])
    np.testing.assert_array_equal(a["votes"][order][live], z["live_votes"])
    # affine parameters within 1e-4 relative (north star), in practice ~1e-9
    got = a["params"][order][live]
    np.testing.assert_allclose(got, z["live_params"], rtol=1e-4, atol=1e-6)
    assert np.abs(got - z["live_params"]).max() < 1e-6 * max(1.0, np.abs(z["live_params"]).max())
    # surviving members identical
    goff = z["live_mem_off"]
    li = 0
    for j in order:
        if not a["live"][j]:
            continue
        i = pos[j]
        sl = slice(h["offset"][i], h["offset"][i] + h["count"][i])
        mem = h["members"][sl][a["member_keep"][sl]]
        pairs = z["live_mem"][goff[li]:goff[li + 1]]
        np.testing.assert_array_equal(z["match_q"][mem], pairs[:, 0])
        np.testing.assert_array_equal(z["match_t"][mem], pairs[:, 1])
        li += 1
    assert li == len(z["live_keys"])


def test_multi_group_bin_counts_vs_oracle_stress():
    """SURVEY C5 shape at reduced size: per-object Hough spaces, 90 % outliers; bin -> votes must be
    identical to the oracle's vectorised restatement (itself checked against the scalar one)."""
    from sod_b200 import engine as E
    d = scenes.make_match_stress(103, n_objects=40, per_object=1500)
    bins = 15
    sc = _scene_arrays(d, prefix="", groups=True)
    mq = torch.from_numpy(d["match_q"]).cuda()
    mt = torch.from_numpy(d["match_t"]).cuda()
    res = E.HoughVoter(sc, bins).vote(mq, mt)
    h = res.host()
    osc = O.Scene(d["q_xy"], d["q_angle"], d["q_octave"], d["m_xy"], d["m_angle"], d["m_octave"], d["m_image"],
                  d["img_centroid"], d["img_size"], d["width"], d["height"], d["img_group"])
    _, base = O.hough_base_bins_vectorized(osc, d["match_q"], d["match_t"], bins)
    bb = res.base_bin.cpu().numpy().view(np.uint32)[:len(base)]
    np.testing.assert_array_equal(np.stack([(bb >> s) & 0xFF for s in (0, 8, 16, 24)], 1), base)
    keys, counts = O.vote_counts_vectorized(base, d["img_group"][d["m_image"][d["match_t"]]], bins)
    got = h["group"].astype(np.int64) * bins ** 4 + h["code"]
    o = np.argsort(got)
    np.testing.assert_array_equal(got[o], keys)
    np.testing.assert_array_equal(h["count"][o], counts)
    assert h["n_votes"] == counts.sum()
    # scalar oracle on a sample of groups: members and means
    grp = d["img_group"][d["m_image"][d["match_t"]]]
    sel = np.nonzero(np.isin(grp, [0, 17, 39]))[0]
    table = O.hough_vote(osc, d["match_q"][sel], d["match_t"][sel], bins)
    lut = {(int(g), int(c)): i for i, (g, c) in enumerate(zip(h["group"], h["code"]))}
    for key, b in table.items():
        code = ((key[1] * bins + key[2]) * bins + key[3]) * bins + key[4]
        i = lut[(key[0], code)]
        mem = h["members"][h["offset"][i]:h["offset"][i] + h["count"][i]]
        np.testing.assert_array_equal(mem, sel[b.members])
        np.testing.assert_allclose(h["mean"][i], [b.centroid[0], b.centroid[1], b.angle, b.scale, *b.img_size],
                                   rtol=1e-12, atol=1e-9)


def test_compact_matches_is_stable():
    from sod_b200 import engine as E
    rng = np.random.default_rng(2)
    for nq in (1, 31, 1024, 1025, 70001):
        ok = (rng.random(nq) < 0.3).astype(np.uint8)
        idx = rng.integers(0, 10 ** 6, (nq, 2)).astype(np.int32)
        mq, mt, n = E.compact_matches(torch.from_numpy(idx).cuda(), torch.from_numpy(ok).cuda())
        k = int(n.item())
        want = np.nonzero(ok)[0]
        assert k == len(want)
        np.testing.assert_array_equal(mq[:k].cpu().numpy(), want)
        np.testing.assert_array_equal(mt[:k].cpu().numpy(), idx[want, 0])


def test_bins_above_limit_is_rejected_loudly():
    from sod_b200 import _capi
    from sod_b200 import engine as E
    z = np.load(GOLD / "scene_tiny.npz")
    with pytest.raises(_capi.SodError):
        E.HoughVoter(_scene_arrays(z), 16)


@pytest.mark.parametrize("dims", [(15, 12, 10, 6), (9, 15, 15, 15), (25, 25, 9, 9), (1, 1, 1, 1)])
def test_per_dimension_bin_counts_vs_oracle(dims):
    """sod_hough_vote_dims (legacy perform_hough_transform signature): keys in insertion order,
    votes, members and means against the oracle's per-dimension restatement."""
    from sod_b200 import engine as E
    z = np.load(GOLD / "scene_multi.npz")
    sc = _scene_arrays(z)
    mq = torch.from_numpy(z["match_q"]).cuda()
    mt = torch.from_numpy(z["match_t"]).cuda()
    res = E.HoughVoter(sc, dims).vote(mq, mt)
    h = res.host()
    scene = O.Scene(z["in_q_xy"], z["in_q_angle"], z["in_q_octave"], z["in_m_xy"], z["in_m_angle"],
                    z["in_m_octave"], z["in_m_image"], z["in_img_centroid"], z["in_img_size"],
                    int(z["in_width"]), int(z["in_height"]))
    table = O.hough_vote(scene, z["match_q"], z["match_t"], dims)
    _, by, bt, bs = dims
    code = h["code"].astype(np.int64)
    keys = np.stack([code // (by * bt * bs), code // (bt * bs) % by, code // bs % bt, code % bs], 1)
    assert [tuple(k) for k in keys.tolist()] == [k[1:] for k in table.keys()]
    assert h["count"].tolist() == [b.votes for b in table.values()]
    for i, b in enumerate(table.values()):
        mem = h["members"][h["offset"][i]:h["offset"][i] + h["count"][i]]
        assert mem.tolist() == b.members
    want_mean = np.array([[b.centroid[0], b.centroid[1], b.angle, b.scale] for b in table.values()])
    np.testing.assert_allclose(h["mean"][:, :4], want_mean, rtol=1e-12, atol=1e-9)
    # the affine stage decodes the sigma index with the sigma count
    aff = E.affine_verify(sc, mq, mt, res, 5, 4)
    live = O.affine_verify(scene, z["match_q"], z["match_t"], O.valid_bins(table, 5), 4)
    a = aff.host(h["n_votes"])
    assert int(a["live"].sum()) == len(live)


def test_too_many_counters_is_rejected_loudly():
    from sod_b200 import _capi, engine as E
    z = np.load(GOLD / "scene_tiny.npz")
    with pytest.raises(_capi.SodError):
        E.HoughVoter(_scene_arrays(z), (30, 30, 15, 15))


# ------------------------------------------------------------------------------------------------
# round 2: rank-deficient bins, edge cases of the truncations and of the residual test
# ------------------------------------------------------------------------------------------------
def _pair_batch(z):
    """The fixture's bins as the degenerate Hough output the drop-in uses for caller-built PoseBins."""
    import cv2
    from PoseBin import PoseBin
    from sod_b200 import dropin
    kp = lambda p: cv2.KeyPoint(float(p[0]), float(p[1]), 1.0)  # noqa: E731
    off = z["off"]
    bins = []
    for b in range(len(z["names"])):
        pairs = [(kp(m), kp(q)) for m, q in zip(z["model"][off[b]:off[b + 1]], z["query"][off[b]:off[b + 1]])]
        bins.append(PoseBin((0, 0, 0, int(z["isigma"][b])), (1500, 1000), len(pairs), pairs, (0.0, 0.0, 0.0, 1.0)))
    return dropin._PairBatch(bins, int(z["width"]), int(z["height"])), bins


def _by_bin(a, n_bins):
    """AffineResult.host() rows re-ordered by bin record."""
    pos = np.empty(n_bins, np.int64)
    pos[a["valid_bin"]] = np.arange(len(a["valid_bin"]))
    return pos


def test_affine_rank_deficient_and_ill_conditioned_bins_equal_reference():
    """tests/golden/affine_singular.npz (the reference's own AffineParameters / apply_affine_parameters on
    bins with duplicate model locations, collinear points, cond(S) up to ~1e11, sizes at the threshold,
    sigma bin 0): identical survivor sets, votes and live flags; parameters within 1e-4 relative
    (north star) of numpy's pinv solution - minimum-norm on the rank-deficient bins (SURVEY Q11); the
    near-singular status bit marks exactly the bins whose normal matrix is rank deficient."""
    from sod_b200 import engine as E
    z = np.load(GOLD / "affine_singular.npz")
    batch, bins = _pair_batch(z)
    n = len(bins)
    off = z["off"]
    # one fit, no pruning (AffineParameters(posebin))
    res = E.affine_verify(batch.scene, batch.ids, batch.ids, batch.h, vote_threshold=0, affine_threshold=0,
                          factor=0.0, factor_y=0.0, max_passes=1)
    a = res.host(batch.total)
    pos = _by_bin(a, n)
    scale = np.abs(z["first_params"]).max(1, keepdims=True)
    err = np.abs(a["params"][pos] - z["first_params"]) / scale
    assert err.max() < 1e-4, (z["names"][err.max(1).argmax()], err.max())
    well = np.array([nm.startswith(("generic", "exactly", "outliers", "isigma", "near_collinear_0.01", "near_collinear_0.001"))
                     for nm in z["names"]])
    assert err[well].max() < 1e-9                       # well-conditioned bins agree far below the bar
    deficient = np.array([nm.startswith(("two_locations", "one_location", "collinear_")) for nm in z["names"]])
    np.testing.assert_array_equal(a["singular"][pos][deficient], True)
    np.testing.assert_array_equal(a["singular"][pos][well], False)
    assert a["n_singular"] == int(a["singular"].sum()) >= int(deficient.sum())
    # the whole fixed point (Main.apply_affine_parameters, factor 128 = pos_factor * 4)
    res = E.affine_verify(batch.scene, batch.ids, batch.ids, batch.h, vote_threshold=0,
                          affine_threshold=int(z["threshold"]), factor=128.0, factor_y=128.0)
    a = res.host(batch.total)
    pos = _by_bin(a, n)
    np.testing.assert_array_equal(a["live"][pos], z["live"])
    np.testing.assert_array_equal(a["votes"][pos], z["votes"])
    np.testing.assert_array_equal(a["member_keep"][:batch.total], z["keep"])
    err = np.abs(a["params"][pos] - z["last_params"]) / np.abs(z["last_params"]).max(1, keepdims=True)
    assert err.max() < 1e-4, (z["names"][err.max(1).argmax()], err.max())
    # the oracle on the same bins gives the same answer as the fixture (CPU test) - and as the device:
    for b in (int(np.flatnonzero(deficient)[0]), int(np.flatnonzero(deficient)[-1])):
        fit = np.asarray(O.affine_fit([tuple(map(float, r)) for r in z["model"][off[b]:off[b + 1]]],
                                      [tuple(map(float, r)) for r in z["query"][off[b]:off[b + 1]]]))
        np.testing.assert_array_equal(fit, z["first_params"][b])


def test_residual_decisions_on_the_edge_of_their_limit_are_counted():
    """Exact-fit bins with a limit of 0 px (sigma bin 0): residuals are rounding noise (~1e-13) against
    a limit of 0, the one situation in which a pair's fate depends on the last bits of the solver.
    The device counts those decisions (sod_affine_out.counters[3], status bit 2) instead of hiding them."""
    import cv2
    from PoseBin import PoseBin
    from sod_b200 import dropin, engine as E
    kp = lambda x, y: cv2.KeyPoint(float(x), float(y), 1.0)  # noqa: E731
    pts = [(0, 0), (100, 0), (0, 100), (100, 100), (50, 25), (20, 80)]
    exact = PoseBin((0, 0, 0, 0), (100, 100), 6, [(kp(x, y), kp(2 * x + 10, 2 * y - 5)) for x, y in pts], (0, 0, 0, 1))
    rng = np.random.default_rng(3)
    noisy = PoseBin((0, 0, 0, 2), (100, 100), 6, [(kp(x, y), kp(2 * x + 10 + rng.normal(), 2 * y - 5 + rng.normal()))
                                                  for x, y in pts], (0, 0, 0, 1))
    batch = dropin._PairBatch([exact, noisy], 1280, 960)
    a = E.affine_verify(batch.scene, batch.ids, batch.ids, batch.h, vote_threshold=0, affine_threshold=4,
                        factor=128.0, factor_y=128.0).host(batch.total)
    pos = _by_bin(a, 2)
    assert a["residual_edge"][pos].tolist() == [True, False]
    assert a["n_residual_edge"] >= 6
    assert a["live"][pos][1] and a["votes"][pos][1] == 6


def _boundary_scene(seed=9, n=600, width=1500, height=900, bins=15):
    """Matches whose pose lands EXACTLY on bin boundaries: equal angles (alpha = 0: cos = 1, sin = 0 on
    every libm) and integer coordinates chosen so that x * bins / W and y * bins / H are integers, among
    generic matches, plus generic-angle matches nudged to within ~1e-7 of a boundary (the query x is a
    float32, so that is the closest a real keypoint gets)."""
    rng = np.random.default_rng(seed)
    cent = np.array([[50.0, 40.0]])
    m_xy = rng.integers(0, 100, (n, 2)).astype(np.float32)
    m_angle = rng.uniform(0, 360, n).astype(np.float32)
    m_oct = np.zeros(n, np.int64)
    q_oct = rng.integers(0, 2, n)
    q_angle = m_angle.copy()
    q_xy = np.zeros((n, 2), np.float32)
    s = 2.0 ** (q_oct - m_oct)
    tx, ty = (cent[0, 0] - m_xy[:, 0]) * s, (cent[0, 1] - m_xy[:, 1]) * s
    bx = rng.integers(-1, bins + 1, n) * (width // bins)          # includes x < 0 and x = W (SURVEY Q2/Q3)
    by = rng.integers(-1, bins + 1, n) * (height // bins)
    q_xy[:, 0], q_xy[:, 1] = bx - tx, by - ty                     # alpha = 0: x = tx + qx exactly
    generic = rng.random(n) < 0.4
    q_angle[generic] = rng.uniform(0, 360, int(generic.sum())).astype(np.float32)
    q_xy[generic] = np.stack([rng.uniform(0, width, int(generic.sum())), rng.uniform(0, height, int(generic.sum()))], 1)
    scene = O.Scene(q_xy, q_angle, scenes.pack_octave(q_oct, np.ones(n, np.int64)), m_xy, m_angle,
                    scenes.pack_octave(m_oct, np.ones(n, np.int64)), np.zeros(n, np.int32), cent,
                    np.array([[100, 80]]), width, height)
    # generic-angle matches moved next to a boundary: pick the float32 qx that brings x closest to k * W / bins
    near = np.flatnonzero(generic)[:150]
    for i in near:
        x, y, _, _ = scene.pose_of(int(i), int(i))
        target = round(x / (width / bins)) * (width / bins)
        best = np.float32(scene.q_xy[i, 0] + (target - x))
        cands = [np.nextafter(best, np.float32(-1e9)), best, np.nextafter(best, np.float32(1e9))]
        errs = []
        for c in cands:
            scene.q_xy[i, 0] = c
            errs.append(abs(scene.pose_of(int(i), int(i))[0] - target))
        scene.q_xy[i, 0] = cands[int(np.argmin(errs))]
    return scene, n


def test_matches_on_bin_boundaries_are_resolved_bit_exactly():
    """SURVEY H4.  Poses exactly on (alpha = 0, integer geometry) and within float32 resolution of bin
    boundaries: the device flags them (counters[2] > 0), confirms the truncation for every admissible
    libm (counters[4] == 0) and the Hough dict - keys in insertion order, votes, members - is the
    oracle's (CPython math / glibc) bit for bit."""
    from sod_b200 import engine as E
    scene, n = _boundary_scene()
    sc = E.SceneArrays(scene.q_xy, scene.q_angle, scene.q_octave, scene.m_xy, scene.m_angle, scene.m_octave,
                       scene.m_image, scene.img_centroid, scene.img_size, np.array([[scene.width, scene.height]], np.int32))
    ids = torch.arange(n, dtype=torch.int32, device="cuda")
    res = E.HoughVoter(sc, 15).vote(ids, ids)
    h = res.host()
    assert h["n_near_edge"] >= 300 and h["n_unresolved_edge"] == 0
    flags = res.near_edge[:n].cpu().numpy()
    assert set(np.unique(flags)) <= {0, 1} and flags.sum() == h["n_near_edge"]
    table = O.hough_vote(scene, np.arange(n), np.arange(n), 15)
    np.testing.assert_array_equal(_decode(h["code"], 15), np.array([k[1:] for k in table.keys()]))
    np.testing.assert_array_equal(h["count"], [b.votes for b in table.values()])
    for i, b in enumerate(table.values()):
        np.testing.assert_array_equal(h["members"][h["offset"][i]:h["offset"][i] + h["count"][i]], b.members)
    # base bins one by one, including x < 0 (int() truncates toward zero) and x = W (votes dropped at the top)
    want = np.array([O.bin_index(scene.pose_of(i, i), 15, scene.height, scene.width) for i in range(n)])
    got = res.base_bin[:n].cpu().numpy().astype(np.int64)
    np.testing.assert_array_equal(np.stack([got & 0xFF, got >> 8 & 0xFF, got >> 16 & 0xFF, got >> 24], 1), want)


def test_one_bin_with_60k_votes_single_space():
    """Round-1 advisor finding: with the reference's single Hough space a dominant object puts 10^4-10^5
    matches into ONE bin.  60,000 matches of one rigid instance (+ 5,000 scattered ones): members of every
    bin ascending (the reference's append order), counts and running means equal to the oracle's
    sequential recurrence; the CTA-per-bin bitmap sort and the warp-fed mean chain do the work."""
    from sod_b200 import engine as E
    rng = np.random.default_rng(77)
    n_in, n_out = 60_000, 5_000
    n = n_in + n_out
    W, H = 4032, 3024
    m_xy = rng.uniform(0, 1500, (n, 2)).astype(np.float32)
    cent = np.array([[750.0, 500.0]])
    q_xy = np.empty((n, 2), np.float32)
    q_xy[:n_in] = m_xy[:n_in] + np.float32([1000.25, 800.5])          # scale 1, no rotation: one pose for all
    q_xy[n_in:] = np.stack([rng.uniform(0, W, n_out), rng.uniform(0, H, n_out)], 1)
    ang = rng.uniform(0, 360, n).astype(np.float32)
    q_ang = ang.copy()
    q_ang[n_in:] = rng.uniform(0, 360, n_out).astype(np.float32)
    octv = scenes.pack_octave(np.ones(n, np.int64), np.ones(n, np.int64))
    perm = rng.permutation(n)                                          # inliers and outliers interleaved
    q_xy, q_ang, m_xy, ang = q_xy[perm], q_ang[perm], m_xy[perm], ang[perm]
    size = np.array([[1500.0, 1000.0]])
    sc = E.SceneArrays(q_xy, q_ang, octv, m_xy, ang, octv, np.zeros(n, np.int32), cent, size,
                       np.array([[W, H]], np.int32))
    ids = torch.arange(n, dtype=torch.int32, device="cuda")
    res = E.HoughVoter(sc, 15).vote(ids, ids)
    h = res.host()
    assert h["n_unresolved_edge"] == 0
    big = np.flatnonzero(h["count"] >= n_in)
    assert len(big) == 16 and h["count"].max() <= n
    scene = O.Scene(q_xy, q_ang, octv, m_xy, ang, octv, np.zeros(n, np.int32), cent, size, W, H)
    table = O.hough_vote(scene, np.arange(n), np.arange(n), 15)
    np.testing.assert_array_equal(_decode(h["code"], 15), np.array([k[1:] for k in table.keys()]))
    np.testing.assert_array_equal(h["count"], [b.votes for b in table.values()])
    want_means = np.array([[b.centroid[0], b.centroid[1], b.angle, b.scale, b.img_size[0], b.img_size[1]]
                           for b in table.values()])
    np.testing.assert_allclose(h["mean"], want_means, rtol=1e-12, atol=1e-9)
    for i, b in enumerate(table.values()):                             # thread-, warp- and CTA-finished bins
        np.testing.assert_array_equal(h["members"][h["offset"][i]:h["offset"][i] + h["count"][i]], b.members)
    # the affine stage on the same result: the giant bins survive with (nearly) all inliers
    aff = E.affine_verify(sc, ids, ids, res, 5, 4).host(h["n_votes"])
    assert (aff["votes"][aff["live"]] >= n_in).sum() >= 1
