"""Generate tests/golden/*.npz by running the REAL reference (/root/reference, read-only) on seeded
synthetic scenes.  Run in the authoring container only:

    python tests/golden/make_golden.py

The reference is imported unmodified.  Three workarounds from SURVEY.md §8c: matplotlib is absent
(stub modules), make_kp fails on cv2 >= 4.5.3 and the dataset is absent (Main fields are injected
instead of calling get_query_features).  Keypoints are cv2.KeyPoint objects whose class_id carries
their index so keypoint pairs can be mapped back to indices.

Each fixture stores the inputs and what the reference produced from them:
  knnMatch indices/distances, ratio survivors, the Hough dict in insertion order (key, votes,
  member pairs, running means), the bins surviving apply_affine_parameters with their parameters,
  and final_pose.
"""
import sys
import types
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
REF = Path("/root/reference")
sys.path.insert(0, str(ROOT / "tests"))

import scenes  # noqa: E402


def import_reference():
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.patches"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["matplotlib.pyplot"].subplots = lambda *a, **k: (None, None)
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["matplotlib"].patches = sys.modules["matplotlib.patches"]
    sys.path.insert(0, str(REF))
    import main as refmain  # the reference's main.py
    return refmain


def keypoints(xy, size, angle, octave):
    import cv2
    return [cv2.KeyPoint(float(xy[i, 0]), float(xy[i, 1]), float(size[i]), float(angle[i]), 0.0,
                         int(octave[i]), i) for i in range(len(xy))]


def ragged(lists, dtype=np.int32):
    off = np.zeros(len(lists) + 1, np.int64)
    off[1:] = np.cumsum([len(x) for x in lists])
    flat = np.array([v for x in lists for v in x], dtype).reshape(-1, 2) if lists else np.zeros((0, 2), dtype)
    return off, flat


def run_reference(refmain, sc: scenes.SyntheticScene, bins=15, vote_thr=5, affine_thr=4):
    import cv2
    m = refmain.Main()
    m.kp = keypoints(sc.m_xy, sc.m_size, sc.m_angle, sc.m_octave)
    m.des = sc.m_des.astype(np.float32)
    m.kp_query = keypoints(sc.q_xy, sc.q_size, sc.q_angle, sc.q_octave)
    m.des_query = sc.q_des.astype(np.float32)
    m.img_size_list = [tuple(int(v) for v in sc.img_size[i]) for i in sc.m_image]
    m.img_centroid_list = [tuple(float(v) for v in sc.img_centroid[i]) for i in sc.m_image]
    m.rgb_query = np.zeros((sc.height, sc.width, 3), np.uint8)
    m.image_query_size = (sc.width, sc.height)

    raw = cv2.BFMatcher().knnMatch(m.des_query, m.des, k=2)
    knn_idx = np.array([[a.trainIdx, b.trainIdx] for a, b in raw], np.int32)
    knn_dist = np.array([[a.distance, b.distance] for a, b in raw], np.float32)

    m.run_matcher()
    match_t = np.array([t[0].class_id for t in m.matching_keypoints], np.int32)
    match_q = np.array([t[1].class_id for t in m.matching_keypoints], np.int32)

    m.apply_hough_transform(bins)
    keys = np.array(list(m.hough_transform.keys()), np.int32).reshape(-1, 4)
    hb = list(m.hough_transform.values())
    votes = np.array([b.votes for b in hb], np.int32)
    means = np.array([[b.centroid[0], b.centroid[1], b.angle, b.scale, b.img_size[0], b.img_size[1]]
                      for b in hb], np.float64).reshape(-1, 6)
    mem_off, mem = ragged([[(p[1].class_id, p[0].class_id) for p in b.keypoint_pairs] for b in hb])

    m.get_valid_bins(vote_thr)
    valid_keys = np.array([b.pose for b in m.valid_bins], np.int32).reshape(-1, 4)
    m.apply_affine_parameters(affine_thr)
    live = m.valid_bins
    live_keys = np.array([b.pose for b in live], np.int32).reshape(-1, 4)
    live_votes = np.array([b.votes for b in live], np.int32)
    live_params = np.array([[float(v) for v in b.affine_parameters] for b in live], np.float64).reshape(-1, 6)
    live_off, live_mem = ragged([[(p[1].class_id, p[0].class_id) for p in b.keypoint_pairs] for b in live])
    n_pairs_after = len(m.keypoint_pairs)

    final_pose = np.zeros((0, 6), np.float64)
    try:
        m.post_process()
        final_pose = np.array([[c[0], c[1], o, s, sh[0], sh[1]] for (c, o, s, sh) in m.final_pose],
                              np.float64).reshape(-1, 6)
    except RecursionError:  # SURVEY Q12
        pass
    return dict(knn_idx=knn_idx, knn_dist=knn_dist, match_q=match_q, match_t=match_t,
                bin_keys=keys, bin_votes=votes, bin_means=means, bin_mem_off=mem_off, bin_mem=mem,
                valid_keys=valid_keys, live_keys=live_keys, live_votes=live_votes,
                live_params=live_params, live_mem_off=live_off, live_mem=live_mem,
                n_pairs_after=np.int64(n_pairs_after), final_pose=final_pose,
                bins=np.int32(bins), vote_thr=np.int32(vote_thr), affine_thr=np.int32(affine_thr))


SCENES = {
    # one model image, one instance at scale 1/2 (sigma bins 0/1 only: exercises quirk Q1)
    "scene_single": dict(seed=11, n_images=1, kp_per_image=3000, n_query=1500, n_true=220, scales=(0.5,),
                         n_false=500, jitter_frac=0.15),
    # three model images in ONE Hough space (quirk Q7), instances at scales 2, 1, 4; duplicate rows
    "scene_multi": dict(seed=12, n_images=3, kp_per_image=1500, n_query=2000, n_true=420,
                        scales=(2.0, 1.0, 4.0), n_dup=40, width=4032, height=3024, n_false=600,
                        jitter_frac=0.2, jitter_px=60.0),
    # tiny database: a single 128-row tile, ragged query
    "scene_tiny": dict(seed=13, n_images=1, kp_per_image=100, n_query=37, n_true=30, scales=(2.0,)),
}


def postprocess_bins(seed=21, n=420):
    """Surviving-bin statistics for the post-processing fixture: several object instances, each a
    cloud of bins around its centre (chains of neighbours, touching clusters, values exactly on the
    <= thresholds, orientation runs 1 degree apart), plus isolated bins."""
    rng = np.random.default_rng(seed)
    cx, cy, sc, an, w, h = [], [], [], [], [], []
    sizes = [(1500, 1000), (1500, 2000), (1500, 1125)]
    for inst in range(7):
        m = int(rng.integers(20, 110))
        size = sizes[inst % 3]
        s0 = float(2.0 ** rng.integers(-2, 1))
        x0, y0 = 800 + 1500.0 * inst + rng.uniform(-60, 60), rng.uniform(300, 2700)
        spread = size[0] * s0 / 4
        cx += list(x0 + rng.uniform(-1.2, 1.2, m) * spread)
        cy += list(y0 + rng.uniform(-1.2, 1.2, m) * size[1] * s0 / 4)
        sc += list(s0 * rng.choice([0.5, 1.0, 1.0, 1.0, 2.0], m))
        a0 = rng.uniform(0, 2 * np.pi)
        an += list(a0 + np.radians(rng.choice([0.0, 0.4, 0.9, 1.0, 1.7, 2.5, 30.0], m)
                                   + rng.uniform(-0.05, 0.05, m)))
        w += [size[0]] * m
        h += [size[1]] * m
    k = max(n - len(cx), 40)
    cx += list(rng.uniform(0, 12000, k)); cy += list(rng.uniform(0, 3000, k))
    sc += list(2.0 ** rng.integers(-2, 3, k).astype(np.float64)); an += list(rng.uniform(0, 2 * np.pi, k))
    w += [1500] * k; h += [1000] * k
    cx, cy, sc, an = (np.asarray(v, np.float64) for v in (cx, cy, sc, an))
    # exact-threshold cases: bin 1 sits exactly reach_x away from bin 0, bin 3 exactly 1 degree from bin 2
    sc[0] = sc[1] = 1.0; w[0] = w[1] = 1500; h[0] = h[1] = 1000
    cx[1] = cx[0] + 375.0; cy[1] = cy[0]
    an[3] = an[2] + np.radians(1.0)
    perm = rng.permutation(len(cx))
    return cx[perm], cy[perm], sc[perm], an[perm], np.asarray(w, np.int64)[perm], np.asarray(h, np.int64)[perm]


def make_postprocess():
    """tests/golden/postprocess.npz: the reference's PostProcessing functions on the bins above."""
    import_reference()
    import PostProcessing as ref_pp  # the reference's module
    cx, cy, sc, an, w, h = postprocess_bins()
    bins = [types.SimpleNamespace(centroid=(float(cx[i]), float(cy[i])), scale=float(sc[i]), angle=float(an[i]),
                                  img_size=(int(w[i]), int(h[i])), index=i) for i in range(len(cx))]
    pose_cluster = ref_pp.group_position(bins)
    ori_cluster = ref_pp.group_orientation(pose_cluster)
    ori = ref_pp.find_max_orientation(ori_cluster)
    final = ref_pp.get_final_pose(pose_cluster, ori)
    cl_off = np.cumsum([0] + [len(c) for c in pose_cluster])
    subs = [sub for c in ori_cluster for sub in c]
    sub_off = np.cumsum([0] + [len(sub) for sub in subs])
    np.savez_compressed(
        HERE / "postprocess.npz", cx=cx, cy=cy, scale=sc, angle=an, img_w=w, img_h=h,
        cluster_off=cl_off, cluster_members=np.array([b.index for c in pose_cluster for b in c], np.int32),
        subs_per_cluster=np.array([len(c) for c in ori_cluster], np.int32), sub_off=sub_off,
        sub_members=np.array([b.index for sub in subs for b in sub], np.int32),
        orientation=np.array(ori, np.float64),
        final=np.array([[c[0], c[1], o, s, sh[0], sh[1]] for (c, o, s, sh) in final], np.float64))
    print("postprocess bins", len(bins), "clusters", len(pose_cluster), "largest", max(len(c) for c in pose_cluster),
          "sub-clusters", len(subs))


def singular_bins(seed=31):
    """Bins for the affine stage that the Hough fixtures never produce (SURVEY Q11 / H5): duplicate
    model locations (real SIFT emits several orientations at one location, main.py:43), collinear
    model points, exactly-threshold sizes, ill-conditioned normal matrices from cond ~1e7 to ~1e11, and
    well-conditioned controls.  -> list of dicts(name, model_xy f32 [n,2], query_xy f32 [n,2], isigma)."""
    rng = np.random.default_rng(seed)
    f32 = lambda a: np.asarray(a, np.float32)  # noqa: E731
    sim = lambda m, s, th, t, noise: (s * (m @ np.array([[np.cos(th), np.sin(th)], [-np.sin(th), np.cos(th)]])) + t  # noqa: E731
                                      + rng.normal(0, noise, m.shape))
    out = []
    for k in range(4):
        m = rng.uniform(0, 1500, (7, 2))
        out.append(dict(name=f"generic{k}", model=f32(m), query=f32(sim(m, 2.0, 0.3 * k, [900, 700], 2.0)), isigma=2))
    for k in range(4):                                   # 2 distinct model locations among 5..8 pairs (rank 2)
        base = rng.uniform(100, 1400, (2, 2))
        idx = np.array([0, 1, 0, 0, 1, 1, 0, 1][:5 + k])
        m = base[idx]
        out.append(dict(name=f"two_locations{k}", model=f32(m), query=f32(sim(m, 1.0, 0.5, [300, 200], 1.5)), isigma=2))
    for k in range(3):                                   # a single model location (rank 1)
        m = np.tile(rng.uniform(100, 1400, (1, 2)), (5 + k, 1))
        out.append(dict(name=f"one_location{k}", model=f32(m), query=f32(sim(m, 1.0, 0.0, [50, 60], 1.0)), isigma=1))
    for k in range(3):                                   # exactly collinear integer model points (rank 2)
        m = np.array([[100 + 10 * j * (k + 1), 200 + 20 * j * (k + 1)] for j in range(6)], float)
        out.append(dict(name=f"collinear_int{k}", model=f32(m), query=f32(sim(m, 1.5, 0.2, [400, 100], 1.0)), isigma=2))
    for k in range(3):                                   # collinear up to float32 rounding
        t = rng.uniform(0, 1, (6, 1))
        m = np.array([100.0, 200.0]) + t * np.array([700.0, 300.0 + 50 * k])
        out.append(dict(name=f"collinear_f32_{k}", model=f32(m), query=f32(sim(m, 0.5, 1.0, [800, 900], 0.5)), isigma=1))
    for eps in (1e-2, 1e-3, 1e-4, 1e-5, 1e-6):          # near-collinear: cond(S) from ~1e7 up to ~1e11
        for k in range(2):
            m = np.array([[100 + 10 * j, 200 + 20 * j] for j in range(6)], float) + 1000 * eps * rng.normal(0, 1, (6, 2))
            out.append(dict(name=f"near_collinear_{eps:g}_{k}", model=f32(m),
                            query=f32(sim(m, 1.0, 0.1, [200, 300], 0.5)), isigma=2))
    # sizes around the threshold (4): exactly 4 good pairs; 5 pairs of which one is a gross outlier (4 stay);
    # 5 pairs with two gross outliers (3 stay -> the bin dies)
    m = rng.uniform(0, 1500, (4, 2))
    out.append(dict(name="exactly_threshold", model=f32(m), query=f32(sim(m, 1.0, 0.4, [500, 500], 0.5)), isigma=2))
    for n_out in (1, 2):
        m = rng.uniform(0, 1500, (5, 2))
        q = sim(m, 1.0, 0.4, [500, 500], 0.5)
        q[:n_out] += [[900.0, -700.0], [-800.0, 600.0]][:n_out]
        out.append(dict(name=f"outliers{n_out}_of5", model=f32(m), query=f32(q), isigma=2))
    # sigma bin 0 (every scale factor <= 1, SURVEY Q4): the residual limits are 0, everything is dropped
    m = rng.uniform(0, 1500, (6, 2))
    out.append(dict(name="isigma0", model=f32(m), query=f32(sim(m, 1.0, 0.2, [100, 100], 1.0)), isigma=0))
    return out


def make_affine_singular(width=4032, height=3024, threshold=4):
    """tests/golden/affine_singular.npz: the reference's AffineParameters / remove_outliers /
    Main.apply_affine_parameters on the bins above, bin by bin (the loop is an independent fixed point
    per bin, SURVEY T13) and all together."""
    import cv2
    refmain = import_reference()
    from PoseBin import PoseBin as RefPoseBin  # the reference's class
    cases = singular_bins()
    kp = lambda p: cv2.KeyPoint(float(p[0]), float(p[1]), 1.0)  # noqa: E731
    bins = []
    for c in cases:
        pairs = [(kp(m), kp(q)) for m, q in zip(c["model"], c["query"])]
        bins.append(RefPoseBin((0, 0, 0, int(c["isigma"])), (1500, 1000), len(pairs), pairs, (0.0, 0.0, 0.0, 1.0)))
    first = []
    for b in bins:                                       # one AffineParameters call on the untouched bin
        from AffineParameters import AffineParameters as ref_fit
        ref_fit(b)
        first.append([float(v) for v in b.affine_parameters])
    tags = [[id(p[0]) for p in b.keypoint_pairs] for b in bins]
    m = refmain.Main()
    m.image_query_size = (width, height)
    m.valid_bins = list(bins)
    m.apply_affine_parameters(threshold)
    live = [any(b is v for v in m.valid_bins) for b in bins]
    keep_off, keep = [0], []
    for b, t in zip(bins, tags):
        alive = {id(p[0]) for p in b.keypoint_pairs}
        keep += [i in alive for i in t]
        keep_off.append(len(keep))
    off = np.cumsum([0] + [len(c["model"]) for c in cases])
    np.savez_compressed(
        HERE / "affine_singular.npz", names=np.array([c["name"] for c in cases]), off=off,
        model=np.concatenate([c["model"] for c in cases]), query=np.concatenate([c["query"] for c in cases]),
        isigma=np.array([c["isigma"] for c in cases], np.int32), width=np.int32(width), height=np.int32(height),
        threshold=np.int32(threshold), first_params=np.array(first, np.float64),
        last_params=np.array([[float(v) for v in b.affine_parameters] for b in bins], np.float64),
        votes=np.array([b.votes for b in bins], np.int32), live=np.array(live), keep=np.array(keep))
    print("affine_singular:", len(cases), "bins,", int(np.sum(live)), "live,", int(np.sum(keep)), "of", len(keep), "pairs kept")


def synthetic_image(seed, width, height):
    """Multi-octave noise + random circles / rectangles (SURVEY 8d C1): texture on which SIFT finds
    keypoints on several octaves, many of them with more than one orientation."""
    import cv2
    rng = np.random.default_rng(seed)
    img = np.zeros((height, width), np.float32)
    for octv in range(6):
        h, w = max(height >> octv, 2), max(width >> octv, 2)
        img += cv2.resize(rng.normal(0, 1, (h, w)).astype(np.float32), (width, height), interpolation=cv2.INTER_CUBIC) * (1.6 ** octv)
    img = (img - img.min()) / (img.max() - img.min()) * 160 + 40
    img = img.astype(np.uint8)
    for _ in range(max(width * height // 9000, 20)):
        c = int(rng.integers(0, 256))
        x, y = int(rng.integers(0, width)), int(rng.integers(0, height))
        if rng.random() < 0.5:
            cv2.circle(img, (x, y), int(rng.integers(4, 40)), c, -1 if rng.random() < 0.6 else 2)
        else:
            cv2.rectangle(img, (x, y), (x + int(rng.integers(6, 70)), y + int(rng.integers(6, 70))), c,
                          -1 if rng.random() < 0.6 else 2)
    return cv2.GaussianBlur(img, (0, 0), 0.8)


def make_c1(model_wh=(1500, 1000), scene_wh=(2000, 1500), scale=0.5, angle_deg=25.0):
    """tests/golden/scene_c1.npz - BASELINE configs[0] (main.py as shipped) on a synthetic image pair,
    because the reference's dataset and pickle are not available: a textured model image is pasted at
    `scale` / `angle_deg` into a clutter scene, REAL cv2.SIFT_create() keypoints and descriptors on both
    sides (GenerateDatabaseInfo.py:14-34, main.py:36-46 with the reference's own get_centroid), then the
    unmodified reference Main from run_matcher to post_process.  Pins real octave packing (negative
    octaves, layers) and multi-orientation duplicates (several keypoints at one location)."""
    import cv2
    refmain = import_reference()
    from SiftHelperFunctions import get_centroid
    mw, mh = model_wh
    sw, sh = scene_wh
    model = synthetic_image(1, mw, mh)
    scene_img = synthetic_image(2, sw, sh)
    rot = cv2.getRotationMatrix2D((mw / 2, mh / 2), angle_deg, scale)
    rot[:, 2] += np.array([sw / 2 - mw / 2, sh / 2 - mh / 2])
    warped = cv2.warpAffine(model, rot, (sw, sh), flags=cv2.INTER_LINEAR)
    mask = cv2.warpAffine(np.full((mh, mw), 255, np.uint8), rot, (sw, sh)) > 127
    scene_img[mask] = warped[mask]
    sift = cv2.SIFT_create()
    kp_m, des_m = sift.detectAndCompute(model, None)
    kp_q, des_q = sift.detectAndCompute(scene_img, None)
    assert np.array_equal(des_m, np.rint(des_m)) and des_m.max() <= 255
    arr = lambda kps, f: np.array([f(k) for k in kps])  # noqa: E731
    sc = scenes.SyntheticScene(
        m_des=des_m.astype(np.uint8), m_xy=arr(kp_m, lambda k: k.pt).astype(np.float32),
        m_angle=arr(kp_m, lambda k: k.angle).astype(np.float32), m_octave=arr(kp_m, lambda k: k.octave).astype(np.int32),
        m_size=arr(kp_m, lambda k: k.size).astype(np.float32), m_image=np.zeros(len(kp_m), np.int32),
        img_size=np.array([[mw, mh]], np.int32), img_centroid=np.array([get_centroid(kp_m)], np.float64),
        q_des=des_q.astype(np.uint8), q_xy=arr(kp_q, lambda k: k.pt).astype(np.float32),
        q_angle=arr(kp_q, lambda k: k.angle).astype(np.float32), q_octave=arr(kp_q, lambda k: k.octave).astype(np.int32),
        q_size=arr(kp_q, lambda k: k.size).astype(np.float32), width=sw, height=sh,
        true_q=np.zeros(0, np.int32), true_t=np.zeros(0, np.int32))
    out = run_reference(refmain, sc)
    dup = len(sc.m_xy) - len(np.unique(sc.m_xy, axis=0))
    inputs = {f"in_{k}": v for k, v in sc.__dict__.items()}
    np.savez_compressed(HERE / "scene_c1.npz", **inputs, **out, paste=np.array([scale, angle_deg]),
                        versions=np.array([cv2.__version__, np.__version__, sys.version.split()[0]]))
    octs = np.unique((sc.m_octave & 0xFF).astype(np.int8))
    print("scene_c1: model kp", len(kp_m), "scene kp", len(kp_q), "duplicate model locations", dup, "octaves", octs.tolist(),
          "matches", len(out["match_q"]), "bins", len(out["bin_votes"]), "valid", len(out["valid_keys"]), "live",
          len(out["live_keys"]), "final", out["final_pose"].round(2).tolist())


LIVE_KEYS = ("knn_idx", "knn_dist", "match_q", "match_t", "bin_keys", "bin_votes", "bin_means", "valid_keys",
             "live_keys", "live_votes", "live_params", "n_pairs_after", "bins", "vote_thr", "affine_thr")


def oracle_outputs(sc: scenes.SyntheticScene, bins, vote_thr, affine_thr):
    """The LIVE_KEYS of run_reference, computed by the oracle (oracle/sod_oracle.py)."""
    from oracle import sod_oracle as O
    scene = O.Scene(sc.q_xy, sc.q_angle, sc.q_octave, sc.m_xy, sc.m_angle, sc.m_octave, sc.m_image,
                    sc.img_centroid, sc.img_size, sc.width, sc.height)
    idx, d2 = O.knn2(sc.q_des, sc.m_des)
    ok = O.ratio_pass(d2, idx)
    match_q, match_t = np.nonzero(ok)[0].astype(np.int32), idx[ok, 0].astype(np.int32)
    table = O.hough_vote(scene, match_q, match_t, bins)
    hb = list(table.values())
    hough = dict(bin_keys=np.array([k[1:] for k in table.keys()], np.int32).reshape(-1, 4),
                 bin_votes=np.array([b.votes for b in hb], np.int32),
                 bin_means=np.array([[b.centroid[0], b.centroid[1], b.angle, b.scale, b.img_size[0], b.img_size[1]]
                                     for b in hb], np.float64).reshape(-1, 6))
    vb = O.valid_bins(table, vote_thr)
    valid_keys = np.array([b.pose for b in vb], np.int32).reshape(-1, 4)
    live = O.affine_verify(scene, match_q, match_t, vb, affine_thr)     # updates the bins of `table` in place
    return dict(knn_idx=idx.astype(np.int32), knn_dist=O.match_distance(d2), match_q=match_q, match_t=match_t,
                **hough, valid_keys=valid_keys, live_keys=np.array([b.pose for b in live], np.int32).reshape(-1, 4),
                live_votes=np.array([b.votes for b in live], np.int32),
                live_params=np.array([b.affine for b in live], np.float64).reshape(-1, 6),
                n_pairs_after=np.int64(sum(b.votes for b in live)),
                bins=np.int32(bins), vote_thr=np.int32(vote_thr), affine_thr=np.int32(affine_thr))


def make_live_cases(refmain=None):
    """tests/golden/live_<seed>.npz for test_oracle_live_reference: the expected outputs of each case,
    from the reference's Main when `refmain` is given, else from the oracle (`source` records which), and
    the digest of the inputs: the test regenerates the inputs themselves from the seed."""
    sys.path.insert(0, str(ROOT))
    from test_oracle_live_reference import CASES, input_digest
    for seed, kw, bins, vote_thr, affine_thr in CASES:
        sc = scenes.make_scene(seed, **kw)
        if refmain is not None:
            out = run_reference(refmain, sc, bins=bins, vote_thr=vote_thr, affine_thr=affine_thr)
            out = {k: out[k] for k in LIVE_KEYS}
        else:
            out = oracle_outputs(sc, bins, vote_thr, affine_thr)
        np.savez_compressed(HERE / f"live_{seed}.npz", **out, input_digest=np.array(input_digest(sc)),
                            source=np.array("reference" if refmain is not None else "oracle"))
        print(f"live_{seed}: matches", len(out["match_q"]), "bins", len(out["bin_votes"]), "valid",
              len(out["valid_keys"]), "live", len(out["live_keys"]))


def main():
    if "--c1-only" in sys.argv:
        return make_c1()
    if "--postprocess-only" in sys.argv:
        return make_postprocess()
    if "--affine-singular-only" in sys.argv:
        return make_affine_singular()
    if "--live-cases-from-oracle" in sys.argv:
        return make_live_cases()
    refmain = import_reference()
    import cv2
    for name, kw in SCENES.items():
        sc = scenes.make_scene(**kw)
        out = run_reference(refmain, sc)
        inputs = {f"in_{k}": v for k, v in sc.__dict__.items()}
        np.savez_compressed(HERE / f"{name}.npz", **inputs, **out,
                            versions=np.array([cv2.__version__, np.__version__, sys.version.split()[0]]))
        print(name, "matches", len(out["match_q"]), "bins", len(out["bin_votes"]), "valid",
              len(out["valid_keys"]), "live", len(out["live_keys"]), "final", len(out["final_pose"]))

    make_postprocess()
    make_affine_singular()
    make_c1()
    make_live_cases(refmain)

    # known-answer facts (SURVEY.md §4 T4, T5, T8) taken from the reference's own libraries
    import math
    from HoughTransformHelperFunctions import calculate_bin_index
    kat = {}
    kat["sigma_k"] = np.arange(-12, 13)
    kat["sigma_bin15"] = np.array([calculate_bin_index((0.0, 0.0, 0.0, 2.0 ** int(k)), 15, (1, 1))[3]
                                   for k in kat["sigma_k"]], np.int32)
    rng = np.random.default_rng(5)
    d = rng.integers(1, 400000, (20000, 2))
    d.sort(1)
    near = np.arange(1, 3000)
    d = np.concatenate([d, np.stack([9 * near * 2, 16 * near * 2], 1), np.stack([9 * near * 2 + 1, 16 * near * 2], 1),
                        np.stack([9 * near * 2 - 1, 16 * near * 2], 1), np.array([[18, 32]])])
    dist = np.sqrt(d.astype(np.float32))
    kat["ratio_d2"] = d.astype(np.int64)
    kat["ratio_pass"] = np.array([float(a) < 0.75 * float(b) for a, b in dist])
    np.savez_compressed(HERE / "kat.npz", **kat)
    print("kat: sigma", kat["sigma_bin15"].tolist(), "ratio cases", len(d),
          "int-test disagreements", int((kat["ratio_pass"] != (16 * d[:, 0] < 9 * d[:, 1])).sum()))


if __name__ == "__main__":
    main()
