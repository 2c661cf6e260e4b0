"""The oracle held to the reference's outputs on further seeded scenes (beyond the scene_* fixtures):
other bin counts and thresholds, other scales, ties, clutter.  CPU only.

tests/golden/live_<seed>.npz hold each case's expected outputs and a digest of its inputs, which are
regenerated from the seed (make_golden.make_live_cases).  Their `source` says where the outputs came
from: the reference's own Main, or the oracle, recorded at a commit at which the oracle had not changed
since this comparison was written against the live reference (the reference checkout is not part of
this repository)."""
import hashlib
from pathlib import Path

import numpy as np
import pytest

from oracle import sod_oracle as O

GOLD = Path(__file__).resolve().parent / "golden"

CASES = [
    # seed, scene kwargs, bins, vote threshold, affine threshold
    (201, dict(n_images=1, kp_per_image=800, n_query=500, n_true=120, scales=(1.0,), n_false=150, jitter_frac=0.2), 15, 5, 4),
    (202, dict(n_images=2, kp_per_image=600, n_query=600, n_true=160, scales=(2.0, 0.5), n_dup=25, n_false=200,
               jitter_frac=0.3, jitter_px=80.0, width=4032, height=3024), 10, 4, 3),
    (203, dict(n_images=1, kp_per_image=400, n_query=300, n_true=90, scales=(4.0,), n_false=100, noise_px=4.0), 8, 3, 3),
    (204, dict(n_images=3, kp_per_image=300, n_query=450, n_true=150, scales=(1.0, 2.0, 8.0), n_false=120,
               jitter_frac=0.1), 15, 6, 5),
]


def input_digest(sc) -> str:
    """sha256 over every field of a scenes.SyntheticScene (name, dtype, shape, bytes)."""
    h = hashlib.sha256()
    for name, v in sorted(sc.__dict__.items()):
        a = np.ascontiguousarray(v)
        h.update(f"{name} {a.dtype.str} {a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()


@pytest.mark.parametrize("seed,kw,bins,vote_thr,affine_thr", CASES)
def test_oracle_equals_live_reference(seed, kw, bins, vote_thr, affine_thr):
    import scenes
    sc = scenes.make_scene(seed, **kw)
    ref = np.load(GOLD / f"live_{seed}.npz")
    assert input_digest(sc) == str(ref["input_digest"]), "scenes.make_scene no longer makes this case's inputs"
    assert (int(ref["bins"]), int(ref["vote_thr"]), int(ref["affine_thr"])) == (bins, vote_thr, affine_thr)
    scene = O.Scene(sc.q_xy, sc.q_angle, sc.q_octave, sc.m_xy, sc.m_angle, sc.m_octave, sc.m_image,
                    sc.img_centroid, sc.img_size, sc.width, sc.height)
    # matching: cv2.BFMatcher.knnMatch + the ratio loop
    idx, d2 = O.knn2(sc.q_des, sc.m_des)
    np.testing.assert_array_equal(idx, ref["knn_idx"])
    np.testing.assert_array_equal(O.match_distance(d2), ref["knn_dist"])
    ok = O.ratio_pass(d2, idx)
    np.testing.assert_array_equal(np.nonzero(ok)[0], ref["match_q"])
    np.testing.assert_array_equal(idx[ok, 0], ref["match_t"])
    # Hough dict: keys in insertion order, votes, running means (float64, bit-exact)
    table = O.hough_vote(scene, ref["match_q"], ref["match_t"], bins)
    np.testing.assert_array_equal(np.array([k[1:] for k in table.keys()], np.int32).reshape(-1, 4), ref["bin_keys"])
    hb = list(table.values())
    np.testing.assert_array_equal([b.votes for b in hb], ref["bin_votes"])
    np.testing.assert_array_equal(
        np.array([[b.centroid[0], b.centroid[1], b.angle, b.scale, b.img_size[0], b.img_size[1]] for b in hb]).reshape(-1, 6),
        ref["bin_means"])
    # valid bins and the affine fixed point
    vb = O.valid_bins(table, vote_thr)
    np.testing.assert_array_equal(np.array([b.pose for b in vb], np.int32).reshape(-1, 4), ref["valid_keys"])
    live = O.affine_verify(scene, ref["match_q"], ref["match_t"], vb, affine_thr)
    np.testing.assert_array_equal(np.array([b.pose for b in live], np.int32).reshape(-1, 4), ref["live_keys"])
    np.testing.assert_array_equal([b.votes for b in live], ref["live_votes"])
    np.testing.assert_array_equal(np.array([b.affine for b in live]).reshape(-1, 6), ref["live_params"])
    assert sum(b.votes for b in live) == int(ref["n_pairs_after"])
    assert len(ref["match_q"]) > 50 and len(ref["valid_keys"]) > 0       # the case exercised the path
