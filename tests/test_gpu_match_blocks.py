"""GPU parity of the u8 matcher at the edges of its query blocks: a CTA sweeps 512 query rows (four tiles of 128),
a CTA pair 1024.  Batch sizes around those boundaries, including an odd number of blocks (the last pair then has
a phantom block), and ties whose tied database rows lie in consecutive stored tiles, each with and without a
caller-held threshold array."""
import numpy as np
import pytest
import torch

from conftest import sift_like
from oracle import sod_oracle as O

pytestmark = pytest.mark.gpu

BLOCK_SIZES = [511, 512, 513, 1023, 1024, 1025, 1537]


def _top2(q, db, carry):
    from sod_b200 import engine as E
    m = E.Matcher(E.prepare_db(torch.from_numpy(db).cuda()))
    thr = m.new_thresholds(len(q)) if carry else None
    idx, d2 = m.top2(torch.from_numpy(q).cuda(), None, thr)
    torch.cuda.synchronize()
    return idx.cpu().numpy(), d2.cpu().numpy().astype(np.int64), thr


def _assert_oracle(q, db, idx, d2):
    ridx, rd2 = O.knn2(q, db)
    bad = np.nonzero((idx != ridx).any(1) | (d2 != rd2).any(1))[0]
    assert bad.size == 0, (f"{bad.size} rows differ, first {bad[:5]}: got {idx[bad[:5]]} {d2[bad[:5]]} "
                           f"want {ridx[bad[:5]]} {rd2[bad[:5]]}")


@pytest.mark.parametrize("carry", [False, True], ids=["plain", "thresholds"])
@pytest.mark.parametrize("nq", BLOCK_SIZES)
def test_query_block_boundaries(nq, carry):
    rng = np.random.default_rng(nq)
    db = sift_like(rng, 12_000)
    q = sift_like(rng, nq)
    # near-copies of database rows in every query tile of every block, the last row included
    hit = np.unique(np.concatenate([np.arange(0, nq, 97), [nq - 1]]))
    q[hit] = np.clip(db[rng.integers(0, len(db), len(hit))].astype(np.int16) + rng.integers(-2, 3, (len(hit), 128)),
                     0, 255).astype(np.uint8)
    idx, d2, thr = _top2(q, db, carry)
    _assert_oracle(q, db, idx, d2)
    if carry:
        # what the sweep leaves in the array: an upper bound of the row's 2nd best (d^2 - |q|^2) for every
        # real row - the exact one where a single unit swept the whole database
        qn = (q.astype(np.int64) ** 2).sum(1)
        left = thr[:nq].cpu().numpy().astype(np.int64)
        assert (left >= d2[:, 1] - qn).all() and (left < 0x7F7F7F7F).all()


def _stored_tile(db):
    """Stored tile of every database row, as sod_db_prepare lays them out: rows sorted by |t|^2 (stable), cut
    into tiles of 128, and stored tile t holding norm-rank tile (t * stride) mod n_tiles."""
    from math import gcd
    n = len(db)
    tiles = (n + 127) // 128
    stride = int(0.6180339887498949 * tiles) | 1
    while gcd(stride, tiles) != 1:
        stride += 2
    rank_tile = np.empty(n, np.int64)
    rank_tile[np.argsort((db.astype(np.int64) ** 2).sum(1), kind="stable")] = np.arange(n) // 128
    stored_of_rank = np.empty(tiles, np.int64)
    stored_of_rank[(np.arange(tiles) * stride) % tiles] = np.arange(tiles)
    return stored_of_rank[rank_tile]


@pytest.mark.parametrize("carry", [False, True], ids=["plain", "thresholds"])
@pytest.mark.parametrize("nq", [513, 1537])
def test_ties_across_consecutive_tiles(nq, carry):
    """Four identical database rows whose sorted positions straddle a tile boundary: the two lowest indices
    lie in consecutive stored tiles, so one query row's thread meets them in consecutive tile steps (and with
    them the other two copies).  Every query tile of every block asks for them: lowest index first."""
    rng = np.random.default_rng(3)
    db = sift_like(rng, 300)                  # 3 tiles: stored in norm order (stride 1)
    norms = (db.astype(np.int64) ** 2).sum(1)
    order = np.argsort(norms, kind="stable")
    want = None
    for cand in order[120:135]:               # a row whose 4 copies sort into positions that straddle 127 | 128
        trial = db.copy()
        copies = [int(cand), 10, 150, 290]
        trial[copies] = db[cand]
        tile = _stored_tile(trial)
        if len({int(tile[c]) for c in copies}) == 2 and tile[min(copies)] + 1 == tile[sorted(copies)[1]]:
            db, want = trial, sorted(copies)
            break
    assert want is not None
    q = sift_like(rng, nq)
    rows = np.arange(0, nq, 61)               # every query tile, every block of 512 rows
    q[rows] = db[want[0]]
    idx, d2, _ = _top2(q, db, carry)
    assert (idx[rows] == want[:2]).all() and (d2[rows] == 0).all()
    _assert_oracle(q, db, idx, d2)
