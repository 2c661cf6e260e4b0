"""GPU parity: sod_match_top2 / sod_top2_merge vs the oracle (bit-exact indices, distances, flags)."""
import numpy as np
import pytest
import torch

from conftest import sift_like
from exact_top2 import direct_d2, exact_top2
from oracle import sod_oracle as O

pytestmark = pytest.mark.gpu


def _run(q, db, index_base=0):
    from sod_b200 import engine as E
    dq = torch.from_numpy(q).cuda()
    shard = E.prepare_db(torch.from_numpy(db).cuda(), index_base)
    idx, d2, dist, ok = E.knn_match_ratio(dq, E.Matcher(shard))
    torch.cuda.synchronize()
    return idx.cpu().numpy(), d2.cpu().numpy(), dist.cpu().numpy(), ok.cpu().numpy().astype(bool)


def _check(q, db, index_base=0):
    idx, d2, dist, ok = _run(q, db, index_base)
    ridx, rd2 = O.knn2(q, db)
    ridx = np.where(ridx >= 0, ridx + index_base, -1)
    bad = np.nonzero((idx != ridx).any(1) | (d2.astype(np.int64) != rd2).any(1))[0]
    assert bad.size == 0, (f"{bad.size} rows differ, first {bad[:5]}: got {idx[bad[:5]]} {d2[bad[:5]]} "
                           f"want {ridx[bad[:5]]} {rd2[bad[:5]]}")
    np.testing.assert_array_equal(dist[ridx[:, 1] >= 0], O.match_distance(rd2)[ridx[:, 1] >= 0])
    np.testing.assert_array_equal(ok, O.ratio_pass(rd2, ridx))


@pytest.mark.parametrize("nq,ndb", [(1, 2), (5, 3), (128, 128), (256, 1000), (257, 129), (300, 4097),
                                    (1000, 20000), (77, 50001)])
def test_uniform_u8(nq, ndb):
    rng = np.random.default_rng(nq * 1000003 + ndb)
    _check(rng.integers(0, 256, (nq, 128), dtype=np.uint8), rng.integers(0, 256, (ndb, 128), dtype=np.uint8))


def test_extreme_values():
    """All-255 vs all-0 rows reach the largest possible distance 128*255^2."""
    q = np.zeros((4, 128), np.uint8); q[1] = 255; q[2, ::2] = 255
    db = np.zeros((300, 128), np.uint8); db[7] = 255; db[9, 1::2] = 255
    _check(q, db)


def test_ties_duplicates_lowest_index_first():
    """SURVEY T4: identical database rows -> lowest index first, also for 2nd place and across tiles."""
    rng = np.random.default_rng(4)
    db = sift_like(rng, 1000)
    q = sift_like(rng, 40)
    for r in (7, 30, 40, 130, 131, 700, 999):
        db[r] = q[0]
    db[5] = db[600] = q[1]       # tie across tiles (5 in tile 0, 600 in tile 4)
    db[128] = db[127] = q[2]     # tie across a tile boundary
    db[256] = db[0] = q[3]       # column 0 of a later tile vs column 0 of the first
    idx, d2, _, _ = _run(q, db)
    assert idx[0].tolist() == [7, 30] and d2[0].tolist() == [0, 0]
    assert idx[1].tolist() == [5, 600]
    assert idx[2].tolist() == [127, 128]
    assert idx[3].tolist() == [0, 256]
    _check(q, db)


def test_sift_like_with_true_matches_and_index_base():
    rng = np.random.default_rng(100)
    db = sift_like(rng, 30000)
    q = sift_like(rng, 3000)
    hit = rng.choice(3000, 300, replace=False)
    src = rng.integers(0, 30000, 300)
    q[hit] = np.clip(db[src].astype(np.int16) + rng.integers(-3, 4, (300, 128)), 0, 255).astype(np.uint8)
    _check(q, db, index_base=123456)
    idx, _, _, ok = _run(q, db)
    assert ok[hit].mean() > 0.9 and (idx[hit, 0] == src).mean() > 0.99


def test_ratio_edge_T5():
    """(d1^2, d2^2) = (18, 32): float32 sqrt makes the reference pass it although 16*18 == 9*32."""
    from sod_b200 import engine as E
    pi = torch.tensor([[[0, 1]], [[2, 3]]], dtype=torch.int32).cuda()
    pd = torch.tensor([[[18, 40]], [[32, 50]]], dtype=torch.int32).cuda()
    idx, d2, dist, ok = E.merge_top2(pi, pd)
    assert idx.cpu().tolist() == [[0, 2]] and d2.cpu().tolist() == [[18, 32]]
    want = O.ratio_pass(np.array([[18, 32]]))
    assert bool(ok.cpu()[0]) == bool(want[0]) == True


def test_merge_matches_oracle_random():
    from sod_b200 import engine as E
    rng = np.random.default_rng(9)
    g, nq = 8, 5000
    pi = rng.permuted(np.tile(np.arange(g * 2 * 4, dtype=np.int32), (nq, 1)), axis=1)[:, :g * 2]
    pi = pi.reshape(nq, g, 2).transpose(1, 0, 2).copy()
    pd = rng.integers(0, 6, (g, nq, 2)).astype(np.int32)      # many equal distances -> index tie-break
    drop = rng.random((g, nq, 2)) < 0.2
    pi[drop] = -1; pd[drop] = -1
    idx, d2, _, ok = E.merge_top2(torch.from_numpy(pi).cuda(), torch.from_numpy(pd).cuda())
    ri, rd = O.merge_top2(pi, pd.astype(np.int64))
    np.testing.assert_array_equal(idx.cpu().numpy(), ri)
    np.testing.assert_array_equal(d2.cpu().numpy().astype(np.int64), rd)
    np.testing.assert_array_equal(ok.cpu().numpy().astype(bool), O.ratio_pass(rd, ri))


def test_pack_from_f32_rejects_non_integer():
    from sod_b200 import engine as E
    x = np.random.default_rng(1).integers(0, 256, (100, 128)).astype(np.float32)
    got = E.pack_descriptors(x).cpu().numpy()
    np.testing.assert_array_equal(got, x.astype(np.uint8))
    x[3, 5] = 1.5
    with pytest.raises(ValueError):
        E.pack_descriptors(x)


def test_random_shapes_soak():
    """Many random shapes, including the few-queries / large-database ones whose segments share their
    thresholds through global memory, each run twice: results must be exact and repeatable."""
    from sod_b200 import engine as E
    rng = np.random.default_rng(2024)
    g = torch.Generator(device="cuda").manual_seed(7)
    shapes = [(int(rng.integers(1, 3000)), int(rng.integers(2, 60000))) for _ in range(24)]
    shapes += [(int(rng.integers(1, 600)), int(rng.integers(100000, 400000))) for _ in range(8)]
    for nq, ndb in shapes:
        hi = int(rng.choice([2, 16, 256]))       # small alphabets make ties frequent
        q = torch.randint(0, hi, (nq, 128), dtype=torch.uint8, device="cuda", generator=g)
        db = torch.randint(0, hi, (ndb, 128), dtype=torch.uint8, device="cuda", generator=g)
        db[torch.randint(0, ndb, (min(nq, 50),), device="cuda", generator=g)] = q[:min(nq, 50)]
        m = E.Matcher(E.prepare_db(db))
        idx1, d1 = m.top2(q)
        idx2, d2 = m.top2(q)
        ridx, rd = exact_top2(q, db)
        assert torch.equal(idx1, ridx) and torch.equal(d1, rd), (nq, ndb, hi)
        assert torch.equal(direct_d2(q, db, idx1), d1), (nq, ndb, hi)
        assert torch.equal(idx1, idx2) and torch.equal(d1, d2), (nq, ndb, hi)


def test_tile_ranges_and_carried_thresholds_stay_exact():
    """sod_match_top2_range: (a) lists of disjoint tile ranges merge to the full result, with and
    without a carried threshold array; (b) a threshold array preset to the exact final 2nd best (the
    tightest bound another shard could ever supply) still yields the exact top-2, ties included."""
    from sod_b200 import engine as E
    g = torch.Generator(device="cuda").manual_seed(11)
    for nq, ndb, hi in ((700, 30000, 256), (3000, 9000, 4), (130, 70000, 256)):
        q = torch.randint(0, hi, (nq, 128), dtype=torch.uint8, device="cuda", generator=g)
        db = torch.randint(0, hi, (ndb, 128), dtype=torch.uint8, device="cuda", generator=g)
        db[torch.randint(0, ndb, (64,), device="cuda", generator=g)] = q[:64]
        m = E.Matcher(E.prepare_db(db, index_base=5))
        full_i, full_d = m.top2(q)
        nt = m.n_tiles
        cut = max(1, nt // 8)
        for carry in (False, True):
            thr = m.new_thresholds(nq) if carry else None
            i1, d1 = m.top2(q, (0, cut), thr)
            i2, d2 = m.top2(q, (cut, nt), thr, prepared=True)
            mi, md = E.merge_top2(torch.stack([i1, i2]), torch.stack([d1, d2]))[:2]
            assert torch.equal(mi, full_i) and torch.equal(md, full_d), (nq, ndb, carry)
        # thresholds as tight as they can ever get: d2 of the true 2nd best minus |q|^2
        qn = (q.int() ** 2).sum(1)
        thr = m.new_thresholds(nq)
        thr[:nq] = full_d[:, 1] - qn
        ti, td = m.top2(q, None, thr)
        assert torch.equal(ti, full_i) and torch.equal(td, full_d), (nq, ndb, "preset")
        # an empty range returns empty lists and leaves the thresholds alone
        before = thr.clone()
        ei, ed = m.top2(q, (3, 3), thr)
        assert (ei == -1).all() and torch.equal(thr, before)


def test_key_exchange_equals_list_merge():
    """sod_top2_keys / sod_top2_merge_keys / sod_top2_from_keys with tensor copies standing in for the
    all-to-all and the all-gather: identical to sod_top2_merge over the gathered lists (ties, one-row
    and empty shards, a batch that does not divide by the number of ranks)."""
    from sod_b200 import engine as E
    g = torch.Generator(device="cuda").manual_seed(5)
    nq = 1001
    q = torch.randint(0, 4, (nq, 128), dtype=torch.uint8, device="cuda", generator=g)      # many ties
    db = torch.randint(0, 4, (2500, 128), dtype=torch.uint8, device="cuda", generator=g)
    db[torch.randint(0, 2500, (200,), device="cuda", generator=g)] = q[:200]
    cuts = [0, 1, 1, 900, 2500]                                                             # 1-row and empty shards
    world = len(cuts) - 1
    none = torch.full((nq, 2), -1, dtype=torch.int32, device="cuda")
    lists = [E.Matcher(E.prepare_db(db[a:b].contiguous(), index_base=a)).top2(q) if b > a else (none, none)
             for a, b in zip(cuts[:-1], cuts[1:])]
    want = E.merge_top2(torch.stack([i for i, _ in lists]), torch.stack([d for _, d in lists]))
    per = (nq + world - 1) // world
    keys = [E.top2_keys(i, d, per * world) for i, d in lists]                  # every rank's send buffer
    merged = torch.cat([E.merge_keys(torch.stack([k[r * per:(r + 1) * per] for k in keys]))
                        for r in range(world)])                                # rank r merges slice r; gather
    for got, ref in zip(E.top2_from_keys(merged, nq), want):
        assert torch.equal(got, ref)
    # the engine wrapper on one rank (both collectives are copies) reproduces the single-shard merge
    i1, d1 = E.Matcher(E.prepare_db(db)).top2(q)
    copy = lambda out, inp: out.copy_(inp)  # noqa: E731
    for got, ref in zip(E.exchange_merge_top2(i1, d1, 1, copy, copy), E.merge_top2(i1[None], d1[None])):
        assert torch.equal(got, ref)


def test_peer_exchange_kernels_with_one_rank():
    """sod_top2_exchange_peer with world = 1 (the own buffer is the only peer): the push / flag / merge
    kernels run for real and must reproduce sod_top2_merge of the same single list, call after call (the
    key slots alternate with the call parity); the multi-rank form is tests/dist_check.py."""
    import ctypes as C
    from sod_b200 import engine as E
    from sod_b200._capi import check, lib
    rng = np.random.default_rng(31)
    db = torch.from_numpy(sift_like(rng, 3000)).cuda()
    matcher = E.Matcher(E.prepare_db(db, index_base=500))
    cap = 700
    buf = C.c_void_p()
    check(lib.sod_exchange_alloc(int(lib.sod_exchange_bytes(cap, 1)), C.byref(buf)), "sod_exchange_alloc")
    table = (C.c_void_p * 1)(buf.value)
    try:
        for call, nq in enumerate((700, 1, 333, 700)):
            q = torch.from_numpy(sift_like(rng, nq)).cuda()
            if nq > 10:
                q[:10] = db[100:110]
            idx, d2 = matcher.top2(q)
            want = E.merge_top2(idx[None], d2[None])
            oi = torch.empty_like(idx); od = torch.empty_like(d2)
            of = torch.empty((nq, 2), dtype=torch.float32, device="cuda"); ok = torch.empty(nq, dtype=torch.uint8, device="cuda")
            check(lib.sod_top2_exchange_peer(E._ptr(idx), E._ptr(d2), nq, 0, 1, C.cast(table, C.c_void_p), cap,
                                             E._ptr(oi), E._ptr(od), E._ptr(of), E._ptr(ok), 0.75, E._stream()),
                  "sod_top2_exchange_peer")
            for g, w in zip((oi, od, of, ok), want):
                assert torch.equal(g, w), f"call {call}"
        rc = lib.sod_top2_exchange_peer(E._ptr(idx), E._ptr(d2), cap + 1, 0, 1, C.cast(table, C.c_void_p), cap,
                                        E._ptr(oi), E._ptr(od), None, None, 0.75, E._stream())
        assert rc == -1 and b"capacity" in lib.sod_last_error()
    finally:
        torch.cuda.synchronize()
        check(lib.sod_exchange_free(buf), "sod_exchange_free")


def test_threshold_publishing_with_rotated_block_order():
    """sod_match_top2_peer on ONE GPU playing two ranks in turn: rank 0 sweeps shard 0 and min-reduces every
    finished block's 2nd best into both ranks' arrays, rank 1 then sweeps shard 1 with those bounds (and a
    rotated block order).  The merged result equals the unsharded one; the bounds really travelled (rank 1's
    array holds rank 0's values before rank 1 starts) and really pruned (rank 1 returns fewer candidates)."""
    import ctypes as C
    from sod_b200 import engine as E
    from sod_b200._capi import lib
    nq, ndb = 151_552, 20_000               # 296 block pairs = 4 full waves of 74 clusters: single-segment sweeps
    g = torch.Generator(device="cuda").manual_seed(5)
    def sift_gpu(n):
        x = torch.randn((n, 128), device="cuda", generator=g).abs_()
        x /= x.norm(dim=1, keepdim=True); x.clamp_(max=0.2); x /= x.norm(dim=1, keepdim=True)
        return (x * 512).round_().clamp_(0, 255).to(torch.uint8)
    db, q = sift_gpu(ndb), sift_gpu(nq)
    q[:500] = db[torch.randint(0, ndb, (500,), device="cuda", generator=g)]
    whole_i, whole_d = E.Matcher(E.prepare_db(db)).top2(q)
    half = ndb // 2
    m0 = E.Matcher(E.prepare_db(db[:half].contiguous(), index_base=0))
    m1 = E.Matcher(E.prepare_db(db[half:].contiguous(), index_base=half))
    thr0, thr1 = m0.new_thresholds(nq), m1.new_thresholds(nq)
    table = (C.c_void_p * 2)(thr0.data_ptr(), thr1.data_ptr())
    blocks = (nq + 255) // 256
    i0, d0 = m0.top2(q, None, thr0, peer_table=table, block_rotation=0)
    torch.cuda.synchronize()
    assert torch.equal(thr0, thr1) and int((thr1[:nq] < 0x7F7F7F7F).sum()) == nq    # published to both arrays
    qn = (q.int() ** 2).sum(1)
    # what was published: the smaller of the 2nd bests of the row's two threads (each sees every other tile) -
    # never below the shard's true 2nd best, and equal to it for most rows
    second0 = d0[:, 1] - qn
    assert bool((thr0[:nq] >= second0).all()) and float((thr0[:nq] == second0).float().mean()) > 0.3
    i1, d1 = m1.top2(q, None, thr1, peer_table=table, block_rotation=blocks // 2)
    plain_i1, _ = m1.top2(q)
    assert int((i1 < 0).sum()) > int((plain_i1 < 0).sum())                           # the bounds pruned candidates
    mi, md, _, _ = E.merge_top2(torch.stack([i0, i1]), torch.stack([d0, d1]))
    assert torch.equal(mi, whole_i) and torch.equal(md, whole_d)
    assert torch.equal(thr0, thr1)
    full_second = whole_d[:, 1] - qn
    assert bool((thr0[:nq] >= full_second).all())                                    # always upper bounds
