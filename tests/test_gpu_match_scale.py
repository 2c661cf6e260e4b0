"""The matcher on every row at the sizes it is measured at and on hostile data, against tests/exact_top2.py.

match_top2_kernel's results depend on the data: the epilogue prunes 32-column chunks against each row's running
2nd best, the database is sorted by |t|^2 and its tiles stored in an interleaved order, thresholds pass between
segments (row_thr), between launches (a caller-held array) and between shards (peer memory), and only the exact
comparison `> thr` lets a tie through.  Every case here compares every row's indices and squared distances with
the exact reference, the ratio flags with the oracle's ratio test on the exact distances, and the kernel's
distances with a direct recomputation; every case asserts the dispatch class (segments, instance) it targets.

  a. the hostile input kinds of tools/bench_match.py x three dispatch classes, each run twice (bit-identical);
  b. bench.py's own batch (1.28M queries x 1M rows) through the matcher and DetectionPipeline, every frame's
     Hough + affine against the oracle;
  c. groups of two and three equidistant database rows whose lowest index is swept last, unsharded (one
     wave and 13 waves of segments sharing row_thr), database-sharded through one caller-held threshold array, and through peer tables;
  d. the bf16 path on integer-valued hostile data, bit-exact.
Each case prints what it asserted and how many rows it compared (run with -s to see it)."""
import ctypes as C
import importlib.util
import time
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from conftest import ROOT
from exact_top2 import chunk_rows, direct_d2, exact_top2, full_fp32_matmul
from oracle import sod_oracle as O

SMS = 148                   # B200
PAIRS = SMS // 2            # the matcher's persistent grid: one CTA pair per TPC
UNIT_ROWS = 1024            # query rows a CTA pair sweeps per unit


def _bench_match():
    spec = importlib.util.spec_from_file_location("bench_match", ROOT / "tools" / "bench_match.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def dispatch(nq: int, rows: int, caller_thr: bool = False) -> tuple[int, str]:
    """(n_seg, instance) sod_match_top2_peer picks for nq queries over `rows` database rows, read back from the
    workspace size: n_seg * nq * 16 + sod_row_thr_ints(nq) * 4 + 16 bytes.  The instance follows the launch's
    rules: "share" when the rows' sweep is split into several segments (they share row_thr), "seeded" for a
    single segment with a caller-held threshold array, "plain" for a single segment without."""
    from sod_b200._capi import lib
    ws = int(lib.sod_match_workspace_bytes(nq, rows))
    n_seg, rem = divmod(ws - 16 - 4 * int(lib.sod_row_thr_ints(nq)), 16 * nq)
    assert rem == 0 and n_seg >= 1, (nq, rows, ws)
    return n_seg, "share" if n_seg > 1 else ("seeded" if caller_thr else "plain")


def waves(nq: int, n_seg: int) -> float:
    return (nq + UNIT_ROWS - 1) // UNIT_ROWS * n_seg / PAIRS


def _first_bad(got_i, got_d, want_i, want_d):
    bad = torch.nonzero((got_i != want_i).any(1) | (got_d != want_d).any(1)).flatten()
    r = bad[:5].tolist()
    return (f"{bad.numel()} rows differ, first {r}: got {got_i[r].tolist()} {got_d[r].tolist()} "
            f"want {want_i[r].tolist()} {want_d[r].tolist()}")


def check_exact(q, db, idx, d2, ok=None, index_base=0, ref=None):
    """Every row's (idx, d2) equals exact_top2, d2 equals the direct recomputation, ok (if given) equals the
    oracle's ratio test on the exact distances.  Returns the reference."""
    ridx, rd2 = exact_top2(q, db, index_base) if ref is None else ref
    assert torch.equal(idx, ridx) and torch.equal(d2, rd2), _first_bad(idx, d2, ridx, rd2)
    dd = direct_d2(q, db, idx, index_base)
    assert torch.equal(dd, d2), _first_bad(idx, dd, idx, d2)
    if ok is not None:
        want = O.ratio_pass(rd2.cpu().numpy().astype(np.int64), ridx.cpu().numpy())
        np.testing.assert_array_equal(ok.cpu().numpy().astype(bool), want)
    return ridx, rd2


# ------------------------------------------------------------------------------------------------
# exact_top2 itself (CPU: rehearsal at toy sizes; GPU: the same plus one medium shape)
# ------------------------------------------------------------------------------------------------
def _oracle_top2(q, db, index_base=0, db_chunk=None):
    """O.knn2 over database chunks of db_chunk rows, merged by O.merge_top2 (as bench.oracle_spot_check)."""
    q, db = q.cpu().numpy(), db.cpu().numpy()
    step = db_chunk or max(len(db), 1)
    pi, pd = [], []
    for s in range(0, len(db), step):
        i, d = O.knn2(q, db[s:s + step])
        pi.append(np.where(i >= 0, i + s + index_base, -1))
        pd.append(d)
    if not pi:
        return np.full((len(q), 2), -1, np.int32), np.full((len(q), 2), -1, np.int64)
    return O.merge_top2(np.stack(pi), np.stack(pd))


def _tie_cases(device):
    g = torch.Generator(device="cpu").manual_seed(3)
    r = lambda hi, n: torch.randint(0, hi, (n, 128), dtype=torch.uint8, generator=g)  # noqa: E731
    out = []
    for hi, nq, ndb in ((2, 40, 300), (4, 70, 257), (2, 33, 1), (4, 9, 2), (256, 5, 1), (256, 17, 2), (4, 20, 0)):
        out.append((r(hi, nq), r(hi, ndb)))
    q, db = r(4, 50), r(4, 400)
    db[[3, 99, 100, 250, 399]] = q[0]          # duplicated rows: lowest index first, also in 2nd place
    db[[7, 8]] = q[1]
    db[200:260] = db[10]                       # one row repeated across chunks
    out.append((q, db))
    return [(a.to(device), b.to(device)) for a, b in out]


def _check_against_oracle(device):
    for k, (q, db) in enumerate(_tie_cases(device)):
        for base, budget in ((0, None), (1000, 12 * 64 * 3)):     # the small budget: blocks of 64 x 3 rows
            kw = {} if budget is None else {"budget": budget}
            idx, d2 = exact_top2(q, db, base, **kw)
            ri, rd = _oracle_top2(q, db, base)
            np.testing.assert_array_equal(idx.cpu().numpy(), ri, err_msg=f"case {k}")
            np.testing.assert_array_equal(d2.cpu().numpy().astype(np.int64), rd, err_msg=f"case {k}")
            assert torch.equal(direct_d2(q, db, idx, base), d2)


def test_exact_top2_equals_oracle_on_ties_cpu():
    """Alphabets of 2 and 4, duplicated rows, 0, 1 and 2 database rows, chunked and whole, with an index base."""
    _check_against_oracle("cpu")


def test_exact_top2_float64_form_cpu():
    g = torch.Generator(device="cpu").manual_seed(4)
    q = torch.randint(0, 256, (300, 128), dtype=torch.uint8, generator=g)
    db = torch.randint(0, 256, (5000, 128), dtype=torch.uint8, generator=g)
    db[:64] = q[:64]
    a = exact_top2(q, db, 7, budget=12 * 128 * 1000)
    b = exact_top2(q, db, 7, dtype=torch.float64)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert torch.equal(direct_d2(q, db, a[0], 7), a[1])


def test_exact_top2_helpers_cpu():
    assert chunk_rows(1_280_000, 1_000_000) == (87381, 16384)
    cq, cd = chunk_rows(1_280_000, 1_000_000)
    assert cq * cd * 12 <= 16 << 30
    before = (torch.get_float32_matmul_precision(), torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        with full_fp32_matmul():
            assert not torch.backends.cuda.matmul.allow_tf32
            assert torch.get_float32_matmul_precision() == "highest"
        assert torch.backends.cuda.matmul.allow_tf32
    finally:
        torch.set_float32_matmul_precision(before[0])
        torch.backends.cuda.matmul.allow_tf32 = before[1]
    # an index outside the database is flagged, never read
    q = torch.zeros((2, 128), dtype=torch.uint8)
    db = torch.ones((3, 128), dtype=torch.uint8)
    assert direct_d2(q, db, torch.tensor([[0, 3], [-1, 2]], dtype=torch.int32)).tolist() == [[128, -2], [-1, 128]]


def test_dispatch_classes_of_the_shapes_used_here():
    """The shapes below land in the classes they are meant for (148 SMs; also what the library assumes
    without a device)."""
    # the adversarial profile's shape: 64 units alone would leave 10 of the 74 pairs idle for 7,819 tile steps;
    # make_plan splits each query block's sweep into 15 segments instead (13 waves of 527 steps)
    assert dispatch(65_536, 1_000_000) == (15, "share")
    n_seg, inst = dispatch(600, 1_000_000)
    assert inst == "share" and n_seg >= 32
    n_seg, inst = dispatch(151_552, 100_000)
    assert inst == "plain" and waves(151_552, n_seg) >= 2
    assert dispatch(151_552, 977 * 128, caller_thr=True) == (1, "seeded")
    assert dispatch(151_552, 3907 * 128, caller_thr=True) == (1, "seeded")
    n_seg, inst = dispatch(1_280_000, 1_000_000)
    assert waves(1_280_000, n_seg) > 16


@pytest.mark.gpu
def test_exact_top2_equals_oracle_on_ties_gpu():
    _check_against_oracle("cuda")


@pytest.mark.gpu
def test_exact_top2_float64_form_gpu():
    g = torch.Generator(device="cuda").manual_seed(5)
    bm = _bench_match()
    q, db = bm.sift_like_gpu(4096, g), bm.sift_like_gpu(262_144, g)
    db[torch.randint(0, 262_144, (512,), device="cuda", generator=g)] = q[:512]
    a = exact_top2(q, db)
    b = exact_top2(q, db, dtype=torch.float64)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert torch.equal(direct_d2(q, db, a[0]), a[1])
    print(f"\n[exact_top2] float32 = float64 form on 4096 x 262144 ({q.shape[0]} rows)")


# ------------------------------------------------------------------------------------------------
# a. hostile legs x dispatch classes
# ------------------------------------------------------------------------------------------------
SHAPES_A = {"adversarial": (65_536, 1_000_000, "share"), "one_unit": (600, 1_000_000, "share"),
            "waves": (151_552, 100_000, "plain")}


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(SHAPES_A))
@pytest.mark.parametrize("kind", ["uniform", "sift", "selfmatch", "cluster", "dup", "noevent"])
def test_hostile_legs_every_row_exact(kind, shape):
    from sod_b200 import engine as E
    nq, ndb, want = SHAPES_A[shape]
    n_seg, inst = dispatch(nq, ndb)
    assert inst == want
    if shape == "adversarial":
        assert n_seg == 15 and waves(nq, n_seg) > 12      # make_plan: 15 segments sharing row_thr, 13 waves
    if shape == "waves":
        assert waves(nq, n_seg) >= 2
    bm = _bench_match()
    q, db = bm.make_inputs(kind, nq, ndb, torch.Generator(device="cuda").manual_seed(1))
    m = E.Matcher(E.prepare_db(db))
    i1, d1 = m.top2(q)
    i2, d2 = m.top2(q)
    ok = E.merge_top2(i1[None], d1[None])[3]
    check_exact(q, db, i1, d1, ok)
    assert torch.equal(i1, i2) and torch.equal(d1, d2), "two runs differ"
    print(f"\n[a] {kind} {nq}x{ndb}: n_seg={n_seg} instance={inst} waves={waves(nq, n_seg):.2f}, "
          f"{nq} rows compared, 2 runs bit-identical")


# ------------------------------------------------------------------------------------------------
# b. bench.py's own batch
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_benchmark_batch_every_row_and_every_frame():
    """bench.make_workload with bench.py's defaults.  Every one of the 1.28M rows of E.Matcher.top2 equals
    exact_top2; DetectionPipeline.detect returns the same idx and ok.  Hough + affine: for EVERY frame the
    scalar oracle (O.hough_vote, O.valid_bins, O.affine_verify) runs on that frame's own matches; its valid
    bins (frame, object, code) and their votes and live flags equal the pipeline's, and the live bins'
    parameters agree within 1e-4."""
    import bench
    from sod_b200 import engine as E
    from sod_b200.pipeline import DetectionPipeline
    args = SimpleNamespace(frames=256, per_frame=5000, objects=1000, kp_per_object=1000, instances=4,
                           inlier_frac=0.10, false_frac=0.01)
    wl = bench.make_workload(args, torch.device("cuda"))
    q, db = wl["q_des"], wl["db_des"]
    nq, ndb = q.shape[0], db.shape[0]
    n_seg, inst = dispatch(nq, ndb)
    assert nq == 1_280_000 and ndb == 1_000_000 and inst == "plain" and waves(nq, n_seg) > 16
    m = E.Matcher(E.prepare_db(db))
    idx, d2 = m.top2(q)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ref = exact_top2(q, db)
    torch.cuda.synchronize()
    t_ref = time.perf_counter() - t0
    ok = E.merge_top2(idx[None], d2[None])[3]
    check_exact(q, db, idx, d2, ok, ref=ref)
    print(f"\n[b] matcher {nq}x{ndb}: n_seg={n_seg} instance={inst} waves={waves(nq, n_seg):.2f}, {nq} rows "
          f"compared; exact_top2 took {t_ref:.1f} s")

    pipe = DetectionPipeline(bench.make_database(wl), nq, wl["frame_wh"])
    res = pipe.detect(q, wl["q_xy"], wl["q_angle"], wl["q_octave"], wl["q_frame"])
    ridx = ref[0].cpu().numpy()
    rok = ok.cpu().numpy().astype(bool)
    np.testing.assert_array_equal(res["idx"], ridx)
    np.testing.assert_array_equal(res["ok"].astype(bool), rok)
    assert res["n_unresolved_edge"] == 0 and res["n_residual_edge"] == 0   # parity is unconditional

    per, spf, bins = args.per_frame, pipe.spaces_per_frame, 15
    assert spf == args.objects
    frame = res["valid_group"] // spf
    live_got = (res["status"] & 1) == 1
    t0 = time.perf_counter()
    n_valid = n_live = n_matches = 0
    for f in range(args.frames):
        rows = np.arange(f * per, (f + 1) * per)
        okf = rok[rows]
        mq, mt = rows[okf], ridx[rows][okf, 0]
        scene = O.Scene(wl["q_xy"], wl["q_angle"], wl["q_octave"], wl["m_xy"], wl["m_angle"], wl["m_octave"],
                        wl["m_image"], wl["img_centroid"], wl["img_size"], int(wl["frame_wh"][f, 0]),
                        int(wl["frame_wh"][f, 1]), np.arange(args.objects, dtype=np.int32))
        valid = O.valid_bins(O.hough_vote(scene, mq.tolist(), mt.tolist(), bins), 5)
        live = {id(b) for b in O.affine_verify(scene, mq.tolist(), mt.tolist(), valid, 4)}
        code = lambda p: ((p[0] * bins + p[1]) * bins + p[2]) * bins + p[3]  # noqa: E731
        want = {(int(b.group), code(b.pose)): (int(b.votes), id(b) in live, b) for b in valid}
        sel = np.flatnonzero(frame == f)
        got = {(int(res["valid_group"][v] % spf), int(res["valid_code"][v])): v for v in sel}
        assert set(got) == set(want), f"frame {f}: valid bins differ"
        for key, (votes, is_live, b) in want.items():
            v = got[key]
            assert (int(res["votes"][v]), bool(live_got[v])) == (votes, is_live), f"frame {f} bin {key}"
            if is_live:
                np.testing.assert_allclose(res["params"][v], b.affine, rtol=1e-4, atol=1e-6,
                                           err_msg=f"frame {f} bin {key}")
        n_valid += len(want)
        n_live += len(live)
        n_matches += len(mq)
    t_oracle = time.perf_counter() - t0
    assert n_live >= args.frames * args.instances // 2
    print(f"[b] pipeline: {nq} rows of idx/ok compared; scalar Hough + affine oracle on all {args.frames} frames "
          f"({n_matches} matches, {n_valid} valid bins, {n_live} live) in {t_oracle:.1f} s of host time")


# ------------------------------------------------------------------------------------------------
# c. ties built to meet the pruning rule
# ------------------------------------------------------------------------------------------------
E_VALUES = (3, -2, 1)           # the offset vector e, |e|^2 = 14, and its permutations
E_NORM = sum(v * v for v in E_VALUES)


CQ_TILE_INTS, CQ_PERM = 260, 132   # include/sod.h: per tile 128 norms, 4 chunk minima, 128 original rows


def _storage_tile(shard, ndb):
    """Original row -> the stored tile that holds it, from the shard's permutation cq[tile * 260 + 132 + col]."""
    perm = shard.cq.view(-1, CQ_TILE_INTS)[:, CQ_PERM:]
    tiles = torch.arange(perm.shape[0], device=perm.device)[:, None].expand_as(perm)
    out = torch.full((ndb,), -1, dtype=torch.int64, device=perm.device)
    have = perm >= 0
    out[perm[have].long()] = tiles[have]
    assert bool((out >= 0).all())
    return out


def _tie_groups(q_np, n_groups, ndb, rng):
    """Group j (query j): 2 or 3 database rows q_j + a permutation of e at distinct distinct positions, at
    random distinct original indices.  -> (rows {index: u8 row}, groups [list of indices])."""
    idx = rng.choice(ndb, 3 * n_groups, replace=False)
    rows, groups, k = {}, [], 0
    for j in range(n_groups):
        qj = q_np[j].astype(np.int16)
        pos = np.flatnonzero((qj >= 3) & (qj <= 252))
        size = 3 if j % 2 == 0 else 2
        made = set()
        members = []
        while len(members) < size:
            p = rng.choice(pos, 3, replace=False)
            t = qj.copy()
            t[p] += np.array(E_VALUES, np.int16)[rng.permutation(3)]
            if t.tobytes() in made:
                continue
            made.add(t.tobytes())
            rows[int(idx[k])] = t.astype(np.uint8)
            members.append(int(idx[k]))
            k += 1
        groups.append(sorted(members))
    return rows, groups


def _write(db, rows):
    keys = torch.tensor(list(rows), dtype=torch.int64, device=db.device)
    db[keys] = torch.from_numpy(np.stack(list(rows.values()))).to(db.device)


def _build_tie_problem(nq, ndb, n_groups, seed, sweep_order=None):
    """Queries and a database with n_groups tie groups.  sweep_order (original row -> position in the sweep,
    or None): the contents of each group are re-assigned so that its lowest index is swept last."""
    bm = _bench_match()
    g = torch.Generator(device="cuda").manual_seed(seed)
    db, q = bm.sift_like_gpu(ndb, g), bm.sift_like_gpu(nq, g)
    rng = np.random.default_rng(seed)
    rows, groups = _tie_groups(q[:n_groups].cpu().numpy(), n_groups, ndb, rng)
    _write(db, rows)
    if sweep_order is not None:
        order = sweep_order(db).cpu().numpy()
        new = {}
        for mem in groups:
            by_sweep = sorted(mem, key=lambda i: -order[i])         # swept last first
            for dst, src in zip(mem, by_sweep):                     # lowest index <- the row swept last
                new[dst] = rows[src]
        rows = new
        _write(db, rows)
    return q, db, groups


def _assert_ties_exact(q, db, groups):
    """The reference sees each group's two lowest indices at |e|^2: no other row is nearer."""
    ridx, rd2 = exact_top2(q, db)
    want = torch.tensor([mem[:2] for mem in groups], dtype=torch.int32, device=q.device)
    assert torch.equal(ridx[:len(groups)], want)
    assert bool((rd2[:len(groups)] == E_NORM).all())
    return ridx, rd2


def _count_lowest_last(groups, order):
    order = order.cpu().numpy()
    return sum(1 for mem in groups if all(order[mem[0]] > order[i] for i in mem[1:]))


@pytest.mark.gpu
@pytest.mark.parametrize("nq,want", [(600, "share"), (65_536, "share")])
def test_ties_lowest_index_swept_last(nq, want):
    from sod_b200 import engine as E
    ndb = 1_000_000
    n_seg, inst = dispatch(nq, ndb)
    assert inst == want
    n_groups = min(nq, 8192)
    n_tiles = (ndb + 127) // 128
    q, db, groups = _build_tie_problem(nq, ndb, n_groups, 21,
                                       sweep_order=lambda d: _storage_tile(E.prepare_db(d), ndb))
    shard = E.prepare_db(db)
    tile = _storage_tile(shard, ndb)
    seg = torch.div(tile * n_seg, n_tiles, rounding_mode="floor")
    # segment s holds the tiles [s * n / n_seg, (s + 1) * n / n_seg): compare (segment, tile) pairs
    later_tile = _count_lowest_last(groups, tile)
    later_seg = _count_lowest_last(groups, seg) if n_seg > 1 else 0
    assert later_tile >= 300 and (n_seg == 1 or later_seg >= 300), (later_tile, later_seg)
    ref = _assert_ties_exact(q, db, groups)
    m = E.Matcher(shard)
    idx, d2 = m.top2(q)
    ok = E.merge_top2(idx[None], d2[None])[3]
    check_exact(q, db, idx, d2, ok, ref=ref)
    print(f"\n[c] ties {nq}x{ndb}: n_seg={n_seg} instance={inst}, {len(groups)} groups, lowest index in a later "
          f"tile for {later_tile}, in a later segment for {later_seg}; {nq} rows compared")


@pytest.mark.gpu
def test_ties_across_shards_swept_in_reverse():
    """Eight object-aligned shards of 125,000 rows swept from the last to the first through ONE caller-held
    threshold array (the seeded instance): the shard with a group's lowest index runs after the others, with
    the threshold already at the tie distance.  Then two halves through sod_match_top2_peer with a two-entry
    peer table and a rotated block order, also the upper half first."""
    from sod_b200 import engine as E
    nq, ndb, per = 151_552, 1_000_000, 125_000
    q, db, groups = _build_tie_problem(nq, ndb, 8192, 22)
    ref = _assert_ties_exact(q, db, groups)
    rows = torch.arange(ndb, device="cuda")
    later = _count_lowest_last(groups, -torch.div(rows, per, rounding_mode="floor"))
    assert later >= 300, later

    thr = None
    parts = [None] * 8
    for r in reversed(range(8)):
        m = E.Matcher(E.prepare_db(db[r * per:(r + 1) * per].contiguous(), index_base=r * per))
        assert dispatch(nq, m.n_tiles * 128, caller_thr=True) == (1, "seeded")
        thr = m.new_thresholds(nq) if thr is None else thr
        parts[r] = m.top2(q, None, thr)
    idx, d2, _, ok = E.merge_top2(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]))
    check_exact(q, db, idx, d2, ok, ref=ref)
    print(f"\n[c] ties {nq}x{ndb} in 8 shards, reverse order, one threshold array: instance=seeded n_seg=1, "
          f"{len(groups)} groups, lowest index in a shard swept later for {later}; {nq} rows compared")

    half = ndb // 2
    later = _count_lowest_last(groups, -torch.div(rows, half, rounding_mode="floor"))
    assert later >= 300, later
    m0 = E.Matcher(E.prepare_db(db[:half].contiguous(), index_base=0))
    m1 = E.Matcher(E.prepare_db(db[half:].contiguous(), index_base=half))
    assert dispatch(nq, m0.n_tiles * 128, caller_thr=True) == (1, "seeded")
    thr0, thr1 = m0.new_thresholds(nq), m1.new_thresholds(nq)
    table = (C.c_void_p * 2)(thr0.data_ptr(), thr1.data_ptr())
    blocks = (nq + 255) // 256
    i1, e1 = m1.top2(q, None, thr1, peer_table=table, block_rotation=0)
    i0, e0 = m0.top2(q, None, thr0, peer_table=table, block_rotation=blocks // 2)
    idx, d2, _, ok = E.merge_top2(torch.stack([i0, i1]), torch.stack([e0, e1]))
    check_exact(q, db, idx, d2, ok, ref=ref)
    assert torch.equal(thr0, thr1)
    print(f"[c] ties {nq}x{ndb} in 2 halves through peer tables, upper half first, rotation {blocks // 2}: "
          f"lowest index in the half swept later for {later}; {nq} rows compared")


# ------------------------------------------------------------------------------------------------
# d. the bf16 path on integer-valued hostile data
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("split", [True, False])
@pytest.mark.parametrize("nq,ndb", [(65_536, 250_000), (600, 1_000_000)])
@pytest.mark.parametrize("kind", ["selfmatch", "cluster", "dup"])
def test_bf16_integer_valued_hostile_bit_exact(kind, nq, ndb, split):
    from sod_b200 import engine as E
    bm = _bench_match()
    q, db = bm.make_inputs(kind, nq, ndb, torch.Generator(device="cuda").manual_seed(1))
    m = E.FloatMatcher(E.prepare_db_float(db.float(), split=split))
    idx, d2f, dist, ok = E.knn_match_ratio_float(q.float(), m)
    assert bool((d2f == d2f.round()).all())
    d2 = d2f.to(torch.int32)
    check_exact(q, db, idx, d2, ok)
    np.testing.assert_array_equal(dist.cpu().numpy(), O.match_distance(d2.cpu().numpy().astype(np.int64)))
    print(f"\n[d] bf16 split={split} {kind} {nq}x{ndb}: {nq} rows compared bit-exact")
