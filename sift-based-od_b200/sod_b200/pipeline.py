"""Array-level public API of the hot path: match -> ratio -> Hough -> affine for a batch of query
frames against a (possibly sharded) model database.  This is what bench.py and multi-GPU callers
use; main.Main is the object-level drop-in on top of the same engine.

Multi-GPU (SURVEY.md §8e): one process per GPU; the database rows are split contiguously and
object-aligned across ranks, the query batch is replicated, every rank computes shard-local top-2
with global indices, and one exchange merges them: packed (d2, row) keys go to the rank that merges
their slice of the query rows (all-to-all), the merged slices are gathered (sod_top2_keys /
sod_top2_merge_keys / sod_top2_from_keys) - or, exchange="gather", every rank gathers all lists and
merges them itself (sod_top2_merge); both reproduce the single-GPU result, ties included.  The bf16
path uses the gather form with sod_top2_merge_f32.  Each rank then runs Hough + affine for the matches of its own objects only.
There is no other collective.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from . import engine as E


def shard_bounds(n_objects: int, rows_per_object: np.ndarray | int, rank: int, world: int) -> tuple[int, int, int, int]:
    """Object-aligned contiguous split -> (obj_lo, obj_hi, row_lo, row_hi) of `rank`."""
    obj_lo = n_objects * rank // world
    obj_hi = n_objects * (rank + 1) // world
    if np.isscalar(rows_per_object):
        return obj_lo, obj_hi, obj_lo * int(rows_per_object), obj_hi * int(rows_per_object)
    starts = np.concatenate([[0], np.cumsum(rows_per_object)])
    return obj_lo, obj_hi, int(starts[obj_lo]), int(starts[obj_hi])


SEED_ROWS = 16384          # size of the threshold-seeding sample of a database sharded over 8 ranks
SEED_ROWS_PER_RANK = 2048  # default sample size = this x world: a rank seeds 1/world of the query rows, so the
                           # seeding sweep costs every rank the same ~0.45 ms per 1.28 M query rows
SEED_MIN_DB_ROWS = 262144  # smaller databases are not seeded by default: the sweep is short anyway
SEED_MIN_QUERIES = 65536   # smaller batches skip the seeding sweep: a launch and an all-reduce cost more
PEER_MAX_QUERIES = 65536   # largest batch whose shard merge goes through peer memory (exchange="auto" / "peer")
QUERY_BLOCK = 256          # query rows per matcher unit: threshold slices must start on this boundary


def seed_sample_rows(n_db_rows: int, n_seed: int = SEED_ROWS) -> np.ndarray:
    """Row numbers of the seeding sample: an even stride over the WHOLE database (the same on every rank)."""
    n_seed = min(int(n_seed), int(n_db_rows))
    return (np.arange(n_seed, dtype=np.int64) * int(n_db_rows)) // max(n_seed, 1)


def seed_query_slice(n_query: int, rank: int, world: int) -> tuple[int, int]:
    """The query rows whose thresholds `rank` establishes on the seeding sample: whole matcher blocks,
    split evenly; the slices of all ranks tile [0, n_query)."""
    blocks = (int(n_query) + QUERY_BLOCK - 1) // QUERY_BLOCK
    lo = blocks * rank // world * QUERY_BLOCK
    hi = blocks * (rank + 1) // world * QUERY_BLOCK
    return min(lo, int(n_query)), min(hi, int(n_query))


def local_hough_spaces(object_of_image, obj_lo: int, obj_hi: int) -> tuple[np.ndarray, int]:
    """Hough spaces of one rank of a database-sharded run: only the rank's own objects [obj_lo, obj_hi)
    can receive votes there, so they are numbered 0..n_local-1 -> (image_group int32 [n_images],
    n_local).  object_of_image: the object of every model image (an int n means n images, each its own
    object).  Images of other ranks never occur in the rank's matches; they map to space 0."""
    n_local = max(int(obj_hi) - int(obj_lo), 1)
    obj = np.arange(object_of_image, dtype=np.int64) if np.isscalar(object_of_image) else \
        np.asarray(object_of_image).astype(np.int64)
    grp = obj - int(obj_lo)
    grp[(grp < 0) | (grp >= n_local)] = 0
    return grp.astype(np.int32), n_local


def global_space_ids(local_ids: np.ndarray, n_local: int, n_objects: int, obj_lo: int) -> np.ndarray:
    """Rank-local space ids (frame * n_local + local object) -> the single-GPU numbering
    (frame * n_objects + object)."""
    local_ids = np.asarray(local_ids).astype(np.int64)
    return ((local_ids // n_local) * n_objects + obj_lo + local_ids % n_local).astype(np.int32)


@dataclass
class ModelDatabase:
    """Host-side description of the model database (what GenerateDatabaseInfo pickles, as arrays)."""
    des: np.ndarray | torch.Tensor   # u8 [N,128]
    xy: np.ndarray                   # f32 [N,2]
    angle: np.ndarray                # f32 [N]
    octave: np.ndarray               # i32 [N]
    image: np.ndarray                # i32 [N] model image (= object) of each row, non-decreasing
    img_centroid: np.ndarray         # f64 [n_images,2]
    img_size: np.ndarray             # [n_images,2] (w,h)
    object_of_image: np.ndarray | None = None   # i32 [n_images] object of every model image, non-decreasing;
                                                # None = the reference's database: training views of ONE object


class DetectionPipeline:
    def __init__(self, db: ModelDatabase, max_queries: int, frame_wh: np.ndarray, rank: int = 0,
                 world: int = 1, group=None, bins: int = 15, vote_threshold: int = 5,
                 affine_threshold: int = 4, per_object_spaces: bool | None = None,
                 device: str | torch.device = "cuda", shard: str = "db", seed_rows: int | None = None,
                 exchange: str = "auto", replicated_host: bool = True, result_rows: str = "all",
                 sweep_stages: int | None = None, thresholds: str = "auto"):
        """Hough spaces.  The reference votes ALL model images into one dict (main.py:30,113-119: the
        database is several training views of one object), and that is the default here: one space
        per frame.  A multi-object database names the object of every model image in
        db.object_of_image; every (frame, object) pair then gets its own space (SURVEY Q7: the key is
        extended to (object, pose); with one object it is the reference).  per_object_spaces=None
        follows the database (object map present -> per object); True without a map treats every image
        as its own object; False forces the single space.
        shard="db": database rows split over the ranks at object boundaries, one exchange of the
        shard-local top-2 (SURVEY §8e); needs per-object spaces when world > 1, because the votes of
        one space must meet on one rank.  shard="frames": database replicated on every rank, the caller
        gives each rank its own frames (no collective at all); the pipeline then behaves exactly like a
        single-GPU one.
        seed_rows (shard="db", several ranks): size of a replicated sample of the whole database that
        seeds the pruning thresholds (see detect_device); 0 = off; None = 0 with the thresholds in peer memory,
        SEED_ROWS_PER_RANK x world with the NCCL form, when the database has at least SEED_MIN_DB_ROWS rows.  Batches below SEED_MIN_QUERIES rows skip the seeding sweep.
        thresholds (seeded runs): how the ranks share pruning thresholds.  "peer" = over peer memory
        (sod_match_top2_peer): a sweep min-reduces the 2nd best of every finished query block into every rank's
        array with reductions over NVLink, and rank r visits the blocks in an order rotated by r/G, so that
        each block is swept with what the earlier visitors found in their shards - no all-reduce, no stages;
        "allreduce" = NCCL MIN all-reduces after the seeding sweep and between sweep_stages tile ranges;
        "auto" = peer where the node can map peer memory, else allreduce.
        sweep_stages (thresholds="allreduce" only): the shard sweep runs in this many tile ranges with a MIN all-reduce
        of the thresholds between them - after half of every shard the bound is the best 2nd best any rank
        has seen in half of the WHOLE database (B200, 8 x 125k rows: 14.5 ms in two stages against 15.7 ms
        in one, profiles/r02_seed_staged.txt); None = 2 for shards of up to 262,144 rows, else 1.
        replicated_host (shard="db", several ranks): every rank is handed the same HOST batch, so each
        uploads only its 1/G slice of the rows over its own PCIe link and one all-gather over NVLink
        replicates it on the devices (load_queries); False = every rank uploads the whole batch.
        result_rows (shard="db", several ranks): "all" = fetch() returns the match lists of every query
        row on every rank; "own" = only the rows of the rank's slice (out["row_lo"] is the first), which
        is all a caller that collects the ranks' answers needs.
        exchange (shard="db"): "scatter" = all-to-all of packed keys, slice merge, all-gather of the merged
        slices (NCCL); "gather" = all-gather of every rank's lists + sod_top2_merge on every rank (NCCL);
        "peer" = packed keys stored straight into every rank's exchange buffer over NVLink + a flag barrier,
        two kernels and no collective call (sod_b200/peer.py; batches up to PEER_MAX_QUERIES rows);
        "auto" (default) = peer for batches up to PEER_MAX_QUERIES rows, scatter above (G x 16 B per row
        and rank against 2 x 16 B) - and scatter throughout if the node cannot map peer memory
        (self.peer_error says why)."""
        if shard not in ("db", "frames"):
            raise ValueError("shard must be 'db' or 'frames'")
        if exchange not in ("scatter", "gather", "peer", "auto"):
            raise ValueError("exchange must be 'auto', 'peer', 'scatter' or 'gather'")
        if result_rows not in ("all", "own"):
            raise ValueError("result_rows must be 'all' or 'own'")
        if thresholds not in ("auto", "peer", "allreduce"):
            raise ValueError("thresholds must be 'auto', 'peer' or 'allreduce'")
        self.exchange = exchange
        self.replicated_host, self.result_rows = bool(replicated_host), result_rows
        self.seed_min_queries = SEED_MIN_QUERIES
        self._sweep_stages_arg = sweep_stages
        self.shard_mode = shard
        if shard == "frames":
            rank, world = 0, 1
        self.rank, self.world, self.group = rank, world, group
        self.device = torch.device(device)
        self.bins, self.vote_threshold, self.affine_threshold = bins, vote_threshold, affine_threshold
        n_images = int(db.img_centroid.shape[0])
        image = np.asarray(db.image)
        if np.any(np.diff(image) < 0):
            raise ValueError("database rows must be grouped by model image")
        if per_object_spaces is None:
            per_object_spaces = db.object_of_image is not None
        if per_object_spaces:
            obj_of_img = (np.arange(n_images, dtype=np.int32) if db.object_of_image is None
                          else np.asarray(db.object_of_image).astype(np.int32))
            if obj_of_img.shape != (n_images,) or np.any(np.diff(obj_of_img) < 0) or (n_images and obj_of_img[0] < 0):
                raise ValueError("object_of_image must give a non-decreasing object id >= 0 for every model image")
        else:
            obj_of_img = np.zeros(n_images, np.int32)
        if world > 1 and not per_object_spaces:
            # one Hough space for all model images: its votes would be spread over the ranks and never
            # meet in a bin, so counts, thresholds and running means would differ from one GPU
            raise ValueError("shard='db' over several ranks needs per-object Hough spaces (give the database an "
                             "object_of_image map); use shard='frames' for the reference's single space")
        n_objects = int(obj_of_img.max()) + 1 if n_images else 1
        rows = np.bincount(obj_of_img[image], minlength=n_objects) if len(image) else np.zeros(n_objects, np.int64)
        self.obj_lo, self.obj_hi, self.row_lo, self.row_hi = shard_bounds(n_objects, rows, rank, world)
        des = db.des[self.row_lo:self.row_hi]
        des_dev = (des if isinstance(des, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(des)))
        des_dev = des_dev.to(self.device).contiguous()
        # u8 descriptors (what OpenCV SIFT produces) take the exact kind::i8 matcher; float32 descriptors
        # the bf16 path with its stated tolerance (include/sod.h) - queries must then be float32 too.
        self.float_path = des_dev.dtype == torch.float32
        self.seed_matcher = None
        if self.float_path:
            self.shard = E.prepare_db_float(des_dev, index_base=self.row_lo)
            self.matcher = E.FloatMatcher(self.shard)
        else:
            self.shard = E.prepare_db(des_dev, index_base=self.row_lo)
            self.matcher = E.Matcher(self.shard)
        # two stages pay on short shard sweeps (<= 256k rows: 8 ranks x 125k gain 1.1 ms of 15.7); on a 500k-row
        # shard the second launch costs what the tighter bound saves (measured at 2 ranks)
        self.sweep_stages = (2 if self.row_hi - self.row_lo <= 262144 else 1) if self._sweep_stages_arg is None \
            else max(1, int(self._sweep_stages_arg))
        self.max_queries = int(max_queries)
        # capacity of the query-side buffers: whole slices of ceil(n / world) rows for every n <= max_queries
        nq = self.max_queries + (world - 1 if world > 1 else 0)
        dev = self.device
        # query-side device buffers (filled by copy for host inputs, pointers stay stable)
        self.q_des = torch.empty((nq, 128), dtype=torch.float32 if self.float_path else torch.uint8, device=dev)
        # One Hough space per (frame, object) - or per frame.  Results number them frame * spaces_per_frame +
        # object; on the device a rank only carries the spaces of its own objects (the Hough stage scans
        # all spaces of a batch, and a rank of a database-sharded run owns 1/G of the objects).
        self.n_images = n_images
        self.n_objects = n_objects
        self.spaces_per_frame = n_objects if per_object_spaces else 1
        img_group, self._local_spaces = (local_hough_spaces(obj_of_img, self.obj_lo, self.obj_hi)
                                         if per_object_spaces else (None, 1))
        self.scene = E.SceneArrays(
            torch.zeros((nq, 2), dtype=torch.float32), torch.zeros(nq, dtype=torch.float32),
            torch.zeros(nq, dtype=torch.int32), db.xy, db.angle, db.octave, db.image, db.img_centroid,
            np.asarray(db.img_size, np.float64), frame_wh, q_frame=torch.zeros(nq, dtype=torch.int32),
            img_group=img_group, groups_per_frame=self._local_spaces, device=dev)
        self.voter = E.HoughVoter(self.scene, bins)
        # Outputs of the Hough and affine stages are sized ONCE for max_queries: a later, larger batch
        # must never meet buffers that were sized for an earlier, smaller one.
        # Two sets, alternating with the query-buffer set: detect_batches keeps step i+1 enqueued while the
        # results of step i are read back.
        self._hough = [self.voter.reserve(self.max_queries), None]
        self._aff = [E.AffineResult(self._hough[0], self.vote_threshold, self.device), None]
        # two sets of query-side buffers: set 0 is the one allocated above; set 1 appears on first use
        self._qsets = [dict(des=self.q_des, xy=self.scene.q_xy, angle=self.scene.q_angle,
                            octave=self.scene.q_octave, frame=self.scene.q_frame), None]
        self._copy_stream = None
        self._fetch_stream = None
        self._pinned: dict = {}
        self._loaded = [None, None]      # event: the set's host->device copies have landed
        self._consumed = [None, None]    # event: the kernels that read the set have been enqueued and finished
        self.peer, self.peer_error = None, None
        if world > 1 and not self.float_path and self.exchange in ("peer", "auto"):
            from .peer import PeerExchange
            try:
                self.peer = PeerExchange(min(self.max_queries, PEER_MAX_QUERIES), rank, world, group, dev)
            except Exception as exc:      # e.g. a container that forbids CUDA IPC between its processes
                if self.exchange == "peer":
                    raise
                self.peer_error = repr(exc)
        self.peer_thr = None
        self.share_thresholds = (world > 1 and not self.float_path and
                                 (bool(seed_rows) or len(image) >= SEED_MIN_DB_ROWS or thresholds == "peer"))
        if self.share_thresholds and thresholds in ("auto", "peer"):
            from .peer import PeerThresholds
            try:
                self.peer_thr = PeerThresholds(self.max_queries, rank, world, group, dev)
            except Exception as exc:
                if thresholds == "peer":
                    raise
                self.peer_error = repr(exc)
        # Database-sharded runs may keep a small even sample of the WHOLE database on every rank; it only seeds
        # pruning thresholds (detect_device).  With the thresholds in peer memory the default is NO sample: the
        # rotation makes every rank the first visitor of 1/G of the query blocks, and sweeping those without a
        # seed costs less than the seeding sweep (8 x 125k rows: 13.4 ms per step against 13.8).  The choice
        # depends on the whole database and on the arguments alone, so it is the same on every rank.
        if not self.float_path:
            if seed_rows is None:
                seed_rows = 0 if (self.peer_thr is not None or len(image) < SEED_MIN_DB_ROWS) else \
                    SEED_ROWS_PER_RANK * world
            if world > 1 and seed_rows > 0:
                rows = seed_sample_rows(len(image), seed_rows)
                sample = db.des[torch.from_numpy(rows)] if isinstance(db.des, torch.Tensor) else \
                    torch.from_numpy(np.ascontiguousarray(np.asarray(db.des)[rows]))
                self.seed_matcher = E.Matcher(E.prepare_db(sample.to(self.device).contiguous(), index_base=0))
        self._graphs: dict = {}
        self._poses: dict = {}           # capacity -> engine.FinalPoses of final_poses_device
        if world > 1 and (self.float_path or self.exchange == "gather"):
            self._gather_idx = torch.empty((world, self.max_queries, 2), dtype=torch.int32, device=dev)
            self._gather_d2 = torch.empty((world, self.max_queries, 2),
                                          dtype=torch.float32 if self.float_path else torch.int32, device=dev)
        # our kernels per detect_device call (see DESIGN.md); the key exchange of a database-sharded run is
        # three kernels instead of the one merge, a seeding sweep adds the norms of its query slice, one
        # match launch and its list merge
        # (18 = norms, match, list merge, ratio merge, 3 x compaction, pose, scan, scatter, vote, 3 x finish, 3 x affine,
        # records; +2 when the Hough spaces of a batch need the tiled three-launch scan)
        self.launches_per_call = 18 + (2 if self.scene.n_groups > 16384 else 0) + \
            (2 if world > 1 and not self.float_path and exchange != "gather" else 0) + \
            (3 + (3 if self.sweep_stages > 1 and self.peer_thr is None else 0) if self.seed_matcher is not None else 0)

    # ---------------------------------------------------------------- device-resident inputs
    def _qset(self, slot: int) -> dict:
        if self._qsets[slot] is None:
            self._qsets[slot] = {k: torch.empty_like(v) for k, v in self._qsets[0].items()}
        return self._qsets[slot]

    def own_rows(self, n: int) -> tuple[int, int, int]:
        """(rows per slice, first row, end row) of the slice of an n-row batch this rank uploads and,
        with result_rows="own", answers for."""
        if self.world == 1:
            return n, 0, n
        per = (n + self.world - 1) // self.world
        lo = min(self.rank * per, n)
        return per, lo, min(lo + per, n)

    def load_queries(self, des, xy, angle, octave, frame, slot: int = 0, overlap: bool = False) -> int:
        """Copy one batch of query frames (host or device arrays) into query-buffer set `slot`.
        overlap=True issues the copies on the pipeline's copy stream, so that (with pinned host
        memory) they run while the kernels of the other set are busy; detect_device(n, slot) waits
        for them on the device.  Database-sharded over several ranks with replicated_host: a HOST
        batch is the same on every rank (the query is broadcast, SURVEY §8e), so each rank uploads
        rows [lo, hi) of it only and an all-gather over NVLink fills in the rest."""
        n = int(des.shape[0])
        if n > self.max_queries:
            raise ValueError("batch larger than max_queries")
        t = lambda a: a if isinstance(a, torch.Tensor) else torch.from_numpy(a)  # noqa: E731
        srcs = (("des", t(des)), ("xy", t(xy)), ("angle", t(angle)), ("octave", t(octave)), ("frame", t(frame)))
        q = self._qset(slot)
        if overlap and self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(self.device)
        stream = self._copy_stream if overlap else torch.cuda.current_stream(self.device)
        if overlap:
            stream.wait_stream(torch.cuda.current_stream(self.device)) if self._consumed[slot] is None else \
                stream.wait_event(self._consumed[slot])
        sliced = (self.world > 1 and self.shard_mode == "db" and self.replicated_host and n > 0 and
                  not any(a.is_cuda for _, a in srcs))
        with torch.cuda.stream(stream):
            if sliced:
                import torch.distributed as dist
                per, lo, hi = self.own_rows(n)
                for key, src in srcs:
                    q[key][lo:hi].copy_(src[lo:hi], non_blocking=True)
                for key, _ in srcs:      # in place: this rank's slice already sits at its offset
                    buf = q[key][:per * self.world]
                    dist.all_gather_into_tensor(buf, buf[self.rank * per:(self.rank + 1) * per], group=self.group)
            else:
                for key, src in srcs:
                    q[key][:n].copy_(src, non_blocking=True)
            if overlap:
                self._loaded[slot] = torch.cuda.Event()
                self._loaded[slot].record(stream)
        if not overlap:
            self._loaded[slot] = None
        return n

    def detect_replay(self, n: int, slot: int = 0):
        """detect_device(n, slot) as ONE CUDA-graph launch: the ~20 kernels of a small batch are launch-bound
        (BASELINE configs[2]: 10k query rows), so the first call with a given (n, slot) runs the path a few
        times, captures it, and every later call replays the graph.  The result tensors are the graph's own
        and are overwritten by the next replay.  All ranks of a database-sharded run must call it alike.
        Batches that would use an NCCL exchange or threshold seeding are not captured (they are not
        launch-bound): they fall through to detect_device."""
        uses_nccl = self.world > 1 and not (self.peer is not None and n <= self.peer.max_query)
        # shared thresholds alternate between two arrays on the HOST side (PeerThresholds.begin_batch): a
        # captured graph would freeze one of them
        shares = (self.seed_matcher is not None or self.peer_thr is not None) and n >= self.seed_min_queries
        if uses_nccl or shares or n == 0:
            return self.detect_device(n, slot)
        cur = torch.cuda.current_stream(self.device)
        if self._loaded[slot] is not None:
            cur.wait_event(self._loaded[slot])
        entry = self._graphs.get((n, slot))
        if entry is None:
            side = torch.cuda.Stream(self.device)
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                for _ in range(3):
                    self.detect_device(n, slot, _events=False)
            cur.wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                result = self.detect_device(n, slot, _events=False)
            entry = self._graphs[(n, slot)] = (graph, result)
        entry[0].replay()
        self._consumed[slot] = torch.cuda.Event()
        self._consumed[slot].record()
        return entry[1]

    def detect_device(self, n: int, slot: int = 0, _events: bool = True, n_dev: torch.Tensor | None = None):
        """Run the path on the first n rows of query-buffer set `slot`; everything stays on the device.
        n_dev (device int32 [1], at most n): the true row count, read on the device.  The matcher and the ratio
        merge then run on all n rows, and only the compaction reads n_dev: matches of rows past it are dropped,
        so those rows may hold anything (a captured graph's previous frame)."""
        qs = self._qset(slot)
        if _events and self._loaded[slot] is not None:
            torch.cuda.current_stream(self.device).wait_event(self._loaded[slot])
        sc = self.scene
        self.q_des, sc.q_xy, sc.q_angle, sc.q_octave, sc.q_frame = (qs["des"], qs["xy"], qs["angle"], qs["octave"],
                                                                    qs["frame"])
        q = self.q_des[:n]
        merge = E.merge_top2_float if self.float_path else E.merge_top2
        if (self.seed_matcher is not None or self.peer_thr is not None) and n >= self.seed_min_queries:
            # Threshold seeding.  A shard-local sweep has to establish every query row's pruning threshold
            # from scratch - about 2 ln(rows) slow-path updates per row and SHARD, i.e. G times the
            # threshold work of one GPU holding the whole database.  Instead every rank sweeps the small
            # replicated sample of the whole database for 1/G of the query rows only, the ranks min-reduce
            # the thresholds (4 B per query row), and each rank sweeps its shard with the bound of a global
            # sample from its first tile on.  The sample's rows are database rows, so its 2nd best is an
            # upper bound of the final 2nd best and pruning with it is exact (ties pass); the sample's own
            # candidate lists are dropped - every sample row is found again by the rank that owns it.
            import torch.distributed as dist
            s_lo, s_hi = seed_query_slice(n, self.rank, self.world)
            if self.peer_thr is not None:
                # Thresholds over peer memory.  The seeding sweep publishes the bounds of this rank's slice of the
                # query rows into every rank's array; the shard sweep starts with the blocks of that same slice
                # (rotation r/G) and publishes every finished block's 2nd best to everybody: a rank reaches the
                # other slices after their seeds - and the other ranks' shard results for them - have arrived.
                thr = self.peer_thr.begin_batch()
                if self.seed_matcher is not None and s_hi > s_lo:
                    self.seed_matcher.top2(q[s_lo:s_hi], None, thr[s_lo:], peer_table=self.peer_thr.table(s_lo))
                blocks = (n + QUERY_BLOCK - 1) // QUERY_BLOCK
                idx, d2 = self.matcher.top2(q, None, thr, peer_table=self.peer_thr.table(0),
                                            block_rotation=blocks * self.rank // self.world)
                return self._after_match(idx, d2, n, slot, _events, merge, n_dev)
            thr = self.matcher.new_thresholds(n)       # (reached with a seed sample only: the NCCL form)
            if s_hi > s_lo:
                self.seed_matcher.top2(q[s_lo:s_hi], None, thr[s_lo:])
            dist.all_reduce(thr, op=dist.ReduceOp.MIN, group=self.group)
            # The shard sweep in stages: between two tile ranges the ranks min-reduce their thresholds again.
            # Every rank's value is the 2nd best of rows it has really seen (or the seed's), so the minimum is
            # still an upper bound of the final 2nd best; after the first half of every shard it is nearly the
            # final one, and the second half runs almost without top-2 updates.
            tiles = self.matcher.n_tiles
            stages = min(self.sweep_stages, max(tiles, 1))
            cuts = [tiles * k // stages for k in range(stages + 1)]
            parts = []
            for k in range(stages):
                parts.append(self.matcher.top2(q, (cuts[k], cuts[k + 1]), thr, prepared=k > 0))
                if k + 1 < stages:
                    dist.all_reduce(thr, op=dist.ReduceOp.MIN, group=self.group)
            if stages == 1:
                idx, d2 = parts[0]
            else:
                idx, d2, _, _ = E.merge_top2(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]))
        else:
            idx, d2 = self.matcher.top2(q)
        return self._after_match(idx, d2, n, slot, _events, merge, n_dev)

    def _after_match(self, idx, d2, n: int, slot: int, _events: bool, merge, n_dev=None):
        """Exchange of the shard-local lists, compaction, Hough, affine (the rest of detect_device)."""
        if self.world > 1 and self.peer is not None and n <= self.peer.max_query:
            # The exchange through peer memory: two kernels, no collective call (sod_b200/peer.py).
            idx, d2, dist_f, ok = self.peer.merge(idx, d2)
        elif self.world > 1 and not self.float_path and self.exchange != "gather":
            # The exchange (SURVEY §8e) in scatter form: candidates travel as signed 64-bit keys
            # (d2 << 32 | global row), rank r merges the query rows of slice r from all ranks
            # (all-to-all), the merged slices are gathered: 2 x 16 B per query row instead of G x 16 B.
            import torch.distributed as dist
            idx, d2, dist_f, ok = E.exchange_merge_top2(
                idx, d2, self.world,
                lambda out, inp: dist.all_to_all_single(out, inp, group=self.group),
                lambda out, inp: dist.all_gather_into_tensor(out, inp, group=self.group))
        elif self.world > 1:
            import torch.distributed as dist
            gi, gd = self._gather_idx[:, :n], self._gather_d2[:, :n]
            if n != self.max_queries:
                gi = torch.empty((self.world, n, 2), dtype=torch.int32, device=self.device)
                gd = torch.empty((self.world, n, 2), dtype=d2.dtype, device=self.device)
            dist.all_gather_into_tensor(gi, idx, group=self.group)
            dist.all_gather_into_tensor(gd, d2, group=self.group)
            idx, d2, dist_f, ok = merge(gi, gd)
        else:
            idx, d2, dist_f, ok = merge(idx[None], d2[None])
        lo, hi = (self.row_lo, self.row_hi) if self.world > 1 else (0, 2 ** 31 - 1)
        mq, mt, n_dev = E.compact_matches(idx, ok, lo, hi, n_dev=n_dev)
        if self._hough[slot] is None:
            self._hough[slot] = self.voter.new_result(self.max_queries)
            self._aff[slot] = E.AffineResult(self._hough[slot], self.vote_threshold, self.device)
        hough = self.voter.vote(mq, mt, n_dev, detail_min_count=self.vote_threshold, result=self._hough[slot])
        aff = E.affine_verify(self.scene, mq, mt, hough, self.vote_threshold, self.affine_threshold,
                              result=self._aff[slot])
        records = aff.records(hough)        # what fetch() reads of the surviving bins, gathered on the device
        counters = torch.cat([n_dev, hough.counters, aff.counters])
        done = None
        if _events:
            self._consumed[slot] = done = torch.cuda.Event()
            done.record()
        return dict(idx=idx, d2=d2, dist=dist_f, ok=ok, match_q=mq, match_t=mt, n_matches=n_dev,
                    hough=hough, affine=aff, n=n, records=records, counters=counters, done=done)

    # ---------------------------------------------------------------- host in, host out
    def detect(self, des, xy, angle, octave, frame) -> dict:
        """Host buffers in (pinned for full copy speed), host results out."""
        n = self.load_queries(des, xy, angle, octave, frame)
        r = self.detect_device(n)
        return self.fetch(r)

    def detect_batches(self, batches):
        """Host batches in, host results out, pipelined one step deep: while the results of batch i are read
        back, the kernels of batch i+1 are already enqueued (two query-buffer sets, two Hough / affine output
        sets, one copy stream), so neither the host->device copy, nor the device->host read, nor the launch
        overhead of a step leaves the GPU idle.  `batches` yields (des, xy, angle, octave, frame) tuples of
        pinned host arrays; results are yielded in order."""
        it = iter(batches)
        slot = 0
        pending = None
        for batch in it:
            n = self.load_queries(*batch, slot=slot, overlap=True)
            r = self.detect_device(n, slot)
            if pending is not None:
                yield self.fetch(pending)
            pending = r
            slot ^= 1
        if pending is not None:
            yield self.fetch(pending)

    def _host_copy(self, name: str, src: torch.Tensor) -> np.ndarray:
        """src -> a pinned staging buffer (grown on demand) on the fetch stream; the caller synchronises the
        stream and copies the view out before the next fetch reuses the buffer."""
        n = src.numel()
        buf = self._pinned.get(name)
        if buf is None or buf.numel() < n or buf.dtype != src.dtype:
            buf = torch.empty(max(n, 1) * 2, dtype=src.dtype, pin_memory=True)
            self._pinned[name] = buf
        view = buf[:n].view(src.shape)
        view.copy_(src, non_blocking=True)
        return view.numpy()

    def fetch(self, r: dict) -> dict:
        """Device -> host read of one result: matches, counters, verified bins of this rank.  Plain copies on
        a stream of their own that only waits for the step that produced `r`: kernels of a later step that
        are already enqueued (detect_batches) keep running underneath."""
        if self._fetch_stream is None:
            self._fetch_stream = torch.cuda.Stream(self.device)
            self._pinned = {}
        st = self._fetch_stream
        st.wait_event(r["done"]) if r.get("done") is not None else st.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(st):
            c_host = self._host_copy("counters", r["counters"])
            st.synchronize()
            n_m, n_bins, n_votes, n_edge, ovf, n_open = (int(v) for v in c_host[:6])
            n_valid, ovf2, n_singular, n_res_edge = (int(v) for v in c_host[9:13])
            if ovf or ovf2:
                raise RuntimeError("output capacity exceeded")
            a = r["affine"]
            # after the exchange every rank holds the merged lists of ALL query rows; with result_rows="own"
            # a rank reads back only the rows of its slice (the same rows it uploaded)
            _, lo, hi = self.own_rows(r["n"]) if self.result_rows == "own" else (0, 0, r["n"])
            g, code, order, mean = r["records"]
            views = dict(idx=self._host_copy("idx", r["idx"][lo:hi]), ok=self._host_copy("ok", r["ok"][lo:hi]),
                         valid_bin=self._host_copy("valid_bin", a.valid_bin[:n_valid]),
                         params=self._host_copy("params", a.params[:n_valid]),
                         votes=self._host_copy("votes", a.votes[:n_valid]),
                         status=self._host_copy("status", a.status[:n_valid]),
                         valid_group=self._host_copy("valid_group", g[:n_valid]),
                         valid_code=self._host_copy("valid_code", code[:n_valid]),
                         valid_order=self._host_copy("valid_order", order[:n_valid]),
                         valid_mean=self._host_copy("valid_mean", mean[:n_valid]))
            st.synchronize()
        out = {k: v.copy() for k, v in views.items()}
        out.update(row_lo=lo, n_matches=n_m, n_bins=n_bins, n_votes=n_votes, n_near_edge=n_edge,
                   n_unresolved_edge=n_open, n_valid=n_valid, n_singular=n_singular, n_residual_edge=n_res_edge)
        if self._local_spaces != self.spaces_per_frame:
            out["valid_group"] = global_space_ids(out["valid_group"], self._local_spaces, self.n_objects, self.obj_lo)
        return out

    def final_poses(self, out: dict) -> dict[int, list]:
        """Main.post_process (main.py:159-168) for every frame of a fetched result: the bins that
        survived the affine stage are clustered by position and orientation (GPU neighbour graphs,
        sod_b200/postprocess.py) -> {frame: [((cx, cy), orientation, scale, (w, h)), ...]}.  Bins
        enter in the reference's order (Hough insertion order inside a space).  With shard="db"
        this covers the objects of this rank only."""
        from .postprocess import post_process_arrays
        live = (out["status"] & 1).astype(bool)
        group, order, mean = out["valid_group"][live], out["valid_order"][live], out["valid_mean"][live]
        frame = group // self.spaces_per_frame
        o = np.lexsort((order, group, frame))
        mean, frame = mean[o], frame[o].astype(np.int32)
        clusters, _, _, final = post_process_arrays(mean[:, 0], mean[:, 1], mean[:, 3], mean[:, 2], mean[:, 4],
                                                    mean[:, 5], segment=frame, device=self.device)
        poses: dict[int, list] = {}
        for cl, pose in zip(clusters, final):
            poses.setdefault(int(frame[cl[0]]), []).append(pose)
        return poses

    def final_poses_device(self, r: dict, cap: int | None = None) -> dict:
        """final_poses of a detect_device result on the device, with no host step (sod_final_poses_records):
        the live bins of the first min(n_valid, cap) verified bins (cap: the affine output capacity by default,
        at most 65,536) -> device tensors pose float64 [cap][6] (cx, cy, orientation, scale, w, h), frame int32
        [cap], shape_bin int32 [cap] (-1: the reference's (0, 0) shape) and counters int32 [2] (clusters, live
        bins); the first counters[0] rows are the clusters, numbered as final_poses meets them.  The tensors
        belong to `poses` (an engine.FinalPoses kept per capacity) and are overwritten by its next call."""
        if self._local_spaces != self.spaces_per_frame:
            raise ValueError("final_poses_device needs every Hough space of a frame on this rank; a database-sharded "
                             "run with per-object spaces numbers them per rank (use fetch and final_poses)")
        a = r["affine"]
        g, _, order, mean = r["records"]
        k = min(a.cap_valid if cap is None else int(cap), a.cap_valid, E._capi.MAX_CLUSTER_BINS)
        fp = self._poses.get(k)
        if fp is None:
            fp = self._poses[k] = E.FinalPoses(k, self.device)
        fp.run_records(a.status, g, order, mean, k, a.counters[:1], self.spaces_per_frame)
        return dict(pose=fp.pose, frame=fp.segment, shape_bin=fp.shape_bin, counters=fp.counters, poses=fp)

    @staticmethod
    def fetched_bytes(out: dict) -> int:
        return int(sum(v.nbytes for v in out.values() if isinstance(v, np.ndarray)) + 13 * 4)
