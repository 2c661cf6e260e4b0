"""Host layer over the C ABI: torch owns device memory and streams, every kernel is ours.

Nothing here computes on the CPU; a missing GPU or library raises.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _capi
from ._capi import check, lib

RATIO = 0.75  # main.py:82


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t: torch.Tensor | None) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


def _require_cuda(t: torch.Tensor, dtype: torch.dtype, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise ValueError(f"{name} must live on the GPU (no CPU path exists)")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    return t.contiguous()


def pack_descriptors(des, device: torch.device | str = "cuda") -> torch.Tensor:
    """float32/uint8 [n,128] (numpy or torch, host or device) -> device u8 [n,128].

    OpenCV SIFT descriptors are float32 holding integers 0..255 (SURVEY T1); float input is converted
    on the GPU and rejected if any value is not such an integer.
    """
    t = torch.as_tensor(des)
    if t.ndim != 2 or t.shape[1] != _capi.DESC_DIM:
        raise ValueError(f"descriptors must be [n,{_capi.DESC_DIM}], got {tuple(t.shape)}")
    if t.dtype == torch.uint8:
        return t.to(device, non_blocking=True).contiguous()
    if t.dtype != torch.float32:
        raise TypeError(f"descriptors must be float32 or uint8, got {t.dtype}")
    src = t.to(device, non_blocking=True).contiguous()
    dst = torch.empty(src.shape, dtype=torch.uint8, device=src.device)
    flag = torch.zeros(1, dtype=torch.int32, device=src.device)
    check(lib.sod_pack_u8_from_f32(_ptr(src), src.shape[0], _ptr(dst), _ptr(flag), _stream()),
          "sod_pack_u8_from_f32")
    if int(flag.item()) != 0:
        raise NonIntegerDescriptors("descriptors are not integer-valued in 0..255: the exact u8 tensor-core "
                                    "path does not apply (use prepare_db_float / FloatMatcher)")
    return dst


class NonIntegerDescriptors(ValueError):
    """Raised by pack_descriptors for float descriptors the exact u8 path cannot represent."""


@dataclass
class DescriptorShard:
    """A contiguous slice of the model-descriptor database resident in HBM."""
    des: torch.Tensor        # u8 [tiles*128,128]: rows re-ordered by sod_db_prepare, zero padded
    n_rows: int              # number of real rows
    cq: torch.Tensor         # int32 per tile: |t|^2, chunk minima, original rows
    index_base: int          # global index of original row 0

    @property
    def n(self) -> int:
        return self.n_rows


def prepare_db(des_u8: torch.Tensor, index_base: int = 0) -> DescriptorShard:
    des_u8 = _require_cuda(des_u8, torch.uint8, "database descriptors")
    n = int(des_u8.shape[0])
    dev = des_u8.device
    tiles = (n + _capi.TILE_ROWS - 1) // _capi.TILE_ROWS
    cq = torch.empty(max(int(lib.sod_cq_ints(n)), 1), dtype=torch.int32, device=dev)
    des_sorted = torch.empty((max(tiles * _capi.TILE_ROWS, 1), _capi.DESC_DIM), dtype=torch.uint8, device=dev)
    ws = torch.empty(int(lib.sod_db_prepare_workspace_bytes(n)), dtype=torch.uint8, device=dev)
    check(lib.sod_db_prepare(_ptr(des_u8), n, _ptr(des_sorted), _ptr(cq), _ptr(ws), ws.numel(),
                             _stream()), "sod_db_prepare")
    return DescriptorShard(des_sorted, n, cq, int(index_base))


class Matcher:
    """2-NN matcher for one database shard; reuses its scratch between calls."""

    def __init__(self, shard: DescriptorShard):
        self.shard = shard
        self._ws: torch.Tensor | None = None
        self._qn: torch.Tensor | None = None
        self.events: list | None = None   # if a list: (start, end) CUDA events around sod_match_top2

    @property
    def n_tiles(self) -> int:
        return (self.shard.n + _capi.TILE_ROWS - 1) // _capi.TILE_ROWS

    def new_thresholds(self, nq: int) -> torch.Tensor:
        """A caller-held threshold array for top2(..., row_thr=...): all "none yet"."""
        return torch.full((max(int(lib.sod_row_thr_ints(nq)), 1),), 0x7F7F7F7F, dtype=torch.int32,
                          device=self.shard.des.device)

    def _scratch(self, nq: int, rows: int | None = None) -> tuple[torch.Tensor, torch.Tensor]:
        need = int(lib.sod_match_workspace_bytes(nq, self.shard.n if rows is None else rows))
        dev = self.shard.des.device
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=dev)
        if self._qn is None or self._qn.numel() < nq:
            self._qn = torch.empty(max(nq, 1), dtype=torch.int32, device=dev)
        return self._ws, self._qn

    def top2(self, q_u8: torch.Tensor, tiles: tuple[int, int] | None = None, row_thr: torch.Tensor | None = None,
             prepared: bool = False, peer_table=None, block_rotation: int = 0) -> tuple[torch.Tensor, torch.Tensor]:
        """-> (idx int32 [nq,2] global rows or -1, d2 int32 [nq,2] squared distances, -1 if none).
        tiles=(begin, end): sweep only these stored 128-row tiles; row_thr: threshold array from
        new_thresholds(), read at the start and updated (sod_match_top2_range); prepared=True reuses the
        query norms of the previous call with the same queries.  peer_table (a ctypes array of device
        pointers, one per rank, to the arrays that correspond to row_thr on every rank) + block_rotation:
        thresholds travel over peer memory (sod_match_top2_peer)."""
        q_u8 = _require_cuda(q_u8, torch.uint8, "query descriptors")
        nq = int(q_u8.shape[0])
        t0, t1 = (0, self.n_tiles) if tiles is None else (int(tiles[0]), int(tiles[1]))
        ws, qn = self._scratch(nq, (t1 - t0) * _capi.TILE_ROWS)
        idx = torch.empty((nq, 2), dtype=torch.int32, device=q_u8.device)
        d2 = torch.empty((nq, 2), dtype=torch.int32, device=q_u8.device)
        s = self.shard
        if not prepared:
            check(lib.sod_query_prepare(_ptr(q_u8), nq, _ptr(qn), _stream()), "sod_query_prepare")
        if self.events is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        n_peers = 0 if peer_table is None else len(peer_table)
        check(lib.sod_match_top2_peer(_ptr(q_u8), _ptr(qn), nq, _ptr(s.des), _ptr(s.cq), s.n, s.index_base, t0, t1,
                                      _ptr(row_thr), None if peer_table is None else C.cast(peer_table, C.c_void_p),
                                      n_peers, int(block_rotation), _ptr(idx), _ptr(d2), _ptr(ws), ws.numel(),
                                      _stream()), "sod_match_top2_peer")
        if self.events is not None:
            e1.record()
            self.events.append((e0, e1))
        return idx, d2


def merge_top2(parts_idx: torch.Tensor, parts_d2: torch.Tensor, ratio: float = RATIO):
    """[G,nq,2] candidate lists -> (idx [nq,2], d2 [nq,2], dist f32 [nq,2], pass u8 [nq])."""
    parts_idx = _require_cuda(parts_idx, torch.int32, "parts_idx")
    parts_d2 = _require_cuda(parts_d2, torch.int32, "parts_d2")
    if parts_idx.ndim == 2:
        parts_idx, parts_d2 = parts_idx[None], parts_d2[None]
    g, nq = int(parts_idx.shape[0]), int(parts_idx.shape[1])
    dev = parts_idx.device
    idx = torch.empty((nq, 2), dtype=torch.int32, device=dev)
    d2 = torch.empty((nq, 2), dtype=torch.int32, device=dev)
    dist = torch.empty((nq, 2), dtype=torch.float32, device=dev)
    ok = torch.empty(nq, dtype=torch.uint8, device=dev)
    check(lib.sod_top2_merge(_ptr(parts_idx), _ptr(parts_d2), g, nq, _ptr(idx), _ptr(d2), _ptr(dist),
                             _ptr(ok), float(ratio), _stream()), "sod_top2_merge")
    return idx, d2, dist, ok


def top2_keys(idx: torch.Tensor, d2: torch.Tensor, n_rows: int | None = None) -> torch.Tensor:
    """This rank's lists [nq,2] -> packed keys int64 [n_rows,2] (rows past nq: none)."""
    idx = _require_cuda(idx, torch.int32, "idx")
    d2 = _require_cuda(d2, torch.int32, "d2")
    nq = int(idx.shape[0])
    n_rows = nq if n_rows is None else int(n_rows)
    keys = torch.empty((n_rows, 2), dtype=torch.int64, device=idx.device)
    check(lib.sod_top2_keys(_ptr(idx), _ptr(d2), nq, n_rows, _ptr(keys), _stream()), "sod_top2_keys")
    return keys


def merge_keys(parts: torch.Tensor) -> torch.Tensor:
    """Key lists int64 [G,rows,2] -> the two smallest keys per row, [rows,2]."""
    parts = _require_cuda(parts, torch.int64, "parts")
    g, rows = int(parts.shape[0]), int(parts.shape[1])
    out = torch.empty((rows, 2), dtype=torch.int64, device=parts.device)
    check(lib.sod_top2_merge_keys(_ptr(parts), g, rows, _ptr(out), _stream()), "sod_top2_merge_keys")
    return out


def top2_from_keys(keys: torch.Tensor, nq: int, ratio: float = RATIO):
    """Merged keys int64 [>=nq,2] -> (idx [nq,2], d2 [nq,2], dist f32 [nq,2], pass u8 [nq])."""
    keys = _require_cuda(keys, torch.int64, "keys")
    dev = keys.device
    idx = torch.empty((nq, 2), dtype=torch.int32, device=dev)
    d2 = torch.empty((nq, 2), dtype=torch.int32, device=dev)
    dist = torch.empty((nq, 2), dtype=torch.float32, device=dev)
    ok = torch.empty(nq, dtype=torch.uint8, device=dev)
    check(lib.sod_top2_from_keys(_ptr(keys), nq, _ptr(idx), _ptr(d2), _ptr(dist), _ptr(ok), float(ratio),
                                 _stream()), "sod_top2_from_keys")
    return idx, d2, dist, ok


def exchange_merge_top2(idx: torch.Tensor, d2: torch.Tensor, world: int, all_to_all, all_gather,
                        ratio: float = RATIO):
    """Shard merge in exchange form (include/sod.h, K3): this rank's lists [nq,2] -> the global
    (idx, d2, dist, pass) on every rank.  all_to_all(out, inp) and all_gather(out, inp) are the
    collectives over the ranks that hold the other shards (torch.distributed.all_to_all_single /
    all_gather_into_tensor): slice r of every rank's keys goes to rank r, which merges its slice of the
    query rows; the merged slices are gathered.  16 B per query row each way instead of G x 16 B."""
    nq = int(idx.shape[0])
    per = (nq + world - 1) // world
    keys = top2_keys(idx, d2, per * world)                       # [world * per, 2]
    parts = torch.empty_like(keys)
    all_to_all(parts, keys)                                      # [world][per][2]: everyone's slice `rank`
    mine = merge_keys(parts.view(world, per, 2))
    merged = torch.empty_like(keys)
    all_gather(merged, mine)
    return top2_from_keys(merged, nq, ratio)


def knn_match_ratio(q_u8: torch.Tensor, matcher: Matcher, ratio: float = RATIO):
    """Single-shard convenience: knnMatch(k=2) + ratio flags."""
    idx, d2 = matcher.top2(q_u8)
    return merge_top2(idx[None], d2[None], ratio)


# ------------------------------------------------------------------------------------------------
# bf16 fallback for non-integer descriptors (approximate distances, tolerance stated in sod.h)
# ------------------------------------------------------------------------------------------------
@dataclass
class FloatShard:
    """Database slice for the bf16 path: operand [tiles*128, cols] (pre-multiplied by -2) + fp32 norms."""
    op: torch.Tensor         # bf16 bits as int16 [tiles*128, cols]
    norms: torch.Tensor      # f32 [tiles*128], +inf on padding rows
    n_rows: int
    index_base: int
    split: bool

    @property
    def n(self) -> int:
        return self.n_rows


def _bf16_prepare(des_f32: torch.Tensor, side: int, split: bool):
    des_f32 = _require_cuda(des_f32, torch.float32, "float descriptors")
    n = int(des_f32.shape[0])
    dev = des_f32.device
    cols = int(lib.sod_bf16_operand_cols(int(split)))
    rows = int(lib.sod_bf16_db_rows(n)) if side else n
    op = torch.empty((max(rows, 1), cols), dtype=torch.int16, device=dev)
    norms = torch.empty(max(rows, 1), dtype=torch.float32, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    check(lib.sod_bf16_prepare(_ptr(des_f32), n, side, int(split), _ptr(op), _ptr(norms), _ptr(flag), _stream()),
          "sod_bf16_prepare")
    if int(flag.item()) != 0:
        raise ValueError("descriptors contain NaN or infinite values")
    return op, norms


def prepare_db_float(des_f32: torch.Tensor, index_base: int = 0, split: bool = True) -> FloatShard:
    op, norms = _bf16_prepare(des_f32, 1, split)
    return FloatShard(op, norms, int(des_f32.shape[0]), int(index_base), bool(split))


class FloatMatcher:
    """2-NN matcher of the bf16 path for one database shard."""

    def __init__(self, shard: FloatShard):
        self.shard = shard
        self._ws: torch.Tensor | None = None
        self.events: list | None = None

    def top2(self, q_f32: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
        """-> (idx int32 [nq,2] global rows or -1, d2 float32 [nq,2] approximate squared distances)."""
        s = self.shard
        q_op, qn = _bf16_prepare(q_f32, 0, s.split)
        nq = int(q_f32.shape[0])
        need = int(lib.sod_match_bf16_workspace_bytes(nq, s.n))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=q_op.device)
        idx = torch.empty((nq, 2), dtype=torch.int32, device=q_op.device)
        d2 = torch.empty((nq, 2), dtype=torch.float32, device=q_op.device)
        if self.events is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        check(lib.sod_match_top2_bf16(_ptr(q_op), _ptr(qn), nq, _ptr(s.op), _ptr(s.norms), s.n, int(s.split),
                                      s.index_base, _ptr(idx), _ptr(d2), _ptr(self._ws), self._ws.numel(),
                                      _stream()), "sod_match_top2_bf16")
        if self.events is not None:
            e1.record()
            self.events.append((e0, e1))
        return idx, d2


def merge_top2_float(parts_idx: torch.Tensor, parts_d2: torch.Tensor, ratio: float = RATIO):
    """[G,nq,2] float candidate lists -> (idx, d2 f32, dist f32, pass u8)."""
    parts_idx = _require_cuda(parts_idx, torch.int32, "parts_idx")
    parts_d2 = _require_cuda(parts_d2, torch.float32, "parts_d2")
    if parts_idx.ndim == 2:
        parts_idx, parts_d2 = parts_idx[None], parts_d2[None]
    g, nq = int(parts_idx.shape[0]), int(parts_idx.shape[1])
    dev = parts_idx.device
    idx = torch.empty((nq, 2), dtype=torch.int32, device=dev)
    d2 = torch.empty((nq, 2), dtype=torch.float32, device=dev)
    dist = torch.empty((nq, 2), dtype=torch.float32, device=dev)
    ok = torch.empty(nq, dtype=torch.uint8, device=dev)
    check(lib.sod_top2_merge_f32(_ptr(parts_idx), _ptr(parts_d2), g, nq, _ptr(idx), _ptr(d2), _ptr(dist),
                                 _ptr(ok), float(ratio), _stream()), "sod_top2_merge_f32")
    return idx, d2, dist, ok


def knn_match_ratio_float(q_f32: torch.Tensor, matcher: FloatMatcher, ratio: float = RATIO):
    idx, d2 = matcher.top2(q_f32)
    return merge_top2_float(idx[None], d2[None], ratio)


# ------------------------------------------------------------------------------------------------
# Hough voting + affine verification
# ------------------------------------------------------------------------------------------------
import math  # noqa: E402

from ._capi import AffineOut, HoughOut, Keypoints, PosesOut, Scene  # noqa: E402

POS_FACTOR = 32          # main.py:141
N_OCT = 4                # HoughTransformHelperFunctions.py:66


def sigma_lut(bins: int) -> list[int]:
    """isigma of scale factor 2^k for k = -24..24, evaluated with the host libm exactly as
    HoughTransformHelperFunctions.py:66-70 does; the scale ratio of two SIFT octaves is always 2^k."""
    out = []
    for k in range(_capi.SIGMA_LUT_MIN, _capi.SIGMA_LUT_MIN + _capi.SIGMA_LUT_LEN):
        i = int(math.log(2.0 ** k, 2) / (2 * (N_OCT - 1) + 0.5) * bins)
        out.append(min(max(0, i), bins - 1))
    return out


def _dev(x, dtype, device):
    t = torch.as_tensor(x)
    return t.to(device=device, dtype=dtype, non_blocking=True).contiguous()


class SceneArrays:
    """Device-resident structure-of-arrays for the Hough/affine stages (sod_scene in sod.h)."""

    def __init__(self, q_xy, q_angle, q_octave, m_xy, m_angle, m_octave, m_image, img_centroid, img_size,
                 frame_wh, q_frame=None, img_group=None, groups_per_frame: int = 1, device="cuda"):
        d = torch.device(device)
        self.q_xy = _dev(q_xy, torch.float32, d).reshape(-1, 2)
        self.q_angle = _dev(q_angle, torch.float32, d)
        self.q_octave = _dev(q_octave, torch.int32, d)
        self.m_xy = _dev(m_xy, torch.float32, d).reshape(-1, 2)
        self.m_angle = _dev(m_angle, torch.float32, d)
        self.m_octave = _dev(m_octave, torch.int32, d)
        self.m_image = _dev(m_image, torch.int32, d)
        self.img_centroid = _dev(img_centroid, torch.float64, d).reshape(-1, 2)
        self.img_size = _dev(img_size, torch.float64, d).reshape(-1, 2)
        self.frame_wh = _dev(frame_wh, torch.int32, d).reshape(-1, 2)
        self.q_frame = None if q_frame is None else _dev(q_frame, torch.int32, d)
        self.img_group = None if img_group is None else _dev(img_group, torch.int32, d)
        self.groups_per_frame = int(groups_per_frame)
        self.device = d
        n_img = self.img_centroid.shape[0]
        if self.img_size.shape[0] != n_img or self.m_image.numel() != self.m_xy.shape[0]:
            raise ValueError("inconsistent model arrays")

    @property
    def n_frames(self) -> int:
        return int(self.frame_wh.shape[0])

    @property
    def n_groups(self) -> int:
        return self.n_frames * self.groups_per_frame

    def struct(self) -> Scene:
        return Scene(
            Keypoints(_ptr(self.q_xy), _ptr(self.q_angle), _ptr(self.q_octave), self.q_xy.shape[0]),
            _ptr(self.q_frame), _ptr(self.frame_wh), self.n_frames,
            Keypoints(_ptr(self.m_xy), _ptr(self.m_angle), _ptr(self.m_octave), self.m_xy.shape[0]),
            _ptr(self.m_image), _ptr(self.img_centroid), _ptr(self.img_size), _ptr(self.img_group),
            int(self.img_centroid.shape[0]), self.groups_per_frame)


def compact_matches(idx: torch.Tensor, ok: torch.Tensor, t_lo: int = 0, t_hi: int = 2 ** 31 - 1,
                    n_dev: torch.Tensor | None = None):
    """Ratio survivors (whose database row is in [t_lo, t_hi)) in query order ->
    (match_q, match_t, n_dev); stays on the device.  n_dev (device int32 [1]): only the first n_dev[0] rows
    count (sod_compact_matches_dev); the rows past it are ignored whatever they hold."""
    idx = _require_cuda(idx, torch.int32, "idx")
    ok = _require_cuda(ok, torch.uint8, "pass flags")
    nq = int(ok.shape[0])
    dev = idx.device
    mq = torch.empty(max(nq, 1), dtype=torch.int32, device=dev)
    mt = torch.empty(max(nq, 1), dtype=torch.int32, device=dev)
    n = torch.zeros(1, dtype=torch.int32, device=dev)
    scratch = torch.empty(int(lib.sod_compact_scratch_bytes(nq)), dtype=torch.uint8, device=dev)
    if n_dev is None:
        check(lib.sod_compact_matches(_ptr(idx), _ptr(ok), nq, int(t_lo), int(t_hi), _ptr(mq), _ptr(mt), _ptr(n),
                                      _ptr(scratch), _stream()), "sod_compact_matches")
    else:
        n_dev = _require_cuda(n_dev, torch.int32, "n_dev")
        check(lib.sod_compact_matches_dev(_ptr(idx), _ptr(ok), nq, _ptr(n_dev), int(t_lo), int(t_hi), _ptr(mq),
                                          _ptr(mt), _ptr(n), _ptr(scratch), _stream()), "sod_compact_matches_dev")
    return mq, mt, n


class HoughResult:
    """Device outputs of sod_hough_vote plus the host view used to build PoseBin objects."""

    def __init__(self, m_cap: int, n_groups: int, bins, device):
        self.dims = tuple(bins) if isinstance(bins, (tuple, list)) else (int(bins),) * 4
        self.bins = self.dims[3]          # what sod_affine_verify decodes from a bin code: code % bins_sigma
        self.m_cap = m_cap
        nb4 = int(np.prod(self.dims))
        self.cap_bins = max(1, min(16 * m_cap, n_groups * nb4))
        self.cap_votes = max(1, 16 * m_cap)
        e = lambda n, dt: torch.empty(n, dtype=dt, device=device)  # noqa: E731
        self.pose = e((max(m_cap, 1), 4), torch.float64)
        self.base_bin = e(max(m_cap, 1), torch.int32)
        self.near_edge = e(max(m_cap, 1), torch.uint8)
        self.counters = torch.zeros(8, dtype=torch.int32, device=device)
        self.bin_group = e(self.cap_bins, torch.int32)
        self.bin_code = e(self.cap_bins, torch.int32)
        self.bin_count = e(self.cap_bins, torch.int32)
        self.bin_offset = e(self.cap_bins, torch.int32)
        self.bin_order = e(self.cap_bins, torch.int64)
        self.bin_mean = e((self.cap_bins, 6), torch.float64)
        self.members = e(self.cap_votes, torch.int32)

    def struct(self) -> HoughOut:
        return HoughOut(_ptr(self.pose), _ptr(self.base_bin), _ptr(self.near_edge), _ptr(self.counters),
                        _ptr(self.bin_group), _ptr(self.bin_code), _ptr(self.bin_count),
                        _ptr(self.bin_offset), _ptr(self.bin_order), _ptr(self.bin_mean),
                        _ptr(self.members), self.cap_bins, self.cap_votes)

    def host(self) -> dict:
        """Synchronise and return numpy arrays with the bins in reference insertion order."""
        c = self.counters.cpu().numpy()
        if c[3]:
            raise _capi.SodError("Hough output capacity exceeded")
        nb, nv = int(c[0]), int(c[1])
        order = torch.argsort(self.bin_order[:nb])
        g = lambda t: t[:nb][order].cpu().numpy()  # noqa: E731
        return dict(n_bins=nb, n_votes=nv, n_near_edge=int(c[2]), n_unresolved_edge=int(c[4]), rec=order.cpu().numpy(),
                    group=g(self.bin_group), code=g(self.bin_code), count=g(self.bin_count),
                    offset=g(self.bin_offset), mean=g(self.bin_mean), order_key=g(self.bin_order),
                    members=self.members[:nv].cpu().numpy())


class HoughVoter:
    """Caches workspace / outputs across calls of the same capacity."""

    def __init__(self, scene: SceneArrays, bins=15):
        """bins: one count for all four pose dimensions (main.py:89), or (bin_x, bin_y, bin_theta,
        bin_sigma) as the legacy perform_hough_transform takes them (HoughTransform.py:8)."""
        self.dims = tuple(int(b) for b in bins) if isinstance(bins, (tuple, list)) else (int(bins),) * 4
        if len(self.dims) != 4 or min(self.dims) < 1:
            raise ValueError("bins must be a positive int or four positive ints")
        if max(self.dims) > 255 or int(np.prod(self.dims)) > _capi.MAX_BINS ** 4:
            raise _capi.SodError(f"bins={bins}: more than {_capi.MAX_BINS}^4 counters are not supported by the "
                                 f"shared-memory histogram")
        self.scene = scene
        self.bins = self.dims[0] if len(set(self.dims)) == 1 else None
        self.lut = torch.tensor(sigma_lut(self.dims[3]), dtype=torch.int32, device=scene.device)
        self._ws = None
        self._res: HoughResult | None = None

    def reserve(self, m_cap: int) -> HoughResult:
        """Size the outputs for up to m_cap matches now, so that later calls of any smaller size reuse
        the same buffers (callers that keep an AffineResult across calls rely on this)."""
        if self._res is None or self._res.m_cap < int(m_cap):
            self._res = HoughResult(int(m_cap), self.scene.n_groups, self.dims, self.scene.device)
        return self._res

    def new_result(self, m_cap: int) -> HoughResult:
        """A second output set of the same shape (callers that keep two steps in flight alternate them)."""
        return HoughResult(int(m_cap), self.scene.n_groups, self.dims, self.scene.device)

    def vote(self, match_q: torch.Tensor, match_t: torch.Tensor, n_dev: torch.Tensor | None = None,
             detail_min_count: int = 1, result: HoughResult | None = None) -> HoughResult:
        """detail_min_count: bins with fewer votes get a record and a count but no sorted members,
        means or order key (pass the vote threshold when only verified bins matter).
        result: write into this output set instead of the voter's own."""
        match_q = _require_cuda(match_q, torch.int32, "match_q")
        match_t = _require_cuda(match_t, torch.int32, "match_t")
        m = int(match_q.shape[0])
        sc = self.scene
        need = int(lib.sod_hough_workspace_bytes(m, sc.n_groups))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=sc.device)
        if result is not None and result.m_cap < m:
            raise ValueError(f"HoughResult sized for {result.m_cap} matches cannot take {m}")
        res = result if result is not None else self.reserve(m)
        s, o = sc.struct(), res.struct()
        check(lib.sod_hough_vote_dims(C.byref(s), _ptr(match_q), _ptr(match_t), m, _ptr(n_dev), *self.dims,
                                      _ptr(self.lut), int(detail_min_count), C.byref(o), _ptr(self._ws),
                                      self._ws.numel(), _stream()),
              "sod_hough_vote_dims")
        return res


class AffineResult:
    def __init__(self, hough: HoughResult, vote_threshold: int, device):
        # a bin enters with >= vote_threshold votes; with no threshold every record may enter (empty
        # bins of a caller-built list included), so the bound by votes does not apply
        self.cap_valid = max(1, hough.cap_bins if vote_threshold <= 0 else
                             min(hough.cap_bins, hough.cap_votes // vote_threshold))
        self.cap_votes = hough.cap_votes
        self.counters = torch.zeros(4, dtype=torch.int32, device=device)
        self.valid_bin = torch.empty(self.cap_valid, dtype=torch.int32, device=device)
        self.params = torch.empty((self.cap_valid, 6), dtype=torch.float64, device=device)
        self.votes = torch.empty(self.cap_valid, dtype=torch.int32, device=device)
        self.status = torch.empty(self.cap_valid, dtype=torch.int32, device=device)
        self.member_keep = torch.empty(hough.cap_votes, dtype=torch.uint8, device=device)
        self._records = None

    def records(self, hough: "HoughResult"):
        """(group, code, order, mean) of the bins in valid_bin, gathered on the device (sod_valid_bin_records);
        the first counters[0] entries are meaningful."""
        if self._records is None:
            dev = self.valid_bin.device
            self._records = (torch.empty(self.cap_valid, dtype=torch.int32, device=dev),
                             torch.empty(self.cap_valid, dtype=torch.int32, device=dev),
                             torch.empty(self.cap_valid, dtype=torch.int64, device=dev),
                             torch.empty((self.cap_valid, 6), dtype=torch.float64, device=dev))
        g, c, o, m = self._records
        h, a = hough.struct(), self.struct()
        check(lib.sod_valid_bin_records(C.byref(h), C.byref(a), _ptr(g), _ptr(c), _ptr(o), _ptr(m), _stream()),
              "sod_valid_bin_records")
        return self._records

    def struct(self) -> AffineOut:
        return AffineOut(_ptr(self.counters), _ptr(self.valid_bin), _ptr(self.params), _ptr(self.votes),
                         _ptr(self.status), _ptr(self.member_keep), self.cap_valid, self.cap_votes)

    def host(self, n_votes: int) -> dict:
        c = self.counters.cpu().numpy()
        if c[1]:
            raise _capi.SodError("affine output capacity exceeded")
        nv = int(c[0])
        st = self.status[:nv].cpu().numpy()
        return dict(n_valid=nv, valid_bin=self.valid_bin[:nv].cpu().numpy(),
                    params=self.params[:nv].cpu().numpy(), votes=self.votes[:nv].cpu().numpy(),
                    live=(st & 1).astype(bool), singular=((st >> 1) & 1).astype(bool),
                    residual_edge=((st >> 2) & 1).astype(bool), passes=st >> 8,
                    n_singular=int(c[2]), n_residual_edge=int(c[3]),
                    member_keep=self.member_keep[:n_votes].cpu().numpy().astype(bool))


def affine_verify(scene: SceneArrays, match_q: torch.Tensor, match_t: torch.Tensor, hough: HoughResult,
                  vote_threshold: int = 5, affine_threshold: int = 4, factor: float = POS_FACTOR * 4,
                  result: AffineResult | None = None, factor_y: float | None = None,
                  max_passes: int = 0) -> AffineResult:
    res = result or AffineResult(hough, vote_threshold, scene.device)
    if res.cap_votes < hough.cap_votes:
        raise ValueError(f"AffineResult sized for {res.cap_votes} votes cannot take a Hough result of "
                         f"{hough.cap_votes}: build it from this HoughResult (or reserve the voter first)")
    s, h, o = scene.struct(), hough.struct(), res.struct()
    check(lib.sod_affine_verify(C.byref(s), _ptr(match_q), _ptr(match_t), C.byref(h), hough.bins,
                                int(vote_threshold), int(affine_threshold), float(factor),
                                float(factor if factor_y is None else factor_y), int(max_passes),
                                C.byref(o), _stream()), "sod_affine_verify")
    return res


class FinalPoses:
    """sod_final_poses / sod_final_poses_records for up to `cap` bins, with the workspace and the outputs kept
    across calls.  The outputs of a call on n bins are views of the first bytes of one device buffer, so one copy of
    that many bytes reads all of them back; they are overwritten by the next call."""

    _NAMES = ("counters", "cluster_offset", "cluster_bins", "sub_bins", "sub_first", "shape_bin", "segment")

    def __init__(self, cap: int, device):
        cap = int(cap)
        if not 1 <= cap <= _capi.MAX_CLUSTER_BINS:
            raise _capi.SodError(f"sod_final_poses: {cap} bins, the limit is {_capi.MAX_CLUSTER_BINS}")
        self.cap, self.device = cap, torch.device(device)
        self.ws = torch.empty(int(lib.sod_final_poses_workspace_bytes(cap)), dtype=torch.uint8, device=self.device)
        self.buf = torch.empty(self._bytes(cap), dtype=torch.uint8, device=self.device)
        v = self.views(cap)
        self.pose, self.counters, self.shape_bin, self.segment = v["pose"], v["counters"], v["shape_bin"], v["segment"]

    @staticmethod
    def _bytes(n: int) -> int:
        return n * 6 * 8 + (2 + (n + 1) + 5 * n) * 4

    def views(self, n: int, buf=None) -> dict:
        """The outputs of a call on n bins as views of buf (the device buffer, or a host copy of its first bytes)."""
        buf = self.buf if buf is None else buf
        tensor = isinstance(buf, torch.Tensor)
        f8 = n * 6 * 8
        pose = buf[:f8].view(torch.float64 if tensor else np.float64).reshape(n, 6)
        iv = buf[f8:self._bytes(n)].view(torch.int32 if tensor else np.int32)
        out, o = dict(pose=pose), 0
        for name, size in zip(self._NAMES, (2, n + 1, n, n, n, n, n)):
            out[name] = iv[o:o + size]
            o += size
        return out

    def struct(self, n: int) -> PosesOut:
        v = self.views(n)
        return PosesOut(*(_ptr(v[name]) for name in ("counters", "cluster_bins", "cluster_offset", "sub_bins",
                                                     "sub_first", "pose", "shape_bin", "segment")), n)

    def run(self, mean: torch.Tensor, segment: torch.Tensor | None, n: int, n_dev: torch.Tensor | None = None):
        """mean: device float64 [>= n][6] (cx, cy, angle, scale, img_w, img_h); segment: device int32 [>= n] or
        None; n_dev: device int32 count (clamped to n), or None for n.  Outputs: views(n)."""
        mean = _require_cuda(mean, torch.float64, "mean")
        o = self.struct(int(n))
        check(lib.sod_final_poses(_ptr(mean), _ptr(segment), int(n), _ptr(n_dev), C.byref(o), _ptr(self.ws),
                                  self.ws.numel(), _stream()), "sod_final_poses")
        return self

    def run_records(self, status, group, order, mean, cap: int, n_dev: torch.Tensor, groups_per_frame: int):
        """The live bins of the affine stage's first min(n_dev, cap) records, in (group, order key) order.
        Outputs: views(cap)."""
        o = self.struct(int(cap))
        check(lib.sod_final_poses_records(_ptr(status), _ptr(group), _ptr(order), _ptr(mean), int(cap), _ptr(n_dev),
                                          int(groups_per_frame), C.byref(o), _ptr(self.ws), self.ws.numel(),
                                          _stream()), "sod_final_poses_records")
        return self

    def host(self, n: int) -> dict:
        """The outputs of the last call on n bins, read back with one copy of their bytes (synchronises)."""
        return self.views(n, self.buf[:self._bytes(n)].cpu().numpy())
