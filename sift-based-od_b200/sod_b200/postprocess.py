"""Pose clustering after the affine stage (SURVEY.md §8f N1) on arrays.

post_process_arrays runs all four steps of Main.post_process on the device (csrc/sod_cluster.cu,
sod_final_poses): one upload, one call, one read-back.  The walks there follow the reference's depth-first
visiting order - which fixes the order of its float sums, the order of the clusters and the tie-break of
find_max_orientation - so results are identical to the reference's and there is no recursion limit
(SURVEY Q12).

The step-by-step functions (cluster_positions, orientation_subclusters) serve the drop-in's group_position /
group_orientation on caller-built lists: the O(V^2) neighbour tests run on the GPU (bit-matrix adjacency +
union-find labels) and the visiting order is recovered here from the bit rows with integer bitsets (V steps of
V/64-word operations).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _capi
from ._capi import check, lib
from .engine import FinalPoses, _ptr, _stream

_final: dict = {}      # device -> FinalPoses kept for later calls (up to _KEEP_BINS bins)
_KEEP_BINS = 4096      # workspace about 2.4 MB; larger calls get a FinalPoses of their own, freed after the call


def _graph(kind: str, arrays, segment, n: int, device, limit: float = 1.0):
    words = (n + 31) // 32
    adj = torch.empty((n, words), dtype=torch.int32, device=device)
    label = torch.empty(n, dtype=torch.int32, device=device)
    dev = [torch.as_tensor(np.ascontiguousarray(a, np.float64)).to(device) for a in arrays]
    seg = None if segment is None else torch.as_tensor(np.ascontiguousarray(segment, np.int32)).to(device)
    if kind == "position":
        check(lib.sod_pose_adjacency(_ptr(dev[0]), _ptr(dev[1]), _ptr(dev[2]), _ptr(dev[3]),
                                     _ptr(seg) if seg is not None else 0, n, _ptr(adj), _ptr(label), _stream()),
              "sod_pose_adjacency")
    else:
        check(lib.sod_angle_adjacency(_ptr(dev[0]), _ptr(seg) if seg is not None else 0, n, float(limit),
                                      _ptr(adj), _ptr(label), _stream()), "sod_angle_adjacency")
    return adj.cpu().numpy().view(np.uint32), label.cpu().numpy()


def _row_bitsets(adj: np.ndarray) -> list[int]:
    """uint32 [n][words] -> one Python int per row (bit j = edge to j)."""
    raw = np.ascontiguousarray(adj.astype("<u4"))
    return [int.from_bytes(raw[i].tobytes(), "little") for i in range(raw.shape[0])]


def preorder_components(rows: list[int]) -> list[list[int]]:
    """Connected components in the reference's order: start nodes ascending, pre-order depth-first
    walk that always takes the lowest unvisited neighbour (PostProcessing.py:4-11 over ascending
    neighbour lists)."""
    n = len(rows)
    seen = 0
    comps = []
    for s in range(n):
        if (seen >> s) & 1:
            continue
        seen |= 1 << s
        comp, stack = [s], [s]
        while stack:
            cand = rows[stack[-1]] & ~seen
            if cand:
                nb = (cand & -cand).bit_length() - 1
                seen |= 1 << nb
                comp.append(nb)
                stack.append(nb)
            else:
                stack.pop()
        comps.append(comp)
    return comps


def cluster_positions(cx, cy, scale, img_w, img_h, segment=None, device="cuda"):
    """group_position on arrays -> (clusters as lists of bin indices in visiting order, labels)."""
    n = len(cx)
    if n == 0:
        return [], np.zeros(0, np.int32)
    # the reference's expression img_size[0] * scale / 4 with Python int * float semantics
    reach_x = [img_w[i] * float(scale[i]) / 4 for i in range(n)]
    reach_y = [img_h[i] * float(scale[i]) / 4 for i in range(n)]
    adj, label = _graph("position", (cx, cy, reach_x, reach_y), segment, n, torch.device(device))
    return preorder_components(_row_bitsets(adj)), label


def orientation_subclusters(angles_per_cluster, device="cuda", max_degrees: float = 1.0):
    """group_orientation: for every position cluster (a list of angles in the cluster's visiting
    order) the sub-clusters as lists of POSITIONS in that list, in the reference's order.  All
    clusters go through one launch: angles are laid out back to back with the cluster number as
    segment id, so a cluster's rows and columns are one contiguous range of the bit matrix."""
    sizes = [len(a) for a in angles_per_cluster]
    n = sum(sizes)
    if n == 0:
        return [[] for _ in sizes]
    flat = np.concatenate([np.asarray(a, np.float64) for a in angles_per_cluster if len(a)])
    segment = np.repeat(np.arange(len(sizes), dtype=np.int32), sizes)
    adj, _ = _graph("angle", (flat,), segment, n, torch.device(device), max_degrees)
    rows = _row_bitsets(adj)
    out, off = [], 0
    for m in sizes:
        mask = (1 << m) - 1
        out.append(preorder_components([(rows[off + p] >> off) & mask for p in range(m)]))
        off += m
    return out


def cluster_orientations(angle, clusters, device="cuda", max_degrees: float = 1.0):
    """group_orientation on arrays: per position cluster, sub-clusters as lists of bin indices."""
    pos = orientation_subclusters([[float(angle[i]) for i in cl] for cl in clusters], device, max_degrees)
    return [[[cl[p] for p in comp] for comp in comps] for cl, comps in zip(clusters, pos)]


def _final_poses(n: int, device) -> FinalPoses:
    device = torch.device(device)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    if n > _KEEP_BINS:
        return FinalPoses(n, device)
    fp = _final.get(device)
    if fp is None or fp.cap < n:
        fp = _final[device] = FinalPoses(max(n, 256), device)
    return fp


def post_process_arrays(cx, cy, scale, angle, img_w, img_h, segment=None, device="cuda"):
    """The four reference steps on arrays -> (clusters, sub_clusters, orientations, final) with
    final[c] = ((cx, cy), orientation, scale, (w, h)) exactly as get_final_pose returns it.  segment (one id
    per bin, e.g. its frame) keeps bins of different segments apart."""
    n = len(cx)
    if n == 0:
        return [], [], [], []
    if n > _capi.MAX_CLUSTER_BINS:
        raise _capi.SodError(f"sod_final_poses: n = {n}, the limit is {_capi.MAX_CLUSTER_BINS}")
    # one upload: the means [n][6] (the sod_hough_out.bin_mean layout) and the segment ids behind them
    host = np.empty(n * 52, np.uint8)
    mean = host[:n * 48].view(np.float64).reshape(n, 6)
    for f, a in enumerate((cx, cy, angle, scale, img_w, img_h)):
        mean[:, f] = np.asarray(a, np.float64)
    host[n * 48:].view(np.int32)[:] = 0 if segment is None else np.asarray(segment, np.int32)
    fp = _final_poses(n, device)
    with torch.cuda.device(fp.device):
        dev = torch.from_numpy(host).to(fp.device)
        fp.run(dev[:n * 48].view(torch.float64), dev[n * 48:].view(torch.int32) if segment is not None else None, n)
        h = fp.host(n)
    nc = int(h["counters"][0])
    off = h["cluster_offset"][:nc + 1].tolist()
    bins, sub_bins = h["cluster_bins"][:n].tolist(), h["sub_bins"][:n].tolist()
    starts = np.flatnonzero(h["sub_first"][:n])
    per_cluster = np.diff(np.searchsorted(starts, off)).tolist()     # sub-clusters per cluster
    bounds = starts.tolist() + [n]
    clusters = [bins[off[c]:off[c + 1]] for c in range(nc)]
    subs, s = [], 0
    for m in per_cluster:
        subs.append([sub_bins[bounds[u]:bounds[u + 1]] for u in range(s, s + m)])
        s += m
    pose = h["pose"][:nc].tolist()
    orientations = [p[2] for p in pose]
    final = [((p[0], p[1]), p[2], p[3], (img_w[k], img_h[k]) if k >= 0 else (0, 0))
             for p, k in zip(pose, h["shape_bin"][:nc].tolist())]
    return clusters, subs, orientations, final
