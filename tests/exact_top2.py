"""Exact 2-NN reference in torch, independent of the project's kernels: the checker for matcher runs too large
for the numpy oracle (up to the benchmark's 1.28M queries x 1M rows on one GPU).

cv2.BFMatcher semantics as oracle/sod_oracle.knn2: ascending squared L2 distance, ties -> lowest index, a
missing 2nd entry is -1.  q.t runs as a float32 matmul (cuBLAS on the GPU), which is exact here: every term
is a non-negative integer and every partial sum is at most 128 * 255^2 < 2^24.  Distances are then formed in
int32 as |t|^2 - 2 q.t (|q|^2 does not change the order) and packed into int64 keys (d << 32 | column),
whose signed order is the (distance, index) order; the two smallest keys per row are kept across chunks.
"""
from __future__ import annotations

from contextlib import contextmanager

import torch

CHUNK_BYTES = 16 << 30      # temporaries of one (query chunk x database chunk) block
# bytes per element of a block at the peak: the float32 (or float64) product and the int32 distances, then
# the int32 distances and the int64 keys
_BYTES_PER_ELEMENT = {torch.float32: 12, torch.float64: 16}


@contextmanager
def full_fp32_matmul():
    """Float32 matmuls in full float32 (no TF32) inside the block; the previous settings come back after."""
    prev_prec = torch.get_float32_matmul_precision()
    prev_cuda = torch.backends.cuda.matmul.allow_tf32
    prev_cudnn = torch.backends.cudnn.allow_tf32
    try:
        torch.set_float32_matmul_precision("highest")
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        yield
    finally:
        torch.set_float32_matmul_precision(prev_prec)
        torch.backends.cuda.matmul.allow_tf32 = prev_cuda
        torch.backends.cudnn.allow_tf32 = prev_cudnn


def chunk_rows(nq: int, ndb: int, dtype=torch.float32, budget: int = CHUNK_BYTES) -> tuple[int, int]:
    """(query rows, database rows) of one block, so that a block's temporaries stay under `budget` bytes."""
    per = _BYTES_PER_ELEMENT[dtype]
    cd = max(1, min(ndb, 1 << 14, budget // (per * 64)))
    cq = max(1, min(nq, budget // (per * cd)))
    return cq, cd


def exact_top2(q_u8: torch.Tensor, db_u8: torch.Tensor, index_base: int = 0, dtype=torch.float32,
               budget: int = CHUNK_BYTES) -> tuple[torch.Tensor, torch.Tensor]:
    """-> (idx int32 [nq,2] = index_base + database row or -1, d2 int32 [nq,2] squared distances or -1), on the
    device of the inputs.  dtype: the matmul's type (float64 is the cross-check of the float32 form)."""
    if q_u8.dtype != torch.uint8 or db_u8.dtype != torch.uint8 or q_u8.ndim != 2 or db_u8.ndim != 2:
        raise TypeError("exact_top2 takes u8 [n,128] descriptors")
    dev = q_u8.device
    nq, ndb = int(q_u8.shape[0]), int(db_u8.shape[0])
    idx = torch.full((nq, 2), -1, dtype=torch.int32, device=dev)
    d2 = torch.full((nq, 2), -1, dtype=torch.int32, device=dev)
    if nq == 0 or ndb == 0:
        return idx, d2
    if index_base < 0 or index_base + ndb >= 2 ** 31:
        raise ValueError("index_base + database rows must fit int32")
    cq, cd = chunk_rows(nq, ndb, dtype, budget)
    tn = (db_u8.to(torch.int32) ** 2).sum(1, dtype=torch.int32)
    qn = (q_u8.to(torch.int32) ** 2).sum(1, dtype=torch.int32)
    k = min(2, ndb)
    with full_fp32_matmul():
        for qs in range(0, nq, cq):
            qf = q_u8[qs:qs + cq].to(dtype)
            best = None
            for ds in range(0, ndb, cd):
                tf = db_u8[ds:ds + cd].to(dtype)
                dot = qf @ tf.T
                d = dot.to(torch.int32)                      # exact integers: the conversion loses nothing
                del dot
                d.mul_(-2).add_(tn[None, ds:ds + cd])          # |t|^2 - 2 q.t, in int32
                key = d.to(torch.int64)
                del d
                col = torch.arange(index_base + ds, index_base + ds + tf.shape[0], dtype=torch.int64, device=dev)
                key.bitwise_left_shift_(32).bitwise_or_(col[None, :])
                top = torch.topk(key, min(2, key.shape[1]), dim=1, largest=False, sorted=True).values
                del key
                best = top if best is None else torch.topk(torch.cat([best, top], 1), k, dim=1, largest=False,
                                                           sorted=True).values
            rows = slice(qs, qs + qf.shape[0])
            idx[rows, :k] = (best & 0xFFFFFFFF).to(torch.int32)
            d2[rows, :k] = (best >> 32).to(torch.int32) + qn[rows, None]
    return idx, d2


def direct_d2(q_u8: torch.Tensor, db_u8: torch.Tensor, idx: torch.Tensor, index_base: int = 0,
              rows_per_chunk: int = 1 << 18) -> torch.Tensor:
    """Squared distances of the candidates idx [nq,2] (index_base + database row, or -1) recomputed directly as
    sum((q - t)^2) in int32 from the gathered rows, no matmul; -1 where idx is -1.  Checks every reported
    distance, whichever code produced the candidates.  An index outside the database gives -2, which no
    distance equals."""
    nq, ndb = int(q_u8.shape[0]), int(db_u8.shape[0])
    out = torch.full((nq, idx.shape[1]), -1, dtype=torch.int32, device=q_u8.device)
    if ndb == 0:
        return torch.where(idx < 0, -1, -2).to(torch.int32)
    for s in range(0, nq, rows_per_chunk):
        i = idx[s:s + rows_per_chunk].to(torch.int64) - index_base
        inside = (i >= 0) & (i < ndb)
        t = db_u8[i.clamp(0, max(ndb - 1, 0))].to(torch.int32)                   # [n, 2, 128]
        diff = q_u8[s:s + rows_per_chunk, None, :].to(torch.int32) - t
        d = (diff * diff).sum(-1, dtype=torch.int32)
        none = idx[s:s + rows_per_chunk] < 0
        out[s:s + rows_per_chunk] = torch.where(inside, d, torch.where(none, -1, -2).to(torch.int32))
    return out
