"""Dev tool: time sod_match_top2 alone on device-resident inputs (CUDA events)."""
import hashlib
import os
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "sift-based-od_b200"))
from sod_b200 import engine as E  # noqa: E402


def sift_like_gpu(n, g):
    x = torch.randn((n, 128), device="cuda", generator=g).abs_()
    x /= x.norm(dim=1, keepdim=True)
    x.clamp_(max=0.2)
    x /= x.norm(dim=1, keepdim=True)
    return (x * 512).round_().clamp_(0, 255).to(torch.uint8)


KINDS = ("uniform", "sift", "selfmatch", "cluster", "dup", "noevent")


def make_inputs(kind, nq, ndb, g):
    """(q, db) u8 [n,128] on the GPU for one data kind, drawn from generator g.  The timed legs below and the
    tests (tests/test_gpu_match_scale.py) build their inputs here, so the data that is timed is the data
    that is checked."""
    if kind == "uniform":
        q = torch.randint(0, 256, (nq, 128), dtype=torch.uint8, device="cuda", generator=g)
        db = torch.randint(0, 256, (ndb, 128), dtype=torch.uint8, device="cuda", generator=g)
    elif kind == "selfmatch":
        # hostile leg 1: EVERY query is a database row + integer noise (100 % true matches)
        db = sift_like_gpu(ndb, g)
        src = torch.randint(0, ndb, (nq,), device="cuda", generator=g)
        noise = torch.randint(-3, 4, (nq, 128), device="cuda", generator=g, dtype=torch.int16)
        q = (db[src].to(torch.int16) + noise).clamp_(0, 255).to(torch.uint8)
    elif kind == "cluster":
        # hostile leg 2: dense near-duplicates - 1024 clusters of ndb/1024 rows within +-2 of their centre,
        # queries = centres + noise: hundreds of database rows sit at almost the distance of the 2nd best
        centres = sift_like_gpu(1024, g)
        lab = torch.randint(0, 1024, (ndb,), device="cuda", generator=g)
        db = (centres[lab].to(torch.int16) + torch.randint(-2, 3, (ndb, 128), device="cuda", generator=g,
                                                            dtype=torch.int16)).clamp_(0, 255).to(torch.uint8)
        ql = torch.randint(0, 1024, (nq,), device="cuda", generator=g)
        q = (centres[ql].to(torch.int16) + torch.randint(-2, 3, (nq, 128), device="cuda", generator=g,
                                                          dtype=torch.int16)).clamp_(0, 255).to(torch.uint8)
    elif kind == "dup":
        # the floor: ONE descriptor repeated ndb times and every query equal to it - every distance is 0, every
        # chunk ties with the threshold and takes the exact path, the lowest indices win one tile at a time
        row = sift_like_gpu(1, g)
        db = row.expand(ndb, 128).contiguous()
        q = row.expand(nq, 128).contiguous()
    elif kind == "noevent":
        # all-zero queries + two all-zero database rows (smallest norm -> first tile): the threshold is 0
        # after the first tile and nothing passes the bound any more: the shipped binary without updates
        q = torch.zeros((nq, 128), dtype=torch.uint8, device="cuda")
        db = sift_like_gpu(ndb, g)
        db[:2] = 0
    elif kind == "sift":
        q, db = sift_like_gpu(nq, g), sift_like_gpu(ndb, g)
    else:
        raise ValueError(f"unknown input kind {kind!r}: one of {', '.join(KINDS)}")
    return q, db


def input_hash(q, db):
    """First 16 hex digits of the SHA-256 of q's and db's bytes: identifies a leg's exact inputs."""
    h = hashlib.sha256()
    for t in (q, db):
        h.update(t.contiguous().cpu().numpy().tobytes())
    return h.hexdigest()[:16]


def run(nq, ndb, iters=10, kind="uniform"):
    g = torch.Generator(device="cuda").manual_seed(1)
    q, db = make_inputs(kind, nq, ndb, g)
    m = E.Matcher(E.prepare_db(db))
    for _ in range(3):
        m.top2(q)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(iters + 1)]
    ev[0].record()
    for i in range(iters):
        m.top2(q)
        ev[i + 1].record()
    torch.cuda.synchronize()
    ts = [ev[i].elapsed_time(ev[i + 1]) for i in range(iters)]
    ms = float(np.median(ts))
    ops = 2.0 * nq * ndb * 128
    print(f"{kind:>8} nq={nq:>8} ndb={ndb:>8}  {ms:9.3f} ms (min {min(ts):.3f})  {ops / ms / 1e9:8.1f} TOPS  "
          f"{nq / ms * 1e3 / 1e6:8.3f} Mq/s  inputs {input_hash(q, db)}", flush=True)


def run_float(nq, ndb, split, iters=10):
    """bf16 fallback path on RootSIFT-style float descriptors; the timed region is the match kernel
    call alone (operands prepared outside)."""
    g = torch.Generator(device="cuda").manual_seed(1)
    q = sift_like_gpu(nq, g).float().sqrt_()
    db = sift_like_gpu(ndb, g).float().sqrt_()
    m = E.FloatMatcher(E.prepare_db_float(db, split=split))
    m.events = []
    for _ in range(3 + iters):
        m.top2(q)
    torch.cuda.synchronize()
    ts = [a.elapsed_time(b) for a, b in m.events[3:]]
    ms = float(np.median(ts))
    k = 384 if split else 128
    print(f"bf16 split={int(split)} nq={nq:>8} ndb={ndb:>8}  {ms:9.3f} ms (min {min(ts):.3f})  "
          f"{2.0 * nq * ndb * k / ms / 1e9:8.1f} TFLOP/s issued  {nq / ms * 1e3 / 1e6:8.3f} Mq/s", flush=True)


if __name__ == "__main__":
    shapes = [(10000, 100000), (10000, 1000000), (65536, 1000000)]
    if len(sys.argv) > 1 and sys.argv[1] != "--adversarial":
        shapes = [tuple(int(x) for x in a.split("x")) for a in sys.argv[1:]]
    kinds = os.environ.get("SOD_BENCH_KINDS", "uniform,sift").split(",")
    if "--adversarial" in sys.argv:     # the hostile-data legs beside the friendly one (VERDICT r1, item 3)
        sys.argv.remove("--adversarial")
        kinds = ["sift", "selfmatch", "cluster", "dup"]
        shapes = [(65536, 1000000)]
    for kind in kinds:
        for nq, ndb in shapes:
            if kind in ("bf16", "bf16x3"):
                run_float(nq, ndb, kind == "bf16x3")
            else:
                run(nq, ndb, kind=kind)
