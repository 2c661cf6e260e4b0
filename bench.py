#!/usr/bin/env python
"""Headline benchmark: query descriptors/s through kNN2 + ratio + Hough + affine against a
1M-descriptor model database (BASELINE.json), one process per GPU.

    python bench.py --gpus N --steps K --warmup W            # our arm (torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path, rank 0 only
    python bench.py ... --dump-outputs DIR                   # + the last timed step's outputs, DIR/<name>.npy

Workload (BASELINE.json configs[3], "throughput mode"): 256 scene frames x 5,000 SIFT descriptors
against 1,000 model objects x 1,000 descriptors, u8 128-d, synthetic (seeded).  Every frame contains
4 planted object instances (10 % of its descriptors are true matches) plus 1 % descriptor-only false
matches; Hough spaces are per (frame, object).  A step is one pass of the whole path over the batch.
N > 1, two ways to partition the same fixed total work ("scaling": "strong"):
  --shard db (default)      the north star's layout: database rows sharded object-aligned across the ranks,
                            the query batch replicated (each rank uploads 1/N of it, one all-gather over
                            NVLink), shard-local top-2 merged by ONE exchange (16 B per query row), pruning
                            thresholds shared over peer memory, Hough + affine for each rank's own objects;
  --shard frames            the 128 MB database is replicated and every rank takes 1/N of the frames: no
                            data-path collective at all.  The default run reports it as `alt_partition`.
The scaling figures are stated once, in DESIGN.md §5 (builder runs under profiles/r02_bench_n*.json); the
driver's SCALE_rNN.json is the authority.

Timed regions
  value : inputs resident in HBM; CUDA events on the launching stream, barrier + synchronize on both
          sides, max over ranks.
  e2e   : the public API (sod_b200.pipeline.DetectionPipeline.detect_batches) with pinned HOST buffers:
          H2D of descriptors + keypoints and D2H of matches + verified bins inside the region, every step;
          pipelined one step deep (the copies of step i+1 overlap the kernels of step i).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT / "sift-based-od_b200"))
sys.path.insert(0, str(ROOT))

METRIC = "query descriptors/sec (kNN2+ratio+Hough+affine), 1M-desc DB"
UNIT = "query descriptors/s"


# ------------------------------------------------------------------------------------------------
# synthetic workload
# ------------------------------------------------------------------------------------------------
def sift_like_torch(n, gen, device):
    import torch
    x = torch.randn((n, 128), device=device, generator=gen).abs_()
    x /= x.norm(dim=1, keepdim=True)
    x.clamp_(max=0.2)
    x /= x.norm(dim=1, keepdim=True)
    return (x * 512).round_().clamp_(0, 255).to(torch.uint8)


def make_workload(args, device):
    """Deterministic (seed 102) on every rank.  Descriptors are generated with torch on `device`
    (fast for 1M x 128); geometry with numpy."""
    import torch
    n_obj, kpo, frames, per = args.objects, args.kp_per_object, args.frames, args.per_frame
    ndb, nq = n_obj * kpo, frames * per
    rng = np.random.default_rng(102)
    mw, mh, W, H = 1500, 1000, 4032, 3024
    m_xy = np.stack([rng.uniform(0, mw, ndb), rng.uniform(0, mh, ndb)], 1).astype(np.float32)
    m_angle = rng.uniform(0, 360, ndb).astype(np.float32)
    m_oct = rng.integers(0, 3, ndb)
    m_image = np.repeat(np.arange(n_obj, dtype=np.int32), kpo)
    cent = m_xy.astype(np.float64).reshape(n_obj, kpo, 2).mean(1)
    q_xy = np.stack([rng.uniform(0, W, nq), rng.uniform(0, H, nq)], 1).astype(np.float32)
    q_angle = rng.uniform(0, 360, nq).astype(np.float32)
    q_oct = rng.integers(-1, 5, nq)
    q_frame = np.repeat(np.arange(frames, dtype=np.int32), per)
    inst, n_in = args.instances, int(per * args.inlier_frac) // args.instances
    src_q, src_t = [], []
    for f in range(frames):
        rows = f * per + rng.choice(per, inst * n_in + int(per * args.false_frac), replace=False)
        objs = rng.choice(n_obj, inst, replace=False)
        for j, o in enumerate(objs):
            qi = rows[j * n_in:(j + 1) * n_in]
            t = o * kpo + rng.choice(kpo, n_in, replace=False)
            k = int(rng.integers(0, 3))
            s, th = 2.0 ** k, rng.uniform(0, 2 * math.pi)
            c = np.array([rng.uniform(0.25, 0.75) * W, rng.uniform(0.25, 0.75) * H])
            rel = (m_xy[t].astype(np.float64) - cent[o]) * s
            rot = np.stack([math.cos(th) * rel[:, 0] - math.sin(th) * rel[:, 1],
                            math.sin(th) * rel[:, 0] + math.cos(th) * rel[:, 1]], 1)
            q_xy[qi] = (rot + c + rng.normal(0, 2.0, rot.shape)).astype(np.float32)
            a = np.mod(m_angle[t].astype(np.float64) + math.degrees(th), 360.0).astype(np.float32)
            q_angle[qi] = np.where(a >= 360.0, 0.0, a)
            q_oct[qi] = m_oct[t] + k
            src_q.append(qi)
            src_t.append(t)
        fq = rows[inst * n_in:]
        src_q.append(fq)
        src_t.append(rng.integers(0, ndb, len(fq)))
    src_q = np.concatenate(src_q)
    src_t = np.concatenate(src_t)
    gen = torch.Generator(device=device).manual_seed(102)
    db_des = sift_like_torch(ndb, gen, device)
    q_des = sift_like_torch(nq, gen, device)
    noise = torch.randint(-3, 4, (len(src_q), 128), device=device, generator=gen, dtype=torch.int16)
    sq = torch.from_numpy(src_q).to(device)
    st = torch.from_numpy(src_t).to(device)
    q_des[sq] = (db_des[st].to(torch.int16) + noise).clamp_(0, 255).to(torch.uint8)
    pack = lambda o: ((o.astype(np.int64) & 0xFF) | (1 << 8)).astype(np.int32)  # noqa: E731
    return dict(db_des=db_des, m_xy=m_xy, m_angle=m_angle, m_octave=pack(m_oct), m_image=m_image,
                img_centroid=cent, img_size=np.tile(np.array([[mw, mh]], np.int32), (n_obj, 1)),
                q_des=q_des, q_xy=q_xy, q_angle=q_angle, q_octave=pack(q_oct), q_frame=q_frame,
                frame_wh=np.tile(np.array([[W, H]], np.int32), (frames, 1)), n_true=len(src_q))


def make_database(wl):
    """The workload's model database for DetectionPipeline: every model image is its own object, so the
    Hough spaces are per (frame, object) and the database shards at object boundaries."""
    from sod_b200.pipeline import ModelDatabase
    return ModelDatabase(wl["db_des"], wl["m_xy"], wl["m_angle"], wl["m_octave"], wl["m_image"],
                         wl["img_centroid"], wl["img_size"],
                         object_of_image=np.arange(len(wl["img_centroid"]), dtype=np.int32))


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons of one GPU DURING the timed region: an NVML polling thread
    (2 ms period, so even an 8-GPU step of ~15 ms is sampled); `nvidia-smi -lms` as fallback."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None
        self.nvml, self.handle, self.samples, self.mask, self.max_mhz = None, None, [], 0, None
        self._stop = threading.Event()
        self._thread = None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:  # CUDA_VISIBLE_DEVICES may renumber the devices: go through the UUID
            uuid = str(torch.cuda.get_device_properties(self.gpu).uuid)
            handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid if not uuid.startswith("GPU-") else uuid).encode())
        except Exception:
            handle = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
        return pynvml, handle

    def start(self):
        try:
            self.nvml, self.handle = self._nvml_handle()
            self.max_mhz = float(self.nvml.nvmlDeviceGetMaxClockInfo(self.handle, self.nvml.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._poll, daemon=True)
            self._thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self._stop.is_set():
            try:
                self.samples.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                self.mask |= int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.nvml is not None:
            self._stop.set()
            self._thread.join(timeout=1.0)
            n = self.nvml
            flags = {"hw_slowdown": n.nvmlClocksEventReasonHwSlowdown,
                     "hw_thermal_slowdown": n.nvmlClocksEventReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": n.nvmlClocksEventReasonSwThermalSlowdown,
                     "sw_power_cap": n.nvmlClocksEventReasonSwPowerCap,
                     "hw_power_brake": n.nvmlClocksEventReasonHwPowerBrakeSlowdown}
            return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(k for k, v in flags.items() if self.mask & v), "samples": len(self.samples),
                    "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 8:
                continue
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
            except ValueError:
                continue
            for n, v in zip(names, r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# CPU path of the reference (cv2.BFMatcher + the Python Hough / affine loops, restated in oracle/)
# ------------------------------------------------------------------------------------------------
class CpuReference:
    def __init__(self, wl, args):
        import cv2
        from oracle import sod_oracle as O
        self.cv2, self.O = cv2, O
        cv2.setNumThreads(os.cpu_count() or 1)
        self.threads = cv2.getNumThreads()
        db = wl["db_des"].cpu().numpy()
        self.db_f32 = db.astype(np.float32)
        self.chunk = (1 << 18) - 1  # cv2 asserts on >= 2^18 train rows (SURVEY T6)
        self.chunks = [self.db_f32[s:s + self.chunk] for s in range(0, len(db), self.chunk)]
        self.offsets = np.arange(0, len(db), self.chunk)
        self.wl, self.args = wl, args
        self.q_des = wl["q_des"].cpu().numpy()
        self.scene = O.Scene(wl["q_xy"], wl["q_angle"], wl["q_octave"], wl["m_xy"], wl["m_angle"], wl["m_octave"],
                             wl["m_image"], wl["img_centroid"], wl["img_size"], int(wl["frame_wh"][0, 0]),
                             int(wl["frame_wh"][0, 1]), np.arange(args.objects, dtype=np.int32))
        # The reference itself is not part of this repository: the Hough / affine leg times the oracle's
        # port of the same single-threaded loops.
        self.kind = "port"
        self.hough_what = "oracle port of the reference's single-threaded Python Hough/affine loops"

    def run(self, q_rows: np.ndarray) -> dict:
        """main.py:180-185 on the given query rows (all from one frame)."""
        cv2, O = self.cv2, self.O
        t0 = time.perf_counter()
        q = self.q_des[q_rows].astype(np.float32)
        bf = cv2.BFMatcher()
        bf.add(self.chunks)
        matches = bf.knnMatch(q, k=2)                                   # main.py:70-71
        mq, mt = [], []
        for m, n in matches:                                            # main.py:81-86
            if m.distance < 0.75 * n.distance:
                mq.append(int(q_rows[m.queryIdx]))
                mt.append(int(self.offsets[m.imgIdx] + m.trainIdx))
        t1 = time.perf_counter()
        table = O.hough_vote(self.scene, mq, mt, 15)                    # main.py:89-119
        vb = O.valid_bins(table, 5)                                     # main.py:121-132
        n_live = len(O.affine_verify(self.scene, mq, mt, vb, 4))        # main.py:139-157
        t2 = time.perf_counter()
        return dict(n=len(q_rows), t_match=t1 - t0, t_hough_affine=t2 - t1, matches=len(mq), live=n_live)

    def sample_rows(self, step: int, n: int) -> np.ndarray:
        per = self.args.per_frame
        f = step % self.args.frames
        return np.arange(f * per, f * per + min(n, per))

    def calibrate(self, target_s: float) -> int:
        r = self.run(self.sample_rows(0, 16))
        per_q = (r["t_match"] + r["t_hough_affine"]) / r["n"]
        return int(max(16, min(self.args.per_frame, target_s / max(per_q, 1e-9))))


# ------------------------------------------------------------------------------------------------
def measure_int8_cublas_tops(device):
    """cuBLASLt int8 GEMM rate on this GPU: informational denominator (MEASURED_PEAKS.json has no
    int8 entry)."""
    import torch
    try:
        a = torch.randint(-8, 8, (8192, 8192), dtype=torch.int8, device=device)
        b = torch.randint(-8, 8, (8192, 8192), dtype=torch.int8, device=device).t().contiguous().t()
        for _ in range(3):
            torch._int_mm(a, b)
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch._int_mm(a, b)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2 * 8192 ** 3 / (best * 1e-3) / 1e12
    except Exception:
        return None


def _stage_ms(stage):
    from sod_b200 import _capi
    return _capi.timing_read(stage)


def measure(args, wl, shard, rank, world, local, device, barrier, with_clocks=True):
    """One partition of the workload over the ranks: device-resident leg + end-to-end leg.
    Returns per-rank-reduced numbers (times = max over ranks)."""
    import torch
    import torch.distributed as dist
    from sod_b200 import _capi
    from sod_b200.pipeline import DetectionPipeline

    nq_total = args.frames * args.per_frame
    q = {k: wl[k] for k in ("q_des", "q_xy", "q_angle", "q_octave", "q_frame")}
    nq = nq_total
    if shard == "frames" and world > 1:
        # database replicated, frames split: rank r owns frames [r*F/N, (r+1)*F/N); no collective
        f_lo, f_hi = args.frames * rank // world, args.frames * (rank + 1) // world
        lo, hi = f_lo * args.per_frame, f_hi * args.per_frame
        q = {k: v[lo:hi] for k, v in q.items()}
        nq = hi - lo
    pipe = DetectionPipeline(make_database(wl), nq, wl["frame_wh"], rank=rank, world=world, device=device,
                             shard=shard, exchange=args.exchange, result_rows="own", seed_rows=args.seed_rows,
                             sweep_stages=args.sweep_stages, thresholds=args.thresholds)
    host = {k: torch.from_numpy(np.ascontiguousarray(q[k])).pin_memory()
            for k in ("q_xy", "q_angle", "q_octave", "q_frame")}
    host["q_des"] = q["q_des"].cpu().pin_memory()
    order = ("q_des", "q_xy", "q_angle", "q_octave", "q_frame")
    # bytes this rank really copies host -> device per step (its slice of the batch when database-sharded)
    _, r_lo, r_hi = pipe.own_rows(nq) if (shard == "db" and world > 1) else (nq, 0, nq)
    h2d_rank = int(sum(host[k][r_lo:r_hi].numel() * host[k].element_size() for k in order))

    # ---------------- device-resident leg
    pipe.load_queries(q["q_des"], host["q_xy"], host["q_angle"], host["q_octave"], host["q_frame"])
    for _ in range(args.warmup):
        r = pipe.detect_device(nq)
    barrier()
    _capi.timing_enable(True)
    sampler = ClockSampler(local) if with_clocks else None
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        r = pipe.detect_device(nq)
    e1.record()
    barrier()
    clocks = sampler.stop() if sampler else None
    stage = {k: _stage_ms(k) for k in _capi.STAGES}
    _capi.timing_enable(False)
    # a seeded database-sharded step launches the matcher several times: the seeding sweep, then the shard
    # sweep in pipe.sweep_stages tile ranges; kernel_ms is the SUM of the shard-sweep launches of a step
    big = nq >= pipe.seed_min_queries
    seeded = pipe.seed_matcher is not None and big            # a seeding sweep in front of the shard sweep
    shared = big and (pipe.seed_matcher is not None or pipe.peer_thr is not None)
    stages = pipe.sweep_stages if (shared and pipe.peer_thr is None) else 1
    per_step = (1 if seeded else 0) + stages
    mm = stage["match"][: len(stage["match"]) // per_step * per_step]
    sweeps = [sum(mm[i * per_step + (1 if seeded else 0):(i + 1) * per_step]) for i in range(len(mm) // per_step)]
    seeds = mm[0::per_step] if seeded else []
    loc = torch.tensor([e0.elapsed_time(e1), float(np.mean(sweeps)) if sweeps else 0.0,
                        float(np.mean(seeds)) if seeds else 0.0,
                        float(np.mean(stage["hough_vote"])) if stage["hough_vote"] else 0.0,
                        float(np.mean(stage["hough_prep"]) + np.mean(stage["hough_finish"])) if stage["hough_prep"] else 0.0,
                        float(np.mean(stage["affine"])) if stage["affine"] else 0.0], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(loc, op=dist.ReduceOp.MAX)
    ms_total, sweep_ms, seed_ms, vote_ms, hough_other_ms, affine_ms = (float(v) for v in loc.tolist())
    res = pipe.fetch(r)

    # ---------------- end-to-end leg: host buffers in, host results out
    # Every step copies its inputs from pinned host memory and reads its result back; detect_batches
    # overlaps the host->device copy of step i+1 with the kernels of step i (two query-buffer sets).
    def host_steps(k):
        for _ in range(k):
            yield tuple(host[key] for key in order)

    for out in pipe.detect_batches(host_steps(max(3, args.warmup))):   # both buffer sets, staging, NCCL paths warm
        pass
    barrier()
    t0 = time.perf_counter()
    stamps = [t0]
    for out in pipe.detect_batches(host_steps(args.steps)):
        stamps.append(time.perf_counter())
    barrier()
    e2e = torch.tensor([time.perf_counter() - t0], device=device, dtype=torch.float64)
    batch_ms = [round((b - a) * 1e3, 3) for a, b in zip(stamps, stamps[1:])]   # this rank's result-to-result intervals
    byt = torch.tensor([h2d_rank, DetectionPipeline.fetched_bytes(out)], device=device, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(e2e, op=dist.ReduceOp.MAX)
        dist.all_reduce(byt, op=dist.ReduceOp.SUM)
    return dict(pipe=pipe, nq=nq, nq_total=nq_total, ms_total=ms_total, sweep_ms=sweep_ms, seed_ms=seed_ms,
                vote_ms=vote_ms, hough_other_ms=hough_other_ms, affine_ms=affine_ms, e2e_s=float(e2e.item()),
                h2d=int(byt[0]), d2h=int(byt[1]), res=res, clocks=clocks, host=host, order=order, batch_ms=batch_ms,
                launches=pipe.launches_per_call)


def latency_record(pipe, n, world, device, barrier, iters=30):
    """BASELINE configs[2]: one small query batch (n rows) against the sharded 1M database - latency of
    the whole path per call (median, max over ranks): eager (one launch per kernel) and as one CUDA-graph
    replay (DetectionPipeline.detect_replay), + the matcher kernel's own duration."""
    import torch
    import torch.distributed as dist
    from sod_b200 import _capi

    def timed(fn):
        ts = []
        for _ in range(iters):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if world > 1:
                dist.barrier()
            a.record()
            fn(n)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))

    for _ in range(3):
        pipe.detect_device(n)
    barrier()
    _capi.timing_enable(True)
    eager = timed(pipe.detect_device)
    stages = {k: _stage_ms(k) for k in _capi.STAGES}
    m = stages["match"]
    _capi.timing_enable(False)       # event records must not be captured into the graph
    barrier()
    pipe.detect_replay(n)            # first call captures
    barrier()
    graph = timed(pipe.detect_replay)
    loc = torch.tensor([eager, graph, float(np.median(m))], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(loc, op=dist.ReduceOp.MAX)
    return float(loc[0]), float(loc[1]), float(loc[2]), {k: float(np.median(v)) for k, v in stages.items() if v}


def oracle_spot_check(wl, res, pipe, args, rows=64):
    """Outside every timed region: `rows` query rows of the batch against the oracle's exact 2-NN over the
    whole database (cv2.BFMatcher semantics, oracle/sod_oracle.py) - indices, squared distances and ratio
    flags - and frame 0 through the oracle's Hough + affine restatement (bins, votes, surviving bins of the
    objects this rank owns)."""
    from oracle import sod_oracle as O
    rng = np.random.default_rng(7)
    n_own = len(res["idx"])
    pick = np.unique(np.concatenate([np.nonzero(res["ok"])[0][:rows // 2], rng.integers(0, n_own, rows)]))[:rows]
    qrows = pick + res["row_lo"]
    qd = wl["q_des"][torch_index(qrows, wl["q_des"])].cpu().numpy()
    db = wl["db_des"].cpu().numpy()
    pi, pd = [], []
    for s in range(0, len(db), 1 << 17):
        i, d = O.knn2(qd, db[s:s + (1 << 17)])
        pi.append(np.where(i >= 0, i + s, -1))
        pd.append(d)
    oi, od = O.merge_top2(np.stack(pi), np.stack(pd))
    ok = O.ratio_pass(od, oi)
    out = {"rows": int(len(pick)), "idx_equal": bool(np.array_equal(res["idx"][pick], oi)),
           "ratio_flags_equal": bool(np.array_equal(res["ok"][pick].astype(bool), ok))}
    # frame 0: the GPU's own matches of that frame -> oracle Hough / valid bins / affine
    per = args.per_frame
    if res["row_lo"] == 0 and n_own >= per:
        okf = res["ok"][:per].astype(bool)
        mq = np.nonzero(okf)[0]
        mt = res["idx"][:per][okf, 0]
        own = (mt >= pipe.row_lo) & (mt < pipe.row_hi) if pipe.world > 1 else np.ones(len(mt), bool)
        scene = O.Scene(wl["q_xy"], wl["q_angle"], wl["q_octave"], wl["m_xy"], wl["m_angle"], wl["m_octave"],
                        wl["m_image"], wl["img_centroid"], wl["img_size"], int(wl["frame_wh"][0, 0]),
                        int(wl["frame_wh"][0, 1]), np.arange(args.objects, dtype=np.int32))
        table = O.hough_vote(scene, mq[own].tolist(), mt[own].tolist(), 15)
        vb = O.valid_bins(table, 5)
        live = O.affine_verify(scene, mq[own].tolist(), mt[own].tolist(), vb, 4)
        want = sorted((int(b.group), tuple(int(v) for v in b.pose), int(b.votes)) for b in live)
        f0 = (res["valid_group"] // pipe.spaces_per_frame == 0) & ((res["status"] & 1) == 1)
        code = res["valid_code"][f0].astype(np.int64)
        got = sorted((int(g % pipe.spaces_per_frame), (int(c // 3375), int(c // 225 % 15), int(c // 15 % 15), int(c % 15)), int(v))
                     for g, c, v in zip(res["valid_group"][f0], code, res["votes"][f0]))
        out.update({"frame0_matches": int(own.sum()), "frame0_verified_bins": len(want),
                    "frame0_hough_affine_equal": bool(got == want)})
    out["parity_check"] = bool(all(v for k, v in out.items() if k.endswith("_equal")))
    return out


def dump_outputs(res, out_dir, budget=60 << 20):   # below 64 MB with the .npy headers
    """--dump-outputs: what the last timed step returned to its caller (DetectionPipeline.fetch), one
    DIR/<name>.npy per array; integers and flags as float64 (exact), floating-point arrays at their own
    precision, counts as 0-d arrays.  The device appends verified bins in whatever order its atomics
    resolve, so the per-bin arrays are written in (Hough space, bin code) order and valid_bin, a position
    in the device's bin table, is left out.  query_rows holds the query row of each entry of the per-query
    arrays (idx, ok); if they would take the total past `budget` bytes, a fixed seeded sample of rows is
    written."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)

    def f(a):
        a = np.asarray(a)
        return a if a.dtype.kind == "f" else a.astype(np.float64)

    order = np.lexsort((res["valid_code"], res["valid_group"]))
    arrays = {k: f(res[k][order]) for k in ("valid_group", "valid_code", "valid_order", "valid_mean", "params",
                                            "votes", "status")}
    arrays.update({k: f(v) for k, v in res.items() if k.startswith("n_")})
    per_query = {"query_rows": f(np.arange(len(res["idx"])) + res["row_lo"]), "idx": f(res["idx"]), "ok": f(res["ok"])}
    n = len(res["idx"])
    row_bytes = sum(a[:1].nbytes for a in per_query.values())
    room = max(budget - sum(a.nbytes for a in arrays.values()), 0) // max(row_bytes, 1)
    if n > room:
        keep = np.sort(np.random.default_rng(0).choice(n, room, replace=False))
        per_query = {k: a[keep] for k, a in per_query.items()}
    arrays.update(per_query)
    for k, a in arrays.items():
        np.save(out / f"{k}.npy", a)


def torch_index(rows, like):
    import torch
    return torch.from_numpy(np.asarray(rows, np.int64)).to(like.device)


def config_records(device, peak_tops, hbm_gbs):
    """The small named configurations of BASELINE.json on ONE GPU (rank 0): C2 (10k x 100k, one object:
    whole path + matcher) and C5 (Hough stress: 2 M ratio-passing matches, 500 objects, 90 % outliers)."""
    import torch
    from sod_b200 import _capi
    from sod_b200 import engine as E
    out = {}
    gen = torch.Generator(device=device).manual_seed(100)
    # ---- C2
    ndb, nq = 100_000, 10_000
    db = sift_like_torch(ndb, gen, device)
    qd = sift_like_torch(nq, gen, device)
    src = torch.randint(0, ndb, (nq // 10,), device=device, generator=gen)
    noise = torch.randint(-3, 4, (nq // 10, 128), device=device, generator=gen, dtype=torch.int16)
    qd[: nq // 10] = (db[src].to(torch.int16) + noise).clamp_(0, 255).to(torch.uint8)
    matcher = E.Matcher(E.prepare_db(db))
    for _ in range(3):
        E.knn_match_ratio(qd, matcher)
    torch.cuda.synchronize()
    _capi.timing_enable(True)
    ts = []
    for _ in range(20):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        E.knn_match_ratio(qd, matcher)
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    km = float(np.median(_stage_ms("match")))
    _capi.timing_enable(False)
    ach = 2.0 * nq * ndb * 128 / (km * 1e-3) / 1e12
    out["C2"] = {"workload": "10,000 query x 100,000 database descriptors, SIFT-like u8, 1 GPU (BASELINE configs[1])",
                 "ms": float(np.median(ts)), "what": "sod_query_prepare + sod_match_top2 + sod_top2_merge (2-NN + ratio)",
                 "kernel_ms": km, "achieved": ach, "unit": "TFLOP/s", "frac": ach / peak_tops,
                 "note": "0.15 ms launch: 40 query blocks x 4 segments on 148 SMs, fill/drain dominated"}
    # ---- C5
    sys.path.insert(0, str(ROOT / "tests"))
    import scenes
    d = scenes.make_match_stress(103, n_objects=500, per_object=4000)
    m = len(d["match_q"])
    sc = E.SceneArrays(d["q_xy"], d["q_angle"], d["q_octave"], d["m_xy"], d["m_angle"], d["m_octave"], d["m_image"],
                       d["img_centroid"], d["img_size"].astype(np.float64),
                       np.array([[d["width"], d["height"]]], np.int32), img_group=d["img_group"], groups_per_frame=500)
    mq, mt = torch.from_numpy(d["match_q"]).to(device), torch.from_numpy(d["match_t"]).to(device)
    voter = E.HoughVoter(sc, 15)
    res = voter.vote(mq, mt)
    aff = E.affine_verify(sc, mq, mt, res, 5, 4)
    torch.cuda.synchronize()
    _capi.timing_enable(True)
    th, ta = [], []
    for _ in range(10):
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        res = voter.vote(mq, mt)
        e1.record()
        aff = E.affine_verify(sc, mq, mt, res, 5, 4, result=aff)
        e2.record()
        torch.cuda.synchronize()
        th.append(e0.elapsed_time(e1))
        ta.append(e1.elapsed_time(e2))
    vote_k = float(np.median(_stage_ms("hough_vote")))
    for k in _capi.STAGES:
        _stage_ms(k)
    _capi.timing_enable(False)
    c = res.counters.cpu().numpy()
    alg = 108.0 * m
    out["C5"] = {"workload": "Hough stress: 2,000,000 ratio-passing matches, 500 objects, 90 % outliers, bins 15 "
                             "(BASELINE configs[4])",
                 "hough_vote_ms": float(np.median(th)), "affine_verify_ms": float(np.median(ta)),
                 "vote_kernel_ms": vote_k, "bins": int(c[0]), "votes": int(c[1]), "near_edge": int(c[2]),
                 "roofline": {"bound": "hbm", "kernel": "hough_vote_kernel", "algorithmic_bytes": alg,
                              "definition": "108 B per match (SURVEY 8d)", "achieved": alg / (vote_k * 1e-3) / 1e9,
                              "peak": hbm_gbs, "unit": "GB/s", "frac": alg / (vote_k * 1e-3) / 1e9 / hbm_gbs,
                              "whole_call_gbs": alg / (float(np.median(th)) * 1e-3) / 1e9}}
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the hot path has no CPU implementation")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    if world != args.gpus and rank == 0:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}", file=sys.stderr)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    wl = make_workload(args, device)
    ndb = args.objects * args.kp_per_object
    int8_tops = measure_int8_cublas_tops(device) if rank == 0 else None
    m = measure(args, wl, args.shard, rank, world, local, device, barrier)
    pipe, nq, nq_total, res = m["pipe"], m["nq"], m["nq_total"], m["res"]
    if args.dump_outputs and rank == 0:
        dump_outputs(res, args.dump_outputs)

    # ---------------- BASELINE configs[2]: 10k-query latency against the (sharded) 1M database
    c3 = None
    if not args.no_configs and nq >= 10_000:
        try:
            c3 = latency_record(pipe, 10_000, world, device, barrier)
        except Exception as exc:   # informational sub-record: never lose the main line over it (all ranks fail alike)
            print(f"C3 latency record failed: {exc!r}", file=sys.stderr)
            c3 = None

    # ---------------- the other partition of the same work, for the record (N > 1 only)
    alt = None
    if world > 1 and not args.no_alt:
        other = "frames" if args.shard == "db" else "db"
        try:
            host_keep = m.pop("host")     # release the pinned buffers of the main run first
            del host_keep
            a = measure(args, wl, other, rank, world, local, device, barrier, with_clocks=False)
            alt = {"parallelism": (f"frame-shard{world}, database replicated, no collective" if other == "frames"
                                   else f"db-shard{world}"),
                   "value": a["nq_total"] * args.steps / (a["ms_total"] * 1e-3), "ms_per_step": a["ms_total"] / args.steps,
                   "kernel_ms": a["sweep_ms"], "e2e": {"value": a["nq_total"] * args.steps / a["e2e_s"], "unit": UNIT,
                                                       "h2d_bytes_per_step": a["h2d"], "d2h_bytes_per_step": a["d2h"]}}
            del a
        except Exception as exc:  # the record is informational: never lose the main line over it
            alt = {"error": repr(exc)[:200]}

    # ---------------- CPU baseline + oracle spot check (rank 0; the baseline only in a single-GPU run)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(wl, args)
        n = ref.calibrate(args.cpu_seconds)
        rr = ref.run(ref.sample_rows(1, n))
        cpu = {"value": rr["n"] / (rr["t_match"] + rr["t_hough_affine"]), "unit": UNIT, "cores": ref.threads,
               "kind": ref.kind,
               "sample": (f"{rr['n']} query descriptors of one frame vs the full {ndb}-row database: "
                          f"cv2.BFMatcher.knnMatch on {ref.threads} OpenCV threads ({rr['t_match']:.2f} s, the call the "
                          f"reference makes, database added in <2^18-row chunks) + {ref.hough_what} "
                          f"({rr['t_hough_affine']:.2f} s, {rr['matches']} matches)"),
               "host_cpus": os.cpu_count()}
    check = None
    if rank == 0 and not args.no_parity_check:
        try:
            check = oracle_spot_check(wl, res, pipe, args)
        except Exception as exc:
            check = {"parity_check": False, "error": repr(exc)[:200]}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:
            pass
        traffic = None
        try:  # dram__bytes_read+write of one match_top2 launch, from the committed ncu --set full capture
            tj = json.loads((ROOT / "profiles" / "r02_match_top2_traffic.json").read_text())
            if world == 1 and (args.frames, args.per_frame, args.objects, args.kp_per_object) == (256, 5000, 1000, 1000):
                traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
        except Exception:
            pass
        bf16_sus = peaks.get("bf16_tflops_sustained", 1400.0)
        hbm = peaks.get("hbm_gbs", 6650.0)
        # MEASURED_PEAKS.json has no int8 entry.  int8 dense is nominally 2 x bf16 dense, and the
        # cuBLASLt int8 GEMM probe of this very run is a second measured ceiling: the denominator is
        # the LARGER of the two, so that the fraction never flatters the kernel.
        peak = max(2.0 * bf16_sus, int8_tops or 0.0)
        shard_rows = pipe.row_hi - pipe.row_lo
        ops = 2.0 * nq * shard_rows * 128
        achieved = ops / (m["sweep_ms"] * 1e-3) / 1e12
        par = ("single" if world == 1 else
               f"db-shard{world}: database rows split at object boundaries, query batch replicated (1/{world} uploaded per "
               f"rank + NVLink all-gather), pruning thresholds shared over peer memory, NCCL "
               f"{'scatter' if args.exchange in ('auto', 'peer') else args.exchange} exchange of the shard-local top-2, Hough+affine by object"
               if args.shard == "db" else f"frame-shard{world}, database replicated, no collective")
        line = {
            "metric": METRIC, "value": nq_total * args.steps / (m["ms_total"] * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": m["ms_total"] / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": (f"{args.frames} frames x {args.per_frame} query descriptors vs {args.objects} objects x "
                                    f"{args.kp_per_object} = {ndb} database descriptors (BASELINE configs[3])"),
                       "n_query": nq_total, "n_db": ndb, "bins": 15, "ratio": 0.75, "hough_spaces": "per (frame, object)",
                       "parallelism": par,
                       "l2": "inputs larger than L2 (128 MB database + 164 MB queries per step)"},
            "e2e": {"value": nq_total * args.steps / m["e2e_s"], "unit": UNIT, "h2d_bytes_per_step": m["h2d"],
                    "d2h_bytes_per_step": m["d2h"], "bytes": "summed over all ranks",
                    "batch_ms_rank0": m["batch_ms"]},
            "gpu_launches": m["launches"] * args.steps,
            "clocks": m["clocks"],
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "traffic": traffic, "kernel": "match_top2_kernel",
                         "algorithmic": {"ops": ops, "definition": "2 * n_query * n_db_shard * 128 int8 ops per launch",
                                         "min_bytes": nq * 128 + shard_rows * 128},
                         "kernel_ms": m["sweep_ms"],
                         "kernel_ms_what": "mean CUDA-event duration of the match_top2_kernel launch alone (sod_timing_*), "
                                           "max over ranks",
                         "seed_sweep_ms": m["seed_ms"],
                         "thresholds": ("peer memory, rotated block order" + ("" if pipe.seed_matcher is not None else ", no seeding sweep")
                                        if pipe.peer_thr is not None and world > 1 else
                                        f"NCCL MIN all-reduce, {pipe.sweep_stages} sweep stage(s)" if pipe.seed_matcher is not None
                                        else "none"),
                         "peak_source": ("max(2 x MEASURED_PEAKS.bf16_tflops_sustained = %.1f, cuBLASLt int8 8192^3 GEMM "
                                         "measured in this run = %.1f); MEASURED_PEAKS.json has no int8 entry%s"
                                         % (2.0 * bf16_sus, int8_tops or 0.0, "" if peaks else " (file absent: 1400 fallback)")),
                         "frac_of_nominal_int8_4500": achieved / 4500.0,
                         "int8_cublaslt_8192_tops": int8_tops},
            "stages_ms": {"match_sweep": m["sweep_ms"], "seed_sweep": m["seed_ms"], "hough_vote_kernel": m["vote_ms"],
                          "hough_other": m["hough_other_ms"], "affine": m["affine_ms"]},
            "result_check": {"matches": res["n_matches"], "bins": res["n_bins"], "valid_bins": res["n_valid"],
                             "verified_bins": int((res["status"] & 1).sum()), "near_edge": res["n_near_edge"],
                             "planted": wl["n_true"], "scope": "this rank's objects" if world > 1 and args.shard == "db" else "all"},
        }
        if check is not None:
            line["parity_check"] = check.pop("parity_check")
            line["parity"] = check
        configs = {}
        if c3 is not None:
            ach3 = 2.0 * 10_000 * shard_rows * 128 / (c3[2] * 1e-3) / 1e12
            xchg = ("none" if world == 1 else "peer memory (sod_top2_exchange_peer: 2 kernels, no collective call)"
                    if pipe.peer is not None else f"NCCL scatter (peer memory unavailable: {pipe.peer_error})")
            configs["C3"] = {"workload": f"10,000-descriptor query vs the 1M-descriptor database on {world} GPU(s) "
                                         "(BASELINE configs[2]), whole path per call (2-NN + ratio + Hough + affine)",
                             "ms": c3[1], "ms_what": "one CUDA-graph replay of the path (DetectionPipeline.detect_replay), "
                                                     "median of 30, max over ranks",
                             "ms_eager": c3[0], "kernel_ms": c3[2], "achieved": ach3, "unit": "TFLOP/s",
                             "frac": ach3 / peak, "exchange": xchg, "stages_ms_rank0": c3[3]}
        if world == 1 and not args.no_configs:
            try:
                configs.update(config_records(device, peak, hbm))
            except Exception as exc:
                configs["error"] = repr(exc)[:200]
        if configs:
            line["configs"] = configs
        if alt is not None:
            line["alt_partition"] = alt
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_reference(args):
    """The reference's own CPU implementation of the path on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    import torch
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0"))) if torch.cuda.is_available() else torch.device("cpu")
    wl = make_workload(args, device)   # same synthetic inputs; only data generation touches the GPU
    ref = CpuReference(wl, args)
    n = ref.calibrate(args.cpu_seconds)
    for w in range(args.warmup):
        ref.run(ref.sample_rows(w, max(16, n // 8)))
    t0 = time.perf_counter()
    tot = 0
    for s in range(args.steps):
        tot += ref.run(ref.sample_rows(s, n))["n"]
    dt = time.perf_counter() - t0
    nq, ndb = args.frames * args.per_frame, args.objects * args.kp_per_object
    v = tot / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": (f"{args.frames} frames x {args.per_frame} query descriptors vs {args.objects} objects x "
                                    f"{args.kp_per_object} = {ndb} database descriptors (BASELINE configs[3])"),
                       "n_query": nq, "n_db": ndb, "bins": 15, "ratio": 0.75},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": ref.threads, "kind": ref.kind, "host_cpus": os.cpu_count(),
                             "sample": (f"each step = {n} query descriptors of ONE frame vs the full database, the rate "
                                        f"extrapolates linearly to the {nq}-descriptor batch: "
                                        f"cv2.BFMatcher.knnMatch ({ref.threads} threads, chunks < 2^18 rows) + "
                                        f"{ref.hough_what} (1 thread)")},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--per-frame", type=int, default=5000)
    ap.add_argument("--objects", type=int, default=1000)
    ap.add_argument("--kp-per-object", type=int, default=1000)
    ap.add_argument("--instances", type=int, default=4)
    ap.add_argument("--inlier-frac", type=float, default=0.10)
    ap.add_argument("--false-frac", type=float, default=0.01)
    ap.add_argument("--shard", default="db", choices=["db", "frames"],
                    help="N > 1: split the database rows (default: the north star's layout, one exchange of the "
                         "shard-local top-2) or the frames (database replicated, no collective)")
    ap.add_argument("--seed-rows", type=int, default=None,
                    help="--shard db: rows of the replicated threshold-seeding sample (0 = off; default: pipeline's)")
    ap.add_argument("--sweep-stages", type=int, default=None,
                    help="--shard db with seeding: tile ranges of the shard sweep with a threshold all-reduce between them")
    ap.add_argument("--thresholds", default="auto", choices=["auto", "peer", "allreduce"],
                    help="--shard db with seeding: thresholds over peer memory (rotated block order) or NCCL all-reduces")
    ap.add_argument("--no-alt", action="store_true", help="N > 1: skip the sub-record of the other partition")
    ap.add_argument("--no-configs", action="store_true", help="skip the C2 / C3 / C5 sub-records")
    ap.add_argument("--no-parity-check", action="store_true", help="skip the oracle spot check")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "scatter", "gather"],
                    help="--shard db: how the shard-local top-2 are merged (DetectionPipeline)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU work per baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0's result) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
