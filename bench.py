#!/usr/bin/env python
"""bench.py — plans/sec of the batched plan-generation-and-validation path (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2|c3|c5]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...      (N > 1)

Workloads (benchmarks/workloads.py; weak scaling: the per-GPU share is fixed):
  c2 (default, BASELINE.json configs[1], the configuration the metric is quoted on): 500 m x 200 m field +
     the two obstacles of mlp3:1629-1632, W = 3.2 m, 4096 candidates per GPU = 4 start corners x 1024 radii,
     h = 0.1 m, every path and speed profile MATERIALISED in HBM;
  c3 (configs[2]): 4096 tilted parallelograms per GPU x 180 headings, summary only, argmin per field;
  c5 (configs[4]): 2 km x 1 km field at h = 0.05 m, 8192 candidates per GPU (65 536 over 8), summary only.
One step = one pass of the full chain over the batch: layout -> path sampling -> speed planning -> kinematic +
geofence validation -> coverage rasterisation -> per-field argmin (+ the cross-GPU argmin merge for N > 1).

value      candidates/s over EXACTLY K steps, inputs resident in HBM (CUDA events, max over ranks)
sustained  the same step repeated for >= --sustain seconds (default 2 s) with no host synchronisation inside,
           SM clocks sampled under load — the burst of K steps may run at boost clocks a long job does not keep
e2e        same metric through the public API plan_batch(host numpy fields + candidate axes, winners=True) -> host
           numpy: host set-up, pinned H2D copies, kernels, D2H of all summaries + the argmin + every field's WINNING
           path and speeds, every step.  e2e.value = the throughput form of the call (wait=False: batch k+1 is
           submitted before the result of batch k is collected), e2e.serial_value = one call at a time
argmin_ok  the (merged) per-field argmin of the timed steps equals the argmin of the whole job's candidates
           evaluated shard by shard on one GPU and merged in numpy (outside the timed region)
roofline   the dominant kernel: issue-slot and FP64-pipe utilisation from the committed ncu capture of this
           build (the binding limits) next to algorithmic bytes / CUDA-event duration vs the measured HBM peak
cpu_baseline  the CPU oracle port process-parallel on all host cores over a bounded sample, split into
           plan_only (generation + speed planning + validation, vectorised numpy) and coverage_only
           (BRUTE-FORCE per-cell integer raster in C: a checker, not an optimised CPU rasteriser)
--impl reference   the same CPU arm as its own JSON line (the reference is pure Python + Shapely and cannot be
           installed here; the oracle port is what runs — see DESIGN.md), same `config` as the GPU arm
--dump-outputs DIR   after the K timed steps, write what the last of them computed as DIR/<name>.npy (float64): the
           per-field argmin, the summary columns and the paths + speed profiles of a fixed, seeded sample of candidates
           (see dump_outputs).  The inputs are generated deterministically, so two builds can be compared file by file.
           With N > 1 rank 0 writes: the argmin is the merged one, summaries and paths cover rank 0's candidate range.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from benchmarks import workloads as wl  # noqa: E402

METRIC = "plans/sec (gen+speed+geofence+coverage)"
UNIT = "plans/s"


def make_config(w: wl.Workload, n_gpus: int):
    """`config` of the JSON line — identical for the GPU arm and the reference arm."""
    return {"workload": w.text, "name": w.name, "candidates_per_step": w.n_cand, "n_gpus": n_gpus,
            "outputs": ("paths+speeds materialised in HBM (24 B/point) + 176 B summaries + argmin"
                        if w.outputs == "paths" else "176 B summaries + per-field argmin (no paths)"),
            "l2": "256 MB flush write between timed steps"}


# ------------------------------------------------------------------------------------------------
# CPU arm (oracle port), used by cpu_baseline and by --impl reference
# ------------------------------------------------------------------------------------------------
def _cpu_one(job):
    """One candidate with the CPU oracle: (seconds without coverage, seconds with coverage, cost)."""
    from oracle import batch as ob, ref_planner as rp
    verts, R, heading, corner, obst, h = job
    t0 = time.perf_counter()
    ob.evaluate_candidate(verts, rp.VehicleParams(), R=R, heading=heading, start_corner=corner, obstacles=obst,
                          grid_h=h, coverage=False)
    t1 = time.perf_counter()
    o = ob.evaluate_candidate(verts, rp.VehicleParams(), R=R, heading=heading, start_corner=corner, obstacles=obst,
                              grid_h=h, coverage=True)
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1, (o["len_main"] + o["len_head"]) if o["status"] == 0 else float("inf")


def cpu_sample(w: wl.Workload, n_sample: int):
    idx = np.linspace(0, w.n_cand - 1, min(n_sample, w.n_cand)).astype(int)
    return [w.oracle_args(int(i)) for i in idx]


def run_cpu(pool, cores, sample):
    """-> dict(total, plan_only, coverage_only plans/s, wall).  total = the sample's wall clock (every candidate is
    evaluated once with and — for the split — once without coverage; the latter, ~1 %, is subtracted)."""
    t0 = time.perf_counter()
    res = pool.map(_cpu_one, sample, chunksize=1)
    wall = time.perf_counter() - t0
    t_plan = sum(r[0] for r in res)
    t_full = sum(r[1] for r in res)
    busy = t_plan + t_full
    wall_full = wall * t_full / busy                     # the share of the wall clock spent in the full evaluations
    n = len(sample)
    par = min(cores, n)
    return {"total": n / wall_full, "plan_only": n / (t_plan / par), "coverage_only": n / (max(t_full - t_plan, 1e-9) / par),
            "wall": wall}


def make_pool():
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    from oracle import raster
    raster.build()
    return mp.get_context("fork").Pool(cores), cores


def default_cpu_sample(w: wl.Workload, cores: int, per_step: bool):
    """Bounded sample sizes (about 10-20 s of CPU work on 16 cores): the brute-force band raster costs ~0.25 s per
    candidate at config 2 / 3 and ~22 s at config 5 (19 million cells)."""
    if w.name == "c5":
        return cores
    return 256 if per_step else 1024


CPU_NOTE = ("CPU oracle port of the reference (the pure-Python reference needs Shapely, not installable here); "
            "coverage_only is a brute-force per-cell x per-segment integer raster (a checker), plan_only is "
            "vectorised numpy — the reference's own per-point Python loops are ~15x slower (SURVEY.md §6.2)")


# ------------------------------------------------------------------------------------------------
# clocks (NVML sampled DURING the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index: int, period: float = 0.005):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.sm, self.reasons, self.max_mhz, self.power = [], set(), None, []
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    NAMES = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
             0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
             0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def run(self):
        if self.nv is None:
            return
        while not self._halt.is_set():
            try:
                self.sm.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                try:
                    self.power.append(self.nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                except Exception:
                    pass
                try:
                    r = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    r = int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in self.NAMES.items():
                    if r & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        return {"sm_mhz": int(statistics.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "power_w_max": round(max(self.power), 1) if self.power else None}


def ncu_metrics(kernel: str, workload: str):
    """Per-launch metrics of `kernel` from the committed `ncu --set full` capture of this build and workload
    (profiles/ncu_metrics.json, written by profiles/summarize.py): DRAM bytes, issue-slot and FP64-pipe
    utilisation.  {} if absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_metrics.json")) as f:
            t = json.load(f)
        return t.get(workload, t).get(kernel, {})
    except Exception:
        return {}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def numpy_merge(parts):
    """[(best_cost[F], best_cand[F])] of the shards -> the job's per-field argmin: lowest cost, ties to the lowest
    global candidate index, -1 when no shard has a valid candidate."""
    cost = np.full_like(parts[0][0], np.inf)
    cand = np.full_like(parts[0][1], -1)
    for c, k in parts:
        better = (k >= 0) & ((cand < 0) | (c < cost) | ((c == cost) & (k < cand)))
        cost = np.where(better, c, cost)
        cand = np.where(better, k, cand)
    return cost, cand


DUMP_LIMIT_BYTES = 64 << 20
DUMP_SUMMARY_ROWS = 65536     # candidates whose summaries --dump-outputs writes (a seeded sample above that)
DUMP_PATH_ROWS = 256          # candidates whose paths and speed profiles it writes


def dump_outputs(bufs, n_cand: int, n_fields: int, cand_base: int, with_paths: bool):
    """What one device step left in ``bufs`` (the arrays run_device_batch hands its caller), as float64 host arrays:
      best_cost, best_cand            [F]       per-field argmin (-1: no valid candidate)
      summary_cand                    [S]       global indices of the candidates whose summaries follow
      summary_<column>                [S, ...]  every fcpp_summary column but `reserved`
      path_cand, path_offsets         [P], [P+1]  (paths mode) the candidates whose points follow, and their ranges
      path_xy, speeds_kmh             [n, 2], [n]
    Batches of more than DUMP_SUMMARY_ROWS / DUMP_PATH_ROWS candidates are sampled with fixed seeds, so the same
    arguments give the same rows.  Integer outputs are exact in float64."""
    import torch
    from field_coverage_path_planning_b200 import _lib

    def sample(k: int, seed: int) -> np.ndarray:
        if n_cand <= k:
            return np.arange(n_cand)
        return np.sort(np.random.default_rng(seed).choice(n_cand, k, replace=False))

    out = {"best_cost": bufs.d_cost[:n_fields].cpu().numpy().astype(np.float64),
           "best_cand": bufs.d_best[:n_fields].cpu().numpy().astype(np.float64)}
    rows = sample(DUMP_SUMMARY_ROWS, 1)
    isz = _lib.SUMMARY_DTYPE.itemsize
    raw = bufs.d_sum[:n_cand * isz].view(n_cand, isz)[torch.as_tensor(rows, device=bufs.d_sum.device)]
    s = np.ascontiguousarray(raw.cpu().numpy()).view(_lib.SUMMARY_DTYPE).reshape(-1)
    out["summary_cand"] = (rows + cand_base).astype(np.float64)
    for name in _lib.SUMMARY_DTYPE.names:
        if name != "reserved":
            out["summary_" + name] = s[name].astype(np.float64)
    if with_paths:
        rows = sample(DUMP_PATH_ROWS, 2)
        off = bufs.d_off[:n_cand + 1].cpu().numpy()
        idx = np.concatenate([np.arange(off[b], off[b + 1]) for b in rows] + [np.zeros(0, dtype=np.int64)])
        ti = torch.as_tensor(idx, device=bufs.d_path.device)
        out["path_cand"] = (rows + cand_base).astype(np.float64)
        out["path_offsets"] = np.concatenate([[0], np.cumsum(off[rows + 1] - off[rows])]).astype(np.float64)
        out["path_xy"] = bufs.d_path[ti].cpu().numpy()
        out["speeds_kmh"] = bufs.d_spd[ti].cpu().numpy()
    nbytes = sum(a.nbytes for a in out.values())
    if nbytes > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {nbytes} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    return out


def write_dump(directory: str, arrays) -> None:
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(wl.WORKLOADS))
    ap.add_argument("--sustain", type=float, default=2.0, help="seconds of the sustained region (0: skip)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="candidates in the bounded CPU sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-check", action="store_true", help="skip the argmin check against the whole job")
    ap.add_argument("--e2e-explicit", action="store_true",
                    help="e2e leg with explicit per-candidate arrays instead of the factored candidate axes")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (GPU arm, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the GPU arm (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1 and args.impl == "b200":
        raise SystemExit("bench.py --gpus N (N > 1) must be launched with one process per GPU:\n  python -m torch.distributed.run "
                         "--nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...")
    n_gpus = max(args.gpus, world)
    w = wl.WORKLOADS[args.workload](n_gpus)
    config = make_config(w, n_gpus)

    if args.impl == "reference":
        if rank != 0:
            return 0
        pool, cores = make_pool()
        sample = cpu_sample(w, args.cpu_sample or default_cpu_sample(w, cores, True))
        for _ in range(min(args.warmup, 1)):
            run_cpu(pool, cores, sample[:cores])
        first = run_cpu(pool, cores, sample)
        # a bounded run: at most ~3 minutes of steps (config 5 costs ~22 s per candidate and core)
        steps = max(1, min(args.steps, int(180.0 / max(first["wall"], 1e-3))))
        runs = [first] + [run_cpu(pool, cores, sample) for _ in range(steps - 1)]
        pool.close()
        n = len(sample)
        tot = n * steps / sum(n / r["total"] for r in runs)
        split = {k: n * steps / sum(n / r[k] for r in runs) for k in ("plan_only", "coverage_only")}
        desc = (f"{n} candidates evenly spaced over the {w.n_cand} of the job per step, {steps} steps, full chain "
                f"incl. the brute-force integer coverage raster, {cores} processes")
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": tot, "unit": UNIT, "n_gpus": n_gpus, "steps": steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sum(n / r["total"] for r in runs) / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config,
            "cpu_baseline": {"value": tot, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc,
                             "plan_only": split["plan_only"], "coverage_only": split["coverage_only"],
                             "note": CPU_NOTE},
            "e2e": {"value": tot, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return 0

    # ---------------------------------------------------------------- GPU arm
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    import ctypes as C
    import field_coverage_path_planning_b200 as fc
    from field_coverage_path_planning_b200 import _lib
    from field_coverage_path_planning_b200.batch import BatchBuffers, DeviceBatch, prepare_batch, run_device_batch
    from field_coverage_path_planning_b200 import dist as fdist

    veh = fc.VehicleParams()
    F = len(w.fields)
    cands, lo = fdist.shard_candidates(w.cands, world, rank)
    B = len(cands["field_id"])
    hi = lo + B
    h = _lib.handle(local_rank)
    h.check(h.lib.fcpp_set_profiling(h.h, 1))

    # resident inputs + reusable output buffers (first run sizes them)
    pb = prepare_batch(w.fields, veh, cands, w.obstacles, None, w.grid_h, True)
    db = DeviceBatch(pb, dev)
    first = run_device_batch(db, w.outputs, cand_base=lo)
    total_pts = int(first.offsets[-1]) if w.outputs == "paths" else 0
    n_pts_mean = float((first.summary["n_main"] + first.summary["n_head"]).mean())
    bufs = BatchBuffers(dev, B, F, total_pts)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def step_device():
        run_device_batch(db, w.outputs, cand_base=lo, buffers=bufs, fetch=False)
        if world > 1:
            fdist.reduce_best(bufs.d_cost, bufs.d_best)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    align_token = torch.zeros(1, dtype=torch.int32, device=dev)

    def align_start():
        """Last part of the barrier in front of a timed region: a device-side barrier (one tiny all-reduce ENQUEUED
        behind the host barrier + synchronize).  The ranks' hosts leave the host barrier up to a millisecond apart;
        without it that skew lands in the first timed step's collective (rank 0 at N = 8: 2.09 ms for step 1, 1.07 ms
        for every other step)."""
        if world > 1:
            dist.all_reduce(align_token)

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step_device()
    # ---- the K timed steps (CUDA events per step; per-kernel event times at N = 1) ----
    # everything that takes host time (NVML initialisation, event creation) happens BEFORE the barrier: ranks that
    # leave it at different times would spend the difference inside the first step's collective
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sync_all()
    align_start()
    sampler.sm.clear()
    sampler.power.clear()
    sampler.reasons.clear()
    ktimes = []
    l0 = h.launches
    t_wall0 = time.perf_counter()
    for k in range(args.steps):
        flush.zero_()                                       # L2 flush between timed iterations
        ev[k][0].record()
        step_device()
        ev[k][1].record()
        if world == 1:
            ev[k][1].synchronize()
            ms3 = (C.c_float * 3)()
            h.check(h.lib.fcpp_kernel_times(h.h, C.byref(ms3)))
            ktimes.append(list(ms3))
        # N > 1: no host synchronisation inside the timed region — every step ends in a collective, and a
        # per-step host sync would add each rank's launch jitter to every rendezvous
    sync_all()
    if world > 1:
        ms3 = (C.c_float * 3)()
        h.check(h.lib.fcpp_kernel_times(h.h, C.byref(ms3)))   # of the last step
        ktimes.append(list(ms3))
    t_wall = time.perf_counter() - t_wall0
    launches = h.launches - l0
    clocks = sampler.stop()
    dev_ms_max = max_over_ranks(sum(a.elapsed_time(b) for a, b in ev))
    total_cands = w.n_cand
    value = total_cands * args.steps / (dev_ms_max / 1e3)
    step_ms = dev_ms_max / args.steps
    # taken before the sustained region runs further steps through the same buffers
    dumped = dump_outputs(bufs, B, F, lo, w.outputs == "paths") if args.dump_outputs and rank == 0 else None

    # ---- merged argmin of the timed steps vs the whole job evaluated shard by shard on this GPU ----
    argmin_ok = None
    if not args.no_check:
        got_cost = bufs.d_cost.cpu().numpy()[:F].copy()
        got_cand = bufs.d_best.cpu().numpy()[:F].copy()
        if world == 1:
            # numpy rule on the batch's own summaries: lowest cost per field, ties to the lowest index
            s = first.summary
            fid = cands["field_id"]
            cost = np.where(s["status"] == 0, s["len_main"] + s["len_head"], np.inf)
            want_cost = np.full(F, np.inf)
            np.minimum.at(want_cost, fid, cost)
            hit = np.nonzero(np.isfinite(cost) & (cost == want_cost[fid]))[0]
            want_cand = np.full(F, np.iinfo(np.int64).max, dtype=np.int64)
            np.minimum.at(want_cand, fid[hit], hit + lo)
            want_cand[~np.isfinite(want_cost)] = -1
        else:
            parts = []
            for r in range(world):
                rc, rlo = fdist.shard_candidates(w.cands, world, r)
                rdb = db if r == rank else DeviceBatch(prepare_batch(w.fields, veh, rc, w.obstacles, None, w.grid_h, True), dev)
                rr = run_device_batch(rdb, "summary", cand_base=rlo, copy_summary=False)
                parts.append((rr.best_cost.copy(), rr.best_cand.copy()))
            want_cost, want_cand = numpy_merge(parts)
        ok = bool(np.array_equal(got_cost, want_cost) and np.array_equal(got_cand, want_cand))
        t = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        argmin_ok = bool(t.item())

    # ---- sustained region: the same step for >= args.sustain seconds, no host sync inside ----
    sustained = None
    if args.sustain > 0:
        n_sus = max(args.steps, int(math.ceil(args.sustain * 1e3 / max(step_ms, 1e-3))))
        if world > 1:      # every rank must run the same number of steps (each ends in a collective)
            t = torch.tensor([n_sus], dtype=torch.int64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            n_sus = int(t.item())
        s2 = ClockSampler(local_rank)
        s2.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        align_start()
        s2.sm.clear()
        s2.power.clear()
        s2.reasons.clear()
        t0 = time.perf_counter()
        e0.record()
        for _ in range(n_sus):
            flush.zero_()
            step_device()
        e1.record()
        sync_all()
        sus_wall = time.perf_counter() - t0
        ck = s2.stop()
        # the flush is inside this region (one event pair): subtract its measured cost
        fa, fb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fa.record()
        for _ in range(50):
            flush.zero_()
        fb.record()
        fb.synchronize()
        flush_ms = fa.elapsed_time(fb) / 50
        sus_ms = max_over_ranks(e0.elapsed_time(e1)) - n_sus * flush_ms
        sustained = {"value": total_cands * n_sus / (sus_ms / 1e3), "unit": UNIT, "steps": n_sus,
                     "seconds": sus_wall, "ms_per_step": sus_ms / n_sus, "flush_ms_subtracted": flush_ms,
                     "clocks": ck}

    # ---- e2e through the public API (host numpy in, host numpy out, winners' paths included) ----
    # the candidate set in factored form (field x heading x radius x start corner axes, decoded on the device):
    # the same candidates in the same order as the explicit arrays of the device-timed loop (asserted in
    # tests/test_host_cpu.py); --e2e-explicit passes the per-candidate arrays instead
    if args.e2e_explicit:
        host_cands = {k: v.copy() for k, v in (w.cands if world > 1 else cands).items()}
    else:
        host_cands = w.axes                 # the whole job; plan_batch(distributed=True) takes each rank's range

    def step_e2e(wait=True):
        return fc.plan_batch(w.fields, veh, host_cands, obstacles=w.obstacles, outputs=w.outputs, grid_h=w.grid_h,
                             device=dev, distributed=world > 1, winners=True, wait=wait)

    for _ in range(3):
        r = step_e2e()
    sync_all()
    e2e_steps = args.steps
    # (a) one call after the other: every call waits for its own result
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        r = step_e2e()
    sync_all()
    e2e_serial = total_cands * e2e_steps / max_over_ranks(time.perf_counter() - t0)
    e2e_value, e2e_mode = e2e_serial, "one call at a time"
    if True:
        # (b) the throughput form of the same public call: batch k+1 is submitted (wait=False) before the result of
        # batch k is collected, so the host side of one call overlaps the kernels of the other.  Every step still
        # prepares its inputs on the host, copies them from pinned memory and reads its whole result back.
        pend = step_e2e(wait=False)          # warm-up: device path buffers and pinned result buffers of two
        for _ in range(6):                   # batches in flight come from the allocators' caches afterwards
            nxt = step_e2e(wait=False)
            r = pend.result()
            pend = nxt
        r = pend.result()
        sync_all()
        t0 = time.perf_counter()
        pend = step_e2e(wait=False)
        for _ in range(e2e_steps - 1):
            nxt = step_e2e(wait=False)
            r = pend.result()
            pend = nxt
        r = pend.result()
        sync_all()
        e2e_value = total_cands * e2e_steps / max_over_ranks(time.perf_counter() - t0)
        e2e_mode = "two calls in flight (plan_batch(..., wait=False) / PendingBatch.result())"
    h2d = int(r.extras.get("h2d_bytes", pb.h2d_bytes()))
    d2h = int(r.extras.get("d2h_bytes", 0))
    e2e_ok = bool(np.array_equal(r.best_cand, got_cand)) if not args.no_check else None

    # ---- roofline of the dominant kernel ----
    kt = np.asarray(ktimes[1:] if len(ktimes) > 1 else ktimes, dtype=np.float64)
    k_layout, k_plan, k_cover = float(kt[:, 0].mean()), float(kt[:, 1].mean()), float(kt[:, 2].mean())
    s = first.summary
    g = s["corner_g"].astype(np.int64)
    G_cells = s["cov_total"].astype(np.int64) + 4 * g * g
    npts = (s["n_main"] + s["n_head"]).astype(np.int64)
    bytes_plan = float((24 * npts * (1 if w.outputs == "paths" else 0) + 176 + 1008).sum())
    bytes_cover = float((2 * ((G_cells + 7) // 8) + 176 + 1008).sum())
    peak, peak_src = measured_peak_gbs()
    if k_cover >= k_plan:
        dom, ach = "cover_kernel", bytes_cover / (k_cover * 1e-3) / 1e9
    else:
        dom, ach = "plan_kernel", bytes_plan / (k_plan * 1e-3) / 1e9
    nm = ncu_metrics("plan_gen_kernel" if dom == "plan_kernel" else dom, w.name) or ncu_metrics(dom, w.name)
    roofline = {"bound": "issue", "kernel": dom,
                "issue_slot_frac": nm.get("issue_slot_frac"), "fp64_pipe_frac": nm.get("fp64_pipe_frac"),
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": nm.get("dram_bytes"), "peak_source": peak_src,
                "kernel_ms": {"layout+scan": k_layout, "plan_kernel": k_plan, "cover_kernel": k_cover, "step": step_ms},
                "algorithmic_bytes_per_launch": {"plan_kernel": bytes_plan, "cover_kernel": bytes_cover},
                "per_kernel": {
                    "plan_gen_kernel": {"ms": k_plan, "achieved": bytes_plan / (k_plan * 1e-3) / 1e9,
                                        "frac": bytes_plan / (k_plan * 1e-3) / 1e9 / peak,
                                        **{k: ncu_metrics("plan_gen_kernel", w.name).get(k) for k in ("issue_slot_frac", "fp64_pipe_frac")}},
                    "cover_kernel": {"ms": k_cover, "achieved": bytes_cover / (k_cover * 1e-3) / 1e9,
                                     "frac": bytes_cover / (k_cover * 1e-3) / 1e9 / peak,
                                     **{k: (ncu_metrics("cover_kernel", w.name) or ncu_metrics("cover_work_kernel", w.name)).get(k)
                                        for k in ("issue_slot_frac", "fp64_pipe_frac")}}},
                "ncu_source": nm.get("source"),
                "note": "both hot kernels are instruction-issue bound (FP64 + integer), not HBM bound: the occupancy grid "
                        "lives in shared memory and most of the band is counted in closed form, so `frac` (algorithmic "
                        "bytes of SURVEY.md §8(d) over the measured HBM peak) is a labelled throughput yardstick that can "
                        "exceed 1; issue_slot_frac / fp64_pipe_frac (ncu, same build) are the binding limits"}

    # ---- CPU baseline on the box's host cores (rank 0, N = 1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        pool, cores = make_pool()
        sample = cpu_sample(w, args.cpu_sample or default_cpu_sample(w, cores, False))
        run_cpu(pool, cores, sample[:cores])
        rc = run_cpu(pool, cores, sample)
        pool.close()
        cpu = {"value": rc["total"], "unit": UNIT, "cores": cores, "kind": "port",
               "plan_only": rc["plan_only"], "coverage_only": rc["coverage_only"],
               "sample": f"{len(sample)} candidates evenly spaced over the batch, full chain (gen+speed+validation+"
                         f"brute-force integer coverage raster) with the CPU oracle, {cores} processes, {rc['wall']:.1f} s wall",
               "note": CPU_NOTE}

    if dumped is not None:
        write_dump(args.dump_outputs, dumped)
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
            "warmup": warm, "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config,
            "detail": {"points_per_plan": n_pts_mean, "fields": F,
                       "wall_ms_per_step_incl_flush": 1e3 * t_wall / args.steps,
                       "step_ms_rank0": [round(a.elapsed_time(b), 4) for a, b in ev]},
            "clocks": clocks, "sustained": sustained, "argmin_ok": argmin_ok,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "argmin_ok": e2e_ok, "mode": e2e_mode, "serial_value": e2e_serial,
                    "speculative_sizes": bool(r.extras.get("speculative", False)),
                    "api": "plan_batch(host numpy fields + "
                           + ("per-candidate arrays" if args.e2e_explicit else "candidate axes (candidate_axes)")
                           + ", winners=True) -> summaries + argmin + every field's winning path and speeds on the host"},
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu}))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
