#!/usr/bin/env python
"""What the segment-level obstacle sweep costs (DESIGN.md §3.9), one GPU, steady state.

    python benchmarks/sweep_bench.py [--workloads c2,hs,paths] [--steps 20] [--rounds 3] [--fields 1024] [--out FILE]

Workloads:
  c2     benchmarks/workloads.py c2: 4 096 candidates on the 500 x 200 m field with two obstacles, paths materialised
  hs     a heading search (180 headings) of c3's seeded parallelograms (--fields of them) with one to three seeded
         obstacles per field, summary only
  paths  the caller-path form: 320 ragged paths (the first c2 plans) and one path of 30 000 points
Per workload, one JSON line:
  step_ms          device time of one step (layout .. coverage + argmin, inputs and buffers resident) with the sweep
                   off and on, CUDA events over --steps steps; the two arms alternate --rounds times, medians
  sweep_us         the sweep kernel alone over the step's records (or the paths), CUDA events over 200 launches
  e2e_plans_s      plans/s through plan_batch(..., winners=True) with two calls in flight (wait=False), sweep off / on
  launches         kernels per step, sweep off / on
  gpu, power_limit_w   read in the same run
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from benchmarks import workloads as wl  # noqa: E402


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return float(out[0])
    except Exception:
        return None


def heading_search(F: int):
    fields = wl.c3_fields(F)
    rng = np.random.default_rng(4321)
    obstacles = []
    for f in fields:
        c = f.mean(axis=0)
        obst = []
        for _ in range(int(rng.integers(1, 4))):
            cx, cy = c + rng.uniform(-40, 40, 2)
            a, b = rng.uniform(3, 15, 2)
            obst.append([(cx - a, cy - b), (cx + a, cy - b), (cx + a, cy + b), (cx - a, cy + b)])
        obstacles.append(obst)
    heads = np.deg2rad(np.arange(180.0))
    return wl.Workload("hs", f"{F} c3 parallelograms x 180 headings, 1-3 obstacles per field, summary only", fields,
                       {"field_id": np.repeat(np.arange(F, dtype=np.int32), 180), "heading": np.tile(heads, F)},
                       obstacles, 0.1, "summary", {"axes": True, "n_fields": F, "heading": heads})


def events_ms(st, fn, reps):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(reps):
        fn()
    b.record(st)
    b.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2,hs,paths")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--fields", type=int, default=1024)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sweep_bench.py needs a CUDA device")
    import field_coverage_path_planning_b200 as fc
    from field_coverage_path_planning_b200 import _lib
    from field_coverage_path_planning_b200.batch import (BatchBuffers, DeviceBatch, _pack_to_dev, prepare_batch,
                                                         run_device_batch)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    gpu, plim = torch.cuda.get_device_name(dev), power_limit_w()
    veh = fc.VehicleParams()
    h = _lib.handle(0)
    st = torch.cuda.current_stream(dev)
    sptr = C.c_void_p(st.cuda_stream)
    lines = []
    for name in args.workloads.split(","):
        if name == "paths":
            w = wl.c2(1)
            res = fc.plan_batch(w.fields, veh, w.cands, obstacles=w.obstacles, outputs="paths")
            ragged = [res.path(b)[0] for b in range(320)]
            long_p, k = [], 0
            while sum(len(p) for p in long_p) < 30000:
                long_p.append(res.path(k)[0])
                k += 1
            one = np.concatenate(long_p)[:30000]
            line = {"workload": "paths", "gpu": gpu, "power_limit_w": plim}
            for tag, paths in (("ragged320", ragged), ("one30000", [one])):
                n = len(paths)
                offs = np.concatenate([[0], np.cumsum([len(p) for p in paths])]).astype(np.int64)
                polys = [np.asarray(o, dtype=np.float64) for o in wl.OBST2]
                t = _pack_to_dev({"path": np.concatenate(paths), "offsets": offs,
                                  "vs": np.array([0, 4, 8], dtype=np.int32), "verts": np.concatenate(polys)}, dev)
                d_out = torch.empty(n * 24, dtype=torch.uint8, device=dev)

                def sweep_fn():
                    h.check(h.lib.fcpp_obstacle_sweep_paths(h.h, t["path"].data_ptr(), t["offsets"].data_ptr(), n, None,
                                                            t["vs"].data_ptr(), t["verts"].data_ptr(), 2, veh.working_width / 2,
                                                            d_out.data_ptr(), sptr))
                for _ in range(5):
                    sweep_fn()
                us = [1e3 * events_ms(st, sweep_fn, 200) for _ in range(args.rounds)]
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    fc.obstacle_sweep(paths, wl.OBST2, veh.working_width)
                rate = n * args.steps / (time.perf_counter() - t0)
                line[tag] = {"points": int(offs[-1]), "sweep_us": statistics.median(us), "sweep_us_all": us,
                             "e2e_paths_s": rate, "launches": 1}
            print(json.dumps(line), flush=True)
            lines.append(line)
            continue
        w = heading_search(args.fields) if name == "hs" else wl.WORKLOADS[name](1)
        F = len(w.fields)
        B = len(w.cands["field_id"])
        pb = prepare_batch(w.fields, veh, w.cands, w.obstacles, None, w.grid_h, True)
        db = DeviceBatch(pb, dev)
        first = run_device_batch(db, w.outputs)
        total_pts = int(first.offsets[-1]) if w.outputs == "paths" else 0
        bufs = BatchBuffers(dev, B, F, total_pts)

        def step(sweep):
            return lambda: run_device_batch(db, w.outputs, buffers=bufs, fetch=False, obstacle_sweep=sweep)
        for s in (False, True):
            for _ in range(2):
                step(s)()
        steps = {"off": [], "on": []}
        for _ in range(args.rounds):
            steps["off"].append(events_ms(st, step(False), args.steps))
            steps["on"].append(events_ms(st, step(True), args.steps))
        launches = {}
        for s, k in ((False, "off"), (True, "on")):
            l0 = h.launches
            step(s)()
            launches[k] = h.launches - l0
        torch.cuda.synchronize(dev)

        def sweep_fn():   # the records of the last step stay valid: same batch, same stream
            h.check(h.lib.fcpp_obstacle_sweep(h.h, C.byref(db.c), bufs.d_sweep.data_ptr(), sptr))
        for _ in range(5):
            sweep_fn()
        kern = [1e3 * events_ms(st, sweep_fn, 200) for _ in range(args.rounds)]

        def e2e_rate(sweep):
            def call(wait):
                return fc.plan_batch(w.fields, veh, w.axes, obstacles=w.obstacles, outputs=w.outputs, grid_h=w.grid_h,
                                     device=dev, winners=True, wait=wait, obstacle_sweep=sweep)
            pend = call(False)
            for _ in range(3):
                nxt = call(False)
                pend.result()
                pend = nxt
            pend.result()
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            pend = call(False)
            for _ in range(args.steps - 1):
                nxt = call(False)
                pend.result()
                pend = nxt
            pend.result()
            torch.cuda.synchronize(dev)
            return B * args.steps / (time.perf_counter() - t0)
        e2e = {"off": [], "on": []}
        for _ in range(args.rounds):
            e2e["off"].append(e2e_rate(False))
            e2e["on"].append(e2e_rate(True))
        med = {k: statistics.median(v) for k, v in steps.items()}
        sw_us = statistics.median(kern)
        line = {"workload": name, "text": w.text, "n_cand": B, "n_fields": F, "step_ms": med, "step_ms_all": steps,
                "sweep_us": sw_us, "sweep_us_all": kern, "sweep_share_of_step": sw_us / 1e3 / med["off"],
                "e2e_plans_s": {k: statistics.median(v) for k, v in e2e.items()}, "launches": launches,
                "gpu": gpu, "power_limit_w": plim}
        print(json.dumps(line), flush=True)
        lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
