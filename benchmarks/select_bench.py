#!/usr/bin/env python
"""What the per-field top-k selection costs: plan_batch(select=Selection(top_k=8, ...)) against cost='length' on
the c2, c3 and c5 workloads of benchmarks/workloads.py, one GPU, steady state.

    python benchmarks/select_bench.py [--workloads c2,c3,c5] [--steps 20] [--rounds 3] [--out FILE]

Per workload, one JSON line:
  step_ms          device time of one step (layout .. coverage + argmin or selection, inputs and buffers resident),
                   CUDA events over --steps steps; the two arms alternate --rounds times, the median is reported
  e2e_plans_s      plans/s through plan_batch(..., winners=True) with two calls in flight (wait=False), alternating
  kernel_us        fcpp_field_select alone over the step's resident summaries, CUDA events over 200 calls each:
                   "argmin" = Selection() (a plain selection: the argmin kernels), "select_k1" = its twin with a
                   limit no candidate reaches (the ranking pipeline at k = 1), "select_k8" = the selection above
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2,c3,c5")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("select_bench.py needs a CUDA device")
    import field_coverage_path_planning_b200 as fc
    from field_coverage_path_planning_b200 import _lib
    from field_coverage_path_planning_b200.batch import BatchBuffers, DeviceBatch, prepare_batch, run_device_batch
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    gpu, plim = torch.cuda.get_device_name(dev), power_limit_w()
    veh = fc.VehicleParams()
    h = _lib.handle(0)
    lines = []
    for name in args.workloads.split(","):
        w = wl.WORKLOADS[name](1)
        F = len(w.fields)
        pb = prepare_batch(w.fields, veh, w.cands, w.obstacles, None, w.grid_h, True)
        db = DeviceBatch(pb, dev)
        first = run_device_batch(db, w.outputs)
        ok = first.summary["status"] == 0
        share = first.summary["cov_cells"][ok] / np.maximum(first.summary["cov_total"][ok], 1)
        sel = fc.Selection(top_k=8, w_time=1.0, max_boundary_viol=int(np.median(first.summary["n_boundary_viol"][ok])),
                           min_coverage=float(np.quantile(share, 0.3)))
        total_pts = int(first.offsets[-1]) if w.outputs == "paths" else 0
        bufs = BatchBuffers(dev, len(w.cands["field_id"]), F, total_pts)
        st = torch.cuda.current_stream(dev)

        def device_ms(select):
            for _ in range(2):
                run_device_batch(db, w.outputs, buffers=bufs, fetch=False, select=select)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st)
            for _ in range(args.steps):
                run_device_batch(db, w.outputs, buffers=bufs, fetch=False, select=select)
            b.record(st)
            b.synchronize()
            return a.elapsed_time(b) / args.steps

        def e2e_rate(select):
            def call(wait):
                return fc.plan_batch(w.fields, veh, w.axes, obstacles=w.obstacles, outputs=w.outputs,
                                     grid_h=w.grid_h, device=dev, winners=True, wait=wait, select=select)
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
            return len(w.cands["field_id"]) * args.steps / (time.perf_counter() - t0)

        steps = {"length": [], "select": []}
        e2e = {"length": [], "select": []}
        for _ in range(args.rounds):
            steps["length"].append(device_ms(None))
            steps["select"].append(device_ms(sel))
            e2e["length"].append(e2e_rate(None))
            e2e["select"].append(e2e_rate(sel))

        # the ranking kernels alone, over the resident summaries of the last step
        run_device_batch(db, w.outputs, buffers=bufs, fetch=False)
        torch.cuda.synchronize(dev)
        B = len(w.cands["field_id"])
        cf = db.t["cand_field"].data_ptr()
        sptr = C.c_void_p(st.cuda_stream)
        d_tk = torch.empty(2 * F * 32, dtype=torch.int64, device=dev)

        def kernel_us(fn, reps=200):
            for _ in range(5):
                fn()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st)
            for _ in range(reps):
                fn()
            b.record(st)
            b.synchronize()
            return 1e3 * a.elapsed_time(b) / reps

        def select_fn(s):
            sc = s.c_struct(w.grid_h)
            return lambda: h.check(h.lib.fcpp_field_select(h.h, bufs.d_sum.data_ptr(), cf, B, F, C.byref(sc), 0,
                                                           d_tk.data_ptr(), d_tk.data_ptr() + 8 * F * s.top_k, sptr))

        argmin_fn = select_fn(fc.Selection())
        kern = {"argmin": kernel_us(argmin_fn),
                "select_k1": kernel_us(select_fn(fc.Selection(max_accel_viol=2**31 - 1))),
                "select_k8": kernel_us(select_fn(sel))}
        l0 = h.launches
        select_fn(sel)()
        launches_select = h.launches - l0
        l0 = h.launches
        argmin_fn()
        launches_argmin = h.launches - l0
        med = {k: statistics.median(v) for k, v in steps.items()}
        line = {"workload": name, "n_cand": B, "n_fields": F, "selection": sel.__dict__,
                "step_ms": med, "step_ms_all": steps, "select_share_of_step": kern["select_k8"] / 1e3 / med["length"],
                "e2e_plans_s": {k: statistics.median(v) for k, v in e2e.items()},
                "kernel_us": kern, "launches": {"argmin": launches_argmin, "select": launches_select},
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
