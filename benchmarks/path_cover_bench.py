#!/usr/bin/env python
"""What the whole-field / headland-band path coverage costs (DESIGN.md §3.10), one GPU, steady state.

    python benchmarks/path_cover_bench.py [--workloads c2,paths,c5plan] [--steps 20] [--rounds 3] [--out FILE]

Workloads:
  c2      benchmarks/workloads.py c2: 4 096 candidates on the 500 x 200 m field with two obstacles, paths materialised
  paths   caller paths: 320 ragged paths (the first c2 plans) and one path of 30 000 points, on c2's field, h = 0.1 m
  c5plan  one config-5 plan (2 000 x 1 000 m field, h = 0.05 m, R = 8 m), paths materialised: ~3 300 row slabs
Per workload, one JSON line:
  step_ms          (c2) device time of one step (layout .. coverage + ranking, inputs and buffers resident) with
                   field_coverage off and on, CUDA events over --steps steps; the two arms alternate --rounds times
  cover_us         the three path coverage kernels alone over the step's plans (or the paths), CUDA events
  launches         kernels per step, off / on (or per call)
  gpu, power_limit_w   read in the same run
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from benchmarks import workloads as wl  # noqa: E402
from benchmarks.sweep_bench import events_ms, power_limit_w  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2,paths,c5plan")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("path_cover_bench.py needs a CUDA device")
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
        line = {"workload": name, "gpu": gpu, "power_limit_w": plim}
        if name == "paths":
            w = wl.c2(1)
            res = fc.plan_batch(w.fields, veh, w.cands, obstacles=w.obstacles, outputs="paths")
            ragged = [res.path(b)[0] for b in range(320)]
            long_p, k = [], 0
            while sum(len(p) for p in long_p) < 30000:
                long_p.append(res.path(k)[0])
                k += 1
            one = np.concatenate(long_p)[:30000]
            for tag, paths in (("ragged320", ragged), ("one30000", [one])):
                n = len(paths)
                offs = np.concatenate([[0], np.cumsum([len(p) for p in paths])]).astype(np.int64)
                polys = [np.asarray(o, dtype=np.float64) for o in wl.OBST2]
                t = _pack_to_dev({"path": np.concatenate(paths), "offsets": offs,
                                  "field": np.zeros(n, dtype=np.int32), "hw": np.full(n, 8.0),
                                  "ps": np.array([0, 2], dtype=np.int32), "vs": np.array([0, 4, 8], dtype=np.int32),
                                  "verts": np.concatenate(polys), "fv": np.asarray(w.fields, dtype=np.float64)}, dev)
                d_out = torch.empty(n * _lib.PATH_COVER_DTYPE.itemsize, dtype=torch.uint8, device=dev)

                def cover_fn():
                    h.check(h.lib.fcpp_path_coverage(h.h, t["path"].data_ptr(), t["offsets"].data_ptr(), n, None,
                                                     t["field"].data_ptr(), t["hw"].data_ptr(), 1, t["fv"].data_ptr(),
                                                     t["ps"].data_ptr(), t["vs"].data_ptr(), t["verts"].data_ptr(),
                                                     veh.working_width / 2, 0.1, d_out.data_ptr(), sptr))
                for _ in range(3):
                    cover_fn()
                us = [1e3 * events_ms(st, cover_fn, 20) for _ in range(args.rounds)]
                line[tag] = {"points": int(offs[-1]), "cover_us": statistics.median(us), "cover_us_all": us,
                             "launches": 3}
        elif name == "c5plan":
            big = wl.BIG
            cand = {"field_id": np.zeros(1, dtype=np.int32), "R": np.array([8.0]), "start_corner": np.zeros(1, np.int32)}
            pb = prepare_batch([big], veh, cand, None, None, 0.05, True)
            db = DeviceBatch(pb, dev)
            first = run_device_batch(db, "paths", field_coverage=True)
            bufs = BatchBuffers(dev, 1, 1, int(first.offsets[-1]))
            run_device_batch(db, "paths", buffers=bufs, fetch=False, field_coverage=True)
            out = _lib.Outputs()
            out.summary, out.offsets = bufs.d_sum.data_ptr(), bufs.d_off.data_ptr()
            out.path_xy, out.speeds_kmh = bufs.d_path.data_ptr(), bufs.d_spd.data_ptr()

            def cover_fn():
                h.check(h.lib.fcpp_plan_coverage(h.h, C.byref(db.c), C.byref(out), bufs.d_fcov.data_ptr(), sptr))
            for _ in range(3):
                cover_fn()
            us = [1e3 * events_ms(st, cover_fn, 10) for _ in range(args.rounds)]
            rec = first.field_cover[0]
            line.update({"points": int(first.offsets[-1]), "field_total": int(rec["field_total"]),
                         "field_cells": int(rec["field_cells"]), "band_total": int(rec["band_total"]),
                         "cover_us": statistics.median(us), "cover_us_all": us, "launches": 3})
        else:
            w = wl.WORKLOADS[name](1)
            F, B = len(w.fields), len(w.cands["field_id"])
            pb = prepare_batch(w.fields, veh, w.cands, w.obstacles, None, w.grid_h, True)
            db = DeviceBatch(pb, dev)
            first = run_device_batch(db, "paths")
            bufs = BatchBuffers(dev, B, F, int(first.offsets[-1]))

            def step(on):
                return lambda: run_device_batch(db, "paths", buffers=bufs, fetch=False, field_coverage=on)
            for on in (False, True):
                for _ in range(2):
                    step(on)()
            steps = {"off": [], "on": []}
            for _ in range(args.rounds):
                steps["off"].append(events_ms(st, step(False), args.steps))
                steps["on"].append(events_ms(st, step(True), args.steps))
            launches = {}
            for on, k in ((False, "off"), (True, "on")):
                l0 = h.launches
                step(on)()
                launches[k] = h.launches - l0
            out = _lib.Outputs()
            out.summary, out.offsets = bufs.d_sum.data_ptr(), bufs.d_off.data_ptr()
            out.path_xy, out.speeds_kmh = bufs.d_path.data_ptr(), bufs.d_spd.data_ptr()

            def cover_fn():   # the plans of the last step stay valid: same batch, same stream
                h.check(h.lib.fcpp_plan_coverage(h.h, C.byref(db.c), C.byref(out), bufs.d_fcov.data_ptr(), sptr))
            for _ in range(3):
                cover_fn()
            kern = [1e3 * events_ms(st, cover_fn, args.steps) for _ in range(args.rounds)]
            med = {k: statistics.median(v) for k, v in steps.items()}
            line.update({"n_cand": B, "step_ms": med, "step_ms_all": steps, "cover_us": statistics.median(kern),
                         "cover_us_all": kern, "cover_share_of_step": statistics.median(kern) / 1e3 / med["off"],
                         "launches": launches})
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
