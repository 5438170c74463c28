"""Load balance of the coverage grid, from a trace build of the library (-DFCPP_COVER_TRACE): every coverage task
(candidate, part; part A10 = corner windows, A11 = headland band) records its start and end on %globaltimer and its SM.

    python benchmarks/cover_balance.py [--workload c2 c5 c3] [--steps 5] [--lib PATH] [--mode M]

Per workload (one GPU, the per-GPU share of bench.py's workloads) it prints one JSON line with the medians over the
traced steps of
    kernel_ms        the coverage kernel's span: first task start to last task end
    utilisation      busy time of all tasks / (CTA slots x span), CTA slots = 2 per SM
    tail_ms          from the first slot that goes idle with no task left to start (the earliest task end after
                     the last task start) to the end of the kernel
    by_R             per part, task durations (mean / max, us) in eight bins of R (c3: one bin, all R are equal)
and the event time of the whole coverage stage (de-duplication kernels included) for reference.
--lib takes an already built trace library; without it the script builds one (make VARIANT=trace) under
field_coverage_path_planning_b200/variants/.  --mode sets fcpp_set_cover_mode for the run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", nargs="+", default=["c2", "c5", "c3"])
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--lib", default=None)
    ap.add_argument("--mode", type=int, default=0)
    args = ap.parse_args()
    lib = args.lib
    if lib is None:
        csrc = os.path.join(ROOT, "field_coverage_path_planning_b200", "csrc")
        subprocess.check_call(["make", "-s", "-C", csrc, "-j8", "VARIANT=trace", "DEFS=-DFCPP_COVER_TRACE"],
                              stdout=subprocess.DEVNULL)
        lib = os.path.join(ROOT, "field_coverage_path_planning_b200", "variants", "libfcpp_trace.so")
    os.environ["FCPP_LIB"] = os.path.abspath(lib)

    import numpy as np
    import torch
    import field_coverage_path_planning_b200 as fc
    from benchmarks import workloads as wl
    from field_coverage_path_planning_b200 import _lib
    from field_coverage_path_planning_b200.batch import BatchBuffers, DeviceBatch, prepare_batch, run_device_batch

    assert torch.cuda.is_available(), "cover_balance.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    h = _lib.handle(0)
    take = h.lib.fcpp_cover_trace_take
    take.restype = C.c_int
    take.argtypes = [C.c_void_p, C.c_int]
    cap = 1 << 18
    buf = np.zeros((cap, 4), dtype=np.uint64)
    slots = 2 * torch.cuda.get_device_properties(dev).multi_processor_count
    h.check(h.lib.fcpp_set_profiling(h.h, 1))
    h.check(h.lib.fcpp_set_cover_mode(h.h, args.mode))
    for name in args.workload:
        w = wl.WORKLOADS[name](1)
        db = DeviceBatch(prepare_batch(w.fields, fc.VehicleParams(), w.axes, w.obstacles, None, w.grid_h, True), dev)
        first = run_device_batch(db, w.outputs)
        bufs = BatchBuffers(dev, db.pb.n_cand, db.pb.n_fields, int(first.offsets[-1]) if w.outputs == "paths" else 0)
        for _ in range(3):
            run_device_batch(db, w.outputs, buffers=bufs, fetch=False)
        torch.cuda.synchronize()
        take(buf.ctypes.data, cap)
        R = np.asarray(w.cands["R"]) if "R" in w.cands else None
        rows = []
        for _ in range(args.steps):
            run_device_batch(db, w.outputs, buffers=bufs, fetch=False)
            torch.cuda.synchronize()
            ms3 = (C.c_float * 3)()
            h.check(h.lib.fcpp_kernel_times(h.h, C.byref(ms3)))
            n = take(buf.ctypes.data, cap)
            assert 0 < n <= cap, n
            t = buf[:n].astype(np.int64)
            t0, t1 = t[:, 0] - t[:, 0].min(), t[:, 1] - t[:, 0].min()
            span = int(t1.max())
            busy = int((t1 - t0).sum())
            tail_from = int(t1[t1 >= t0.max()].min())
            part = t[:, 3] & 3
            cand = t[:, 3] >> 2
            by_r = {}
            if R is not None:
                rc = R[cand]
                edges = np.linspace(R.min(), R.max(), 9)
                binr = np.clip(np.searchsorted(edges, rc, side="right") - 1, 0, 7)
            else:
                binr = np.zeros(n, dtype=np.int64)
                edges = None
            for p, pname in ((1, "A10"), (2, "A11")):
                out = []
                for k in range(8 if R is not None else 1):
                    m = (part == p) & (binr == k)
                    if not m.any():
                        continue
                    d = (t1[m] - t0[m]) / 1e3
                    out.append({"R": f"{edges[k]:.2f}-{edges[k + 1]:.2f}" if edges is not None else "all",
                                "tasks": int(m.sum()), "mean_us": round(float(d.mean()), 1),
                                "max_us": round(float(d.max()), 1)})
                by_r[pname] = out
            rows.append({"kernel_ms": span / 1e6, "utilisation": busy / (slots * span), "tail_ms": (span - tail_from) / 1e6,
                         "tasks": int(n), "sms_used": int(len(np.unique(t[:, 2] & 0xffff))), "cover_stage_ms": float(ms3[2]),
                         "by_R": by_r})
        med = lambda k: float(np.median([r[k] for r in rows]))
        mid = sorted(rows, key=lambda r: r["kernel_ms"])[len(rows) // 2]
        print(json.dumps({"workload": name, "mode": args.mode, "lib": os.path.basename(lib), "gpu": torch.cuda.get_device_name(dev),
                          "kernel_ms": round(med("kernel_ms"), 4), "utilisation": round(med("utilisation"), 4),
                          "tail_ms": round(med("tail_ms"), 4), "tail_share": round(med("tail_ms") / med("kernel_ms"), 4),
                          "cover_stage_ms": round(med("cover_stage_ms"), 4), "tasks": mid["tasks"],
                          "sms_used": mid["sms_used"], "by_R": mid["by_R"]}), flush=True)


if __name__ == "__main__":
    main()
