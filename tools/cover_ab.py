"""A/B of coverage launch modes (fcpp_set_cover_mode: 0 default, 64 one coverage CTA per listed task, 128 the persistent
work list over the listed representatives, ...) per workload and output mode.
python tools/cover_ab.py [mode ...]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import field_coverage_path_planning_b200 as fc  # noqa: E402
from benchmarks import workloads as wl  # noqa: E402
from field_coverage_path_planning_b200 import _lib  # noqa: E402
from field_coverage_path_planning_b200.batch import BatchBuffers, DeviceBatch, prepare_batch, run_device_batch  # noqa: E402

dev = torch.device("cuda", 0)
h = _lib.handle(0)
h.check(h.lib.fcpp_set_profiling(h.h, 1))
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
for name, w in (("c2", wl.c2(1)), ("c5", wl.c5(1)), ("c3/512 fields", wl.c3(1, 512))):
    for outputs in (("paths", "summary") if name == "c2" else ("summary",)):
        db = DeviceBatch(prepare_batch(w.fields, fc.VehicleParams(), w.axes, w.obstacles, None, w.grid_h, True), dev)
        first = run_device_batch(db, outputs)
        bufs = BatchBuffers(dev, db.pb.n_cand, db.pb.n_fields, int(first.offsets[-1]) if outputs == "paths" else 0)
        for mode in ([int(x) for x in sys.argv[1:]] or [0, 64, 128, 0, 64, 128]):
            h.check(h.lib.fcpp_set_cover_mode(h.h, mode))
            for _ in range(3):
                run_device_batch(db, outputs, buffers=bufs, fetch=False)
            torch.cuda.synchronize()
            tot = 0.0
            n = 10 if name.startswith("c3") else 40
            for _ in range(n):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                run_device_batch(db, outputs, buffers=bufs, fetch=False)
                b.record()
                b.synchronize()
                tot += a.elapsed_time(b)
            import ctypes as C
            ms3 = (C.c_float * 3)()
            h.check(h.lib.fcpp_kernel_times(h.h, C.byref(ms3)))
            print(f"{name:14s} {outputs:8s} mode {mode}  {tot / n:.4f} ms/step "
                  f"(last step: layout {ms3[0]:.3f} plan {ms3[1]:.3f} cover {ms3[2]:.3f})", flush=True)
        h.check(h.lib.fcpp_set_cover_mode(h.h, 0))
