"""Where the end-to-end time of plan_batch(host numpy, winners=True) goes, per bench workload and per
candidate form (explicit per-candidate arrays vs factored axes): host set-up, packed H2D, kernels,
read-back, winners' paths.   python tools/e2e_profile.py [c2|c3|c5 ...]"""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import field_coverage_path_planning_b200 as fc  # noqa: E402
from benchmarks import workloads as wl  # noqa: E402
from field_coverage_path_planning_b200 import batch as B  # noqa: E402

dev = torch.device("cuda", 0)
veh = fc.VehicleParams()


def T(f, n):
    keep = [f() for _ in range(3)]      # warm-up incl. the pinned result pool (a kept result pins its buffer)
    del keep
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        r = f()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n * 1e3, r


for name in (sys.argv[1:] or ["c2", "c3", "c5"]):
    w = wl.WORKLOADS[name](1)
    n = 5 if name == "c3" else 30
    for form, cands in (("explicit", w.cands), ("axes", w.axes)):
        t_all, res = T(lambda: fc.plan_batch(w.fields, veh, cands, obstacles=w.obstacles, outputs=w.outputs,
                                             grid_h=w.grid_h, device=dev, winners=True), n)
        t_prep, pb = T(lambda: B.prepare_batch(w.fields, veh, cands, w.obstacles, None, w.grid_h, True), n)
        t_h2d, db = T(lambda: B.DeviceBatch(pb, dev), n)
        t_launch, lb = T(lambda: B._launch_device_batch(db, w.outputs, False, B.Selection(), 0, None), n)
        bufs, offs = lb
        t_fetch, r = T(lambda: B._finish_fetch(B._enqueue_fetch(db, bufs, w.outputs, offs, True, 0), False), n)
        t_win, _ = T(lambda: B.fetch_winner_paths(db, r, w.outputs), n)
        t_nosum, _ = T(lambda: B.run_device_batch(db, w.outputs, copy_summary=False), n)
        print(f"{name} {form:8s} plan_batch(winners) {t_all:8.3f} ms = prepare {t_prep:.3f} + DeviceBatch/H2D {t_h2d:.3f} "
              f"+ launch+kernels {t_launch:.3f} + fetch {t_fetch:.3f} + winners {t_win:.3f}   "
              f"[h2d {pb.h2d_bytes()} B; run without summary copy {t_nosum:.3f} ms]  "
              f"-> {w.n_cand / t_all / 1e3:.3f} M plans/s", flush=True)

if os.environ.get("FCPP_CPROFILE"):
    import cProfile
    import pstats
    w = wl.WORKLOADS[os.environ["FCPP_CPROFILE"]](1)
    call = lambda: fc.plan_batch(w.fields, veh, w.axes, obstacles=w.obstacles, outputs=w.outputs, grid_h=w.grid_h,  # noqa: E731
                                 device=dev, winners=True)
    for _ in range(5):
        r = call()
    pr = cProfile.Profile()
    pr.enable()
    for _ in range(200):
        r = call()
    pr.disable()
    pstats.Stats(pr).sort_stats("cumulative").print_stats(45)
