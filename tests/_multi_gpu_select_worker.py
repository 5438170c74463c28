"""torchrun worker of tests/test_gpu_select.py::test_select_on_two_or_more_gpus (needs >= 2 GPUs).

plan_batch(distributed=True, select=...) over the whole job == the single-GPU plan_batch of the same global candidate
set: the merged ranking (candidates and cost bits) and the summary record of every ranked candidate byte for byte,
for a config-2 shape (explicit arrays, paths) and a config-3 shape (factored heading search, summary only).
Prints "MULTI GPU SELECT OK" on rank 0 and exits 0, or exits 1.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import field_coverage_path_planning_b200 as fc  # noqa: E402
from benchmarks import workloads as wl  # noqa: E402


def main():
    import faulthandler
    # a hang (a collective some rank never reaches) must not hold the GPUs: stacks of all threads, then exit
    faulthandler.dump_traceback_later(int(os.environ.get("FCPP_WORKER_WATCHDOG_S", "150")), exit=True)
    rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(lr)
    dev = torch.device("cuda", lr)
    dist.init_process_group("nccl", device_id=dev)
    ok = True
    veh = fc.VehicleParams()
    w2 = wl.c2(world, radii_per_gpu=128)
    w3 = wl.c3(world, fields_per_gpu=32)
    cases = [(w2.fields, w2.cands, w2.obstacles, "paths",
              fc.Selection(top_k=8, w_time=1.0, w_obstacle=50.0, max_boundary_viol=40, min_coverage=0.99)),
             (w2.fields, w2.axes, w2.obstacles, "summary", fc.Selection(top_k=32, w_uncovered=1.0)),
             (w3.fields, w3.axes, None, "summary", fc.Selection(top_k=5, w_boundary=2.0, max_boundary_viol=10)),
             (w3.fields, w3.cands, None, "summary", fc.Selection(top_k=1, max_boundary_viol=0))]
    for it, (fields, cands, obst, outputs, sel) in enumerate(cases):
        single = fc.plan_batch(fields, veh, cands, obstacles=obst, outputs=outputs, device=dev, select=sel)
        shard = fc.plan_batch(fields, veh, cands, obstacles=obst, outputs=outputs, device=dev, distributed=True,
                              select=sel)
        good = (np.array_equal(single.topk_cand, shard.topk_cand) and
                single.topk_cost.tobytes() == shard.topk_cost.tobytes() and
                single.topk_summary.tobytes() == shard.topk_summary.tobytes() and
                np.array_equal(single.best_cand, shard.best_cand))
        lo, hi = shard.extras["shard"]
        good = good and shard.summary.tobytes() == single.summary[lo:hi].tobytes()
        good = good and (single.topk_cand >= 0).any()
        if not good:
            ok = False
            print("SHARDED SELECT MISMATCH rank", rank, "case", it, flush=True)
    flag = torch.tensor([0 if ok else 1], device=dev)
    dist.all_reduce(flag)
    dist.destroy_process_group()
    if int(flag.item()) == 0:
        if rank == 0:
            print("MULTI GPU SELECT OK", flush=True)
        sys.exit(0)
    sys.exit(1)


if __name__ == "__main__":
    main()
