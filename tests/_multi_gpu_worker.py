"""torchrun worker of tests/test_gpu_multi.py (needs >= 2 GPUs): results of the multi-GPU path on hardware.

1. reduce_best (NCCL all-gather + fcpp_field_select_merge at k = 1) against the numpy rule, 40 back-to-back calls
   with many ties, F = 1, 7, 4096;
2. plan_batch(distributed=True) over the whole job == the single-process plan_batch of the same global
   candidate set (merged per-field argmin, costs, the winner's summary record), for config 2 at 512
   candidates per rank and a 3-field batch with a field that has no valid candidate.
Prints "MULTI GPU CHECK OK" on rank 0 and exits 0, or exits 1.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import field_coverage_path_planning_b200 as fc  # noqa: E402
from benchmarks import workloads as wl  # noqa: E402
from field_coverage_path_planning_b200 import dist as fdist  # noqa: E402


def main():
    import faulthandler
    # a hang (a collective some rank never reaches) must not hold the GPUs: stacks of all threads, then exit
    faulthandler.dump_traceback_later(int(os.environ.get("FCPP_WORKER_WATCHDOG_S", "150")), exit=True)
    rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(lr)
    dev = torch.device("cuda", lr)
    dist.init_process_group("nccl", device_id=dev)
    ok = True
    # ---- 1. NCCL all-gather + merge vs numpy rule ----
    for F in (1, 7, 4096):
        for it in range(40):
            # every rank derives ALL ranks' inputs from the same seed: the expected result is local numpy
            rng = np.random.default_rng(1000 * F + it)
            cost_all = rng.integers(0, 5, size=(world, F)).astype(np.float64)
            cand_all = rng.integers(-1, 1000, size=(world, F)).astype(np.int64) * world + np.arange(world)[:, None]
            none = cand_all < 0
            cand_all[none] = -1
            cost_all[none] = np.inf
            want_c, want_k = np.full(F, np.inf), np.full(F, -1, dtype=np.int64)
            for r in range(world):
                better = (cand_all[r] >= 0) & ((want_k < 0) | (cost_all[r] < want_c) |
                                               ((cost_all[r] == want_c) & (cand_all[r] < want_k)))
                want_c = np.where(better, cost_all[r], want_c)
                want_k = np.where(better, cand_all[r], want_k)
            cb = torch.empty(2 * F, dtype=torch.int64, device=dev)
            c, k = cb[:F].view(torch.float64), cb[F:]
            c.copy_(torch.from_numpy(cost_all[rank]))
            k.copy_(torch.from_numpy(cand_all[rank]))
            fdist.reduce_best(c, k)
            if not (np.array_equal(c.cpu().numpy(), want_c) and np.array_equal(k.cpu().numpy(), want_k)):
                ok = False
                print("MISMATCH rank", rank, "F", F, "it", it, flush=True)
    # ---- 2. sharded plan_batch == single-process plan_batch ----
    veh = fc.VehicleParams()
    w = wl.c2(world, radii_per_gpu=128)
    cases = [(w.fields, w.cands, w.obstacles, "paths")]
    rect = [(0, 0), (500, 0), (500, 200), (0, 200)]
    small = [(0, 0), (100, 0), (100, 80), (0, 80)]
    tiny = [(0, 0), (12, 0), (12, 9), (0, 9)]
    cases.append(([rect, small, tiny], fc.make_candidates(3, radii=[5.0, 8.0, 8.0, 11.0], start_corners=[0, 1, 2, 3]),
                  None, "summary"))
    for fields, cands, obst, outputs in cases:
        single = fc.plan_batch(fields, veh, cands, obstacles=obst, outputs=outputs, device=dev)
        shard = fc.plan_batch(fields, veh, cands, obstacles=obst, outputs=outputs, device=dev, distributed=True)
        good = np.array_equal(single.best_cand, shard.best_cand) and np.array_equal(single.best_cost, shard.best_cost)
        win = shard.extras["winner_summary"]
        for f in range(len(single.best_cand)):
            if single.best_cand[f] >= 0:
                good = good and win[f].tobytes() == single.summary[single.best_cand[f]].tobytes()
        lo, hi = shard.extras["shard"]
        good = good and shard.summary.tobytes() == single.summary[lo:hi].tobytes()
        if not good:
            ok = False
            print("SHARDED MISMATCH rank", rank, flush=True)
    # ---- 3. factored candidate sets, remembered launch sizes, two sharded batches in flight, collective repeat ----
    from field_coverage_path_planning_b200 import batch as fbatch
    fbatch._Hints._c.clear()
    small_ax = fc.candidate_axes(1, radii=np.linspace(5.0, 6.0, 16 * world), start_corners=[0, 1, 2, 3])
    # same shape, but ONE rank's shard holds longer headlands: its remembered sizes do not fit -> all ranks repeat
    radii = np.linspace(5.0, 6.0, 16 * world)
    radii[-8:] = np.linspace(11.0, 12.0, 8)
    odd_ax = fc.candidate_axes(1, radii=radii, start_corners=[0, 1, 2, 3])
    heads_ax = fc.candidate_axes(3, headings=np.deg2rad(np.arange(0.0, 180.0, 5.0)))
    jobs = [([rect], small_ax, "paths"), ([rect], odd_ax, "paths"), ([rect, small, tiny], heads_ax, "summary"),
            ([rect], small_ax, "summary")]
    want = [fc.plan_batch(f, veh, fc.expand_axes(c), outputs=o, device=dev) for f, c, o in jobs]
    for rounds in range(2):
        pend = [fc.plan_batch(f, veh, c, outputs=o, device=dev, distributed=True, winners=True, wait=False) for f, c, o in jobs]
        for k in (1, 0, 2, 3):                      # the same order on every rank (a repeat is collective)
            got = pend[k].result()
            lo, hi = got.extras["shard"]
            good = (np.array_equal(got.best_cand, want[k].best_cand) and np.array_equal(got.best_cost, want[k].best_cost)
                    and got.summary.tobytes() == want[k].summary[lo:hi].tobytes())
            for f, (pth, spd, _) in got.winner_paths.items():
                wp, ws, _ = want[k].path(int(want[k].best_cand[f])) if want[k].d_path is not None else (None, None, None)
                if wp is not None:
                    good = good and np.array_equal(pth, wp) and np.array_equal(spd, ws)
            if not good:
                ok = False
                print("PIPELINED SHARDED MISMATCH rank", rank, "job", k, "round", rounds, flush=True)
    t = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("MULTI GPU CHECK", "OK" if t.item() else "FAILED", flush=True)
    faulthandler.cancel_dump_traceback_later()
    dist.destroy_process_group()
    return 0 if t.item() else 1


if __name__ == "__main__":
    sys.exit(main())
