"""Collecting batches submitted with plan_batch(..., wait=False): every read-back lands in host memory of its own,
and single-GPU and sharded batches are collected through the same pending batch."""
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RECT = [(0, 0), (500, 0), (500, 200), (0, 200)]
SMALL = [(0, 0), (100, 0), (100, 80), (0, 80)]
TINY = [(0, 0), (12, 0), (12, 9), (0, 9)]                 # no valid candidate
OBST2 = [[(200, 80), (250, 80), (250, 120), (200, 120)], [(350, 140), (380, 140), (380, 170), (350, 170)]]


@pytest.fixture(scope="module")
def fc():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import field_coverage_path_planning_b200 as pkg
    return pkg


def _assert_same(got, want):
    """Summaries, argmin and the winners' paths byte for byte."""
    assert got.summary.tobytes() == want.summary.tobytes()
    assert np.array_equal(got.best_cand, want.best_cand) and np.array_equal(got.best_cost, want.best_cost)
    assert got.winner_paths.keys() == want.winner_paths.keys()
    for f, (path, speeds, n_main) in got.winner_paths.items():
        w_path, w_speeds, w_n_main = want.winner_paths[f]
        assert path.tobytes() == w_path.tobytes() and speeds.tobytes() == w_speeds.tobytes() and n_main == w_n_main


def test_results_past_the_pool_cap_keep_their_own_buffers(fc, monkeypatch):
    """Past _ResultPool.MAX_BYTES every read-back still gets pinned memory of its own: two batches in flight with
    their winners' paths (slices of materialised paths, and a re-planned winners' batch), collected in reverse order
    and in order, each equal their own synchronous result.  The two batches differ in shape and the remembered
    sizes are cleared, so both are launched from their own layout pass: a result is never repeated, which would
    hide a read-back that another one overwrote."""
    from field_coverage_path_planning_b200 import batch as B
    veh = fc.VehicleParams()
    cands = [fc.candidate_axes(1, radii=np.linspace(5.0, 9.0, 33), start_corners=[0, 1]),
             fc.candidate_axes(1, radii=np.linspace(6.0, 12.0, 31), start_corners=[2, 3])]
    for outputs in ("paths", "summary"):
        want = [fc.plan_batch([RECT], veh, c, obstacles=[OBST2], outputs=outputs, winners=True) for c in cands]
        assert want[0].summary.tobytes() != want[1].summary.tobytes()
        with monkeypatch.context() as m:
            m.setattr(B._ResultPool, "MAX_BYTES", 0)
            m.setattr(B._ResultPool, "_bufs", [])
            for order in ((1, 0), (0, 1)):
                B._Hints._c.clear()
                pend = [fc.plan_batch([RECT], veh, c, obstacles=[OBST2], outputs=outputs, winners=True, wait=False)
                        for c in cands]
                for k in order:
                    got = pend[k].result()
                    _assert_same(got, want[k])
                    assert not got.extras["speculative"]
            assert B._ResultPool._bufs == []          # past the cap nothing is kept by the pool


def test_sharded_batches_in_flight_world1_nccl(fc):
    """plan_batch(distributed=True, winners=True, wait=False) through a world-size-1 NCCL group: four batches in
    flight, collected out of order, one of them repeated because the remembered launch sizes do not fit it; each
    equals the single-process call."""
    import torch
    import torch.distributed as dist
    from field_coverage_path_planning_b200 import _lib, batch as B
    created = not dist.is_initialized()
    if created:
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1,
                                device_id=torch.device("cuda", 0))
    try:
        veh = fc.VehicleParams()
        rec = _lib.SUMMARY_DTYPE.itemsize
        small_ax = fc.candidate_axes(1, radii=np.linspace(5.0, 6.0, 16), start_corners=[0, 1, 2, 3])
        long_ax = fc.candidate_axes(1, radii=np.linspace(11.0, 12.0, 16), start_corners=[0, 1, 2, 3])  # same shape
        heads_ax = fc.candidate_axes(3, headings=np.deg2rad(np.arange(0.0, 180.0, 5.0)))
        jobs = [([RECT], small_ax, "paths"), ([RECT], long_ax, "paths"), ([RECT, SMALL, TINY], heads_ax, "summary"),
                ([RECT], small_ax, "summary")]
        want = [fc.plan_batch(f, veh, c, outputs=o, device="cuda:0", winners=True) for f, c, o in jobs]
        B._Hints._c.clear()
        for rounds in range(2):
            pend = [fc.plan_batch(f, veh, c, outputs=o, device="cuda:0", distributed=True, winners=True, wait=False)
                    for f, c, o in jobs]
            for k in (1, 0, 3, 2):
                got = pend[k].result()
                assert got is pend[k].result()
                w, F, n = want[k], len(jobs[k][0]), len(want[k].summary)
                _assert_same(got, w)
                assert got.extras["shard"] == (0, n)
                for f in range(F):
                    if w.best_cand[f] >= 0:
                        assert got.extras["winner_summary"][f].tobytes() == w.summary[w.best_cand[f]].tobytes()
                # the sharded read-back carries the winners' records and the flag-count word on top of the
                # single-process one: summaries + 16 F + F records + 16 (+ offsets), plus the winners' paths
                assert got.extras["d2h_bytes"] == w.extras["d2h_bytes"] + F * rec + 16
                if rounds == 0:
                    # sized from its own layout pass; job 1 was sized from job 0's and repeated
                    assert not got.extras["speculative"]
                elif k != 0:
                    # sized from its own earlier run (job 0 runs with job 1's sizes, which may not fit it)
                    assert got.extras["speculative"]
    finally:
        if created:
            dist.destroy_process_group()
