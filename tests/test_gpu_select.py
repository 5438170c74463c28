"""Per-field top-k selection on the device (fcpp_field_select, plan_batch(select=...)) against the numpy statement
in oracle/select.py: same candidates, same cost bits."""
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RECT = [(0, 0), (500, 0), (500, 200), (0, 200)]
OBST2 = [[(200, 80), (250, 80), (250, 120), (200, 120)], [(350, 140), (380, 140), (380, 170), (350, 170)]]


@pytest.fixture(scope="module")
def fc():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import field_coverage_path_planning_b200 as pkg
    return pkg


def _sel(fc, ns):
    return fc.Selection(**vars(ns))


def _device_rank(fc, summ, fid, F, sel, grid_h=0.1, base=0):
    """fcpp_field_select on host arrays -> (cost [F, k], cand [F, k])."""
    import ctypes as C
    import torch
    from field_coverage_path_planning_b200 import _lib
    h = _lib.handle(0)
    B, k = len(summ), sel.top_k
    d_s = torch.from_numpy(np.ascontiguousarray(summ).view(np.uint8).reshape(-1).copy()).cuda()
    d_f = torch.from_numpy(np.ascontiguousarray(fid, dtype=np.int32)).cuda()
    d_tk = torch.empty(2 * max(F, 1) * k, dtype=torch.int64, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    sc = sel.c_struct(grid_h)
    h.check(h.lib.fcpp_field_select(h.h, d_s.data_ptr() if B else None, d_f.data_ptr() if B else None, B, F,
                                    C.byref(sc), base, d_tk.data_ptr(), d_tk.data_ptr() + 8 * max(F, 1) * k, st))
    out = d_tk.cpu().numpy()
    n = max(F, 1) * k
    return out[:n].view(np.float64)[:F * k].reshape(F, k), out[n:][:F * k].reshape(F, k), sc.cell_area


def _check(fc, summ, fid, F, ns, base=0):
    from oracle import select as osel
    sel = _sel(fc, ns)
    cost, cand, cell_area = _device_rank(fc, summ, fid, F, sel, base=base)
    want_c, want_i = osel.rank(summ, fid, F, ns, cell_area, base=base)
    assert np.array_equal(cand, want_i), (ns, np.argwhere(cand != want_i)[:5])
    assert cost.tobytes() == want_c.tobytes(), ns


@pytest.mark.parametrize("seed,B,F,shuffle", [(0, 0, 0, True), (1, 0, 9, True), (2, 1, 1, True), (3, 700, 1, True),
                                              (4, 5000, 37, False), (4, 5000, 37, True), (5, 3000, 2000, True),
                                              (6, 40000, 3, True)])
def test_select_kernel_matches_oracle(fc, seed, B, F, shuffle):
    """Ties, limits at n == max and max + 1, coverage at the threshold, all-ineligible fields, fewer than k, any
    field order, k in {1, 2, 7, 32}."""
    from oracle import select as osel
    summ, fid = osel.adversarial_summaries(seed, B, F, shuffle=shuffle)
    for ns in osel.adversarial_selections():
        _check(fc, summ, fid, F, ns, base=1000 * seed)


def test_select_kernel_skewed_fields(fc):
    """One field of half the candidates, the rest spread over many tiny fields, shuffled: fields run across the
    tiles of the tree reduction and share tiles with many complete ones."""
    from oracle import select as osel
    rng = np.random.default_rng(7)
    summ, _ = osel.adversarial_summaries(7, 200000, 1)
    F = 5000
    fid = np.where(rng.random(len(summ)) < 0.5, 4321, rng.integers(0, F, size=len(summ))).astype(np.int32)
    fid[rng.random(len(summ)) < 0.2] = 17
    for ns in osel.adversarial_selections()[2:5]:
        _check(fc, summ, fid, F, ns)


def test_select_kernel_one_field_of_a_million(fc):
    from oracle import select as osel
    summ, fid = osel.adversarial_summaries(8, 1 << 20, 1)
    for ns in (osel.adversarial_selections()[0], osel.adversarial_selections()[3], osel.adversarial_selections()[-1]):
        _check(fc, summ, fid, 1, ns)


def test_select_kernel_c3_shape(fc):
    """4096 fields x 180 candidates (config 3's shape), shuffled and field-major, deterministic on repeat."""
    from oracle import select as osel
    for shuffle in (False, True):
        summ, fid = osel.adversarial_summaries(9, 4096 * 180, 4096, shuffle=shuffle)
        for ns in osel.adversarial_selections()[1:4]:
            _check(fc, summ, fid, 4096, ns)
    sel = _sel(fc, osel.adversarial_selections()[4])
    a = _device_rank(fc, summ, fid, 4096, sel)
    b = _device_rank(fc, summ, fid, 4096, sel)
    assert a[0].tobytes() == b[0].tobytes() and np.array_equal(a[1], b[1])


def _same_as_argmin(fc, fields, cands, obstacles, outputs, grid_h=0.1):
    """cost= and the plain selection (the argmin kernels), and the plain selection's twin with a limit no candidate
    reaches (the ranking pipeline at k = 1): the same bytes."""
    veh = fc.VehicleParams()
    for cost, plain in (("length", fc.Selection()), ("time", fc.Selection(w_length=0.0, w_time=1.0))):
        want = fc.plan_batch(fields, veh, cands, obstacles=obstacles, outputs=outputs, grid_h=grid_h, cost=cost)
        assert want.topk_cand is None and want.topk_cost is None and want.topk_summary is None
        for sel in (plain, fc.Selection(**{**plain.__dict__, "max_accel_viol": 2**31 - 1})):
            got = fc.plan_batch(fields, veh, cands, obstacles=obstacles, outputs=outputs, grid_h=grid_h, select=sel)
            assert got.summary.tobytes() == want.summary.tobytes()
            assert np.array_equal(got.best_cand, want.best_cand), (cost, sel)
            assert got.best_cost.tobytes() == want.best_cost.tobytes(), (cost, sel)
            assert got.topk_cand.shape == (len(fields), 1)


def test_default_selections_equal_the_argmin(fc):
    """Selection() is cost='length' and the time-only selection cost='time', bit for bit, through the argmin kernels
    and through the ranking pipeline: config 2's shape (explicit arrays and factored) and a heading search over
    parallelograms (factored, coverage de-duplicated per heading)."""
    from benchmarks import workloads as wl
    w = wl.c2(1, radii_per_gpu=256)
    _same_as_argmin(fc, w.fields, w.cands, w.obstacles, "paths")
    _same_as_argmin(fc, w.fields, w.axes, w.obstacles, "summary")
    w3 = wl.c3(1, fields_per_gpu=96)
    from field_coverage_path_planning_b200 import batch as B
    assert B.prepare_batch(w3.fields, fc.VehicleParams(), w3.axes).dedupe == 2
    _same_as_argmin(fc, w3.fields, w3.axes, None, "summary")


def _limits_selection(fc, summary, k):
    """A selection whose limits and coverage threshold cut through the batch's own values."""
    ok = summary["status"] == 0
    share = summary["cov_cells"][ok] / np.maximum(summary["cov_total"][ok], 1)
    return fc.Selection(w_length=1.0, w_time=0.5, w_boundary=3.0, w_obstacle=100.0, w_uncovered=0.25,
                        max_boundary_viol=int(np.median(summary["n_boundary_viol"][ok])),
                        min_coverage=float(np.quantile(share, 0.3)), top_k=k)


def _check_result(fc, res, sel, fields_of, base=0):
    from oracle import select as osel
    F = res.n_fields
    cost, cand = osel.rank(res.summary, fields_of, F, sel, sel.c_struct(0.1).cell_area, base=base)
    assert np.array_equal(res.topk_cand, cand) and res.topk_cost.tobytes() == cost.tobytes()
    assert np.array_equal(res.best_cand, cand[:, 0]) and res.best_cost.tobytes() == cost[:, 0].tobytes()
    own = cand >= 0
    assert res.topk_summary[own].tobytes() == res.summary[cand[own] - base].tobytes()
    assert not res.topk_summary[~own].view(np.uint8).any()


def test_plan_batch_select_end_to_end(fc):
    """Limits and coverage terms on a real batch, summary and paths modes, with the rank-0 winners' paths."""
    from benchmarks import workloads as wl
    veh = fc.VehicleParams()
    w = wl.c2(1, radii_per_gpu=128)
    probe = fc.plan_batch(w.fields, veh, w.cands, obstacles=w.obstacles)
    for k in (1, 7, 32):
        sel = _limits_selection(fc, probe.summary, k)
        for outputs in ("summary", "paths"):
            res = fc.plan_batch(w.fields, veh, w.cands, obstacles=w.obstacles, outputs=outputs, select=sel,
                                winners=True)
            _check_result(fc, res, sel, w.cands["field_id"])
            assert res.extras["d2h_bytes"] >= len(res.summary) * 176 + 16 * k
            b = int(res.topk_cand[0, 0])
            assert b >= 0 and list(res.winner_paths) == [0]
            path, speeds, n_main = res.winner_paths[0]
            s = res.summary[b]
            assert n_main == int(s["n_main"]) and len(path) == int(s["n_main"]) + int(s["n_head"])
            if outputs == "paths":
                p, v, _ = res.path(b)
                assert path.tobytes() == p.tobytes() and speeds.tobytes() == v.tobytes()
    # several fields, factored: fields without an eligible candidate come back as -1 / +inf / zeros
    w3 = wl.c3(1, fields_per_gpu=40)
    probe = fc.plan_batch(w3.fields, veh, w3.axes)
    sel = _limits_selection(fc, probe.summary, 5)
    sel = fc.Selection(**{**sel.__dict__, "max_boundary_viol": 0})
    res = fc.plan_batch(w3.fields, veh, w3.axes, select=sel, winners=True)
    _check_result(fc, res, sel, w3.cands["field_id"])
    assert set(res.winner_paths) == set(np.nonzero(res.best_cand >= 0)[0].tolist())


def test_select_batches_in_flight(fc):
    """Four batches with selections in flight, collected out of order, one of them repeated because the remembered
    launch sizes do not fit it: each equals its synchronous result."""
    from field_coverage_path_planning_b200 import batch as B
    veh = fc.VehicleParams()
    small_ax = fc.candidate_axes(1, radii=np.linspace(5.0, 6.0, 16), start_corners=[0, 1, 2, 3])
    long_ax = fc.candidate_axes(1, radii=np.linspace(11.0, 12.0, 16), start_corners=[0, 1, 2, 3])  # same shape
    heads_ax = fc.candidate_axes(2, headings=np.deg2rad(np.arange(0.0, 180.0, 5.0)))
    two = [RECT, [(0, 0), (100, 0), (130, 80), (30, 80)]]
    sels = [fc.Selection(top_k=4, w_time=1.0, max_obstacle_viol=0), fc.Selection(top_k=7, min_coverage=0.5),
            fc.Selection(top_k=3, w_boundary=1.0), fc.Selection(top_k=32, w_uncovered=2.0)]
    jobs = [([RECT], small_ax, "paths", [OBST2]), ([RECT], long_ax, "paths", [OBST2]), (two, heads_ax, "summary", None),
            ([RECT], small_ax, "summary", [OBST2])]
    want = [fc.plan_batch(f, veh, c, obstacles=o, outputs=out, select=s, winners=True)
            for (f, c, out, o), s in zip(jobs, sels)]
    B._Hints._c.clear()
    pend = [fc.plan_batch(f, veh, c, obstacles=o, outputs=out, select=s, winners=True, wait=False)
            for (f, c, out, o), s in zip(jobs, sels)]
    for k in (1, 0, 3, 2):
        got, w = pend[k].result(), want[k]
        assert got.summary.tobytes() == w.summary.tobytes()
        assert np.array_equal(got.topk_cand, w.topk_cand) and got.topk_cost.tobytes() == w.topk_cost.tobytes()
        assert got.topk_summary.tobytes() == w.topk_summary.tobytes()
        assert got.winner_paths.keys() == w.winner_paths.keys()
        for f in got.winner_paths:
            assert got.winner_paths[f][0].tobytes() == w.winner_paths[f][0].tobytes()
        assert got.extras["d2h_bytes"] == w.extras["d2h_bytes"]
    assert not pend[1].result().extras["speculative"]      # repeated with sizes from its own layout pass


def test_sharded_select_world1_nccl(fc):
    """plan_batch(distributed=True, select=...) through a world-size-1 NCCL group equals the single-process call:
    ranking, records, and the flag-count repeat path."""
    import torch
    import torch.distributed as dist
    from field_coverage_path_planning_b200 import batch as B
    created = not dist.is_initialized()
    if created:
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1,
                                device_id=torch.device("cuda", 0))
    try:
        veh = fc.VehicleParams()
        heads_ax = fc.candidate_axes(3, headings=np.deg2rad(np.arange(0.0, 180.0, 4.0)))
        fields = [RECT, [(0, 0), (100, 0), (130, 80), (30, 80)], [(0, 0), (12, 0), (12, 9), (0, 9)]]
        small_ax = fc.candidate_axes(1, radii=np.linspace(5.0, 6.0, 16), start_corners=[0, 1, 2, 3])
        long_ax = fc.candidate_axes(1, radii=np.linspace(11.0, 12.0, 16), start_corners=[0, 1, 2, 3])
        jobs = [(fields, heads_ax, None, fc.Selection(top_k=6, w_time=1.0, max_boundary_viol=3)),
                ([RECT], small_ax, [OBST2], fc.Selection(top_k=32, min_coverage=0.9, w_uncovered=1.0)),
                ([RECT], long_ax, [OBST2], fc.Selection(top_k=2))]
        B._Hints._c.clear()
        for f, c, o, s in jobs:
            want = fc.plan_batch(f, veh, c, obstacles=o, select=s)
            got = fc.plan_batch(f, veh, c, obstacles=o, select=s, distributed=True, device="cuda:0")
            assert np.array_equal(got.topk_cand, want.topk_cand)
            assert got.topk_cost.tobytes() == want.topk_cost.tobytes()
            assert got.topk_summary.tobytes() == want.topk_summary.tobytes()
            assert got.extras["winner_summary"].tobytes() == want.topk_summary[:, 0].tobytes()
            assert got.extras["d2h_bytes"] == want.extras["d2h_bytes"] + len(f) * s.top_k * 176 + 16
    finally:
        if created:
            dist.destroy_process_group()


def test_select_on_two_or_more_gpus():
    """Sharded top-k over 2 / 4 / 8 ranks == the single-GPU ranking of the whole job (tests/_multi_gpu_select_worker.py)."""
    import os
    import subprocess
    import sys
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    n = 2 if n < 4 else (4 if n < 8 else 8)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(root, "tests", "_multi_gpu_select_worker.py")]
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=root, start_new_session=True)
    try:
        out, err = p.communicate(timeout=300)
    except subprocess.TimeoutExpired:
        import signal
        os.killpg(p.pid, signal.SIGKILL)
        out, err = p.communicate()
        raise AssertionError("multi-GPU select worker timed out\n" + out[-2000:] + err[-4000:])
    assert p.returncode == 0 and "MULTI GPU SELECT OK" in out, out[-2000:] + err[-4000:]
