"""Segment-level obstacle sweep on the device (fcpp_obstacle_sweep, fcpp_obstacle_sweep_paths, plan_batch(...,
obstacle_sweep=True)) against the numpy statement in oracle/sweep.py, and the records form against the paths form."""
import socket

import numpy as np
import pytest

from oracle import batch as ob, ref_planner as rp, sweep as osw

pytestmark = pytest.mark.gpu

RECT = [(0.0, 0.0), (500.0, 0.0), (500.0, 200.0), (0.0, 200.0)]
OBST2 = [[(200, 80), (250, 80), (250, 120), (200, 120)], [(350, 140), (380, 140), (380, 170), (350, 170)]]
W = 3.2


@pytest.fixture(scope="module")
def fc():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import field_coverage_path_planning_b200 as pkg
    return pkg


def _oracle_check(got, field, obst, R=None, heading=None, corner=None, turn_model="arc"):
    """One candidate's device record against the oracle: counts exact unless the plan has knife-edge segments (then
    within their number), lengths to 1e-9 m.  Returns the number of knife-edge segments."""
    o = ob.evaluate_candidate(field, rp.VehicleParams(), R=R, heading=heading, start_corner=corner, obstacles=obst,
                              coverage=False, keep_paths=True, turn_model=turn_model)
    if o["status"]:
        assert got.tobytes() == np.zeros(1, got.dtype).tobytes()
        return 0
    want = osw.sweep(o["path"], obst, W, o["n_main"])
    knife = osw.knife_edges(o["path"], obst, W)
    for k in ("n_seg_main", "n_seg_head"):
        assert abs(int(got[k]) - want[k]) <= knife, (k, int(got[k]), want[k], knife)
    for k in ("len_main", "len_head"):
        assert abs(float(got[k]) - want[k]) <= 1e-9, (k, float(got[k]), want[k])
    return knife


def test_c2_full_batch_matches_oracle(fc):
    """The c2 workload (4 096 candidates): no candidate has an obstacle POINT, every one drives through the
    obstacles; a seeded sample matches the oracle."""
    from benchmarks import workloads as wl
    w = wl.c2(1)
    res = fc.plan_batch(w.fields, fc.VehicleParams(), w.cands, obstacles=w.obstacles, outputs="paths",
                        obstacle_sweep=True)
    sw = res.sweep
    assert len(sw) == w.n_cand == 4096
    assert (res.summary["status"] == 0).all() and (res.summary["n_obstacle_viol"] == 0).all()
    assert (sw["n_seg_main"] > 0).all() and (sw["len_main"] > 1000).all()
    knife = 0
    for i in np.random.default_rng(7).choice(w.n_cand, 16, replace=False):
        knife += _oracle_check(sw[i], RECT, OBST2, R=float(w.cands["R"][i]), corner=int(w.cands["start_corner"][i]))
    print("knife-edge segments in the sample:", knife)


def _fields_and_obstacles(seed):
    """A rotated and a sheared field, each with seeded convex and non-convex obstacles inside."""
    rng = np.random.default_rng(seed)
    out = []
    for shear, phi in ((0.0, 0.6), (60.0, -0.3)):
        q = np.array([(0.0, 0.0), (420.0, 0.0), (420.0 + shear, 230.0), (shear, 230.0)])
        c, s = np.cos(phi), np.sin(phi)
        rot = lambda p: (p[0] * c - p[1] * s + 1000.0, p[0] * s + p[1] * c - 300.0)  # noqa: E731
        obst = []
        for k in range(4):
            cx, cy = rng.uniform(90, 330), rng.uniform(50, 180)
            a, b = rng.uniform(6, 25, 2)
            shape = [(-a, -b), (a, -b), (a, b), (-a, b)] if k % 2 == 0 else \
                [(-a, -b), (a, -b), (a, -b / 3), (-a / 3, -b / 3), (-a / 3, b), (-a, b)]    # L shape
            obst.append([rot((cx + x, cy + y)) for x, y in shape])
        out.append(([rot(p) for p in q], obst))
    return out


def _paths_form(fc, res, obst, n_cand):
    paths = [res.path(b)[0] for b in range(n_cand)]
    return fc.obstacle_sweep(paths, obst, W, n_main=res.summary["n_main"][:n_cand])


@pytest.mark.parametrize("turn_model", ["arc", "clothoid", "omega"])
def test_records_form_equals_paths_form(fc, turn_model):
    """Sweeping the materialised paths with n_main from the summaries gives the records form's bytes, and summary
    mode gives the paths mode's bytes: c2 and two seeded fields with convex and non-convex obstacles."""
    veh = fc.VehicleParams()
    cases = [(RECT, OBST2)] + _fields_and_obstacles(3)
    knife = 0
    for field, obst in cases:
        cand = fc.make_candidates(1, headings=[0.0, 0.4, 1.3] if field is not RECT else None,
                                  radii=[5.0, 7.7, 11.0], start_corners=[0, 1, 2, 3])
        res = fc.plan_batch([field], veh, cand, obstacles=[obst], outputs="paths", turn_model=turn_model,
                            coverage=False, obstacle_sweep=True)
        n = len(res.summary)
        assert (res.summary["status"] == 0).all()
        assert res.sweep.tobytes() == _paths_form(fc, res, obst, n).tobytes()
        summ = fc.plan_batch([field], veh, cand, obstacles=[obst], outputs="summary", turn_model=turn_model,
                             coverage=False, obstacle_sweep=True)
        assert summ.sweep.tobytes() == res.sweep.tobytes()
        assert (res.sweep["n_seg_main"] + res.sweep["n_seg_head"] > 0).any()
        if turn_model == "arc":
            for b in range(0, n, 7):
                knife += _oracle_check(res.sweep[b], field, obst, R=float(cand["R"][b]),
                                       heading=float(cand["heading"][b]) if "heading" in cand else None,
                                       corner=int(cand["start_corner"][b]))
    print("knife-edge segments in the sample:", knife)


def test_heading_search_factored_matches_oracle(fc):
    """A factored heading search (180 headings, de-duplicated coverage) on parallelograms with obstacles."""
    from benchmarks import workloads as wl
    fields = wl.c3_fields(6, seed=11)
    rng = np.random.default_rng(5)
    obstacles = []
    for f in fields:
        c = f.mean(axis=0)
        obst = []
        for _ in range(int(rng.integers(1, 4))):
            cx, cy = c + rng.uniform(-30, 30, 2)
            a = rng.uniform(4, 15)
            obst.append([(cx - a, cy - a), (cx + a, cy - a), (cx + a, cy + a), (cx - a, cy + a)])
        obstacles.append(obst)
    heads = np.deg2rad(np.arange(180.0))
    ax = fc.candidate_axes(len(fields), headings=heads)
    res = fc.plan_batch(fields, fc.VehicleParams(), ax, obstacles=obstacles, obstacle_sweep=True)
    expl = fc.plan_batch(fields, fc.VehicleParams(), fc.make_candidates(len(fields), headings=heads),
                         obstacles=obstacles, obstacle_sweep=True)
    assert res.sweep.tobytes() == expl.sweep.tobytes()
    assert (res.sweep["n_seg_main"] > 0).sum() > 100
    knife = 0
    for g in np.random.default_rng(2).choice(len(res.sweep), 10, replace=False):
        f, h = int(g // 180), float(heads[g % 180])
        knife += _oracle_check(res.sweep[g], fields[f].tolist(), obstacles[f], heading=h)
    print("knife-edge segments in the sample:", knife)


def test_many_obstacles_beyond_shared_memory(fc):
    """~300 obstacle polygons (more than the kernels stage in shared memory): read from global memory, same rule."""
    obst = [[(x, y), (x + 4, y), (x + 4, y + 3), (x, y + 3)] for x in range(40, 460, 21) for y in range(20, 180, 11)]
    assert len(obst) > 256
    cand = fc.make_candidates(1, radii=[5.0, 9.0], start_corners=[0, 3])
    res = fc.plan_batch([RECT], fc.VehicleParams(), cand, obstacles=[obst], outputs="paths", coverage=False,
                        obstacle_sweep=True)
    assert res.sweep.tobytes() == _paths_form(fc, res, obst, len(res.summary)).tobytes()
    assert (res.sweep["n_seg_main"] > 20).all()
    # the oracle segment by segment on a prefix (it takes ~10 ms per segment with 1 200 edges).  The prefix has two
    # knife-edge segments: the swaths at y = 43.4 and 46.6 run parallel to the obstacle edges y = 45 at r = 1.6 up to
    # the last bits; their hit flags are not pinned, every other segment's is
    p = res.path(0)[0][:300]
    knife = osw.knife_mask(p, obst, W)
    print("knife-edge segments:", int(knife.sum()))
    got = fc.obstacle_sweep([p[i:i + 2] for i in range(len(p) - 1)], obst, W)["len_main"]
    want = osw.segment_measures(p, obst, W)
    assert (want[~knife] > 0).sum() > 0
    assert np.array_equal(got[~knife] > 0, want[~knife] > 0)
    assert np.abs(got - want).max() <= 1e-9
    whole, ref = fc.obstacle_sweep(p, obst, W)[0], osw.sweep(p, obst, W)
    assert abs(int(whole["n_seg_main"]) - ref["n_seg_main"]) <= int(knife.sum())
    assert abs(float(whole["len_main"]) - ref["len_main"]) <= 1e-9


def test_no_obstacles_and_dead_candidates_give_zeros(fc):
    fields = [RECT, [(0.0, 0.0), (300.0, 0.0), (300.0, 100.0), (0.0, 100.0)]]
    cand = {"field_id": np.array([0, 0, 1, 1], dtype=np.int32), "R": np.array([6.0, 150.0, 6.0, 7.0])}
    res = fc.plan_batch(fields, fc.VehicleParams(), cand, obstacles=[OBST2, []], obstacle_sweep=True)
    assert res.summary["status"][1] != 0 and res.summary["status"][0] == 0
    z = np.zeros(1, dtype=res.sweep.dtype).tobytes()
    assert res.sweep[0]["n_seg_main"] > 0
    for b in (1, 2, 3):
        assert res.sweep[b].tobytes() == z
    none = fc.plan_batch(fields, fc.VehicleParams(), cand, obstacle_sweep=True)
    assert none.sweep.tobytes() == np.zeros(4, dtype=res.sweep.dtype).tobytes()
    assert fc.obstacle_sweep(np.array([[0.0, 0.0], [500.0, 100.0]]), [], W)[0].tobytes() == z


def test_pipelined_and_repeated_batches(fc):
    """Batches in flight (wait=False), collected out of order, one repeated because the remembered launch sizes do
    not fit it: each sweep equals its synchronous result."""
    from field_coverage_path_planning_b200 import batch as B
    veh = fc.VehicleParams()
    small_ax = fc.candidate_axes(1, radii=np.linspace(5.0, 6.0, 16), start_corners=[0, 1, 2, 3])
    long_ax = fc.candidate_axes(1, radii=np.linspace(11.0, 12.0, 16), start_corners=[0, 1, 2, 3])  # same shape
    jobs = [(small_ax, "paths"), (long_ax, "paths"), (small_ax, "summary"), (long_ax, "summary")]
    want = [fc.plan_batch([RECT], veh, c, obstacles=[OBST2], outputs=o, obstacle_sweep=True) for c, o in jobs]
    B._Hints._c.clear()
    pend = [fc.plan_batch([RECT], veh, c, obstacles=[OBST2], outputs=o, obstacle_sweep=True, wait=False)
            for c, o in jobs]
    for k in (1, 0, 3, 2):
        got = pend[k].result()
        assert got.summary.tobytes() == want[k].summary.tobytes()
        assert got.sweep.tobytes() == want[k].sweep.tobytes()
        assert got.extras["d2h_bytes"] == want[k].extras["d2h_bytes"]
    assert not pend[1].result().extras["speculative"]      # repeated with sizes from its own layout pass


def test_sharded_world1_nccl(fc):
    import torch
    import torch.distributed as dist
    created = not dist.is_initialized()
    if created:
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1,
                                device_id=torch.device("cuda", 0))
    try:
        ax = fc.candidate_axes(1, radii=np.linspace(5.0, 12.0, 32), start_corners=[0, 1, 2, 3])
        want = fc.plan_batch([RECT], fc.VehicleParams(), ax, obstacles=[OBST2], obstacle_sweep=True)
        got = fc.plan_batch([RECT], fc.VehicleParams(), ax, obstacles=[OBST2], obstacle_sweep=True, distributed=True,
                            device="cuda:0")
        assert got.sweep.tobytes() == want.sweep.tobytes()
        assert got.summary.tobytes() == want.summary.tobytes()
    finally:
        if created:
            dist.destroy_process_group()


def test_verify_obstacle_clearance(fc):
    """The mlp3 demo scenario (500 x 200 m, the two obstacles of mlp3:1629-1632): no obstacle point, ~1.1 km inside."""
    pl = fc.TwoLayerPathPlannerV37(field_length=500, field_width=200, obstacles=OBST2)
    plan = pl.plan_complete_coverage()
    v = pl.verify_obstacle_clearance()
    assert v["point_violations"] == 0 and v["segments"] > 0 and not v["pass"]
    assert v["metres"] == v["metres_main"] + v["metres_head"] and v["metres"] > 1000
    p = np.vstack([plan["main_work"]["path"], plan["headland"]["path"]])
    want = osw.sweep(p, OBST2, W, len(plan["main_work"]["path"]))
    assert v["segments_main"] == want["n_seg_main"] and v["segments_head"] == want["n_seg_head"]
    assert abs(v["metres_main"] - want["len_main"]) <= 1e-9 and abs(v["metres_head"] - want["len_head"]) <= 1e-9
    line = np.array([[0.0, 100.0], [500.0, 100.0], [500.0, 10.0]])
    c = pl.verify_obstacle_clearance(line)
    assert c["point_violations"] is None and c["segments"] == 1 and c["segments_head"] == 0
    assert abs(c["metres"] - 53.2) <= 1e-9
    assert pl.verify_obstacle_clearance(line, n_main=0)["segments_head"] == 1      # all headland
    assert pl.verify_obstacle_clearance(line, n_main=1)["segments"] == 0           # the hit is the junction


def test_without_sweep_nothing_changes(fc):
    """Without obstacle_sweep, summaries, rankings and launch counts are those of the same call made before a sweep
    ran on the handle."""
    from field_coverage_path_planning_b200 import _lib
    ax = fc.candidate_axes(1, radii=np.linspace(5.0, 12.0, 64), start_corners=[0, 1, 2, 3])
    h = _lib.handle(0)

    def run(**kw):
        n0 = h.launches
        r = fc.plan_batch([RECT], fc.VehicleParams(), ax, obstacles=[OBST2], select=fc.Selection(top_k=4), **kw)
        return r, h.launches - n0

    run()                               # sizes remembered: the three calls below launch alike
    a, na = run()
    s, ns = run(obstacle_sweep=True)
    b, nb = run()
    assert a.summary.tobytes() == b.summary.tobytes() == s.summary.tobytes()
    assert np.array_equal(a.topk_cand, b.topk_cand) and a.topk_cost.tobytes() == b.topk_cost.tobytes()
    assert na == nb == ns - 1 and a.sweep is None and b.sweep is None
