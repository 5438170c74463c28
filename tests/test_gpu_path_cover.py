"""Whole-field and headland-band coverage on the device (fcpp_path_coverage, fcpp_plan_coverage: verify_paths,
plan_batch(..., field_coverage=True)) against the brute-force integer oracle (tests/_path_cover_oracle.py) and against the
coverage kernel's own band counts."""
import os
import socket
import sys

import numpy as np
import pytest

from oracle import ref_planner as rp

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _path_cover_oracle as pco  # noqa: E402

pytestmark = pytest.mark.gpu

RECT = [(0.0, 0.0), (500.0, 0.0), (500.0, 200.0), (0.0, 200.0)]
OBST2 = [[(200, 80), (250, 80), (250, 120), (200, 120)], [(350, 140), (380, 140), (380, 170), (350, 170)]]
W = 3.2


def _rot(q, phi, ox, oy):
    c, s = np.cos(phi), np.sin(phi)
    return [(x * c - y * s + ox, x * s + y * c + oy) for x, y in q]


TILT = _rot([(0.0, 0.0), (300.0, 0.0), (300.0, 150.0), (0.0, 150.0)], 0.37, 40.0, -20.0)
PARA = [(0.0, 0.0), (260.0, 0.0), (330.0, 120.0), (70.0, 120.0)]
UTM = [(x + 512345.67, y + 4321098.76) for x, y in _rot([(0.0, 0.0), (220.0, 0.0), (220.0, 90.0), (0.0, 90.0)],
                                                        -0.21, 0.0, 0.0)]
FIELDS = [RECT, TILT, PARA, UTM]
OBSTACLES = [OBST2, [_rot([(100.0, 50.0), (130.0, 50.0), (130.0, 80.0), (100.0, 80.0)], 0.37, 40.0, -20.0)], [], []]


@pytest.fixture(scope="module")
def fc():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import field_coverage_path_planning_b200 as pkg
    return pkg


def _walk(rng, field, n, step, leave=False):
    """A random walk from a random point of the field's box (leave: also far outside it)."""
    f = np.asarray(field)
    lo, hi = f.min(0), f.max(0)
    p0 = rng.uniform(lo - (40 if leave else 0), hi + (40 if leave else 0))
    steps = rng.normal(0, step, (max(n - 1, 0), 2))
    return np.vstack([p0[None], p0 + np.cumsum(steps, 0)])[:n]


def _lawnmower(field, W, R):
    f = np.asarray(field)
    lo, hi = f.min(0) + R, f.max(0) - R
    ys = np.arange(lo[1], hi[1], W)
    pts = []
    for k, y in enumerate(ys):
        xs = (lo[0], hi[0]) if k % 2 == 0 else (hi[0], lo[0])
        pts += [(xs[0], y), (xs[1], y)]
    return np.asarray(pts)


def _oracle(field, obst, path, R, n_main, h):
    bt, bc = pco.band_coverage_of(field, R, path, W, h, n_main)
    ft, fcov = pco.field_coverage(field, path, W, h, n_main)
    p = np.asarray(path, dtype=np.float64).reshape(-1, 2)
    return (rp.boundary_violations(p, field), rp.obstacle_violations(p, obst, W), bt, bc, ft, fcov)


def _as_tuple(r):
    return tuple(int(r[k]) for k in ("n_boundary_viol", "n_obstacle_viol", "band_total", "band_cells", "field_total",
                                     "field_cells"))


def _caller_batch(seed):
    rng = np.random.default_rng(seed)
    paths, fid, hw, nm = [], [], [], []
    for f, field in enumerate(FIELDS):
        short = min(np.ptp(np.asarray(field)[:, 0]), np.ptp(np.asarray(field)[:, 1]))
        cases = [(_walk(rng, field, 400, 6.0), 8.0), (_walk(rng, field, 60, 25.0, leave=True), 5.5),
                 (_lawnmower(field, W, 6.0), 6.0), (np.zeros((0, 2)), 8.0), (_walk(rng, field, 1, 1.0), 8.0),
                 (_walk(rng, field, 120, 10.0), short / 2 + 5.0),     # the inset collapses: band = whole field
                 (_walk(rng, field, 120, 10.0), 0.0), (_walk(rng, field, 50, 10.0), -3.0)]   # no band
        for k, (p, R) in enumerate(cases):
            paths.append(p)
            fid.append(f)
            hw.append(R)
            nm.append([0, len(p) // 2, len(p)][k % 3])
    return paths, np.array(fid), np.array(hw), np.array(nm)


@pytest.mark.parametrize("h", [0.1, 0.05])
def test_caller_paths_match_the_brute_force(fc, h):
    """One ragged batch over four fields (the c2 rectangle with its obstacles, a tilted field with an obstacle, a
    parallelogram, a field at UTM-like coordinates): random walks, paths leaving the field, 0- and 1-point paths,
    n_main 0 / mid / len, collapsing insets and widths <= 0.  All seven integers equal the oracle's."""
    paths, fid, hw, nm = _caller_batch(11)
    got = fc.verify_paths(paths, FIELDS, fc.VehicleParams(), path_field=fid, headland_width=hw, obstacles=OBSTACLES,
                          n_main=nm, grid_h=h)
    assert (got["status"] == 0).all()
    assert (got["field_cells"] >= 0).all() and (got["n_boundary_viol"] > 0).any() and (got["n_obstacle_viol"] > 0).any()
    step = 1 if h == 0.1 else 3          # the oracle takes ~1 s per path at 0.05 m
    for i in range(0, len(paths), step):
        want = _oracle(FIELDS[fid[i]], OBSTACLES[fid[i]], paths[i], float(hw[i]), int(nm[i]), h)
        assert _as_tuple(got[i]) == want, (i, _as_tuple(got[i]), want)
    assert (got["band_total"][hw <= 0] == 0).all() and (got["band_total"][hw > 0] > 0).all()
    # without n_main the whole path is headland
    one = fc.verify_paths(paths[:8], FIELDS, path_field=fid[:8], headland_width=hw[:8], obstacles=OBSTACLES, grid_h=h)
    zero = fc.verify_paths(paths[:8], FIELDS, path_field=fid[:8], headland_width=hw[:8], obstacles=OBSTACLES,
                           n_main=np.zeros(8, dtype=np.int64), grid_h=h)
    assert one.tobytes() == zero.tobytes()


@pytest.mark.slow
def test_big_field_thousands_of_slabs(fc):
    """2 km x 1 km at 0.1 m: 20 000-cell rows, 2 500 row slabs, paths crossing all of them."""
    big = [(0.0, 0.0), (2000.0, 0.0), (2000.0, 1000.0), (0.0, 1000.0)]
    rng = np.random.default_rng(3)
    walk = _walk(rng, big, 3000, 40.0, leave=True)
    cross = np.array([[-5.0, -5.0], [2005.0, 1003.0], [1000.0, -2.0], [1001.0, 1002.0]])
    paths = [walk, cross, _lawnmower(big, 25.0, 8.0)]
    got = fc.verify_paths(paths, [big], headland_width=[8.0, 8.0, 8.0], n_main=[1500, 2, 0])
    for i, (p, m) in enumerate(zip(paths, [1500, 2, 0])):
        assert _as_tuple(got[i]) == _oracle(big, [], p, 8.0, m, 0.1), i


def _plans(fc, turn_model, n=256):
    from benchmarks import workloads as wl
    w = wl.c2(1, radii_per_gpu=n // 4)
    res = fc.plan_batch(w.fields, fc.VehicleParams(), w.cands, obstacles=w.obstacles, outputs="paths",
                        turn_model=turn_model, field_coverage=True)
    return w, res


@pytest.mark.parametrize("turn_model", ["arc", "clothoid", "omega"])
def test_generated_plans_two_rasterisers_agree(fc, turn_model):
    """The band counts of fcpp_plan_coverage equal the coverage kernel's cov_total / cov_cells, the D3 counts the
    plan kernel's; every record equals verify_paths on the fetched path byte for byte; the field counts equal the
    oracle's on a sample."""
    w, res = _plans(fc, turn_model)
    s, fcv = res.summary, res.field_cover
    assert len(fcv) == len(s) == w.n_cand
    ok = s["status"] == 0
    assert ok.sum() > 100
    assert np.array_equal(fcv["band_total"][ok], s["cov_total"][ok])
    assert np.array_equal(fcv["band_cells"][ok], s["cov_cells"][ok])
    assert np.array_equal(fcv["n_boundary_viol"][ok], s["n_boundary_viol"][ok])
    assert np.array_equal(fcv["n_obstacle_viol"][ok], s["n_obstacle_viol"][ok])
    assert (fcv["status"][ok] == 0).all() and (fcv["field_cells"] >= fcv["band_cells"]).all()
    assert (fcv["field_cells"][ok] > fcv["band_cells"][ok]).all()
    assert fcv[~ok].tobytes() == np.zeros((~ok).sum(), fcv.dtype).tobytes()
    allp = res.d_path.cpu().numpy()
    paths = [allp[res.offsets[b]:res.offsets[b + 1]] for b in range(len(s))]
    idx = np.nonzero(ok)[0]
    mine = fc.verify_paths([paths[i] for i in idx], w.fields, fc.VehicleParams(), path_field=w.cands["field_id"][idx],
                           headland_width=w.cands["R"][idx], obstacles=w.obstacles, n_main=s["n_main"][idx],
                           grid_h=w.grid_h)
    assert fcv[idx].tobytes() == mine.tobytes()
    for b in np.random.default_rng(5).choice(np.nonzero(ok)[0], 16, replace=False):
        ft, fcov = pco.field_coverage(RECT, paths[b], W, 0.1, int(s["n_main"][b]))
        assert (int(fcv["field_total"][b]), int(fcv["field_cells"][b])) == (ft, fcov), b


def test_verify_field_coverage_after_plan(fc):
    pl = fc.TwoLayerPathPlannerV37(field_length=500, field_width=200, obstacles=OBST2)
    plan = pl.plan_complete_coverage()
    v = pl.verify_field_coverage()
    assert v["band_coverage_rate"] == plan["headland"]["stats"]["coverage_rate"]
    s = plan["validation"]
    assert (v["band_cells"], v["band_total"]) == (s["cov_cells"], s["cov_total"])
    assert (v["boundary_violations"], v["obstacle_violations"]) == (s["n_boundary_viol"], s["n_obstacle_viol"])
    assert 0.9 < v["field_coverage_rate"] <= 1.0 and v["field_cells"] > v["band_cells"]
    # a caller path: all headland by default
    line = np.array([[0.0, 100.0], [500.0, 100.0]])
    c = pl.verify_field_coverage(line)
    assert c["field_cells"] == pco.field_coverage(RECT, line, W)[1]
    assert c["band_cells"] > 0 and pl.verify_field_coverage(line, n_main=2)["band_cells"] == 0


def test_out_of_range_point_flags_only_its_path(fc):
    from field_coverage_path_planning_b200 import _lib
    paths, fid, hw, nm = _caller_batch(21)
    base = fc.verify_paths(paths, FIELDS, path_field=fid, headland_width=hw, obstacles=OBSTACLES, n_main=nm)
    far = np.vstack([paths[0][:10], [[250.0, 2.0e5]], paths[0][10:]])
    got = fc.verify_paths(paths[:5] + [far] + paths[5:], FIELDS, path_field=np.insert(fid, 5, 0),
                          headland_width=np.insert(hw, 5, 8.0), obstacles=OBSTACLES, n_main=np.insert(nm, 5, 3))
    assert got[5]["status"] == _lib.PATH_OUT_OF_RANGE
    assert _as_tuple(got[5]) == (0,) * 6
    assert np.delete(got, 5).tobytes() == base.tobytes()


def test_without_field_coverage_nothing_changes(fc):
    from field_coverage_path_planning_b200 import _lib
    h = _lib.handle(0)
    ax = fc.candidate_axes(1, radii=np.linspace(5.0, 12.0, 32), start_corners=[0, 1, 2, 3])

    def run(**kw):
        n0 = h.launches
        r = fc.plan_batch([RECT], fc.VehicleParams(), ax, obstacles=[OBST2], outputs="paths", **kw)
        return r, h.launches - n0

    run()
    a, na = run()
    c, nc = run(field_coverage=True)
    b, nb = run()
    assert a.summary.tobytes() == b.summary.tobytes() == c.summary.tobytes()
    assert na == nb == nc - 3 and a.field_cover is None and c.field_cover is not None


def test_pipelined_batches(fc):
    veh = fc.VehicleParams()
    small = fc.candidate_axes(1, radii=np.linspace(5.0, 6.0, 16), start_corners=[0, 1, 2, 3])
    large = fc.candidate_axes(1, radii=np.linspace(11.0, 12.0, 16), start_corners=[0, 1, 2, 3])
    want = [fc.plan_batch([RECT], veh, c, obstacles=[OBST2], outputs="paths", field_coverage=True) for c in (small, large)]
    from field_coverage_path_planning_b200 import batch as B
    B._Hints._c.clear()
    pend = [fc.plan_batch([RECT], veh, c, obstacles=[OBST2], outputs="paths", field_coverage=True, wait=False)
            for c in (small, large)]
    for k in (1, 0):
        got = pend[k].result()
        assert got.field_cover.tobytes() == want[k].field_cover.tobytes()


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
        ax = fc.candidate_axes(1, radii=np.linspace(5.0, 12.0, 16), start_corners=[0, 1, 2, 3])
        want = fc.plan_batch([RECT], fc.VehicleParams(), ax, obstacles=[OBST2], outputs="paths", field_coverage=True)
        got = fc.plan_batch([RECT], fc.VehicleParams(), ax, obstacles=[OBST2], outputs="paths", field_coverage=True,
                            distributed=True, device="cuda:0")
        assert got.field_cover.tobytes() == want.field_cover.tobytes()
        assert got.summary.tobytes() == want.summary.tobytes()
    finally:
        if created:
            dist.destroy_process_group()
