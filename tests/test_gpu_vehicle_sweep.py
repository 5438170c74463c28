"""Plan kernels against the CPU oracle across vehicle parameters.

The other suites run (nearly) every plan with the default VehicleParams, under which no lateral-acceleration
violation ever happens, no speed falls to the 0.1 m/s floor of the time sums and the acceleration ramps are short.
A kernel that hard-coded a default (safety factor 0.85, 1.5 m/s^2, the class speeds) or dropped a term that is zero
under the defaults would pass them.  Here every path of the plan kernels runs under named vehicles that reach those
regimes: many violations inside the regular main chains (safety factor 1.5), long ramps (0.02 m/s^2), speeds down to
0.15 km/h (0.001 m/s^2 lateral), speeds of exactly 0 (safety factor or turn speed 0), a ramp increment of 0, three
class speeds distinct from the defaults, and the knife edge of safety factor 1.0.

Knife edge.  At safety factor 1.0 a curvature-limited point has a_lat = (v / 3.6)^2 kappa == max_lateral_accel up to
rounding, and the reference's `a_lat > max_lateral_accel` is decided by the last bits of kappa.  The device computes
kappa with one atan2 (and from per-candidate tables inside congruent pieces), the oracle with the reference's three
atan2 + sin / cos, so such points may count differently.  A point is a knife-edge point when the ORACLE's value has
|a_lat - max_lateral_accel| <= KNIFE_EPS * max_lateral_accel; a candidate's violation count must equal the oracle's
exactly when it has no knife-edge point, and may differ by at most their number otherwise.  Measured on a B200 at
safety factor 1.0 on the 80 candidates of test_plan_batch_vs_oracle_per_vehicle: 644 knife-edge points (all within
4.4e-16 of the limit, relative; every other point is 3e-3 or more away), 31 counts differ, 36 points are classified
differently and the farthest of them lies 2.2e-16 from the limit; KNIFE_EPS = 1e-13 keeps a margin of more than 400.
Every other vehicle here must have no knife-edge point at all, i.e. its counts are compared exactly.

Tolerances as in test_gpu_parity.py: counts exact, FP64 sums rtol 1e-9, points and speeds 1e-9 (1e-7 for the speeds
of the opt-in turn models, whose Fresnel / trigonometric series differ from scipy / numpy in the last bits).
"""
import numpy as np
import pytest

from test_gpu_fullsize import oracle_many

gpu = pytest.mark.gpu

TIGHT = 1e-9
KNIFE_EPS = 1e-13

RECT = [(0, 0), (500, 0), (500, 200), (0, 200)]
OBST2 = [[(200, 80), (250, 80), (250, 120), (200, 120)], [(350, 140), (380, 140), (380, 170), (350, 170)]]
PARA = [(100, 50), (600, 120), (640, 330), (140, 260)]
SMALL = [(0, 0), (100, 0), (100, 80), (0, 80)]
TILT = [(0, 0), (300, 40), (280, 190), (-20, 150)]
HUGE = [(0, 0), (5000, 0), (5000, 3000), (0, 3000)]
FIELDS = [RECT, PARA, SMALL]
OBSTACLES = [OBST2, [], []]
RADII = [5.0, 6.4, 8.0, 11.0]
CORNERS = [0, 1, 2, 3]
TILT_HEADINGS = np.deg2rad([17.0, 90.0])

# changes from the defaults (working_width 3.2, R 8, work / headland / turn 9 / 15 / 4 km/h, lateral 2 m/s^2,
# longitudinal 1.5 m/s^2, safety factor 0.85)
VEHICLES = {
    "default": {},
    "sf1.5": dict(safety_factor=1.5, headland_turn_speed_kmh=20.0),   # violations inside the regular main chains
    "sf1.2": dict(safety_factor=1.2),                                   # a few violations, all in the headland
    "along0.02": dict(max_longitudinal_accel=0.02),                     # long acceleration ramps
    "alat0.001": dict(max_lateral_accel=0.001),                         # speeds below the 0.1 m/s time floor
    "sf0": dict(safety_factor=0.0),                                     # speeds of exactly 0
    "turn0": dict(headland_turn_speed_kmh=0.0),                         # class speed 0
    "along0": dict(max_longitudinal_accel=0.0),                         # ramp increment 0
    "sf1.0": dict(safety_factor=1.0),                                   # the knife edge
    "classes": dict(max_work_speed_kmh=7.0, max_headland_speed_kmh=13.0, headland_turn_speed_kmh=3.0),
}

INT_KEYS = ("n_passes", "n_loops", "n_main", "n_head", "n_boundary_viol", "n_obstacle_viol")
FP_KEYS = ("len_main", "len_head", "time_main", "time_head", "time_main_pre", "time_head_pre", "max_curvature",
           "max_lateral_accel", "max_jump")
COV_KEYS = ("corner_g", "corner_before", "corner_after", "cov_total", "cov_cells")


@pytest.fixture(scope="module")
def fc():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import field_coverage_path_planning_b200 as pkg
    return pkg


def vehicles(fc, name):
    """(device VehicleParams, oracle VehicleParams, the changed fields) of a named vehicle."""
    from oracle import ref_planner as rp
    kw = VEHICLES[name]
    return fc.VehicleParams(**kw), rp.VehicleParams(**kw), kw


def knife_edge_points(path, speeds, oveh):
    """Points of a path whose lateral acceleration (the oracle's values) lies within KNIFE_EPS of the limit."""
    from oracle import ref_planner as rp
    if len(path) < 3:
        return 0
    a_lat = (speeds[1:-1] / 3.6) ** 2 * rp.curvatures(path)
    lim = oveh.max_lateral_accel
    return int(np.count_nonzero(np.abs(a_lat - lim) <= KNIFE_EPS * lim))


def assert_accel_count(got, want, n_knife):
    if n_knife == 0:
        assert got == want, ("n_accel_viol", got, want)
    else:
        assert abs(got - want) <= n_knife, ("n_accel_viol", got, want, n_knife)


def check_candidate(s, o, oveh, path=None, speeds=None, speed_tol=TIGHT):
    """Every non-coverage summary field of one candidate against the oracle (o from keep_paths=True); points and
    speeds too when given.  Returns the number of knife-edge points."""
    assert int(s["status"]) == o["status"]
    if o["status"]:
        return 0
    for k in INT_KEYS:
        assert int(s[k]) == int(o[k]), (k, int(s[k]), o[k])
    n_knife = knife_edge_points(o["path"], o["speeds"], oveh)
    assert_accel_count(int(s["n_accel_viol"]), o["n_accel_viol"], n_knife)
    for k in FP_KEYS:
        np.testing.assert_allclose(float(s[k]), o[k], rtol=1e-9, atol=1e-12, err_msg=k)
    if path is not None:
        assert path.shape == o["path"].shape
        dp = float(np.abs(path - o["path"]).max())
        ds = float(np.abs(speeds - o["speeds"]).max())
        assert dp <= TIGHT and ds <= speed_tol, (dp, ds)
    return n_knife


def oracle_jobs(fields, obstacles, cand, kw, keep=True, extra=None, grid_h=0.1):
    jobs = []
    for b in range(len(cand["field_id"])):
        f = int(cand["field_id"][b])
        args = (fields[f], float(cand["R"][b]) if "R" in cand else None,
                float(cand["heading"][b]) if "heading" in cand else None,
                int(cand["start_corner"][b]) if "start_corner" in cand else None,
                obstacles[f] if obstacles else (), grid_h)
        jobs.append((args, False, keep, kw, extra or {}))
    return jobs


def sweep_batches(fc, veh, outputs):
    """The sweep's two batches: three fields x radii x start corners (explicit candidates) and a tilted quad with a
    heading axis (factored candidates)."""
    cand = fc.make_candidates(len(FIELDS), radii=RADII, start_corners=CORNERS)
    ax = fc.candidate_axes(1, headings=TILT_HEADINGS, radii=RADII, start_corners=CORNERS)
    a = fc.plan_batch(FIELDS, veh, cand, obstacles=OBSTACLES, outputs=outputs)
    t = fc.plan_batch([TILT], veh, ax, outputs=outputs)
    return (a, cand), (t, fc.expand_axes(ax))


_default_coverage = {}


def default_coverage(fc):
    if not _default_coverage:
        (a, _), (t, _) = sweep_batches(fc, fc.VehicleParams(), "summary")
        _default_coverage.update(a=a.summary.copy(), t=t.summary.copy())
    return _default_coverage


@gpu
@pytest.mark.parametrize("name", list(VEHICLES))
def test_plan_batch_vs_oracle_per_vehicle(fc, name):
    """Every non-coverage summary field, points and speeds of 80 candidates (RECT with two obstacles, a sheared
    field, a small field, a tilted quad under two headings; R 5 / 6.4 / 8 / 11; start corners 0-3) against the
    oracle with the same vehicle; summary-only mode gives the same bytes as paths mode (its turns are classified
    separately); coverage does not depend on the speeds: the coverage columns equal the default vehicle's."""
    veh, oveh, kw = vehicles(fc, name)
    paths = sweep_batches(fc, veh, "paths")
    summ = sweep_batches(fc, veh, "summary")
    cov = default_coverage(fc)
    n_knife = 0
    for ((res, cand), fields, obst), (sres, _), key in zip(((paths[0], FIELDS, OBSTACLES), (paths[1], [TILT], None)),
                                                           summ, ("a", "t")):
        assert res.summary.tobytes() == sres.summary.tobytes()
        for k in COV_KEYS:
            assert np.array_equal(res.summary[k], cov[key][k]), k
        recs = oracle_many(oracle_jobs(fields, obst, cand, kw))
        assert all(o["status"] == 0 for o in recs)
        for b, o in enumerate(recs):
            p, s, _ = res.path(b)
            n_knife += check_candidate(res.summary[b], o, oveh, p, s)
    assert (n_knife > 0) == (name == "sf1.0")     # every other vehicle: exact counts everywhere
    if name == "sf1.5":
        assert paths[0][0].summary["n_accel_viol"].min() > 100


@gpu
@pytest.mark.parametrize("name", ["along0.02", "sf1.5"])
def test_plan_longer_than_shared_memory_staging_per_vehicle(fc, name):
    """A 5 km x 3 km field (> 20 000 points per plan, the HBM-staged kernel) next to a small one, against the
    oracle: long ramps under a small longitudinal acceleration, many violations under safety factor 1.5."""
    veh, oveh, kw = vehicles(fc, name)
    fields = [RECT, HUGE]
    cand = fc.make_candidates(2, start_corners=[0, 2])
    res = fc.plan_batch(fields, veh, cand, outputs="paths", grid_h=0.5, coverage=False)
    assert (res.summary["status"] == 0).all() and int(res.summary["n_main"][2]) > 20000
    recs = oracle_many(oracle_jobs(fields, None, cand, kw, grid_h=0.5))
    for b, o in enumerate(recs):
        p, s, _ = res.path(b)
        check_candidate(res.summary[b], o, oveh, p, s)
    if name == "sf1.5":
        assert res.summary["n_accel_viol"][2:].min() > 1000


@gpu
@pytest.mark.parametrize("name", ["sf1.5", "alat0.001"])
def test_fused_plan_cover_kernel_identical_per_vehicle(fc, name):
    """The opt-in fused plan + coverage kernel (fcpp_set_cover_mode bit 2) == the two separate launches, bit for
    bit, under a vehicle with many violations and one with speeds below the time floor."""
    import torch
    from field_coverage_path_planning_b200 import _lib
    h = _lib.handle(0)
    veh, _, _ = vehicles(fc, name)
    tiny = [(0, 0), (30, 0), (30, 15), (0, 15)]
    cases = [
        ([RECT], fc.make_candidates(1, radii=np.linspace(5.0, 12.0, 257), start_corners=CORNERS), [OBST2]),
        ([RECT, tiny, PARA], fc.make_candidates(3, radii=[6.0, 8.0, 11.0], start_corners=[0, 2, 3]), None),
        ([PARA, RECT], fc.make_candidates(2, headings=np.deg2rad(np.arange(0.0, 180.0, 9.0)), radii=[7.0]), None),
        ([RECT], fc.make_candidates(1, radii=np.linspace(5.0, 8.0, 65), start_corners=CORNERS), [OBST2]),
        ([RECT], fc.make_candidates(1, radii=[8.0]), None),
    ]
    n_fused = 0
    for fields, cand, obst in cases:
        a = fc.plan_batch(fields, veh, cand, obstacles=obst, outputs="paths")
        try:
            h.check(h.lib.fcpp_set_cover_mode(h.h, 4))
            b = fc.plan_batch(fields, veh, cand, obstacles=obst, outputs="paths")
            n_fused += int(h.lib.fcpp_last_fused(h.h))
        finally:
            h.check(h.lib.fcpp_set_cover_mode(h.h, 0))
        assert a.summary.tobytes() == b.summary.tobytes()
        assert np.array_equal(a.best_cand, b.best_cand) and np.array_equal(a.best_cost, b.best_cost)
        n = int(a.offsets[-1])
        assert np.array_equal(a.offsets, b.offsets)
        assert torch.equal(a.d_path[:n], b.d_path[:n]) and torch.equal(a.d_speeds[:n], b.d_speeds[:n])
    assert n_fused >= 2


@gpu
@pytest.mark.parametrize("turn_model", ["omega", "clothoid"])
@pytest.mark.parametrize("name", ["sf1.5", "along0.02"])
def test_opt_in_turn_models_vs_oracle_per_vehicle(fc, name, turn_model):
    """Ω skip-row turns (chains evaluated one by one, not from the regular-chain shortcut) and clothoid turns under
    many violations and long ramps, against the oracle; summary-only == paths mode."""
    veh, oveh, kw = vehicles(fc, name)
    cand = fc.make_candidates(len(FIELDS), radii=[5.0, 8.0, 11.0], start_corners=[0, 3])
    res = fc.plan_batch(FIELDS, veh, cand, obstacles=OBSTACLES, outputs="paths", turn_model=turn_model, coverage=False)
    summ = fc.plan_batch(FIELDS, veh, cand, obstacles=OBSTACLES, outputs="summary", turn_model=turn_model,
                         coverage=False)
    assert summ.summary.tobytes() == res.summary.tobytes()
    recs = oracle_many(oracle_jobs(FIELDS, OBSTACLES, cand, kw, extra=dict(turn_model=turn_model)))
    for b, o in enumerate(recs):
        p, s, _ = res.path(b) if o["status"] == 0 else (None, None, None)
        assert check_candidate(res.summary[b], o, oveh, p, s, speed_tol=1e-7) == 0
    if name == "sf1.5":
        assert res.summary["n_accel_viol"].min() > 100


@gpu
@pytest.mark.parametrize("name", list(VEHICLES))
def test_drop_in_planner_per_vehicle(fc, name):
    """TwoLayerPathPlannerV37(veh, ...) on a sheared field with a start point: plan_complete_coverage() against the
    oracle's statement of the reference, verify_curvature_constraints() against rp.verify_curvature_constraints."""
    from oracle import ref_planner as rp
    veh, oveh, _ = vehicles(fc, name)
    start = (500.0, 250.0)
    pl = fc.TwoLayerPathPlannerV37(veh, field_vertices=PARA, start_point=start)
    r = pl.plan_complete_coverage()
    o = rp.plan_complete_coverage(rp.setup_field(oveh, field_vertices=PARA, start_point=start))
    for layer in ("main_work", "headland"):
        assert r[layer]["path"].shape == o[layer]["path"].shape
        assert np.abs(r[layer]["path"] - o[layer]["path"]).max() <= TIGHT
        assert np.abs(r[layer]["speeds"] - o[layer]["speeds"]).max() <= TIGHT
        for k in ("path_length_km", "time_hours", "avg_speed_kmh"):
            np.testing.assert_allclose(r[layer]["stats"][k], o[layer]["stats"][k], rtol=1e-9, err_msg=k)
    allp = np.vstack([r["main_work"]["path"], r["headland"]["path"]])
    alls = np.concatenate([r["main_work"]["speeds"], r["headland"]["speeds"]])
    oallp = np.vstack([o["main_work"]["path"], o["headland"]["path"]])
    oalls = np.concatenate([o["main_work"]["speeds"], o["headland"]["speeds"]])
    cc = pl.verify_curvature_constraints(allp, alls)
    oc = rp.verify_curvature_constraints(oallp, oalls, oveh)
    n_knife = knife_edge_points(oallp, oalls, oveh)
    assert n_knife == 0 or name == "sf1.0"
    assert_accel_count(cc["accel_violations"], oc["accel_violations"], n_knife)
    if cc["accel_violations"] == oc["accel_violations"]:
        np.testing.assert_allclose(cc["accel_violation_rate"], oc["accel_violation_rate"], rtol=1e-12)
    assert cc["pass"] == oc["pass"]
    for k in ("max_curvature", "max_lateral_accel", "max_jump"):
        np.testing.assert_allclose(cc[k], oc[k], rtol=1e-9, atol=1e-12, err_msg=k)
    if name == "sf1.5":
        assert cc["pass"] is False and cc["accel_violation_rate"] > 5


@gpu
@pytest.mark.parametrize("name", ["along0.02", "alat0.001", "sf0"])
def test_caller_path_speed_planning_per_vehicle(fc, name):
    """The speed planner on caller-supplied random walks (duplicates, sharp turns, long jumps) of 3 to 30 000 points
    (30 000: the HBM-staged kernel; long ramps cross the per-thread chunks and warps of the min-plus scan) against
    rp.speed_plan, the work time against rp.work_time, the violation count against rp.verify_curvature_constraints."""
    from oracle import ref_planner as rp
    veh, oveh, _ = vehicles(fc, name)
    rng = np.random.default_rng(17)
    pl = fc.TwoLayerPathPlannerV37(veh, field_length=500, field_width=200)
    for n in (3, 257, 5000, 30000):
        step = rng.normal(0, 1.0, size=(n, 2)) * rng.choice([0.0, 0.3, 1.0, 25.0], size=(n, 1), p=[0.1, 0.3, 0.5, 0.1])
        path = np.cumsum(step, axis=0) + 1000.0
        speeds = rng.choice([2.5, 4.0, 9.0, 15.0], size=n)
        got = pl._apply_curvature_based_speed_limit(path, speeds)
        want = rp.speed_plan(path, speeds, oveh)
        assert np.abs(got - want).max() <= TIGHT, n
        np.testing.assert_allclose(pl._calculate_work_time(path, got), rp.work_time(path, want), rtol=1e-9)
        cc = pl.verify_curvature_constraints(path, got)
        oc = rp.verify_curvature_constraints(path, want, oveh)
        assert knife_edge_points(path, want, oveh) == 0
        assert cc["accel_violations"] == oc["accel_violations"]
        if n == 30000 and name == "along0.02":
            # the ramps are long: the speed limit of a point reaches far beyond its neighbours
            assert np.count_nonzero(want < speeds) > n // 2
        if name != "along0.02" and n > 3:
            assert np.count_nonzero(want < 0.36) > n // 2      # below the 0.1 m/s floor of the time sums


@gpu
@pytest.mark.parametrize("name", ["sf1.5", "alat0.001"])
def test_cost_time_argmin_vs_oracle(fc, name):
    """plan_batch(cost='time'): the per-field winner is numpy's argmin of time_main + time_head (ties to the lowest
    index) over the oracle-checked time columns, for two vehicles whose time ranking differs from the length
    ranking; a batch of more than 16 384 candidates takes the multi-kernel argmin."""
    veh, oveh, kw = vehicles(fc, name)
    cand = fc.make_candidates(len(FIELDS), radii=RADII, start_corners=CORNERS)
    res = fc.plan_batch(FIELDS, veh, cand, obstacles=OBSTACLES, coverage=False, cost="time")
    lres = fc.plan_batch(FIELDS, veh, cand, obstacles=OBSTACLES, coverage=False)
    assert res.summary.tobytes() == lres.summary.tobytes()
    s = res.summary
    recs = oracle_many(oracle_jobs(FIELDS, OBSTACLES, cand, kw, keep=False))
    for b, o in enumerate(recs):
        assert int(s["status"][b]) == o["status"]
        if o["status"] == 0:
            for k in ("time_main", "time_head", "len_main", "len_head"):
                np.testing.assert_allclose(float(s[k][b]), o[k], rtol=1e-9, err_msg=k)
    per = len(cand["field_id"]) // len(FIELDS)
    t = np.where(s["status"] == 0, s["time_main"] + s["time_head"], np.inf).reshape(len(FIELDS), per)
    ln = np.where(s["status"] == 0, s["len_main"] + s["len_head"], np.inf).reshape(len(FIELDS), per)
    want = np.arange(len(FIELDS)) * per + t.argmin(1)
    assert np.array_equal(res.best_cand, want) and np.array_equal(res.best_cost, t.min(1))
    assert np.array_equal(lres.best_cand, np.arange(len(FIELDS)) * per + ln.argmin(1))
    assert (t.argmin(1) != ln.argmin(1)).all()
    ot = np.array([o["time_main"] + o["time_head"] if o["status"] == 0 else np.inf for o in recs]).reshape(t.shape)
    for f in range(len(FIELDS)):
        srt = np.sort(ot[f])
        if srt[1] - srt[0] > 1e-6 * srt[0]:          # a clear minimum: it must be the oracle's
            assert int(res.best_cand[f]) == f * per + int(np.argmin(ot[f]))
    # more than 16 384 candidates: the argmin runs as init / cost / index / final kernels
    big = fc.make_candidates(len(FIELDS), radii=np.linspace(5.0, 12.0, 1400), start_corners=CORNERS)
    res = fc.plan_batch(FIELDS, veh, big, obstacles=OBSTACLES, coverage=False, cost="time")
    s = res.summary
    per = len(big["field_id"]) // len(FIELDS)
    assert per * len(FIELDS) > 16384
    t = np.where(s["status"] == 0, s["time_main"] + s["time_head"], np.inf).reshape(len(FIELDS), per)
    want = np.arange(len(FIELDS)) * per + t.argmin(1)
    assert np.array_equal(res.best_cand, want) and np.array_equal(res.best_cost, t.min(1))
    idx = sorted(set(want.tolist()) | set(np.random.default_rng(3).choice(len(s), 9, replace=False).tolist()))
    sub = {k: v[idx] for k, v in big.items()}
    for b, o in zip(idx, oracle_many(oracle_jobs(FIELDS, OBSTACLES, sub, kw, keep=False))):
        assert int(s["status"][b]) == o["status"]
        if o["status"] == 0:
            np.testing.assert_allclose(float(s["time_main"][b] + s["time_head"][b]), o["time_main"] + o["time_head"],
                                       rtol=1e-9)


def test_plan_batch_rejects_unknown_cost():
    """cost is 'length' or 'time'; anything else is an error raised before a device is looked for (no GPU needed)."""
    import field_coverage_path_planning_b200 as fc
    for bad in ("bogus", "Time", "", None, 1):
        with pytest.raises(ValueError, match="cost"):
            fc.plan_batch([RECT], fc.VehicleParams(), cost=bad)
        with pytest.raises(ValueError, match="cost"):
            fc.plan_batch([RECT], fc.VehicleParams(), cost=bad, distributed=True)
