"""GPU parity tests: the CUDA path (through the C-ABI, via the Python host) against the CPU
oracle on the same inputs, against the committed golden fixtures of the reference, and —
at BASELINE.json's full sizes — through size-independent properties.

Tolerances (north_star): counts bit-exact; points <= 1e-4 m; speeds <= 1e-4 m/s = 3.6e-4 km/h.
The generated points are expected to be BIT-IDENTICAL to numpy's (host-supplied trig tables,
-fmad=false), so the tests assert a much tighter 1e-9 and record the observed maximum.
"""
import glob
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PT_TOL = 1e-4          # m       (north_star)
SPEED_TOL = 3.6e-4     # km/h    (north_star: 1e-4 m/s)
TIGHT = 1e-9           # what the design actually delivers


@pytest.fixture(scope="module")
def fc():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import field_coverage_path_planning_b200 as pkg
    return pkg


def _golden_cases():
    d = os.path.join(os.path.dirname(__file__), "golden")
    return sorted(glob.glob(os.path.join(d, "ref_*.npz")))


def _meta(z):
    meta = json.loads(str(z["meta"]))
    kw = dict(meta["planner"])
    for k in ("start_point", "end_point"):
        if kw.get(k) is not None:
            kw[k] = tuple(kw[k])
    if kw.get("field_vertices") is not None:
        kw["field_vertices"] = [tuple(v) for v in kw["field_vertices"]]
    return meta, kw


@pytest.mark.parametrize("path", _golden_cases(), ids=lambda p: os.path.basename(p)[4:-4])
def test_single_plan_vs_reference_golden(fc, path):
    """Drop-in API vs outputs of the unmodified reference (tests/golden/make_golden.py)."""
    z = np.load(path)
    meta, kw = _meta(z)
    veh = fc.VehicleParams(**meta["vehicle"])
    planner = fc.TwoLayerPathPlannerV37(veh, **kw)
    assert planner.field_shape == meta["field_shape"]
    assert planner.main_work_pattern == meta["pattern"]
    r = planner.plan_complete_coverage()
    assert r["version"] == "V3.5.1"
    assert r["main_work"]["path"].shape == z["main_path"].shape        # integer layout: exact
    assert r["headland"]["path"].shape == z["head_path"].shape
    dm = np.abs(r["main_work"]["path"] - z["main_path"]).max()
    dh = np.abs(r["headland"]["path"] - z["head_path"]).max()
    ds = max(np.abs(r["main_work"]["speeds"] - z["main_speeds"]).max(),
             np.abs(r["headland"]["speeds"] - z["head_speeds"]).max())
    assert dm <= TIGHT and dh <= TIGHT, (dm, dh)
    assert ds <= TIGHT, ds
    assert dm <= PT_TOL and dh <= PT_TOL and ds <= SPEED_TOL
    for layer, key in (("main_work", "main_stats"), ("headland", "head_stats")):
        got = [r[layer]["stats"][k] for k in ("path_length_km", "time_hours", "avg_speed_kmh")]
        np.testing.assert_allclose(got, z[key], rtol=1e-11)
    allp = np.vstack([r["main_work"]["path"], r["headland"]["path"]])
    alls = np.concatenate([r["main_work"]["speeds"], r["headland"]["speeds"]])
    cc = planner.verify_curvature_constraints(allp, alls)
    ref = z["curv"]
    np.testing.assert_allclose([cc["max_curvature"], cc["max_lateral_accel"], cc["max_jump"]],
                               [ref[0], ref[1], ref[4]], rtol=1e-9)
    assert cc["accel_violations"] == int(ref[2])
    assert cc["pass"] == bool(ref[5])
    for name, key in (("approach_path", "approach"), ("departure_path", "departure")):
        if len(z[key]):
            np.testing.assert_allclose(r[name], z[key], rtol=0, atol=TIGHT)
        else:
            assert r[name] is None
    if "corner_cells_float" in z.files:
        cov = planner.verify_all_corners_coverage(r["headland"])
        got = np.array([[c["cells_before"], c["cells_after"]] for c in cov["corners"]])
        assert np.max(np.abs(got - z["corner_cells_float"])) <= 2      # float64 vs exact fixed point (D5)
    # README.md:199: "100.0 %" headland coverage for the rectangles
    assert 0.99 < r["headland"]["stats"]["coverage_rate"] <= 1.0


def _summary_vs_oracle(s, o, coverage=True):
    assert int(s["status"]) == o["status"]
    if o["status"]:
        return
    for k in ("n_passes", "n_loops", "n_main", "n_head", "n_accel_viol", "n_boundary_viol", "n_obstacle_viol"):
        assert int(s[k]) == int(o[k]), (k, int(s[k]), o[k])
    for k in ("len_main", "len_head", "time_main", "time_head", "time_main_pre", "time_head_pre",
              "max_curvature", "max_lateral_accel", "max_jump"):
        np.testing.assert_allclose(float(s[k]), o[k], rtol=1e-9, atol=1e-12, err_msg=k)
    if coverage:
        assert int(s["corner_g"]) == o["corner_g"]
        assert list(map(int, s["corner_before"])) == o["corner_before"]
        assert list(map(int, s["corner_after"])) == o["corner_after"]
        assert (int(s["cov_total"]), int(s["cov_cells"])) == (o["cov_total"], o["cov_cells"])


OBST2 = [[(200, 80), (250, 80), (250, 120), (200, 120)], [(350, 140), (380, 140), (380, 170), (350, 170)]]
RECT = [(0, 0), (500, 0), (500, 200), (0, 200)]


def test_batch_config2_subset_vs_oracle(fc):
    """BASELINE config 2 (500x200 + two obstacles, start corner x radius), a 44-candidate subset
    including the FP64 knife-edge radii of SURVEY.md App. A Q17 — every summary field against
    the oracle, paths and speeds of every candidate too."""
    from oracle import batch as ob, ref_planner as rp
    veh = fc.VehicleParams()
    radii = np.concatenate([np.linspace(5.0, 12.0, 8), [7.2, 9.6, 6.4]])
    cand = fc.make_candidates(1, radii=radii, start_corners=[0, 1, 2, 3])
    res = fc.plan_batch([RECT], veh, cand, obstacles=[OBST2], outputs="paths")
    oveh = rp.VehicleParams()
    assert len(res.summary) == len(radii) * 4
    worst_p = worst_s = 0.0
    for b in range(len(res.summary)):
        o = ob.evaluate_candidate(RECT, oveh, R=cand["R"][b], start_corner=int(cand["start_corner"][b]),
                                  obstacles=OBST2, keep_paths=True)
        _summary_vs_oracle(res.summary[b], o)
        p, s, nm = res.path(b)
        assert p.shape == o["path"].shape
        worst_p = max(worst_p, np.abs(p - o["path"]).max())
        worst_s = max(worst_s, np.abs(s - o["speeds"]).max())
    assert worst_p <= TIGHT and worst_s <= TIGHT, (worst_p, worst_s)
    # obstacles never change the path (Q2) and swaths only carry their two end points, so no path
    # POINT falls into these two obstacles: the point-based count of D3 is 0 here
    assert (res.summary["n_obstacle_viol"] == 0).all()
    # argmin: len_main + len_head, ties to the lowest index
    cost = res.summary["len_main"] + res.summary["len_head"]
    assert int(res.best_cand[0]) == int(np.argmin(cost))
    assert res.best_cost[0] == cost.min()


def test_obstacle_and_boundary_counts_nonzero_vs_oracle(fc):
    """Obstacles placed over swath ends / headland loops (triangle, pentagon, rectangle) and a
    sheared field whose swaths overshoot the slanted sides (Q14): non-zero integer counts."""
    from oracle import batch as ob, ref_planner as rp
    obst = [[(10, 40), (30, 40), (30, 90), (10, 90)], [(480, 100), (499, 120), (470, 150)],
            [(240, 0.5), (260, 0.5), (265, 6), (250, 11), (235, 6)]]
    para = [(0, 0), (500, 0), (580, 200), (80, 200)]
    fields = [RECT, para]
    cand = fc.make_candidates(2, radii=[6.0, 8.0], start_corners=[0, 3])
    res = fc.plan_batch(fields, fc.VehicleParams(), cand, obstacles=[obst, obst], coverage=False)
    for b in range(len(res.summary)):
        o = ob.evaluate_candidate(fields[int(cand["field_id"][b])], rp.VehicleParams(), R=cand["R"][b],
                                  start_corner=int(cand["start_corner"][b]), obstacles=obst, coverage=False)
        _summary_vs_oracle(res.summary[b], o, coverage=False)
    assert res.summary["n_obstacle_viol"].min() > 0
    assert res.summary["n_boundary_viol"][len(res.summary) // 2:].min() > 0   # parallelogram overshoot
    assert (res.summary["n_boundary_viol"][:len(res.summary) // 2] == 0).all()  # rectangle: README "0 points"


def test_batch_config3_parallelograms_headings_vs_oracle(fc):
    """BASELINE config 3 in miniature: seeded tilted parallelograms x headings; counts exact."""
    from oracle import batch as ob, ref_planner as rp
    rng = np.random.default_rng(1234)
    F = 6
    fields = []
    for _ in range(F):
        L, Wd = rng.uniform(200, 800), rng.uniform(100, 400)
        sx, phi = rng.uniform(-0.4, 0.4) * Wd, rng.uniform(0, np.pi)
        o = rng.uniform(0, 5000, 2)
        q = np.array([(0, 0), (L, 0), (L + sx, Wd), (sx, Wd)])
        rot = np.array([[np.cos(phi), -np.sin(phi)], [np.sin(phi), np.cos(phi)]])
        fields.append(q @ rot.T + o)
    fields = np.array(fields)
    heads = np.deg2rad([0.0, 17.0, 45.0, 90.0, 133.0, 179.0])
    cand = fc.make_candidates(F, headings=heads)
    veh = fc.VehicleParams()
    res = fc.plan_batch(fields, veh, cand, outputs="paths", grid_h=0.1)
    oveh = rp.VehicleParams()
    for b in range(len(res.summary)):
        f = int(cand["field_id"][b])
        o = ob.evaluate_candidate(fields[f], oveh, heading=float(cand["heading"][b]), keep_paths=True,
                                  coverage=(b % 6 == 0))
        _summary_vs_oracle(res.summary[b], o, coverage=(b % 6 == 0))
        if not o["status"]:
            p, s, _ = res.path(b)
            assert np.abs(p - o["path"]).max() <= TIGHT
            assert np.abs(s - o["speeds"]).max() <= TIGHT
    # per-field argmin is local to each field's 6 headings
    cost = res.summary["len_main"] + res.summary["len_head"]
    for f in range(F):
        assert int(res.best_cand[f]) == f * 6 + int(np.argmin(cost[f * 6:(f + 1) * 6]))


def test_degenerate_candidates_status(fc):
    """mlp3:597-598 (headland too wide) and mlp3:967-969 (loop skipped) become status bits."""
    from oracle import batch as ob, ref_planner as rp
    fields = [[(0, 0), (30, 0), (30, 15), (0, 15)], RECT]
    cand = fc.make_candidates(2, radii=[8.0, 40.0])
    res = fc.plan_batch(fields, fc.VehicleParams(), cand)
    for b in range(4):
        o = ob.evaluate_candidate(fields[int(cand["field_id"][b])], rp.VehicleParams(), R=cand["R"][b],
                                  coverage=False)
        assert int(res.summary["status"][b]) == o["status"]
    assert res.summary["status"][0] != 0 and res.summary["status"][2] == 0
    with pytest.raises(ValueError):
        fc.TwoLayerPathPlannerV37(fc.VehicleParams(), field_length=30, field_width=15).plan()


def test_full_config2_properties(fc):
    """BASELINE config 2 at full size (4096 candidates): summary-only and paths mode agree bit for
    bit, the run is idempotent, counts obey their closed forms (SURVEY.md App. B) and the path
    buffers are consistent with the summaries."""
    import torch
    veh = fc.VehicleParams()
    radii = np.linspace(5.0, 12.0, 1024)
    cand = fc.make_candidates(1, radii=radii, start_corners=[0, 1, 2, 3])
    a = fc.plan_batch([RECT], veh, cand, obstacles=[OBST2], outputs="summary")
    b = fc.plan_batch([RECT], veh, cand, obstacles=[OBST2], outputs="paths")
    assert a.summary.tobytes() == b.summary.tobytes()
    c = fc.plan_batch([RECT], veh, cand, obstacles=[OBST2], outputs="summary")
    assert a.summary.tobytes() == c.summary.tobytes()
    s = a.summary
    assert (s["status"] == 0).all()
    P = s["n_passes"]
    assert (s["n_main"] == 2 * P + 20 * (P - 1)).all()
    K = np.ceil(cand["R"] / 3.2).astype(int)
    assert (s["n_loops"] == K).all()
    assert (s["n_head"] == 126 * K + s["n_rev"].sum(1)).all()
    assert (s["corner_g"] == (2 * cand["R"] / 0.1).astype(int)).all()
    assert (s["n_accel_viol"] == 0).all()                      # safety_factor < 1 (Q16)
    assert (s["cov_total"] > 0).all() and (s["cov_cells"] <= s["cov_total"]).all()
    assert (s["corner_after"] >= s["corner_before"]).all()
    # start corner only permutes the visiting order: total band cells depend on R alone
    tot = s["cov_total"].reshape(1024, 4)
    assert (tot == tot[:, :1]).all()
    # offsets are the prefix sum of the counts
    n = s["n_main"] + s["n_head"]
    assert (np.diff(b.offsets) == n).all()
    # path length recomputed from the materialised points equals the summary (checksum of checksums)
    d = b.d_path[1:] - b.d_path[:-1]
    seg = torch.sqrt((d * d).sum(1)).cpu().numpy()
    for k in (0, 1234, 4095):
        o0, nm, nt = int(b.offsets[k]), int(s["n_main"][k]), int(n[k])
        np.testing.assert_allclose(seg[o0:o0 + nm - 1].sum(), s["len_main"][k], rtol=1e-12)
        np.testing.assert_allclose(seg[o0 + nm:o0 + nt - 1].sum(), s["len_head"][k], rtol=1e-12)
    assert torch.isfinite(b.d_speeds).all()
    assert float(b.d_speeds.min()) > 0 and float(b.d_speeds.max()) <= 15.0


def test_speed_planner_random_paths_vs_oracle(fc):
    """A7 on caller-supplied paths: random walks with duplicates, sharp turns and long jumps."""
    from oracle import ref_planner as rp
    rng = np.random.default_rng(5)
    veh = fc.VehicleParams()
    oveh = rp.VehicleParams()
    pl = fc.TwoLayerPathPlannerV37(veh, field_length=500, field_width=200)
    for n in (3, 17, 256, 257, 1000, 5000):
        step = rng.normal(0, 1.0, size=(n, 2)) * rng.choice([0.0, 0.3, 1.0, 25.0], size=(n, 1), p=[0.1, 0.3, 0.5, 0.1])
        path = np.cumsum(step, axis=0) + 1000.0
        speeds = rng.choice([2.5, 4.0, 9.0, 15.0], size=n)
        got = pl._apply_curvature_based_speed_limit(path, speeds)
        want = rp.speed_plan(path, speeds, oveh)
        assert np.abs(got - want).max() <= 1e-9, n
        cc = pl.verify_curvature_constraints(path, got)
        oc = rp.verify_curvature_constraints(path, want, oveh)
        assert cc["accel_violations"] == oc["accel_violations"]
        np.testing.assert_allclose(cc["max_curvature"], oc["max_curvature"], rtol=1e-9)
        np.testing.assert_allclose(pl._calculate_path_length(path), rp.path_length(path), rtol=1e-12)
        np.testing.assert_allclose(pl._calculate_work_time(path, got), rp.work_time(path, want), rtol=1e-9)
    # ragged edge cases of the reference: fewer than 3 points are returned untouched (mlp3:480-481)
    p2 = np.array([[0.0, 0.0], [1.0, 0.0]])
    s2 = np.array([9.0, 9.0])
    assert pl._apply_curvature_based_speed_limit(p2, s2) is s2
    assert pl.verify_curvature_constraints(p2, s2) == {'max_curvature': 0, 'violations': 0, 'pass': True}
    assert pl._calculate_path_length(p2[:1]) == 0.0


def test_raster_window_random_polylines_vs_oracle(fc):
    """A10 on caller-supplied polylines vs the brute-force integer oracle (bit-exact grids)."""
    from oracle import raster
    rng = np.random.default_rng(11)
    pl = fc.TwoLayerPathPlannerV37(fc.VehicleParams(), field_length=500, field_width=200)
    R, W = 8.0, 3.2
    g = int(2 * R / 0.1)
    for trial in range(6):
        corner = (float(rng.uniform(0, 400)), float(rng.uniform(0, 150)))
        ci = trial % 4
        n1, n2 = int(rng.integers(2, 40)), int(rng.integers(2, 40))
        base = np.array(corner) + rng.uniform(-4, 12, 2)
        turn = base + np.cumsum(rng.normal(0, 1.5, size=(n1, 2)), axis=0)
        rev = turn[-1] + np.cumsum(rng.normal(0, 1.0, size=(n2, 2)), axis=0)
        if trial == 3:
            rev[5] = rev[4]                                   # zero-length segment
        got = pl.verify_corner_coverage_grid_based(corner, ci, turn, rev)
        ox = corner[0] if ci in (0, 3) else corner[0] - 2 * R
        oy = corner[1] if ci in (0, 1) else corner[1] - 2 * R
        c1, bits = raster.raster_window(turn, W / 2, (ox, oy), 0.1, g, g)
        c2, bits = raster.raster_window(rev, W / 2, (ox, oy), 0.1, g, g, bits)
        assert (got["cells_before"], got["cells_after"]) == (c1, c2)
        want = np.unpackbits(bits, bitorder="little")[:g * g].reshape(g, g).astype(bool)
        assert np.array_equal(got["grid"], want)


def test_tour_lengths_vs_reference_golden_and_oracle(fc, golden_dir):
    from oracle import raster
    z = np.load(os.path.join(golden_dir, "ga_tours.npz"))
    d, f = fc.tour_lengths(z["D"], z["pop"], return_fitness=True)
    assert np.array_equal(d, z["dist"])                       # sequential FP64 sum: bit-exact
    assert np.array_equal(f, z["fitness"])
    # BASELINE config 4: 200 fields + depot, population 8192
    rng = np.random.default_rng(42)
    pos = np.vstack([[100.0, 100.0], rng.uniform(0, 5000, size=(200, 2))])
    D = np.sqrt(((pos[:, None, :] - pos[None, :, :]) ** 2).sum(-1))
    prng = np.random.default_rng(7)
    pop = np.array([prng.permutation(201) for _ in range(8192)], dtype=np.int32)
    got = fc.tour_lengths(D, pop)
    assert np.array_equal(got, raster.tour_lengths(D, pop))
    # invariances: rotating or reversing a closed tour keeps its length up to summation order
    np.testing.assert_allclose(fc.tour_lengths(D, np.roll(pop[:64], 5, axis=1)), got[:64], rtol=1e-12)
    np.testing.assert_allclose(fc.tour_lengths(D, pop[:64, ::-1].copy()), got[:64], rtol=1e-12)
    # ragged sizes
    for n, m in ((2, 1), (3, 5), (33, 129), (64, 128)):
        Dn = D[:n, :n].copy()
        pn = np.array([prng.permutation(n) for _ in range(m)], dtype=np.int32)
        assert np.array_equal(fc.tour_lengths(Dn, pn), raster.tour_lengths(Dn, pn))


def test_ga_solver_improves(fc):
    rng = np.random.default_rng(3)
    pos = rng.uniform(0, 1000, size=(30, 2))
    D = np.sqrt(((pos[:, None, :] - pos[None, :, :]) ** 2).sum(-1))
    solver = fc.GeneticAlgorithmSolver(fc.GAConfig(population_size=120, max_generations=150), seed=1)
    route, stats = solver.solve(D, verbose=False)
    assert sorted(route) == list(range(30)) and route[0] == 0
    rand = fc.tour_lengths(D, np.array([rng.permutation(30) for _ in range(200)], dtype=np.int32)).mean()
    assert stats["best_distance"] < 0.6 * rand
    assert abs(stats["best_distance"] - fc.tour_lengths(D, np.array([route], dtype=np.int32))[0]) < 1e-6


def test_config5_large_field_fine_grid(fc):
    """BASELINE config 5 geometry (2 km x 1 km, h = 0.05 m): one candidate against the oracle,
    and a closed form for the number of band cells."""
    from oracle import batch as ob, ref_planner as rp
    big = [(0, 0), (2000, 0), (2000, 1000), (0, 1000)]
    cand = fc.make_candidates(1, radii=[8.0, 5.0], start_corners=[0, 2])
    res = fc.plan_batch([big], fc.VehicleParams(), cand, grid_h=0.05)
    s = res.summary
    assert (s["status"] == 0).all()
    assert int(s["n_main"][0]) == 6756 and int(s["n_head"][0]) == 435           # SURVEY.md App. B
    assert int(s["cov_total"][0]) == 19097600                                    # SURVEY.md §8(d)
    o = ob.evaluate_candidate(big, rp.VehicleParams(), R=8.0, start_corner=0, grid_h=0.05)
    _summary_vs_oracle(s[0], o)


def test_band_zoned_equals_row_tiled_and_oracle(fc):
    """The coverage kernel evaluates the headland band of fields with axis-aligned straights "zoned"
    (bitmap around the corners + closed-form rows, DESIGN.md §3.3) and every other field row-tiled.
    Both must give the same integers: compared here on BASELINE config 2 at full size, config 5
    geometry, small / offset / sheared / mixed fields and several grid pitches, with a sample of every
    case against the brute-force oracle."""
    from field_coverage_path_planning_b200 import _lib
    from oracle import batch as ob, ref_planner as rp
    h = _lib.handle(0)
    # mode bits other than 0, 1, 6 and 7 are rejected (bit 2 once selected a fused plan + coverage kernel)
    for bad in (4, 5, 8, 16, 32):
        assert h.lib.fcpp_set_cover_mode(h.h, bad) == -1, bad  # FCPP_ERR_INVALID

    def both(fields, veh, cand, modes=(1, 2, 3, 64, 128, 65, 129), **kw):
        """mode bit 0: row-tiled band only; bit 1: no coverage de-duplication (on by default in batches with a
        heading or start-corner axis: corner windows shared per (field, R), bands per (field, R, corner)); bits 6 / 7:
        one coverage CTA per candidate / the persistent work list over the representatives, whichever the batch
        would choose (a heading search takes the work list, every other de-duplicated batch one CTA per candidate)"""
        auto = fc.plan_batch(fields, veh, cand, **kw).summary
        for mode in modes:
            try:
                h.check(h.lib.fcpp_set_cover_mode(h.h, mode))
                other = fc.plan_batch(fields, veh, cand, **kw).summary
            finally:
                h.check(h.lib.fcpp_set_cover_mode(h.h, 0))
            assert auto.tobytes() == other.tobytes(), mode
        return auto

    veh = fc.VehicleParams()
    cand = fc.make_candidates(1, radii=np.linspace(5.0, 12.0, 1024), start_corners=[0, 1, 2, 3])
    s = both([RECT], veh, cand, obstacles=[OBST2])
    assert (s["status"] == 0).all() and (s["cov_cells"] > 0).all()
    # config 5 geometry, radii across the range (zones larger than one tile at R = 12)
    big = [(0, 0), (2000, 0), (2000, 1000), (0, 1000)]
    both([big], veh, fc.make_candidates(1, radii=[5.0, 7.3, 9.6, 12.0], start_corners=[0, 1, 2, 3]), grid_h=0.05)
    # small, offset, sheared (horizontal chains only), tilted (no chains) and non-origin fields in one batch
    fields = [
        [(0, 0), (60, 0), (60, 45), (0, 45)],
        [(1000.3, 2000.7), (1180.3, 2000.7), (1180.3, 2075.7), (1000.3, 2075.7)],
        [(0, 0), (500, 0), (580, 200), (80, 200)],
        [(0, 0), (300, 40), (280, 190), (-20, 150)],
        [(-250.05, -100.02), (249.95, -100.02), (249.95, 99.98), (-250.05, 99.98)],
        [(0, 0), (45, 0), (45, 300), (0, 300)],
    ]
    cand = fc.make_candidates(len(fields), radii=[5.0, 6.4, 8.0, 11.0], start_corners=[0, 1, 2, 3])
    for gh in (0.1, 0.05, 0.25):
        s = both(fields, veh, cand, grid_h=gh)
    for wv in (2.0, 4.5):
        both(fields, fc.VehicleParams(working_width=wv), cand)
    # heading search (BASELINE config 3 in small): the coverage of a field does not depend on the
    # heading, so it is rasterised once per (field, R, start corner) and shared — same integers as
    # rasterising every candidate (mode 2), also with duplicated and dead candidates in the batch
    hc = fc.make_candidates(len(fields), headings=np.deg2rad(np.arange(0.0, 180.0, 15.0)), radii=[6.0, 8.0],
                            start_corners=[0, 2])
    s = both(fields, veh, hc)
    per = s["cov_cells"].reshape(len(fields), 12, 4)
    assert (per == per[:, :1, :]).all() and (s["cov_cells"] > 0).all()
    tiny = [[(0, 0), (30, 0), (30, 15), (0, 15)]] + fields[:2]       # field 0: inset empty -> dead candidates
    tc = fc.make_candidates(3, headings=[0.0, 0.3], radii=[8.0, 8.0], start_corners=[1])
    s = both(tiny, veh, tc, modes=(2, 64, 128))
    assert (s["status"][:4] != 0).all() and (s["cov_total"][:4] == 0).all() and (s["cov_total"][4:] > 0).all()
    # many narrow loops: K = 12, 15 and 16 headland loops (48-64 chain rectangles = the cap)
    narrow = [[(0, 0), (120, 0), (120, 90), (0, 90)]]
    s = both(narrow, fc.VehicleParams(working_width=0.8), fc.make_candidates(1, radii=[9.6, 12.0, 12.8], start_corners=[0, 3]))
    assert (s["status"] == 0).all() and list(s["n_loops"][::2]) == [12, 15, 16]
    o = ob.evaluate_candidate(narrow[0], rp.VehicleParams(working_width=0.8), R=12.8, start_corner=3)
    assert int(s["cov_total"][5]) == o["cov_total"] and int(s["cov_cells"][5]) == o["cov_cells"]
    # the oracle (brute force per cell) on a sample of the last batch set-up
    s = both(fields, veh, cand)
    for b in range(0, len(s), 7):
        if s["status"][b]:
            continue
        o = ob.evaluate_candidate(fields[int(cand["field_id"][b])], rp.VehicleParams(), R=cand["R"][b],
                                  start_corner=int(cand["start_corner"][b]))
        assert int(s["cov_total"][b]) == o["cov_total"] and int(s["cov_cells"][b]) == o["cov_cells"], b


def test_integration_md_ctypes_stub_runs(fc):
    """The reference-side ctypes stub printed in INTEGRATION.md is executed verbatim (only the
    library path is made absolute) and must reproduce the drop-in planner's result."""
    import re
    import types
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    md = open(os.path.join(root, "INTEGRATION.md"), encoding="utf-8").read()
    code = re.search(r"```python\n# fcpp_binding\.py.*?\n(.*?)```", md, re.S).group(1)
    code = code.replace('"libfcpp.so"', repr(os.path.join(root, "field_coverage_path_planning_b200", "libfcpp.so")))
    ns = {}
    exec(compile(code, "INTEGRATION.md", "exec"), ns)
    verts = [(0, 0), (500, 0), (580, 200), (80, 200)]
    ref = fc.TwoLayerPathPlannerV37(fc.VehicleParams(), field_vertices=verts)
    want = ref.plan_complete_coverage()
    shim = types.SimpleNamespace(vehicle=fc.VehicleParams(), field_vertices=verts, field_length=ref.field_length,
                                 field_width=ref.field_width, corner_angles=ref.corner_angles,
                                 _calculate_rotation_angle=lambda: np.arctan2(0.0, 500.0))
    (mp, ms), (hp, hs) = ns["plan_on_gpu"](shim, 0)
    assert np.array_equal(mp, want["main_work"]["path"]) and np.array_equal(hp, want["headland"]["path"])
    assert np.array_equal(ms, want["main_work"]["speeds"]) and np.array_equal(hs, want["headland"]["speeds"])


def test_plan_longer_than_shared_memory_staging(fc):
    """A 5 km x 3 km field has ~20 000 points per plan — more than fits the on-chip staging; such
    plans run through the HBM-staged variant of the same kernel.  Mixed batch (one small, one huge)."""
    from oracle import batch as ob, ref_planner as rp
    huge = [(0, 0), (5000, 0), (5000, 3000), (0, 3000)]
    fields = [RECT, huge]
    cand = fc.make_candidates(2, start_corners=[0, 2])
    res = fc.plan_batch(fields, fc.VehicleParams(), cand, outputs="paths", grid_h=0.5)
    assert (res.summary["status"] == 0).all()
    assert int(res.summary["n_main"][2]) > 20000
    for b in range(4):
        o = ob.evaluate_candidate(fields[int(cand["field_id"][b])], rp.VehicleParams(),
                                  start_corner=int(cand["start_corner"][b]), grid_h=0.5, keep_paths=True)
        _summary_vs_oracle(res.summary[b], o)
        p, s, _ = res.path(b)
        assert np.abs(p - o["path"]).max() <= TIGHT and np.abs(s - o["speeds"]).max() <= TIGHT
    # caller-supplied path longer than the staging (verify_curvature_constraints on 30 000 points)
    rng = np.random.default_rng(9)
    path = np.cumsum(rng.normal(0, 1.0, size=(30000, 2)), axis=0)
    speeds = rng.choice([4.0, 9.0, 15.0], size=len(path))
    pl = fc.TwoLayerPathPlannerV37(fc.VehicleParams(), field_length=500, field_width=200)
    got = pl._apply_curvature_based_speed_limit(path, speeds)
    assert np.abs(got - rp.speed_plan(path, speeds, rp.VehicleParams())).max() <= 1e-9


def test_edge_cases(fc):
    """Empty batch, fields without candidates, invalid grid size."""
    res = fc.plan_batch([RECT], fc.VehicleParams(), {"field_id": np.zeros(0, dtype=np.int32)})
    assert len(res.summary) == 0 and int(res.best_cand[0]) == -1 and np.isinf(res.best_cost[0])
    res = fc.plan_batch([RECT, RECT], fc.VehicleParams(), {"field_id": np.array([1], dtype=np.int32)}, outputs="paths")
    assert int(res.best_cand[0]) == -1 and int(res.best_cand[1]) == 0 and res.offsets[-1] == 1691
    with pytest.raises(fc.FcppError):
        fc.plan_batch([RECT], fc.VehicleParams(), grid_h=0.0333)          # not an even multiple of 1e-4 m
    res = fc.plan_batch([RECT], fc.VehicleParams(), coverage=False)
    assert int(res.summary["cov_total"][0]) == 0 and int(res.summary["n_main"][0]) == 1256
    # the same edge cases in factored form and through the asynchronous call: an empty range of the product, a
    # one-candidate product, winners of an empty batch
    ax = fc.candidate_axes(1, radii=[7.0, 8.0], start_corners=[0, 1])
    for outputs in ("summary", "paths"):
        e = fc.plan_batch([RECT], fc.VehicleParams(), dict(ax, range=(2, 2)), outputs=outputs, winners=True, wait=False).result()
        assert len(e.summary) == 0 and int(e.best_cand[0]) == -1 and e.winner_paths == {}
        one = fc.plan_batch([RECT], fc.VehicleParams(), dict(ax, range=(3, 4)), outputs=outputs, winners=True)
        full = fc.plan_batch([RECT], fc.VehicleParams(), ax, outputs=outputs)
        assert one.summary.tobytes() == full.summary[3:4].tobytes() and int(one.best_cand[0]) == 0
        assert len(one.winner_paths[0][0]) == int(one.summary["n_main"][0] + one.summary["n_head"][0])
    with pytest.raises(fc.FcppError):
        fc.plan_batch([RECT], fc.VehicleParams(), ax, device="cpu")


def test_clothoid_turn_model_vs_scipy_oracle(fc):
    """Row A16 (opt-in, no reference code): clothoid -> arc -> clothoid turns with device-side
    Fresnel series vs oracle/clothoid.py (scipy.special.fresnel).  Parity with the reference is
    unpinned; the layout (point counts) must equal the arc model's."""
    from oracle import batch as ob, ref_planner as rp
    para = [(100, 50), (600, 120), (640, 330), (140, 260)]
    fields = [RECT, para]
    cand = fc.make_candidates(2, radii=[6.0, 8.0], start_corners=[0, 3])
    for lam in (0.5, 1.0, 0.2):
        res = fc.plan_batch(fields, fc.VehicleParams(), cand, outputs="paths", turn_model="clothoid", clothoid_share=lam)
        arc = fc.plan_batch(fields, fc.VehicleParams(), cand, coverage=False)
        assert (res.summary["n_main"] == arc.summary["n_main"]).all()
        for b in range(len(res.summary)):
            o = ob.evaluate_candidate(fields[int(cand["field_id"][b])], rp.VehicleParams(), R=cand["R"][b],
                                      start_corner=int(cand["start_corner"][b]), keep_paths=True,
                                      turn_model="clothoid", clothoid_share=lam, coverage=(b % 3 == 0))
            _summary_vs_oracle(res.summary[b], o, coverage=(b % 3 == 0))
            p, s, _ = res.path(b)
            assert np.abs(p - o["path"]).max() <= TIGHT
            assert np.abs(s - o["speeds"]).max() <= 1e-7
    # the clothoid turn lowers the peak curvature seen by the speed planner
    assert res.summary["max_curvature"].max() <= arc.summary["max_curvature"].max()
    pl = fc.TwoLayerPathPlannerV37(fc.VehicleParams(), field_length=500, field_width=200, turn_model="clothoid")
    r = pl.plan()
    assert len(r["main_work"]["path"]) == 1256
    with pytest.raises(ValueError):
        fc.plan_batch(fields, fc.VehicleParams(), cand, turn_model="bezier")


def test_select_merge_at_k1_vs_numpy_rule(fc):
    """fcpp_field_select_merge at k = 1 (the multi-GPU merge of the per-field argmin after ONE all-gather): lowest
    cost wins, ties go to the lowest global candidate index, ranks without a candidate (-1) are skipped."""
    import ctypes as C
    import torch
    from field_coverage_path_planning_b200 import _lib
    rng = np.random.default_rng(9)
    h = _lib.handle(0)
    for world, F in ((1, 1), (2, 7), (3, 1000), (8, 4096)):
        cost = rng.integers(0, 6, size=(world, F)).astype(np.float64) * 0.5      # many ties
        cand = rng.integers(0, 10 ** 6, size=(world, F)).astype(np.int64)
        none = rng.random((world, F)) < 0.3
        cand[none] = -1
        cost[none] = np.inf
        if F > 5:
            cand[:, 3] = -1                                                        # nobody has field 3
            cost[:, 3] = np.inf
        g = np.concatenate([cost.view(np.int64), cand], axis=1)                    # [world][2F] words
        dg = torch.from_numpy(np.ascontiguousarray(g)).cuda()
        oc = torch.empty(F, dtype=torch.float64, device="cuda")
        ob_ = torch.empty(F, dtype=torch.int64, device="cuda")
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        h.check(h.lib.fcpp_field_select_merge(h.h, dg.data_ptr(), world, F, 1, oc.data_ptr(), ob_.data_ptr(), st))
        want_c, want_i = np.full(F, np.inf), np.full(F, -1, dtype=np.int64)
        for f in range(F):
            for r in range(world):
                if cand[r, f] >= 0 and (want_i[f] < 0 or cost[r, f] < want_c[f] or
                                        (cost[r, f] == want_c[f] and cand[r, f] < want_i[f])):
                    want_c[f], want_i[f] = cost[r, f], cand[r, f]
        assert np.array_equal(oc.cpu().numpy(), want_c) and np.array_equal(ob_.cpu().numpy(), want_i)


def test_distributed_plan_batch_world1_nccl(fc):
    """plan_batch(distributed=True) through a world-size-1 NCCL group == the single-process result
    (all-gather + merge kernel + winner-record exchange on the CUDA path)."""
    import torch
    import torch.distributed as dist
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29533")
    created = not dist.is_initialized()
    if created:
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        rect = [(0, 0), (500, 0), (500, 200), (0, 200)]
        small = [(0, 0), (100, 0), (100, 80), (0, 80)]
        tiny = [(0, 0), (12, 0), (12, 9), (0, 9)]                                  # no valid candidate
        cand = fc.make_candidates(3, radii=[5.0, 8.0, 11.0], start_corners=[0, 1, 2, 3])
        a = fc.plan_batch([rect, small, tiny], fc.VehicleParams(), cand, outputs="summary", device="cuda:0")
        b = fc.plan_batch([rect, small, tiny], fc.VehicleParams(), cand, outputs="summary", device="cuda:0",
                          distributed=True)
        assert np.array_equal(a.best_cand, b.best_cand) and np.array_equal(a.best_cost, b.best_cost)
        assert a.best_cand[2] == -1 and np.isinf(a.best_cost[2])
        win = b.extras["winner_summary"]
        for f in range(2):
            assert win[f].tobytes() == a.summary[a.best_cand[f]].tobytes()
    finally:
        if created:
            dist.destroy_process_group()


def test_big_plan_workspace_survives_layout_passes(fc):
    """Regression (ADVICE r1): the HBM staging of plans longer than shared memory (launch_big) is owned by the
    plan launcher alone — a layout pass that grows the scan workspace in between must not free it.  Sequence:
    long-path speed planning -> plan_batch on a fresh, larger batch -> long-path speed planning again."""
    from oracle import ref_planner as rp
    rng = np.random.default_rng(21)
    pl = fc.TwoLayerPathPlannerV37(fc.VehicleParams(), field_length=500, field_width=200)
    path = np.cumsum(rng.normal(0, 1.0, size=(12000, 2)), axis=0)
    speeds = rng.choice([4.0, 9.0, 15.0], size=len(path))
    want = rp.speed_plan(path, speeds, rp.VehicleParams())
    assert np.abs(pl._apply_curvature_based_speed_limit(path, speeds) - want).max() <= 1e-9
    for n in (3, 9000, 40000):     # growing batches: every one re-allocates candidate records / scan workspace
        cand = fc.make_candidates(1, radii=np.linspace(5.0, 12.0, n))
        res = fc.plan_batch([RECT], fc.VehicleParams(), cand, coverage=False)
        assert (res.summary["status"] == 0).all()
        assert np.abs(pl._apply_curvature_based_speed_limit(path, speeds) - want).max() <= 1e-9


def test_verify_all_corners_returns_grid_and_origin(fc):
    """mlp3:1503-1510, :1561: every corner record of verify_all_corners_coverage carries 'grid' (occupancy after
    the reverse fill) and 'grid_origin' — written out by the coverage kernel, compared bit for bit with the
    brute-force oracle's window raster of the same verification polylines."""
    from oracle import raster, ref_planner as rp
    for R, L, Wd in ((8.0, 500, 200), (9.6, 300, 150), (5.0, 100, 80)):
        pl = fc.TwoLayerPathPlannerV37(fc.VehicleParams(min_turn_radius=R), field_length=L, field_width=Wd)
        r = pl.plan_complete_coverage()
        cov = pl.verify_all_corners_coverage(r["headland"])
        fs = rp.setup_field(rp.VehicleParams(min_turn_radius=R), field_length=L, field_width=Wd)
        g = int(2 * R / 0.1)
        for k, ((cx, cy), ci, arc, rev) in enumerate(rp.verification_corner_paths(fs)):
            c = cov["corners"][k]
            ox = cx if ci in (0, 3) else cx - 2 * R
            oy = cy if ci in (0, 1) else cy - 2 * R
            assert c["grid_origin"] == (ox, oy) and c["grid_resolution"] == 0.1
            n1, bits = raster.raster_window(arc, 3.2 / 2, (ox, oy), 0.1, g, g)
            n2 = n1
            if rev is not None and len(rev) > 0:
                n2, bits = raster.raster_window(rev, 3.2 / 2, (ox, oy), 0.1, g, g, bits)
            want = np.unpackbits(bits, bitorder="little")[:g * g].reshape(g, g).astype(bool)
            assert c["grid"].shape == (g, g) and c["grid"].dtype == bool
            assert np.array_equal(c["grid"], want), (R, k)
            assert (c["cells_before"], c["cells_after"]) == (n1, n2) and int(c["grid"].sum()) == n2


def test_factored_candidate_sets_identical_to_explicit_arrays(fc):
    """fcpp_batch with cand_field == NULL (batch.candidate_axes): the layout kernel decodes every candidate from
    its product index — summaries, offsets, paths, argmin and the winners' paths are byte-identical to the explicit
    per-candidate arrays of make_candidates; ranges of the product (multi-GPU shards) equal slices."""
    import torch
    veh = fc.VehicleParams()
    tiny = [(0, 0), (30, 0), (30, 15), (0, 15)]
    para = [(100, 50), (600, 120), (640, 330), (140, 260)]
    heads = np.deg2rad(np.arange(0.0, 180.0, 11.0))
    cases = [
        ([RECT], dict(radii=np.linspace(5.0, 12.0, 67), start_corners=[0, 1, 2, 3]), [OBST2], "paths"),
        ([RECT, tiny, para], dict(radii=[6.0, 8.0, 11.0], start_corners=[3, 0]), None, "paths"),
        ([para, RECT], dict(headings=heads, radii=[7.0, 9.0]), None, "summary"),
        ([para, RECT, tiny], dict(headings=heads, start_corners=[2, 1]), None, "summary"),
        ([para, RECT], dict(), None, "paths"),
        ([para, RECT], dict(start_corners=[1]), None, "summary"),
    ]
    for fields, axes, obst, outputs in cases:
        ex = fc.make_candidates(len(fields), **axes)
        ax = fc.candidate_axes(len(fields), **axes)
        a = fc.plan_batch(fields, veh, ex, obstacles=obst, outputs=outputs, winners=True)
        b = fc.plan_batch(fields, veh, ax, obstacles=obst, outputs=outputs, winners=True)
        assert a.summary.tobytes() == b.summary.tobytes()
        assert np.array_equal(a.best_cand, b.best_cand) and np.array_equal(a.best_cost, b.best_cost)
        assert b.extras["h2d_bytes"] < a.extras["h2d_bytes"] or len(ex["field_id"]) <= len(fields)
        if outputs == "paths":
            n = int(a.offsets[-1])
            assert np.array_equal(a.offsets, b.offsets)
            assert torch.equal(a.d_path[:n], b.d_path[:n]) and torch.equal(a.d_speeds[:n], b.d_speeds[:n])
        assert a.winner_paths.keys() == b.winner_paths.keys()
        for f in a.winner_paths:
            for x, y in zip(a.winner_paths[f], b.winner_paths[f]):
                assert np.array_equal(x, y)
        # a range of the product == the same slice of the explicit arrays (local indices, cand_base 0)
        n = len(ex["field_id"])
        lo, hi = n // 3, n - n // 4
        if hi > lo:
            s = fc.plan_batch(fields, veh, {k: v[lo:hi] for k, v in ex.items()}, obstacles=obst)
            r = fc.plan_batch(fields, veh, dict(ax, range=(lo, hi)), obstacles=obst, winners=True)
            assert s.summary.tobytes() == r.summary.tobytes() == a.summary[lo:hi].tobytes()
            assert np.array_equal(s.best_cand, r.best_cand)


def test_results_are_views_of_pinned_buffers_that_outlive_later_calls(fc):
    """The read-back hands out numpy views of pooled pinned buffers (no host copy): a result stays intact while any
    of its arrays is alive, however many calls follow, and its buffer is reused once the last view is gone."""
    import gc
    from field_coverage_path_planning_b200.batch import _ResultPool
    veh = fc.VehicleParams()
    ca = fc.candidate_axes(1, radii=np.linspace(5.0, 9.0, 33), start_corners=[0, 1])
    cb = fc.candidate_axes(1, radii=np.linspace(6.0, 12.0, 33), start_corners=[2, 3])
    a = fc.plan_batch([RECT], veh, ca, outputs="paths", winners=True)
    keep = (a.summary.copy(), a.best_cost.copy(), a.offsets.copy(), a.winner_paths[0][0].copy(), a.winner_paths[0][1].copy())
    only_summary = a.summary            # one array of the result kept, the BatchResult itself dropped below
    wp = a.winner_paths[0]
    del a
    others = [fc.plan_batch([RECT], veh, cb, outputs="paths", winners=True) for _ in range(3)]
    assert only_summary.tobytes() == keep[0].tobytes()
    assert np.array_equal(wp[0], keep[3]) and np.array_equal(wp[1], keep[4])
    assert others[0].summary.tobytes() == others[2].summary.tobytes() != keep[0].tobytes()
    del others, only_summary, wp
    gc.collect()
    n_before = len(_ResultPool._bufs)
    for _ in range(4):
        r = fc.plan_batch([RECT], veh, ca, outputs="paths", winners=True)
        assert r.summary.tobytes() == keep[0].tobytes() and np.array_equal(r.offsets, keep[2])
        del r
    assert len(_ResultPool._bufs) <= n_before        # steady state: no new pinned allocations


def test_pipelined_and_speculatively_sized_batches_identical(fc):
    """plan_batch(..., wait=False) / PendingBatch.result() with several batches in flight, and launches sized from
    remembered batches of the same shape (no layout read-back): byte-identical to the synchronous, layout-sized
    call; a batch that does not fit the remembered sizes is detected through the status flags and repeated."""
    import torch
    from field_coverage_path_planning_b200 import batch as B
    veh = fc.VehicleParams()
    B._Hints._c.clear()
    small = fc.candidate_axes(1, radii=np.linspace(5.0, 6.0, 64), start_corners=[0, 1, 2, 3])
    big = fc.candidate_axes(1, radii=np.linspace(11.0, 12.0, 64), start_corners=[0, 1, 2, 3])     # more headland loops
    heads = fc.candidate_axes(2, headings=np.deg2rad(np.arange(0.0, 180.0, 7.0)))
    para = [(100, 50), (600, 120), (640, 330), (140, 260)]
    for outputs in ("paths", "summary"):
        ref_small = fc.plan_batch([RECT], veh, small, obstacles=[OBST2], outputs=outputs, winners=True)     # sized by its layout
        assert not ref_small.extras["speculative"]
        again = fc.plan_batch([RECT], veh, small, obstacles=[OBST2], outputs=outputs, winners=True)         # remembered sizes
        assert again.extras["speculative"]
        assert again.summary.tobytes() == ref_small.summary.tobytes()
        assert np.array_equal(again.winner_paths[0][0], ref_small.winner_paths[0][0])
        # same shape, longer plans: the remembered sizes are too small -> flagged -> repeated from its own layout
        r_big = fc.plan_batch([RECT], veh, big, obstacles=[OBST2], outputs=outputs, winners=True)
        assert not r_big.extras["speculative"] and (r_big.summary["status"] == 0).all()
        assert r_big.summary["n_head"].max() > ref_small.summary["n_head"].max()
        B._Hints._c.clear()
        want_big = fc.plan_batch([RECT], veh, big, obstacles=[OBST2], outputs=outputs, winners=True)
        assert want_big.summary.tobytes() == r_big.summary.tobytes()
        if outputs == "paths":
            n = int(want_big.offsets[-1])
            assert np.array_equal(want_big.offsets, r_big.offsets) and torch.equal(want_big.d_path[:n], r_big.d_path[:n])
    # several batches in flight, collected out of order
    B._Hints._c.clear()
    jobs = [([RECT], small, [OBST2], "paths"), ([para, RECT], heads, None, "summary"), ([RECT], big, [OBST2], "paths"),
            ([RECT], small, [OBST2], "summary")]
    want = [fc.plan_batch(f, veh, c, obstacles=o, outputs=out, winners=True) for f, c, o, out in jobs]
    for rounds in range(2):          # second round: every shape is remembered
        pend = [fc.plan_batch(f, veh, c, obstacles=o, outputs=out, winners=True, wait=False) for f, c, o, out in jobs]
        assert all(isinstance(p, B.PendingBatch) for p in pend)
        for k in (2, 0, 3, 1):
            got = pend[k].result()
            assert got is pend[k].result()
            assert got.summary.tobytes() == want[k].summary.tobytes()
            assert np.array_equal(got.best_cand, want[k].best_cand) and np.array_equal(got.best_cost, want[k].best_cost)
            assert got.winner_paths.keys() == want[k].winner_paths.keys()
            for f in got.winner_paths:
                assert np.array_equal(got.winner_paths[f][0], want[k].winner_paths[f][0])
                assert np.array_equal(got.winner_paths[f][1], want[k].winner_paths[f][1])


def test_omega_skip_row_pattern_vs_oracle(fc):
    """Ω-type skip-row main work (opt-in, the reference has only the label, mlp3:312-320; build-defined, parity
    unpinned): device vs oracle/ref_planner.omega_* — layout counts exact, points <= 1e-9 m, speeds, lengths, times,
    violation counts; rectangles (axis-aligned chains), a sheared field, a heading axis, radii with bulb turns
    (gap < 2R) and plain half circles; summary-only == paths mode; the default pattern is untouched."""
    from oracle import batch as ob, ref_planner as rp
    para = [(100, 50), (600, 120), (640, 330), (140, 260)]
    small = [(0, 0), (100, 0), (100, 80), (0, 80)]
    fields = [RECT, para, small]
    veh = fc.VehicleParams()
    cand = fc.make_candidates(3, radii=[5.0, 8.0, 11.0], start_corners=[0, 1, 2, 3])
    res = fc.plan_batch(fields, veh, cand, outputs="paths", turn_model="omega")
    u = fc.plan_batch(fields, veh, cand, coverage=False)
    assert (res.summary["n_main"] == u.summary["n_main"]).all() and (res.summary["n_head"] == u.summary["n_head"]).all()
    assert (res.summary["len_main"] != u.summary["len_main"]).all()            # another main path ...
    assert res.summary["len_head"].tobytes() == u.summary["len_head"].tobytes()  # ... the same headland
    for b in range(0, len(res.summary), 1):
        o = ob.evaluate_candidate(fields[int(cand["field_id"][b])], rp.VehicleParams(), R=cand["R"][b],
                                  start_corner=int(cand["start_corner"][b]), keep_paths=True, turn_model="omega",
                                  coverage=(b % 5 == 0))
        _summary_vs_oracle(res.summary[b], o, coverage=(b % 5 == 0))
        p, s, n_main = res.path(b)
        assert np.abs(p - o["path"]).max() <= TIGHT
        assert np.abs(s - o["speeds"]).max() <= 1e-7
        # every turn connects the two swath ends it lies between (first / last sample ON them)
        m = p[:n_main].reshape(-1)[: (n_main // 22) * 44].reshape(-1, 22, 2)
        assert np.abs(m[:, 2] - m[:, 1]).max() <= 1e-9
        nxt = p[22:n_main:22]
        assert np.abs(m[:len(nxt), 21] - nxt).max() <= 1e-9
    summ = fc.plan_batch(fields, veh, cand, outputs="summary", turn_model="omega")
    assert summ.summary.tobytes() == res.summary.tobytes()
    # a heading axis (rotated swaths) in factored form
    ax = fc.candidate_axes(2, headings=np.deg2rad([0.0, 17.0, 90.0, 133.0]), radii=[7.0])
    hr = fc.plan_batch([para, RECT], veh, ax, outputs="paths", turn_model="omega")
    ex = fc.expand_axes(ax)
    for b in range(len(hr.summary)):
        o = ob.evaluate_candidate([para, RECT][int(ex["field_id"][b])], rp.VehicleParams(), R=7.0,
                                  heading=float(ex["heading"][b]), keep_paths=True, turn_model="omega", coverage=False)
        _summary_vs_oracle(hr.summary[b], o, coverage=False)
        assert np.abs(hr.path(b)[0] - o["path"]).max() <= TIGHT
    # drop-in class
    pl = fc.TwoLayerPathPlannerV37(fc.VehicleParams(), field_length=500, field_width=200, turn_model="omega")
    r = pl.plan()
    assert len(r["main_work"]["path"]) == 1256 and len(r["headland"]["path"]) == 435
    # the turns respect the turning radius (the reference's U 'turns' are half circles of radius R that do not connect)
    k = rp.curvatures(r["main_work"]["path"])
    assert k.max() <= 1.0 / 8.0 * 1.01
