"""The CPU oracle (oracle/) against the golden fixtures produced by executing the unmodified
reference (tests/golden/make_golden.py) and against the prose known-answers of the reference
(README.md:193-202, doc/V3.5.1 更新日志.md:108-114) — SURVEY.md §8(c)."""
import glob
import json
import os

import numpy as np
import pytest

from oracle import raster, ref_planner as rp

GOLD = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "ref_*.npz")))


def _load(path):
    z = np.load(path)
    meta = json.loads(str(z["meta"]))
    veh = rp.VehicleParams(**meta["vehicle"])
    kw = {k: v for k, v in meta["planner"].items()}
    for k in ("start_point", "end_point"):
        if kw.get(k) is not None:
            kw[k] = tuple(kw[k])
    if kw.get("field_vertices") is not None:
        kw["field_vertices"] = [tuple(v) for v in kw["field_vertices"]]
    return z, meta, veh, kw


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p)[4:-4] for p in GOLD])
def test_oracle_reproduces_reference(path):
    z, meta, veh, kw = _load(path)
    fs = rp.setup_field(veh, **kw)
    assert fs.field_shape == meta["field_shape"]
    assert fs.main_work_pattern == meta["pattern"]
    np.testing.assert_allclose(fs.corner_angles, meta["corner_angles"], rtol=0, atol=1e-12)
    o = rp.plan_complete_coverage(fs)
    # integer layout: bit-exact
    assert o["main_work"]["path"].shape == z["main_path"].shape
    assert o["headland"]["path"].shape == z["head_path"].shape
    # points: the restatement performs the same numpy operations -> <= 1e-12 m (tolerance of
    # north_star is 1e-4 m); speeds <= 1e-12 km/h (north_star: 1e-4 m/s)
    np.testing.assert_allclose(o["main_work"]["path"], z["main_path"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(o["headland"]["path"], z["head_path"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(o["main_work"]["speeds"], z["main_speeds"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(o["headland"]["speeds"], z["head_speeds"], rtol=0, atol=1e-12)
    for layer, key in (("main_work", "main_stats"), ("headland", "head_stats")):
        got = [o[layer]["stats"][k] for k in ("path_length_km", "time_hours", "avg_speed_kmh")]
        np.testing.assert_allclose(got, z[key], rtol=1e-13)
    allp = np.vstack([o["main_work"]["path"], o["headland"]["path"]])
    alls = np.concatenate([o["main_work"]["speeds"], o["headland"]["speeds"]])
    cc = rp.verify_curvature_constraints(allp, alls, veh)
    ref = z["curv"]
    np.testing.assert_allclose([cc["max_curvature"], cc["max_lateral_accel"], cc["max_jump"]],
                               [ref[0], ref[1], ref[4]], rtol=1e-12)
    assert cc["accel_violations"] == int(ref[2])
    assert cc["pass"] == bool(ref[5])
    for name, key in (("approach_path", "approach"), ("departure_path", "departure")):
        if len(z[key]):
            np.testing.assert_allclose(o[name], z[key], rtol=0, atol=1e-12)
        else:
            assert o[name] is None
    if "corner_cells_float" in z.files:
        got, g = raster.corner_coverage(fs)
        ref_cells = z["corner_cells_float"]
        # the reference decides "inside" in float64; the oracle in exact 1e-4 m fixed point (D5):
        # lattice points that sit on the buffer boundary may flip -> allow 2 cells per window
        assert np.max(np.abs(np.array(got) - ref_cells)) <= 2
        assert g * g == 25600 or meta["vehicle"]["min_turn_radius"] != 8.0
        # the averages verify_all_corners_coverage returns (mlp3:1573-1578), stored by make_golden.py
        avg = [100.0 * np.mean([c[k] for c in got]) / (g * g) for k in (0, 1)]
        np.testing.assert_allclose(avg + [avg[1] - avg[0]], z["corner_avg"], rtol=0, atol=100.0 * 2 / (g * g) + 1e-9)
    # headland coverage_rate of the reference (mlp3:1357-1371; the stand-in's D2 area) against the
    # integer raster of the band (D5): observed <= 2.5e-5 on rectangles, 1.3e-4 on the sheared field
    if max(fs.field_length, fs.field_width) <= 600:     # the 3500 m fields take 3.5 s each: covered by the GPU test
        total, cov = raster.band_coverage(fs, z["head_path"], 0.1)
        assert abs(cov / total - float(z["coverage_rate_sampled"])) <= 2e-4


def test_known_answers_readme():
    """README.md:193-202: 1256/435 points, 0 boundary violations, 0.0 % accel violations,
    headland coverage 100.0 %, corner gain +3.2 %."""
    veh = rp.VehicleParams(3.2, 8.0, 9.0, 15.0)
    fs = rp.setup_field(veh, field_length=500, field_width=200)
    o = rp.plan_complete_coverage(fs)
    assert len(o["main_work"]["path"]) == 1256
    assert len(o["headland"]["path"]) == 435
    allp = np.vstack([o["main_work"]["path"], o["headland"]["path"]])
    alls = np.concatenate([o["main_work"]["speeds"], o["headland"]["speeds"]])
    assert rp.boundary_violations(allp, fs.field_vertices) == 0
    assert rp.verify_curvature_constraints(allp, alls, veh)["accel_violations"] == 0
    cells, g = raster.corner_coverage(fs)
    b = np.array(cells)
    gain = (b[:, 1] - b[:, 0]).mean() / (g * g) * 100
    assert abs(gain - 3.2) < 0.1
    total, cov = raster.band_coverage(fs, o["headland"]["path"], 0.1)
    assert total == 1094400                      # SURVEY.md §8(d) G_band
    assert round(cov / total * 100, 1) == 100.0  # README "100.0 %"
    assert (total, cov) == (1094400, 1094113)    # regression KAT of the integer raster


def test_known_answers_changelog_v351():
    """doc/V3.5.1 更新日志.md:109-111: start (10,10) -> corner (4,4) at 8.5 m, approach 11.9 m,
    departure to (490,190) 515.2 m."""
    veh = rp.VehicleParams(3.2, 8.0, 9.0, 14.0)
    fs = rp.setup_field(veh, field_length=500, field_width=200, start_point=(10, 10), end_point=(490, 190))
    assert rp.select_best_start_corner(fs, fs.start_point) == 0
    assert round(float(np.hypot(10 - 4, 10 - 4)), 1) == 8.5
    o = rp.plan_complete_coverage(fs)
    assert round(rp.path_length(o["approach_path"]), 1) == 11.9
    assert round(rp.path_length(o["departure_path"]), 1) == 515.2


def test_knife_edges_q17():
    """SURVEY.md App. A Q17: FP64 knife edges of the integer layout."""
    assert int((200 - 2 * 7.2) / 3.2) == 57              # the closed form sits on a knife edge ...
    fs = rp.setup_field(rp.VehicleParams(3.2, 7.2), field_length=500, field_width=200)
    _, _, info = rp.plan_main_work(fs)
    # ... but the code path goes through the inset bounds: (200-7.2) - 7.2 = 185.60000000000002,
    # /3.2 -> 58.000000000000007 -> P = 59 (the reference run in ref_r72_knife.npz agrees: 1278 pts)
    assert info["P"] == 59
    assert 22 * info["P"] - 20 == 1278
    assert int(2 * 9.6 / 0.1) == 191
    fs = rp.setup_field(rp.VehicleParams(3.2, 9.6), field_length=300, field_width=150)
    _, g = raster.corner_coverage(fs)
    assert g == 191


def test_speed_plan_is_minplus_scan():
    """SURVEY.md App. C: the three-pass planner == u=v² min-plus scans with chain breaks."""
    veh = rp.VehicleParams()
    fs = rp.setup_field(veh, field_length=500, field_width=200)
    o = rp.plan_complete_coverage(fs)
    path = np.vstack([o["main_work"]["path"], o["headland"]["path"]])
    pre = o["_info"]["speeds_pre"]
    kap = np.concatenate([[0.0], rp.curvatures(path), [0.0]])
    lim = pre.copy()
    m = kap > 1e-6
    lim[m] = np.minimum(lim[m], np.sqrt(veh.max_lateral_accel / kap[m]) * veh.safety_factor * 3.6)
    u = (lim / 3.6) ** 2
    ds = np.sqrt((np.diff(path, axis=0) ** 2).sum(1))
    c = np.where(ds < 1e-6, np.inf, 2 * veh.max_longitudinal_accel * ds)
    f = u.copy()
    for i in range(1, len(f)):
        f[i] = min(f[i], f[i - 1] + c[i - 1])
    for i in range(len(f) - 2, -1, -1):
        f[i] = min(f[i], f[i + 1] + c[i])
    got = np.concatenate([o["main_work"]["speeds"], o["headland"]["speeds"]])
    np.testing.assert_allclose(3.6 * np.sqrt(f), got, rtol=0, atol=1e-12)
    assert int((ds < 1e-6).sum()) == 72   # App. C: 72 zero-length segments


def test_ga_tour_lengths_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "ga_tours.npz"))
    d = raster.tour_lengths(z["D"], z["pop"])
    assert np.array_equal(d, z["dist"])          # sequential FP64 sum: bit-exact
    np.testing.assert_array_equal(1.0 / (d + 1e-6), z["fitness"])


def test_inset_error_status():
    fs = rp.setup_field(rp.VehicleParams(3.2, 8.0), field_length=30, field_width=15)
    with pytest.raises(ValueError):
        rp.plan_complete_coverage(fs)


# a checkout of the reference project (qwagrox/field-coverage-path-planning).  The repository contains neither the
# reference nor its output for the scenario below (120 x 60 m, R = 6.4 m, start and end point): without the checkout
# this comparison does not run.  The stored ref_*.npz scenarios are compared above, at atol 1e-12.
REFERENCE_DIR = os.environ.get("FCPP_REFERENCE_DIR")


@pytest.mark.skipif(not REFERENCE_DIR or not os.path.exists(os.path.join(REFERENCE_DIR, "multi_layer_planner_v3.py")),
                    reason="set FCPP_REFERENCE_DIR to a checkout of the reference project")
def test_oracle_vs_reference_executed_live():
    """Execute the UNMODIFIED reference (through the Shapely stand-in) right now and compare:
    proves the committed fixtures are what the reference produces and that the stub pipeline works."""
    import contextlib
    import io
    from oracle import shapely_stub
    m = shapely_stub.load_reference(os.path.join(REFERENCE_DIR, "multi_layer_planner_v3.py"))
    kw = dict(field_length=120, field_width=60, start_point=(110, 50), end_point=(5, 5))
    with contextlib.redirect_stdout(io.StringIO()):
        p = m.TwoLayerPathPlannerV37(m.VehicleParams(3.2, 6.4, 9.0, 14.0), **kw)
        r = p.plan_complete_coverage()
    fs = rp.setup_field(rp.VehicleParams(3.2, 6.4, 9.0, 14.0), **kw)
    o = rp.plan_complete_coverage(fs)
    for layer in ("main_work", "headland"):
        assert np.array_equal(o[layer]["path"], r[layer]["path"])          # 0 ulp
        np.testing.assert_allclose(o[layer]["speeds"], r[layer]["speeds"], rtol=0, atol=1e-12)
    assert np.array_equal(o["approach_path"], r["approach_path"])
    assert np.array_equal(o["departure_path"], r["departure_path"])


@pytest.mark.parametrize("case", ["rect120x80", "rect500x200", "offset_rect", "narrow_loops", "sheared", "tilted"])
def test_zoned_band_model_equals_brute_force(case):
    """The four exactness claims behind the coverage kernel's zoned band evaluation (chains = rectangle +
    end discs, entries inside the R-inset cover no band cell, general entries stay inside their quadrant's
    zone, runs of rows are constant between breakpoints) restated on the CPU (oracle/zoned_model.py) give
    the brute-force counts of raster_oracle.c; fields without axis-aligned chains / with overlapping zones
    are reported as 'fall back' (None), as the kernel does."""
    from dataclasses import replace
    from oracle import raster, ref_planner as rp, zoned_model
    fields = {
        "rect120x80": ([(0, 0), (120, 0), (120, 80), (0, 80)], 3.2, (5.0, 8.0, 11.0), 0.1),
        "rect500x200": ([(0, 0), (500, 0), (500, 200), (0, 200)], 3.2, (7.2,), 0.1),      # BASELINE configs 1-2
        "offset_rect": ([(1000.3, 2000.7), (1180.3, 2000.7), (1180.3, 2075.7), (1000.3, 2075.7)], 3.2, (6.4, 9.6), 0.25),
        "narrow_loops": ([(0, 0), (90, 0), (90, 70), (0, 70)], 0.8, (6.0,), 0.1),
        "sheared": ([(0, 0), (200, 0), (230, 90), (30, 90)], 3.2, (8.0,), 0.25),
        "tilted": ([(0, 0), (150, 20), (140, 95), (-10, 75)], 3.2, (8.0,), 0.25),
    }
    verts, W, radii, h = fields[case]
    got_zoned = 0
    for R in radii:
        for corner in (0, 2):
            fs = rp.setup_field(replace(rp.VehicleParams(), working_width=W, min_turn_radius=R),
                                field_vertices=[tuple(map(float, v)) for v in verts], obstacles=[])
            hp = rp.plan_complete_coverage(fs, start_corner=corner)["headland"]["path"]
            brute = raster.band_coverage(fs, hp, h)
            model = zoned_model.band_zoned(fs, hp, h)
            if model is not None:
                assert model == brute, (case, R, corner, model, brute)
                got_zoned += 1
    # rectangles are evaluated zoned; the slanted straights of sheared / tilted fields are general entries that
    # span the field, the zones overlap and the evaluation falls back to the whole band
    assert (got_zoned > 0) == (case not in ("tilted", "sheared")), (case, got_zoned)


def test_geos_faithful_buffer_vs_exact_round_buffer_quantified():
    """SURVEY.md §8(f) N3: what decisions D2 / D5 (exact round buffer, lattice counts) give away against the polygon
    GEOS builds (16 chords per quadrant, inscribed fillets — restated in oracle/geos_buffer.py, GEOS itself is not
    installable).  On every fixture scenario with the corner-grid verification:
      * the GEOS region is a subset of the exact buffer; the lattice points that differ lie within the deepest
        sliver (r (1 - cos(inc / 2)) <= 2.6 mm) of the exact boundary;
      * per 2R x 2R window at most 4 of ~25 000 lattice points differ (<= 0.02 percentage points of
        coverage_before / coverage_after, mlp3:1477, :1494);
      * for the headland path ALL slivers together are < 1e-4 of the band area (an upper bound of the coverage_rate
        difference, mlp3:1357-1371 — most slivers lie under a neighbouring segment's cover); rasterised over the
        whole band (100 x 80 and 500 x 200 m fields at 0.1 m) the GEOS region and the exact buffer cover the SAME
        lattice points, equal to the integer oracle's count.
    The numbers are printed (pytest -s) and recorded in oracle/README.md."""
    from oracle import geom, geos_buffer as gb
    rows = []
    for path in GOLD:
        z, meta, veh, kw = _load(path)
        if "corner_before" not in z.files and not meta.get("corner_grid"):
            pass
        fs = rp.setup_field(veh, **kw)
        if fs.field_shape != "rectangle":
            continue
        R, W = fs.vehicle.min_turn_radius, fs.vehicle.working_width
        g = int(2 * R / rp.GRID_RESOLUTION)
        I, J = np.meshgrid(np.arange(g), np.arange(g))
        worst = 0
        for (cx, cy), ci, arc, rev in rp.verification_corner_paths(fs):
            ox = cx if ci in (0, 3) else cx - 2 * R
            oy = cy if ci in (0, 1) else cy - 2 * R
            X, Y = ox + I * rp.GRID_RESOLUTION, oy + J * rp.GRID_RESOLUTION
            ex, d = gb.exact_contains(arc, W / 2, X, Y)
            ge = gb.contains(arc, W / 2, X, Y)
            depth = gb.max_sliver_depth(arc, W / 2)
            if rev is not None and len(rev) > 0:
                ex2, d2 = gb.exact_contains(rev, W / 2, X, Y)
                ex, d = ex | ex2, np.minimum(d, d2)
                ge = ge | gb.contains(rev, W / 2, X, Y)
                depth = max(depth, gb.max_sliver_depth(rev, W / 2))
            assert not (ge & ~ex).any()                      # inscribed: GEOS region inside the exact buffer
            diff = ex & ~ge
            assert depth <= 2.6e-3 * (W / 3.2)
            assert (W / 2 - d[diff] <= depth + 1e-9).all()    # only cells inside a sliver differ
            assert diff.sum() <= 4
            worst = max(worst, int(diff.sum()))
        o = rp.plan_complete_coverage(fs)
        head = o["headland"]["path"]
        band = abs(geom.signed_area(fs.field_vertices)) - abs(geom.signed_area(geom.inset_convex(fs.field_vertices, fs.headland_width)))
        rel = gb.sliver_area_bound(head, W / 2) / band
        assert rel < 1e-4
        band_diff = None
        if fs.field_length <= 500 and not kw.get("obstacles") and kw.get("start_point") is None:
            h = 0.1
            nx, ny = int(round(fs.field_length / h)), int(round(fs.field_width / h))
            ge, ex = gb.raster_grid(head, W / 2, h / 2, h / 2, h, nx, ny)
            I2, J2 = np.meshgrid(np.arange(nx), np.arange(ny))
            X2, Y2 = h / 2 + I2 * h, h / 2 + J2 * h
            hw = fs.headland_width
            inb = ~((X2 > hw) & (X2 < fs.field_length - hw) & (Y2 > hw) & (Y2 < fs.field_width - hw))
            assert not (ge & ~ex).any()
            band_diff = int((ex & ~ge & inb).sum())
            total, covered = raster.band_coverage(fs, head, h)
            assert (int(inb.sum()), int((ex & inb).sum())) == (total, covered)    # float exact == integer oracle
            assert band_diff == 0
        rows.append((os.path.basename(path)[4:-4], g * g, worst, rel, band_diff))
    assert len(rows) >= 5
    assert sum(r[4] is not None for r in rows) >= 2
    for name, cells, worst, rel, band_diff in rows:
        print(f"N3 {name:12s} window {cells} lattice points: <= {worst} differ (GEOS fan vs exact round buffer); "
              f"coverage_rate bound {rel:.2e}; band lattice points that differ: {band_diff}")


def test_omega_pattern_oracle_properties():
    """The build-defined Ω (skip-row) pattern of the oracle (the reference has only the label, mlp3:312-320): every row
    exactly once, consecutive rows at most s apart, the U pattern's sample counts and swath ends, turns that start and
    end ON the swath ends with curvature <= 1/R (up to the sampling), equal arc-length spacing."""
    for P in range(1, 40):
        for s_ in (1, 2, 5, 7):
            order = rp.omega_order(P, s_)
            assert sorted(order) == list(range(P))
            assert all(abs(a - b) <= s_ for a, b in zip(order, order[1:]))
    assert rp.omega_skip(8.0, 3.2) == 5 and rp.omega_skip(1.0, 3.2) == 1 and rp.omega_skip(4.8, 3.2) == 3
    for d, R in ((3.2, 8.0), (12.8, 8.0), (16.0, 8.0), (22.4, 8.0), (0.5, 5.0)):
        u, v = rp.omega_turn_local(d, R)
        pts = np.stack([u, v], axis=1)
        assert np.abs(pts[0]).max() == 0.0 and np.abs(pts[-1] - (0.0, d)).max() < 1e-12
        seg = np.linalg.norm(np.diff(pts, axis=0), axis=1)
        assert seg.max() / seg.min() < 1.01
        assert rp.curvatures(pts).max() <= 1.0 / max(R, d / 2) * 1.02
    veh = rp.VehicleParams()
    fo = rp.setup_field(veh, field_length=500, field_width=200, turn_model="omega")
    fu = rp.setup_field(veh, field_length=500, field_width=200)
    po, pu = rp.plan_complete_coverage(fo), rp.plan_complete_coverage(fu)
    mo, mu = po["main_work"]["path"], pu["main_work"]["path"]
    assert mo.shape == mu.shape == (1256, 2)
    assert np.array_equal(po["headland"]["path"], pu["headland"]["path"])
    ends_o = {tuple(np.round(p, 9)) for k in range(0, 1256, 22) for p in mo[k:k + 2]}
    ends_u = {tuple(np.round(p, 9)) for k in range(0, 1256, 22) for p in mu[k:k + 2]}
    assert ends_o == ends_u                                   # the same swaths, another order
    assert rp.curvatures(mo).max() <= 1.0 / 8.0 * 1.01
