"""The coverage rasterisers at exact lattice ties, near-ties and the 2^30 range limit (tests/_raster_ties.py).

Every case is built in integer lattice units and asserts its own minimum of ties and near-ties, so no case can stop
reaching the edge it is named for.  The reference is the integer oracle (oracle/raster_oracle.c) where its int64
products cannot overflow, Python integers otherwise.  Kernels: the A10 window raster (fcpp_raster_window, called as
the planner calls it, for any g, pitch and origin), the whole-field and band coverage of paths (fcpp_path_coverage via
verify_paths) and the coverage kernel of generated plans."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from oracle import raster

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _path_cover_oracle as pco  # noqa: E402
import _raster_ties as rt  # noqa: E402

pytestmark = pytest.mark.gpu

LIM = 1 << 30
GEO = rt.GEO
# cases whose brute-force window (g = max(nx, ny), g² cells) exceeds ~1.2e6 cells run with the slow tests
CASE_PARAMS = [pytest.param(n, marks=pytest.mark.slow) if n in rt.SLOW_CASES else n for n in rt.CASES]


@pytest.fixture(scope="module")
def fc():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import field_coverage_path_planning_b200 as pkg
    return pkg


def gpu_window(paths, r, X0, Y0, H, g, fill=None):
    """fcpp_raster_window over every path in turn, ORing into one g x g grid: (status, count, grid bytes)."""
    import torch
    from field_coverage_path_planning_b200 import _lib
    h = _lib.handle(0)
    nw = (g * g + 31) // 32
    bits = torch.zeros(nw, dtype=torch.int32, device="cuda:0")
    if fill is not None:
        bits.fill_(fill)
    cnt = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    st = C.c_void_p(torch.cuda.current_stream(0).cuda_stream)
    rc = 0
    for p in paths:
        d = torch.from_numpy(rt.metres(p)).to("cuda:0")
        rc = h.lib.fcpp_raster_window(h.h, d.data_ptr(), len(p), r / 1e4, X0 / 1e4, Y0 / 1e4, H / 1e4, g,
                                      bits.data_ptr(), cnt.data_ptr(), st)
        if rc:
            break
    torch.cuda.synchronize()
    return rc, int(cnt.item()), bits.cpu().numpy().view(np.uint8)


def oracle_window(paths, r, X0, Y0, H, g):
    bits = None
    cnt = 0
    for p in paths:
        cnt, bits = raster.raster_window(rt.metres(p), r / 1e4, (X0 / 1e4, Y0 / 1e4), H / 1e4, g, g, bits)
    return cnt, bits


def field_of(X0, Y0, H, nx, ny):
    """Rectangle (units) whose A11 cell centres are the lattice points (X0 + i H, Y0 + j H), i < nx, j < ny."""
    x0, y0, x1, y1 = X0 - H // 2, Y0 - H // 2, X0 + (nx - 1) * H + H // 2, Y0 + (ny - 1) * H + H // 2
    return np.array([(x0, y0), (x1, y0), (x1, y1), (x0, y1)], dtype=np.int64)


def oracle_paths(paths, r, X0, Y0, H, nx, ny, hw):
    """Per path (field cells, covered, band cells, covered) on the rectangle of field_of, headland width hw units with
    hw - H/2 a multiple of H: the inset's edges run through cell centres (closed inset: those are not band cells)."""
    k = (hw - H // 2) // H
    band = np.ones((ny, nx), dtype=bool)
    band[k:ny - k, k:nx - k] = False
    out = []
    for p in paths:
        bits = np.zeros((nx * ny + 7) // 8, dtype=np.uint8)
        pts = np.ascontiguousarray(p, dtype=np.int64)
        raster.lib().fcpo_raster(raster._i64p(pts), len(pts), r, X0, Y0, H, nx, ny, bits.ctypes.data)
        b = np.unpackbits(bits, bitorder="little")[:nx * ny].reshape(ny, nx).astype(bool)
        out.append((nx * ny, int(b.sum()), int(band.sum()), int((b & band).sum())))
    return out


def gpu_paths(fc, paths, field, r, H, hw, off=(0, 0)):
    off = np.asarray(off)
    got = fc.verify_paths([rt.metres(p + off) for p in paths], [rt.metres(field + off)],
                          fc.VehicleParams(working_width=2 * r / 1e4), headland_width=hw / 1e4, grid_h=H / 1e4)
    assert (got["status"] == 0).all()
    return got


def _counts(got):
    return [tuple(int(g[k]) for k in ("field_total", "field_cells", "band_total", "band_cells")) for g in got]


# ---- a-d: end discs, tangent lines, axis-aligned segments; georeferenced copies ----

@pytest.mark.parametrize("name", CASE_PARAMS)
def test_window_ties_vs_oracle(fc, name):
    paths, r, H, X0, Y0, nx, ny, mt, mn = rt.case(name)
    g = max(nx, ny)
    rt.check_ties(paths, r, X0, Y0, H, g, g, mt, mn, name)
    want, wbits = oracle_window(paths, r, X0, Y0, H, g)
    rc, cnt, bits = gpu_window(paths, r, X0, Y0, H, g)
    assert rc == 0 and cnt == want
    nb = (g * g + 7) // 8
    assert np.array_equal(bits[:nb], wbits[:nb]), name
    # georeferenced: the lattice moves with the window origin, so every bit is the same
    rc, cnt2, bits2 = gpu_window([p + GEO for p in paths], r, X0 + int(GEO[0]), Y0 + int(GEO[1]), H, g)
    assert rc == 0 and cnt2 == cnt and np.array_equal(bits2, bits)


@pytest.mark.parametrize("name", CASE_PARAMS)
def test_path_coverage_ties_vs_oracle(fc, name):
    from oracle import ref_planner as rp
    paths, r, H, X0, Y0, nx, ny, mt, mn = rt.case(name)
    rt.check_ties(paths, r, X0, Y0, H, nx, ny, mt, mn, name)
    field = field_of(X0, Y0, H, nx, ny)
    hw = (min(nx, ny) // 4) * H + H // 2
    got = gpu_paths(fc, paths, field, r, H, hw)
    assert _counts(got) == oracle_paths(paths, r, X0, Y0, H, nx, ny, hw), name
    geo = gpu_paths(fc, paths, field, r, H, hw, GEO)
    assert _counts(geo) == _counts(got)
    fm = rt.metres(field + GEO)
    for p, g in zip(paths[:4], geo[:4]):
        assert int(g["n_boundary_viol"]) == rp.boundary_violations(rt.metres(p + GEO), fm)


def test_near_axis_extremes(fc):
    """dy = +-1 over dx = 1 m .. 2^30 - 1 units, and transposed: the window, the field counts and a georeferenced
    copy of the window."""
    r, H, O, g, mt, mn = rt.NEAR_AXIS
    paths = rt.near_axis_case(r, H)
    rt.check_ties(paths, r, O, O, H, g, g, mt, mn, "near_axis")
    want, wbits = oracle_window(paths, r, O, O, H, g)
    rc, cnt, bits = gpu_window(paths, r, O, O, H, g)
    nb = (g * g + 7) // 8
    assert rc == 0 and cnt == want and np.array_equal(bits[:nb], wbits[:nb])
    rc, cnt2, bits2 = gpu_window([p + GEO for p in paths], r, O + int(GEO[0]), O + int(GEO[1]), H, g)
    assert rc == 0 and cnt2 == cnt and np.array_equal(bits2, bits)
    field = field_of(O, O, H, g, g)
    got = gpu_paths(fc, paths, field, r, H, 20 * H + H // 2)
    assert _counts(got) == oracle_paths(paths, r, O, O, H, g, g, 20 * H + H // 2)


# ---- e: the 2^30 range limit ----

def test_range_limit_window(fc):
    r, H, g = 16000, 1000, 48
    ok, far = [], []
    for ax in (0, 1):
        for sgn in (1, -1):
            e = np.zeros(2, dtype=np.int64)
            e[ax] = sgn * (LIM - 1)
            ok.append(np.array([(20000, 24000), e]))
            e2 = e.copy()
            e2[ax] = sgn * LIM
            far.append(np.array([(20000, 24000), e2]))
    for p in ok:
        rc, cnt, bits = gpu_window([p], r, 0, 0, H, g)
        ref = rt.cover_bits([p], r, 0, 0, H, g, g)
        assert rc == 0 and cnt == int(ref.sum())
        assert np.array_equal(np.unpackbits(bits, bitorder="little")[:g * g].reshape(g, g).astype(bool), ref)
    for p in far:   # rejected: count -1, the caller's grid untouched
        rc, cnt, bits = gpu_window([p], r, 0, 0, H, g, fill=0x5A5A5A5A)
        assert rc == 0 and cnt == -1 and (bits.view(np.uint32) == 0x5A5A5A5A).all()
    # a window whose extent reaches 2^30 units is an invalid argument
    import torch
    from field_coverage_path_planning_b200 import _lib
    h = _lib.handle(0)
    d = torch.zeros(4, dtype=torch.float64, device="cuda:0")
    b = torch.zeros(4, dtype=torch.int32, device="cuda:0")
    c = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    assert h.lib.fcpp_raster_window(h.h, d.data_ptr(), 2, 1.6, 0.0, 0.0, (LIM // 8) / 1e4, 8, b.data_ptr(),
                                    c.data_ptr(), None) == -1
    assert h.lib.fcpp_raster_window(h.h, d.data_ptr(), 2, 1.6, 0.0, 0.0, (LIM // 8 - 1) / 1e4, 8, b.data_ptr(),
                                    c.data_ptr(), None) == 0


def test_clamp_demonstration_segments(fc):
    """One segment from (8, 8) m to far away, window g = 160, h = 0.1 m, r = 1.6 m: never the clamped cover.  Beyond
    2^30 units the window is rejected; the same directions ending just inside the range give the exact cover."""
    r, H, g = 16000, 1000, 160
    a = (80000, 80000)
    for b in [(3_080_000_000, 1_500_080_000), (-4_000_000_000, 80_500), (2_000_080_000, -99_920_000)]:
        p = np.array([a, b], dtype=np.int64)
        rc, cnt, bits = gpu_window([p], r, 0, 0, H, g)
        assert rc == 0 and cnt == -1
        # the same direction, scaled to end inside the range
        k = max(abs(b[0] - a[0]), abs(b[1] - a[1])) / (LIM - 100_000)
        q = np.array([a, (a[0] + int((b[0] - a[0]) / k), a[1] + int((b[1] - a[1]) / k))], dtype=np.int64)
        rc, cnt, bits = gpu_window([q], r, 0, 0, H, g)
        ref = rt.cover_bits([q], r, 0, 0, H, g, g)
        assert rc == 0 and cnt == int(ref.sum()), (b, cnt, int(ref.sum()))
        assert np.array_equal(np.unpackbits(bits, bitorder="little")[:g * g].reshape(g, g).astype(bool), ref)


def test_planner_accepts_points_inside_the_range(fc):
    pl = fc.TwoLayerPathPlannerV37(field_length=500, field_width=200)
    turn = np.array([[8.0, 8.0], [9.0, 9.5]])
    ok = pl.verify_corner_coverage_grid_based((8.0, 8.0), 0, turn, np.array([[8.0, 8.0], [107000.0, 8.0]]))
    assert ok["cells_after"] >= ok["cells_before"] > 0


def test_range_limit_path_coverage(fc):
    """Points at +-(2^30 - 1) units from the lattice origin are accepted (a long diagonal whose capsule crosses the
    field with a planted tie: near_seg's t and cr near 2^62 and 2^63), +-2^30 is FCPP_PATH_OUT_OF_RANGE."""
    from field_coverage_path_planning_b200 import _lib
    r, H, n = 16000, 1000, 64
    X0 = Y0 = 0
    field = field_of(X0, Y0, H, n, n)
    M = LIM - 1
    # the diagonal y = x + c passes at exactly r from lattice points when c = r sqrt(2): not an integer, so plant the
    # tie with the (3, 4) direction instead: 4 x - 3 y = 5 r through the lattice point (0, 0) shifted by its normal
    d = (3, 4)
    k = (M - 20000) // 4
    A = np.array([-3 * k, -4 * k], dtype=np.int64)
    base = np.array([4 * r // 5, -3 * r // 5], dtype=np.int64)        # r (4, -3) / 5: perpendicular offset r
    tie = np.array([A + base, A + base + 2 * k * np.array(d)])
    paths = [np.array([(-M, -M), (M, M)]), np.array([(M, -M), (-M, M)]), tie,
             np.array([(20000, 20000), (M, 0)]), np.array([(20000, 20000), (-M, 0)]),
             np.array([(20000, 20000), (0, M)]), np.array([(20000, 20000), (0, -M)])]
    ties, _ = rt.tie_counts(rt.segments(tie), r, X0, Y0, H, n, n)
    print(f"range: {ties} ties")
    assert ties >= 1
    got = gpu_paths(fc, paths, field, r, H, 10 * H + H // 2)
    for p, g in zip(paths, got):
        ref = rt.cover_bits([p], r, X0, Y0, H, n, n)
        assert (int(g["field_total"]), int(g["field_cells"])) == (n * n, int(ref.sum()))
    far = [np.array([(20000, 20000), (s * LIM, 0)]) for s in (1, -1)] + [np.array([(20000, 20000), (0, s * LIM)])
                                                                        for s in (1, -1)]
    got = fc.verify_paths([rt.metres(p) for p in far], [rt.metres(field)], fc.VehicleParams(working_width=3.2),
                          grid_h=0.1)
    assert (got["status"] == _lib.PATH_OUT_OF_RANGE).all()


# ---- f: quad windows (field_total, band_total) with edges through cell centres ----

@pytest.mark.parametrize("name", ["slope_1_2", "slope_3_4", "nearly_flat", "rect_inset"])
def test_quad_edges_through_cell_centres(fc, name):
    from oracle import geom
    H = 200 if name != "rect_inset" else 2000
    if name == "rect_inset":     # R = 3.3 m at h = 0.2 m: the inset's edges run through cell centres
        quad, hw = [(0, 0), (2_000_000, 0), (2_000_000, 1_000_000), (0, 1_000_000)], 33_000
        inset = [tuple(v) for v in raster.q(np.asarray(geom.inset_convex(rt.metres(quad), hw / 1e4)))]
        on = rt.edge_points(inset, H // 2, H // 2, H, 1000, 500)
        print(f"{name}: centres on the inset's edges {on}")
        assert min(on) >= 400
    else:
        quad, hw = rt.quads(H)[name], 10 * H
        xs, ys = [v[0] for v in quad], [v[1] for v in quad]
        nx, ny = -(-(max(xs) - min(xs)) // H), -(-(max(ys) - min(ys)) // H)
        on = rt.edge_points(quad, min(xs) + H // 2, min(ys) + H // 2, H, nx, ny)
        near = rt.edge_margin_points(quad, min(xs) + H // 2, min(ys) + H // 2, H, nx, ny)
        print(f"{name}: centres on the edges {on}, within the 1e-5 cell margin {near}")
        if name == "nearly_flat":
            assert near[2] >= 1        # the 1-unit-over-500-m edge itself
        else:
            assert sum(on) >= 40
    quad = np.asarray(quad, dtype=np.int64)
    path = np.array([quad[0] + (H, H * 3), quad[2] - (H * 2, H)], dtype=np.int64)
    W = 3.2
    got = fc.verify_paths([rt.metres(path)], [rt.metres(quad)], fc.VehicleParams(working_width=W),
                          headland_width=hw / 1e4, grid_h=H / 1e4)[0]
    fm = rt.metres(quad)
    assert (int(got["field_total"]), int(got["field_cells"])) == pco.field_coverage(fm, rt.metres(path), W, H / 1e4)
    assert (int(got["band_total"]), int(got["band_cells"])) == pco.band_coverage_of(fm, hw / 1e4, rt.metres(path), W,
                                                                                    H / 1e4)


# ---- g: slab staging and the work list of fcpp_path_coverage ----

def test_slab_boundaries_and_staging_rounds(fc):
    """nx = 4096 cells: rows per slab = min(1024, 8192 / 128) = 64.  Horizontal segments whose capsule reaches exactly
    one row into the neighbouring slab (r - 1 from it), segments at exactly r from a slab's edge row (they reach no
    row), and one path of > 512 segments inside one slab."""
    r, H, nx, ny = 16000, 200, 4096, 256
    rows = min(1024, 8192 // -(-nx // 32))
    assert rows == 64
    field = field_of(0, 0, H, nx, ny)
    paths = []
    for j0 in (64, 128, 192):
        for dy, x0 in ((-r + 1, 1000), (-r, 300_000), (-H + r - 1, 600_000), (-H + r, 900_000)):
            y = j0 * H + dy
            paths.append(np.array([(x0, y), (x0 + 200_000, y)], dtype=np.int64))
    zig = np.array([(2000 + 1000 * i, 70 * H + (i % 2) * 40 * H) for i in range(700)], dtype=np.int64)
    paths.append(zig)
    got = gpu_paths(fc, paths, field, r, H, 20 * H + H // 2)
    assert _counts(got) == oracle_paths(paths, r, 0, 0, H, nx, ny, 20 * H + H // 2)


def test_work_list_over_many_chunks(fc):
    """> 2048 paths: the scan runs three 1024-path chunks; zero-slab (out-of-range) paths at 0, 1023, 1024 and last.
    Every record equals the same path alone in a batch of one."""
    from field_coverage_path_planning_b200 import _lib
    r, H, nx, ny = 16000, 200, 600, 300
    field = rt.metres(field_of(0, 0, H, nx, ny))
    rng = np.random.default_rng(7)
    uniq = [np.cumsum(rng.integers(-3000, 3000, size=(int(rng.integers(2, 40)), 2)), 0) + (60_000, 30_000)
            for _ in range(12)]
    far = np.array([[1000, 1000], [LIM, 0]])
    n = 2100
    idx = [k % len(uniq) for k in range(n)]
    paths = [uniq[k] for k in idx]
    for i in (0, 1023, 1024, n - 1):
        paths[i] = far
    veh = fc.VehicleParams(working_width=2 * r / 1e4)
    kw = dict(headland_width=2.1, grid_h=H / 1e4)
    got = fc.verify_paths([rt.metres(p) for p in paths], [field], veh, **kw)
    alone = {k: fc.verify_paths([rt.metres(u)], [field], veh, **kw)[0].tobytes() for k, u in enumerate(uniq)}
    far1 = fc.verify_paths([rt.metres(far)], [field], veh, **kw)[0]
    assert far1["status"] == _lib.PATH_OUT_OF_RANGE
    for i in range(n):
        want = far1.tobytes() if i in (0, 1023, 1024, n - 1) else alone[idx[i]]
        assert got[i].tobytes() == want, i
    for k in (0, 5):
        assert (int(got[k + 1]["field_total"]), int(got[k + 1]["field_cells"])) == pco.field_coverage(
            field, rt.metres(paths[k + 1]), veh.working_width, H / 1e4)


def test_n_main_extremes_and_junction(fc):
    """n_main = 1 and N - 1, and a junction segment that alone crosses the field: its cells stay uncovered."""
    r, H, nx, ny = 16000, 200, 500, 300
    field = field_of(0, 0, H, nx, ny)
    p = np.array([(2000, 2000), (20000, 2000), (20000, 50000), (95000, 55000), (95000, 5000), (80000, 5000)])
    veh = fc.VehicleParams(working_width=3.2)
    fm = rt.metres(field)
    for nm in (1, len(p) - 1, 2, 3):
        got = fc.verify_paths([rt.metres(p)], [fm], veh, headland_width=2.1, n_main=[nm], grid_h=0.02)[0]
        assert (int(got["field_total"]), int(got["field_cells"])) == pco.field_coverage(fm, rt.metres(p), 3.2, 0.02, nm)
        assert (int(got["band_total"]), int(got["band_cells"])) == pco.band_coverage_of(fm, 2.1, rt.metres(p), 3.2,
                                                                                        0.02, nm)
    # n_main = 3: the segment (20000, 50000) -> (95000, 55000) joins the layers; alone it crosses the field's middle
    only = fc.verify_paths([rt.metres(p)], [fm], veh, headland_width=2.1, n_main=[3], grid_h=0.02)[0]
    whole = fc.verify_paths([rt.metres(p)], [fm], veh, headland_width=2.1, n_main=[0], grid_h=0.02)[0]
    split = fc.verify_paths([rt.metres(p[:3]), rt.metres(p[3:])], [fm], veh, headland_width=2.1, grid_h=0.02)
    assert int(whole["field_cells"]) > int(only["field_cells"])
    assert int(only["band_cells"]) == int(split[1]["band_cells"])
    pts = rt.cover_bits([p[:3]], r, 0, 0, H, nx, ny) | rt.cover_bits([p[3:]], r, 0, 0, H, nx, ny)
    assert int(only["field_cells"]) == int(pts.sum())


# ---- h: generated plans on a tie lattice (W = 3.3 m, h = 0.2 m) ----

RECT = [(0.0, 0.0), (500.0, 0.0), (500.0, 200.0), (0.0, 200.0)]


def test_generated_plans_on_a_tie_lattice(fc):
    """W = 3.3 m at h = 0.2 m puts ~20 000 (segment, cell centre) pairs of the headland at exactly r.  The coverage
    kernel's band counts equal the path kernel's for every candidate, start corner and turn model, in every cover
    mode and with de-duplication on and off; a sample equals the oracle, and A10 equals oracle.raster."""
    from field_coverage_path_planning_b200 import _lib
    from oracle import batch as ob, ref_planner as rp
    h = _lib.handle(0)
    veh = fc.VehicleParams(working_width=3.3)
    cand = fc.make_candidates(1, radii=[8.0, 6.5, 9.9], start_corners=[0, 1, 2, 3])
    for tm in ("arc", "clothoid", "omega"):
        base = None
        for mode in (0, 1, 2, 3):
            try:
                h.check(h.lib.fcpp_set_cover_mode(h.h, mode))
                res = fc.plan_batch([RECT], veh, cand, outputs="paths", turn_model=tm, grid_h=0.2, field_coverage=True)
            finally:
                h.check(h.lib.fcpp_set_cover_mode(h.h, 0))
            s, fcv = res.summary, res.field_cover
            ok = s["status"] == 0
            assert ok.all()
            assert np.array_equal(fcv["band_total"], s["cov_total"]) and np.array_equal(fcv["band_cells"], s["cov_cells"])
            if base is None:
                base = (s.tobytes(), fcv.tobytes())
            assert (s.tobytes(), fcv.tobytes()) == base, (tm, mode)
        if tm == "arc":
            for b in range(4):        # R = 8.0, the four start corners
                o = ob.evaluate_candidate(RECT, rp.VehicleParams(working_width=3.3), R=8.0, start_corner=b, grid_h=0.2,
                                          keep_paths=True)
                assert (int(s["cov_total"][b]), int(s["cov_cells"][b])) == (o["cov_total"], o["cov_cells"])
                assert list(map(int, s["corner_after"][b])) == o["corner_after"]
                if b == 0:
                    path, _, _ = res.path(b)
                    hp = path[int(s["n_main"][b]):]
                    X0, Y0, H, nx, ny = raster.band_dims(RECT, 0.2)
                    segs = rt.segments(raster.q(hp))
                    ties, _ = rt.tie_counts(segs, int(raster.q(1.65)), X0 + H // 2, Y0 + H // 2, H, nx, ny)
                    print(f"c2 W 3.3 h 0.2 R 8 headland: {ties} ties")
                    assert ties >= 1000


def test_pythagorean_rotated_field(fc):
    """A field with integer vertices along (4, 3) and (-3, 4): slanted segments reach raster_entries in the coverage
    kernel too.  The two rasterisers agree; the tie count is reported, no minimum is demanded."""
    from oracle import raster as orr
    f = [(0.0, 0.0), (240.0, 180.0), (240.0 - 90.0, 180.0 + 120.0), (-90.0, 120.0)]
    veh = fc.VehicleParams(working_width=3.0)
    cand = fc.make_candidates(1, radii=[8.0, 6.0], start_corners=[0, 1, 2, 3])
    res = fc.plan_batch([f], veh, cand, outputs="paths", grid_h=0.2, field_coverage=True)
    s, fcv = res.summary, res.field_cover
    ok = s["status"] == 0
    assert ok.any()
    assert np.array_equal(fcv["band_total"][ok], s["cov_total"][ok])
    assert np.array_equal(fcv["band_cells"][ok], s["cov_cells"][ok])
    b = int(np.nonzero(ok)[0][0])
    path, _, _ = res.path(b)
    X0, Y0, H, nx, ny = orr.band_dims(f, 0.2)
    ties, nears = rt.tie_counts(rt.segments(orr.q(path[int(s["n_main"][b]):])), 15000, X0 + H // 2, Y0 + H // 2, H,
                                nx, ny)
    print(f"rotated (4, 3) field: {ties} ties, {nears} near-ties")
