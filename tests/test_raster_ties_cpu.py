"""The lattice-tie cases without a device: each reaches its edge (its stated minimum of ties and near-ties), the
integer oracle agrees with the Python-integer predicate on them, coordinates survive the 1e-4 m snap at UTM-like
magnitudes, and the planner's window range check runs before any device is looked for."""
import os
import sys

import numpy as np
import pytest

from oracle import raster

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _raster_ties as rt  # noqa: E402


@pytest.mark.parametrize("name", list(rt.CASES))
def test_case_reaches_its_edge_and_oracle_agrees(name):
    paths, r, H, X0, Y0, nx, ny, mt, mn = rt.case(name)
    rt.check_ties(paths, r, X0, Y0, H, nx, ny, mt, mn, name)
    assert (name in rt.SLOW_CASES) == (max(nx, ny) ** 2 > rt.SLOW_CELLS), (name, nx, ny)
    if name.startswith("tan_"):   # every copy (as given, reversed, mirrored in x, in y) reaches its edge on its own
        for k in range(0, len(paths), 2):
            assert rt.tie_counts(rt.segments(paths[k]), r, X0, Y0, H, nx, ny)[0] >= 6
            assert rt.tie_counts(rt.segments(paths[k + 1]), r, X0, Y0, H, nx, ny)[1] >= 1
    for p in paths[:6]:
        rt.metres(p)
        rt.metres(p + rt.GEO)
    # the oracle's brute force == the Python-integer predicate, on the (small) part of the lattice of the first paths
    sub = paths[:4]
    Xs, Ys, nxs, nys = rt.bbox_window(sub, r, H)
    bits = np.zeros((nxs * nys + 7) // 8, dtype=np.uint8)
    for p in sub:
        pts = np.ascontiguousarray(p, dtype=np.int64)
        raster.lib().fcpo_raster(raster._i64p(pts), len(pts), r, Xs, Ys, H, nxs, nys, bits.ctypes.data)
    got = np.unpackbits(bits, bitorder="little")[:nxs * nys].reshape(nys, nxs).astype(bool)
    assert np.array_equal(got, rt.cover_bits(sub, r, Xs, Ys, H, nxs, nys)), name


def test_near_axis_case_reaches_its_edge():
    r, H, O, g, mt, mn = rt.NEAR_AXIS
    rt.check_ties(rt.near_axis_case(r, H), r, O, O, H, g, g, mt, mn, "near_axis")


def test_predicate_at_exact_ties():
    """The strict predicate and the tie test on hand-made ties: end disc (3, 4, 5), tangent line, far segments."""
    r2 = 5 * 5
    seg = (3, 4, 30, 40)
    assert rt.on_boundary(0, 0, seg, r2) and not rt.near(0, 0, seg, r2)
    assert rt.near(0, 1, seg, r2)
    seg = (0, 5, 100, 5)                      # horizontal: the row y = 0 is at exactly r
    assert rt.on_boundary(50, 0, seg, r2) and not rt.near(50, 0, seg, r2) and rt.near(50, 1, seg, r2)
    big = (-(1 << 31), 5, 1 << 31, 6)         # cr and r² dd beyond 2^63: Python integers do not overflow
    assert rt.near(0, 0, big, (6 * 6)) and not rt.near(0, 0, big, 5 * 5)


def test_coordinates_survive_the_snap():
    U = np.array([[0, 0], [1, -1], [(1 << 30) - 1, -((1 << 30) - 1)], [5_123_456_789, 43_210_987_654],
                  [5_123_456_789 + (1 << 30) - 1, 43_210_987_654 - (1 << 30) + 1]], dtype=np.int64)
    assert np.array_equal(raster.q(rt.metres(U)), U)


def test_edge_point_counts():
    for name, quad in rt.quads(200).items():
        xs, ys = [v[0] for v in quad], [v[1] for v in quad]
        dims = (min(xs) + 100, min(ys) + 100, 200, -(-(max(xs) - min(xs)) // 200), -(-(max(ys) - min(ys)) // 200))
        on, near = rt.edge_points(quad, *dims), rt.edge_margin_points(quad, *dims)
        print(name, on, near)
        for k in range(4):   # horizontal edges are decided by an integer test, not by the FP row interval
            if quad[k][1] != quad[(k + 1) % 4][1]:
                assert near[k] >= on[k]
        if name == "nearly_flat":
            assert near[2] >= 1
        else:
            assert sum(on) >= 40


def test_clamp_demonstration_counts():
    """The exact cover of the three demonstration segments differs from the cover of the clamped segment."""
    r, H, g, lim = 16000, 1000, 160, 1 << 30
    a = (80000, 80000)
    clamp = lambda v: max(-lim, min(lim, v))  # noqa: E731
    b = (3_080_000_000, 1_500_080_000)
    exact = rt.cover_bits([np.array([a, b], dtype=object)], r, 0, 0, H, g, g)
    clamped = rt.cover_bits([np.array([a, (clamp(b[0]), clamp(b[1]))], dtype=object)], r, 0, 0, H, g, g)
    assert (int(exact.sum()), int(clamped.sum()), int((exact ^ clamped).sum())) == (3226, 3721, 3035)


def test_planner_rejects_far_points_on_the_host():
    """verify_corner_coverage_grid_based checks its paths before it touches the device: without a GPU this raises
    ValueError naming the path and the point."""
    import field_coverage_path_planning_b200 as fc
    pl = fc.TwoLayerPathPlannerV37(field_length=500, field_width=200)
    turn = np.array([[8.0, 8.0], [9.0, 9.5]])
    with pytest.raises(ValueError, match="turn_path point 1 "):
        pl.verify_corner_coverage_grid_based((8.0, 8.0), 0, np.array([[8.0, 8.0], [308000.0, 150000.0]]))
    with pytest.raises(ValueError, match="reverse_path point 0 "):
        pl.verify_corner_coverage_grid_based((8.0, 8.0), 0, turn, np.array([[0.0, -110000.0], [8.0, 8.0]]))
    # exactly 2^30 units from the origin (8, 8) m along x: rejected
    with pytest.raises(ValueError, match="reverse_path point 1 "):
        pl.verify_corner_coverage_grid_based((8.0, 8.0), 0, turn, np.array([[8.0, 8.0], [8.0 + 107374.1824, 8.0]]))
