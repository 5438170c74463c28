"""CPU tests of the segment-level obstacle sweep's statement (oracle/sweep.py): the closed form of a horizontal swath
through a rectangle on the c2 scenario, dense sampling on hand-made segments, and the relation to D3's point counts.
The device kernels are pinned to the same oracle by tests/test_gpu_sweep.py."""
import math

import numpy as np
import pytest

from oracle import batch as ob, ref_planner as rp, sweep as osw

RECT = [(0.0, 0.0), (500.0, 0.0), (500.0, 200.0), (0.0, 200.0)]
OBST2 = [[(200, 80), (250, 80), (250, 120), (200, 120)], [(350, 140), (380, 140), (380, 170), (350, 170)]]
W = 3.2
r = W / 2


def swath_closed_form(y, xa, xb, rects):
    """m of the horizontal segment (xa, y) -> (xb, y) that spans every rectangle's buffered x-range."""
    m = 0.0
    for o in rects:
        xs, ys = [p[0] for p in o], [p[1] for p in o]
        x0, x1, y0, y1 = min(xs), max(xs), min(ys), max(ys)
        assert xa < x0 - r and xb > x1 + r
        d = max(y0 - y, 0.0, y - y1)
        if d < r:
            m += (x1 - x0) + 2 * math.sqrt(r * r - d * d)
    return m


@pytest.mark.parametrize("R,corner", [(5.0, 0), (8.0, 0), (8.0, 2), (12.0, 0), (6.5, 1), (10.0, 3)])
def test_c2_swaths_match_the_closed_form(R, corner):
    o = ob.evaluate_candidate(RECT, rp.VehicleParams(), R=R, start_corner=corner, obstacles=OBST2, coverage=False,
                              keep_paths=True)
    p, nm = o["path"], o["n_main"]
    knife = osw.knife_mask(p, OBST2, W)
    # R = 8: the swath at y = 8 + 35 * 3.2 runs parallel to the top edge of the first obstacle (y = 120) at r = 1.6 up
    # to a few ulps; its measure hinges on them (closed form 2.7e-7 m, 1e-14 m with y one ulp higher)
    print("knife-edge segments:", int(knife.sum()))
    hits = 0
    for i in range(0, nm - 1, 2 + 20):         # swath i -> i + 1 of every pass
        a, b = p[i], p[i + 1]
        assert a[1] == b[1]
        if knife[i]:
            continue
        m = osw.segment_measure(a, b, osw._polys(OBST2), r)
        want = swath_closed_form(a[1], min(a[0], b[0]), max(a[0], b[0]), OBST2)
        assert abs(m - want) <= 1e-9, (i, m, want)
        hits += m > 0
    # the plan reports no obstacle POINT, yet drives ~1.1 km through the two obstacles
    s = osw.sweep(p, OBST2, W, nm)
    assert o["n_obstacle_viol"] == 0
    assert s["n_seg_main"] >= hits >= 20 and s["len_main"] > 1000


def sampled(a, b, obstacles, n=200001):
    """Dense-sampling estimate of m: the share of n equally spaced parameters whose point is in O, times |b - a|."""
    polys = osw._polys(obstacles)
    t = (np.arange(n) + 0.5) / n
    a, b = np.asarray(a, float), np.asarray(b, float)
    pts = a[None, :] + t[:, None] * (b - a)[None, :]
    inside = np.zeros(n, dtype=bool)
    from oracle import geom
    for o in polys:
        inside |= geom.point_in_polygon_crossing(pts[:, 0], pts[:, 1], o)
        for k in range(len(o)):
            q, s = o[k], o[(k + 1) % len(o)]
            inside |= geom.dist2_point_segment(pts[:, 0], pts[:, 1], q[0], q[1], s[0], s[1]) < r * r
    crossings = int(np.count_nonzero(inside[1:] != inside[:-1]))
    L = float(np.hypot(*(b - a)))
    return inside.mean() * L, (crossings + 2) * L / n


SQUARE = [(0.0, 0.0), (10.0, 0.0), (10.0, 10.0), (0.0, 10.0)]
L_SHAPE = [(0.0, 0.0), (30.0, 0.0), (30.0, 10.0), (10.0, 10.0), (10.0, 30.0), (0.0, 30.0)]
U_SHAPE = [(0.0, 0.0), (40.0, 0.0), (40.0, 30.0), (30.0, 30.0), (30.0, 10.0), (10.0, 10.0), (10.0, 30.0), (0.0, 30.0)]
CASES = {
    "crossing": ((-20.0, 5.0), (30.0, 5.0), [SQUARE]),
    "diagonal": ((-5.0, -7.0), (17.0, 12.0), [SQUARE]),
    "grazing_edge": ((-20.0, 11.0), (30.0, 11.0), [SQUARE]),            # 1 m above the top edge: the strip only
    "vertex_disc_only": ((11.0, -3.0), (13.0, 3.0), [SQUARE]),          # passes the corner (10, 0) at < r
    "ends_inside_disc": ((10.5, -0.5), (10.9, -0.2), [SQUARE]),
    "wholly_inside": ((3.0, 3.0), (7.0, 6.0), [SQUARE]),                # farther than r from every edge
    "starts_inside": ((5.0, 5.0), (25.0, 9.0), [SQUARE]),
    "l_shape_diagonal": ((25.0, 5.0), (5.0, 25.0), [L_SHAPE]),
    "l_shape_enters_twice": ((-5.0, 20.0), (35.0, 5.0), [L_SHAPE]),
    "u_shape_enters_twice": ((-5.0, 20.0), (45.0, 20.0), [U_SHAPE]),
    "overlapping": ((-5.0, 5.0), (25.0, 5.0), [SQUARE, [(6.0, 2.0), (16.0, 2.0), (16.0, 8.0), (6.0, 8.0)]]),
    "overlapping_same": ((-5.0, 5.0), (25.0, 5.0), [SQUARE, SQUARE]),
    "miss": ((-20.0, 20.0), (30.0, 20.0), [SQUARE]),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_measure_matches_dense_sampling(name):
    a, b, obstacles = CASES[name]
    m = osw.segment_measure(a, b, osw._polys(obstacles), r)
    est, bound = sampled(a, b, obstacles)
    assert abs(m - est) <= bound, (m, est, bound)
    assert osw.knife_edges(np.array([a, b]), obstacles, W) == 0
    if name == "miss":
        assert m == 0.0
    if name == "wholly_inside":
        assert m == pytest.approx(5.0, abs=1e-12)


def test_segments_that_enter_twice_are_cut_in_three():
    a, b, obstacles = CASES["u_shape_enters_twice"]
    # inside the two arms of the U (x in [0, 10] and [30, 40]) grown by r at both sides of each arm
    assert osw.segment_measure(a, b, osw._polys(obstacles), r) == pytest.approx(2 * (10 + 2 * r), abs=1e-9)


def test_zero_length_and_empty():
    polys = osw._polys([SQUARE])
    assert osw.segment_measure((5.0, 5.0), (5.0, 5.0), polys, r) == 0.0
    assert osw.segment_measure((0.0, 0.0), (1.0, 0.0), [], r) == 0.0
    s = osw.sweep(np.array([[5.0, 5.0], [5.0, 5.0], [5.0, 5.0]]), [SQUARE], W)
    assert s == {"n_seg_main": 0, "n_seg_head": 0, "len_main": 0.0, "len_head": 0.0}


def test_layers_and_junction():
    p = np.array([[-20.0, 5.0], [30.0, 5.0], [30.0, -20.0], [-20.0, 5.0], [30.0, 5.0]])
    m = osw.segment_measures(p, [SQUARE], W)
    s = osw.sweep(p, [SQUARE], W, n_main=2)    # segment 0 main, 1 the junction, 2 and 3 headland
    assert s["n_seg_main"] == 1 and s["len_main"] == m[0]
    assert s["n_seg_head"] == (m[2] > 0) + (m[3] > 0) and s["len_head"] == (0.0 + m[2]) + m[3]
    assert osw.sweep(p, [SQUARE], W)["n_seg_main"] == int(np.count_nonzero(m))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_point_violations_imply_hit_segments(seed):
    rng = np.random.default_rng(seed)
    obst = []
    for _ in range(3):
        cx, cy = rng.uniform(40, 460), rng.uniform(30, 170)
        w, h = rng.uniform(5, 40, 2)
        obst.append([(cx - w, cy - h), (cx + w, cy - h), (cx + w, cy + h), (cx - w, cy + h)])
    R = float(rng.uniform(5, 12))
    o = ob.evaluate_candidate(RECT, rp.VehicleParams(), R=R, start_corner=int(rng.integers(4)), obstacles=obst,
                              coverage=False, keep_paths=True)
    p, nm = o["path"], o["n_main"]
    print("knife-edge segments:", osw.knife_edges(p, obst, W))
    assert osw.knife_edges(p, obst, W) == 0
    s = osw.sweep(p, obst, W, nm)
    if o["n_obstacle_viol"] > 0:
        assert s["n_seg_main"] + s["n_seg_head"] > 0
    # every point in O is an end of a segment with m > 0 unless both its segments are zero-length
    m = osw.segment_measures(p, obst, W)
    polys = osw._polys(obst)
    for i in range(len(p)):
        if osw.in_region(p[i, 0], p[i, 1], polys, r * r):
            near = [m[j] for j in (i - 1, i) if 0 <= j < len(m) and np.any(p[j] != p[j + 1])]
            assert not near or max(near) > 0, i
