"""Lattice-tie cases for the coverage rasterisers (TEST INFRASTRUCTURE ONLY).

The span rasteriser of csrc/fcpp_cover.cu places capsule and quad boundaries in floating point and decides a lattice
point with the exact integer predicate only when a boundary falls within its certification margin (at least 0.03
lattice units for capsules, 1e-5 cells for quads).  Random inputs almost never put a point there.  Every case here is
built in integer lattice units (1e-4 m) so that it does, and states how often:

  tie        a lattice point at exactly r from a segment (dist² = r²) that no capsule strictly covers: the strict
             predicate leaves it out;
  near-tie   a lattice point that is not a tie but has a capsule boundary of the union within 1 / EPS_SCALE units of
             it on its row (far inside the margin): only the exact fallback classifies it.

Segments are (ax, ay, bx, by) in units on the lattice (i H, j H); ``metres`` hands them to the library as U / 1e4 m
and asserts that the library's snap q(x) = rint(x 1e4) gives U back.  ``near`` is the strict predicate in Python
integers (no overflow at any magnitude): the reference where raster_oracle.c's int64 products would overflow.
"""
import math

import numpy as np

from oracle.raster import q

EPS_SCALE = 100


def metres(U):
    a = np.asarray(U, dtype=np.int64)
    m = a.astype(np.float64) / 1e4
    assert np.array_equal(q(m), a), "a coordinate does not survive the 1e-4 m snap"
    return m


def near(px, py, seg, r2):
    """dist²((px, py), segment) < r2, exactly (oracle/raster_oracle.c near_segment)."""
    ax, ay, bx, by = seg
    dx, dy, wx, wy = bx - ax, by - ay, px - ax, py - ay
    t, dd = wx * dx + wy * dy, dx * dx + dy * dy
    if t <= 0:
        return wx * wx + wy * wy < r2
    if t >= dd:
        return (px - bx) ** 2 + (py - by) ** 2 < r2
    cr = wx * dy - wy * dx
    return cr * cr < r2 * dd


def on_boundary(px, py, seg, r2):
    """dist²((px, py), segment) == r2 exactly."""
    ax, ay, bx, by = seg
    dx, dy, wx, wy = bx - ax, by - ay, px - ax, py - ay
    t, dd = wx * dx + wy * dy, dx * dx + dy * dy
    if t <= 0:
        return wx * wx + wy * wy == r2
    if t >= dd:
        return (px - bx) ** 2 + (py - by) ** 2 == r2
    cr = wx * dy - wy * dx
    return cr * cr == r2 * dd


def _row_span(seg, r, y):
    """Approximate open x-interval of the capsule on the row y (float; only used to find candidate points)."""
    ax, ay, bx, by = seg
    lo, hi = math.inf, -math.inf
    for cx, cy in ((ax, ay), (bx, by)):
        h2 = float(r) * r - float(y - cy) ** 2
        if h2 > 0:
            h = math.sqrt(h2)
            lo, hi = min(lo, cx - h), max(hi, cx + h)
    dx, dy = bx - ax, by - ay
    if dy == 0:
        if abs(y - ay) < r:
            lo, hi = min(lo, min(ax, bx)), max(hi, max(ax, bx))
        return lo, hi
    L = math.hypot(dx, dy)
    s0, s1 = sorted((ax + ((y - ay) * dx - r * L) / dy, ax + ((y - ay) * dx + r * L) / dy))
    if dx != 0:
        t0, t1 = sorted((ax - (y - ay) * dy / dx, ax + (dx * dx + dy * dy - (y - ay) * dy) / dx))
    else:
        t0, t1 = (-math.inf, math.inf) if 0 <= (y - ay) * dy <= dy * dy else (math.inf, -math.inf)
    a, b = max(s0, t0), min(s1, t1)
    if a < b:
        lo, hi = min(lo, a), max(hi, b)
    return lo, hi


def _rows(seg, r, Y0, H, ny):
    lo, hi = min(seg[1], seg[3]) - r, max(seg[1], seg[3]) + r
    return range(max(0, -((Y0 - lo) // H)), min(ny - 1, (hi - Y0) // H) + 1)


def tie_counts(segs, r, X0, Y0, H, nx, ny):
    """(ties, near-ties) of the union of the capsules of ``segs`` (radius r) on the lattice (X0 + i H, Y0 + j H),
    i < nx, j < ny.  Only the points next to each capsule's row boundaries are examined."""
    r2, S = r * r, EPS_SCALE
    by_row = {}
    cand = set()
    for s in segs:
        for j in _rows(s, r, Y0, H, ny):
            by_row.setdefault(j, []).append(s)
            lo, hi = _row_span(s, r, Y0 + j * H)
            if lo > hi:
                continue
            for x in (lo, hi):
                i = math.floor((x - X0) / H)
                for ii in (i - 1, i, i + 1, i + 2):
                    if 0 <= ii < nx:
                        cand.add((ii, j))
    ties = near_ties = 0
    for i, j in cand:
        px, py = X0 + i * H, Y0 + j * H
        row = by_row[j]
        if any(near(px, py, s, r2) for s in row):
            inside = True
        else:
            inside = False
            if any(on_boundary(px, py, s, r2) for s in row):
                ties += 1
                continue
        ss = [tuple(S * v for v in s) for s in row]
        a = any(near(S * px - 1, S * py, s, r2 * S * S) for s in ss)
        b = any(near(S * px + 1, S * py, s, r2 * S * S) for s in ss)
        if a != b or a != inside:
            near_ties += 1
    return ties, near_ties


def cover_bits(paths, r, X0, Y0, H, nx, ny):
    """Brute force in Python integers: bool [ny, nx], point (X0 + i H, Y0 + j H) covered by a segment of a path."""
    r2 = r * r
    out = np.zeros((ny, nx), dtype=bool)
    for p in paths:
        for s in segments(p):
            lox, hix = min(s[0], s[2]) - r, max(s[0], s[2]) + r
            i0, i1 = max(0, -((X0 - lox) // H)), min(nx - 1, (hix - X0) // H)
            for j in _rows(s, r, Y0, H, ny):
                py = Y0 + j * H
                for i in range(i0, i1 + 1):
                    if not out[j, i] and near(X0 + i * H, py, s, r2):
                        out[j, i] = True
    return out


def segments(path):
    p = [tuple(map(int, v)) for v in np.asarray(path, dtype=object).reshape(-1, 2)]
    return [(a[0], a[1], b[0], b[1]) for a, b in zip(p[:-1], p[1:])]


# ---- constructors: every case is a list of paths (integer [n, 2] arrays, units) on the lattice H Z² ----

def _ext_gcd(a, b):
    if b == 0:
        return (1 if a >= 0 else -1), 0, abs(a)
    x, y, g = _ext_gcd(b, a % b)
    return y, x - (a // b) * y, g


def sums_of_two_squares(n, limit=8):
    """Up to ``limit`` (u, v), 0 < u <= v, with u² + v² = n."""
    out = []
    u = 1
    while 2 * u * u <= n and len(out) < limit:
        v = math.isqrt(n - u * u)
        if v * v == n - u * u:
            out.append((u, v))
        u += 1
    return out


def nearest_reps(r):
    """(exact, below, above): representations of r², of the largest n < r² and of the smallest n > r² that are sums
    of two positive squares."""
    n2 = r * r
    exact = sums_of_two_squares(n2, 2)
    below = above = []
    for d in range(1, 10000):
        below = below or sums_of_two_squares(n2 - d, 1)
        above = above or sums_of_two_squares(n2 + d, 1)
        if below and above:
            break
    return exact, below, above


def _orient(u, v):
    return [(su * a, sv * b) for a, b in ((u, v), (v, u)) for su in (1, -1) for sv in (1, -1)]


def disc_case(r, H):
    """Segment ends at a lattice point + (u, v), u² + v² = r² or the nearest sums of two squares on either side, in
    all eight orientations; each segment points straight away from its lattice point (its end disc decides)."""
    exact, below, above = nearest_reps(r)
    step = -(-3 * r // H) * H
    paths, k = [], 0
    for u0, v0 in exact + below + above:
        g = math.gcd(u0, v0)
        kk = max(1, r // (2 * max(u0, v0) // g))
        for u, v in _orient(u0, v0):
            A = ((k % 6) * step + u, (k // 6) * step + v)
            paths.append(np.array([A, (A[0] + u // g * kk, A[1] + v // g * kk)], dtype=np.int64))
            k += 1
    return paths


def tangent_case(a, b, r, H):
    """Direction (a, b), a² + b² = c², c | r: a segment whose left tangent line runs through the lattice points
    k H (a, b), k = 0..5, at perpendicular distance exactly r; and a segment of the nearby primitive direction
    (a m + j, b m), dy >= 200, j >= 1 the first with gcd(dx, dy) = 1, placed so that the lattice origin's cross product is the integer nearest r |d|: its
    row boundary lies within 0.5 / dy units of the point."""
    c = math.isqrt(a * a + b * b)
    assert c * c == a * a + b * b and r % c == 0
    n = (-b * (r // c), a * (r // c))
    A = (-n[0] - a * (H // 2), -n[1] - b * (H // 2))
    tie = np.array([A, (A[0] + a * (5 * H + H), A[1] + b * (5 * H + H))], dtype=np.int64)
    m = -(-200 // b)
    dx, dy = a * m + 1, b * m
    while math.gcd(dx, dy) != 1:
        dx += 1
    dd = dx * dx + dy * dy
    T = math.isqrt(r * r * dd)
    if (T + 1) ** 2 - r * r * dd < r * r * dd - T * T:
        T += 1
    x, y, _ = _ext_gcd(dx, dy)                # dx x + dy y = 1
    Ax, Ay = -T * y, T * x                    # cross((0, 0) - A, d) = T
    s = (-(Ax * dx + Ay * dy)) // dd - 2      # slide along d: the origin projects into the middle of 5 d
    k = -(-6 * r // (H * c))                  # then move it 6 r across, clear of the tie segment, by a lattice vector
    A = (Ax + s * dx + k * H * b, Ay + s * dy - k * H * a)
    return [tie, np.array([A, (A[0] + 5 * dx, A[1] + 5 * dy)], dtype=np.int64)]


def variants(paths, r, H):
    """The case as given, reversed, mirrored in x and mirrored in y (the lattice H Z² maps onto itself), each copy
    moved by a lattice vector on a 2 x 2 layout.  Every copy's capsules lie within M + r of its own origin
    (M = max |coordinate|, mirrors included), and the copies are 2 (M + r) + 2 H apart: no capsule of one copy
    reaches a point within H of another copy's capsules."""
    M = int(np.abs(np.concatenate(paths)).max())
    D = (2 * (M + r) // H + 3) * H
    out = []
    for k, f in enumerate((lambda p: p, lambda p: p[::-1].copy(), lambda p: p * np.array([-1, 1]),
                           lambda p: p * np.array([1, -1]))):
        out += [f(p) + np.array([(k % 2) * D, (k // 2) * D]) for p in paths]
    return out


def axis_case(r, H):
    """Exactly horizontal and vertical segments with lattice rows / columns at exactly r on both sides and
    disc ties at their ends (the end lies at a lattice point + (u, v), u² + v² = r²)."""
    u, v = (sums_of_two_squares(r * r, 1) or [(0, r)])[0]
    L = 20 * H
    paths = []
    for k, (ex, ey) in enumerate(((u, v), (v, u))):
        y0 = 4 * k * r - (4 * k * r) % H
        A = (ex, y0 + r)
        paths.append(np.array([A, (A[0] + L, A[1])], dtype=np.int64))        # row y0 at exactly r below
        A = (8 * H * (k + 2) + r, -ey)
        paths.append(np.array([A, (A[0], A[1] - L)], dtype=np.int64))        # column at exactly r to the left
    return paths


def near_axis_case(r, H, dxs=(10_000, 123_457, 10_000_019, (1 << 30) - 1)):
    """dy = +-1 with dx from 1 m to 2^30 - 1 units, and the transposed segments.  Each starts r above a lattice row
    (or r right of a lattice column) at a lattice point, so its tangent line grazes that row next to the start; the
    far end stays below 2^30 units from the lattice origin.  The interesting part lies in [-r, 12 r]²."""
    paths = []
    step = -(-3 * r // H) * H
    for k, dx in enumerate(dxs):
        for n, sgn in enumerate((1, -1)):
            y = (2 * k + n) * step // 2 // H * H + step
            paths.append(np.array([(0, y + r), (dx - 1, y + r + sgn)], dtype=np.int64))
            paths.append(np.array([(y + r, 0), (y + r + sgn, dx - 1)], dtype=np.int64))
    return paths


def bbox_window(paths, r, H, pad=2):
    """(X0, Y0, nx, ny): the lattice points (X0 + i H, Y0 + j H) around every capsule, X0 and Y0 multiples of H."""
    P = np.concatenate(paths)
    lo = P.min(0) - r
    hi = P.max(0) + r
    X0, Y0 = (int(lo[0]) // H - pad) * H, (int(lo[1]) // H - pad) * H
    nx, ny = (int(hi[0]) - X0) // H + pad + 1, (int(hi[1]) - Y0) // H + pad + 1
    return X0, Y0, nx, ny


def edge_points(quad, Xc0, Yc0, H, nx, ny):
    """Per edge of a closed quad (integer vertices), the lattice points lying exactly on it."""
    out = []
    for k in range(4):
        (ax, ay), (bx, by) = quad[k], quad[(k + 1) % 4]
        g = math.gcd(bx - ax, by - ay)
        sx, sy = (bx - ax) // g, (by - ay) // g
        n = 0
        for t in range(g + 1):
            x, y = ax + t * sx, ay + t * sy
            if (x - Xc0) % H == 0 and (y - Yc0) % H == 0 and 0 <= (x - Xc0) // H < nx and 0 <= (y - Yc0) // H < ny:
                n += 1
        out.append(n)
    return out


def edge_margin_points(quad, Xc0, Yc0, H, nx, ny, margin=1e-5):
    """Per edge of a closed quad (integer vertices), the lattice points whose row meets the edge within ``margin``
    cells of them (quad_row_interval's AMBIG_Q: only the exact in_quad decides them), exactly on it included.
    Horizontal edges count 0: quad_row_interval decides them with an integer comparison.
    Exact: |x_edge(y) - x| < margin H  <=>  |(ax - x) ey + (y - ay) ex| < margin H |ey|."""
    inv = round(1 / margin)
    out = []
    for k in range(4):
        (ax, ay), (bx, by) = quad[k], quad[(k + 1) % 4]
        ex, ey = bx - ax, by - ay
        n = 0
        if ey != 0:
            for j in range(max(0, -((Yc0 - min(ay, by)) // H)), min(ny - 1, (max(ay, by) - Yc0) // H) + 1):
                y = Yc0 + j * H
                num = ax * ey + (y - ay) * ex            # x_edge(y) = num / ey
                i = round((num / ey - Xc0) / H)
                for ii in (i - 1, i, i + 1):
                    if 0 <= ii < nx and inv * abs(num - (Xc0 + ii * H) * ey) < H * abs(ey):
                        n += 1
        out.append(n)
    return out


# ---- the cases of test_gpu_raster_ties.py / test_raster_ties_cpu.py ----

GEO = np.array([5_123_456_789, 43_210_987_654])   # ~(512 345.6789, 4 321 098.7654) m

# name -> (constructor, r, H, min ties, min near-ties); the lattices are the cases' bounding boxes
CASES = {
    "disc_r16000_H200": (lambda: disc_case(16000, 200), 16000, 200, 48, 14),
    "disc_r16000_H1000": (lambda: disc_case(16000, 1000), 16000, 1000, 16, 14),
    "disc_r16000_H2000": (lambda: disc_case(16000, 2000), 16000, 2000, 16, 14),
    "disc_r17500_H200": (lambda: disc_case(17500, 200), 17500, 200, 44, 12),
    "disc_r17500_H1000": (lambda: disc_case(17500, 1000), 17500, 1000, 16, 12),
    "disc_r17500_H2000": (lambda: disc_case(17500, 2000), 17500, 2000, 16, 12),
    "disc_r180000_H2000": (lambda: disc_case(180000, 2000), 180000, 2000, 62, 14),
    "disc_r1500_H200": (lambda: disc_case(1500, 200), 1500, 200, 16, 8),
    "disc_r1500_H1000": (lambda: disc_case(1500, 1000), 1500, 1000, 16, 8),
}
for _a, _b, _r in ((3, 4, 15000), (5, 12, 13000), (8, 15, 17000), (7, 24, 25000), (20, 21, 29000)):
    for _H in (1000, 200):
        CASES[f"tan_{_a}_{_b}_H{_H}"] = (lambda a=_a, b=_b, r=_r, H=_H: variants(tangent_case(a, b, r, H), r, H),
                                        _r, _H, 48, 4)   # per copy: 12 ties, 1 near-tie
CASES["axis_H200"] = (lambda: axis_case(16000, 200), 16000, 200, 80, 0)
CASES["axis_H1000"] = (lambda: axis_case(16000, 1000), 16000, 1000, 42, 0)
# cases whose brute-force window (g = max(nx, ny), g² lattice points) exceeds 1.2e6 points: marked slow
SLOW_CASES = {"disc_r16000_H200", "disc_r17500_H200", "disc_r180000_H2000", "tan_3_4_H200", "tan_5_12_H200",
              "tan_8_15_H200", "tan_7_24_H200", "tan_20_21_H200"}
SLOW_CELLS = 1_200_000
# r, H, window origin (both axes: the far ends stay below 2^30 units from it), g, min ties, min near-ties
NEAR_AXIS = (16000, 1000, 0, 300, 2, 190)


def case(name):
    make, r, H, mt, mn = CASES[name]
    paths = make()
    X0, Y0, nx, ny = bbox_window(paths, r, H)
    return paths, r, H, X0, Y0, nx, ny, mt, mn


def check_ties(paths, r, X0, Y0, H, nx, ny, mt, mn, name):
    segs = [s for p in paths for s in segments(p)]
    ties, nears = tie_counts(segs, r, X0, Y0, H, nx, ny)
    print(f"{name}: {ties} ties, {nears} near-ties")
    assert ties >= mt and nears >= mn, (name, ties, nears)


def quads(H):
    """Fields with integer vertices whose edges run through cell centres (slopes 1:2, 3:4 and 1:1; centres at
    min + H/2 + (i H, j H)), and one whose 500 m long top edge rises by 1 unit from a cell centre."""
    L, s = 100 * H + H // 2, 40 * H + H // 2
    return {
        "slope_1_2": [(0, 0), (L, 0), (L + 2 * s, s), (s, s)],
        "slope_3_4": [(0, 0), (L, 0), (L + 4 * s, 3 * s), (3 * s, 3 * s)],
        "nearly_flat": [(0, 0), (5_000_000 + H // 2, 0), (5_000_000 + H // 2, s + 1), (5 * H + H // 2, s)],
    }
