"""Segment-level obstacle sweep (DESIGN.md §3.9): how far each segment of a path drives through the obstacle region
O, stated in numpy / Python floats.  The CUDA kernels of csrc/fcpp_sweep.cu evaluate the same expressions in the
same order (the library is built with -fmad=false), so their per-segment measures are the same doubles.

O is the set of points D3 counts (ref_planner.obstacle_violations): inside some obstacle polygon (even-odd
crossing) or at squared distance < r^2 from one of its edges, r = W / 2.

Measure of a segment a -> b:
  1. for every polygon edge, the parameter interval on which a + t (b - a) lies within r of the edge (the capsule
     is convex: the hull of its two vertex-disc intervals and its strip interval), clipped to [0, 1];
  2. breakpoints {0, 1} and the interval ends, distinct, ascending;
  3. every sub-interval classified by the D3 predicate at its midpoint;
  4. m = (sum of the inside sub-intervals' lengths, left to right) * |b - a|.
A zero-length segment measures 0.  Per layer: the number of segments with m > 0 and the sum of m, left to right in
segment order.
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import numpy as np

KNIFE_REL = 1e-12


def _polys(obstacles) -> List[np.ndarray]:
    return [np.asarray(o, dtype=np.float64).reshape(-1, 2) for o in obstacles if len(o)]


def in_region(x: float, y: float, polys: Sequence[np.ndarray], r2: float) -> bool:
    """The D3 point predicate (oracle/geom.py point_in_polygon_crossing, dist2_point_segment) for one point."""
    for o in polys:
        n = len(o)
        inside = False
        for k in range(n):
            ax, ay = float(o[k, 0]), float(o[k, 1])
            bx, by = float(o[(k + 1) % n, 0]), float(o[(k + 1) % n, 1])
            if (ay > y) != (by > y):
                xi = ax + (y - ay) * (bx - ax) / (by - ay)
                if x < xi:
                    inside = not inside
            dx, dy, wx, wy = bx - ax, by - ay, x - ax, y - ay
            dd = dx * dx + dy * dy
            tt = wx * dx + wy * dy
            u = tt / dd if dd > 0.0 else 0.0
            u = min(max(u, 0.0), 1.0)
            qx, qy = wx - u * dx, wy - u * dy
            if qx * qx + qy * qy < r2:
                return True
        if inside:
            return True
    return False


def capsule_interval_raw(ax, ay, dx, dy, A, px, py, qx, qy, r, r2) -> Tuple[float, float]:
    """Parameter interval [lo, hi] of the whole line a + t d within r of the edge p q (lo > hi: empty)."""
    lo, hi = math.inf, -math.inf
    for cx, cy in ((px, py), (qx, qy)):
        wx, wy = ax - cx, ay - cy
        B = dx * wx + dy * wy
        Cc = (wx * wx + wy * wy) - r2
        disc = B * B - A * Cc
        if disc >= 0.0:
            s = math.sqrt(disc)
            lo = min(lo, (-B - s) / A)
            hi = max(hi, (-B + s) / A)
    ex, ey = qx - px, qy - py
    ee = ex * ex + ey * ey
    if ee > 0.0:
        wx, wy = ax - px, ay - py
        s_lo, s_hi = -math.inf, math.inf
        w0, w1 = wx * ex + wy * ey, dx * ex + dy * ey       # projection on the edge, times |e|: in [0, ee]
        h0, h1 = ex * wy - ey * wx, ex * dy - ey * dx       # distance from the edge's line, times |e|: in [-rl, rl]
        rl = r * math.sqrt(ee)
        ok = True
        if w1 == 0.0:
            ok = 0.0 <= w0 <= ee
        else:
            ta, tb = (0.0 - w0) / w1, (ee - w0) / w1
            if w1 < 0.0:
                ta, tb = tb, ta
            s_lo, s_hi = max(s_lo, ta), min(s_hi, tb)
        if h1 == 0.0:
            ok = ok and abs(h0) <= rl
        else:
            ta, tb = (-rl - h0) / h1, (rl - h0) / h1
            if h1 < 0.0:
                ta, tb = tb, ta
            s_lo, s_hi = max(s_lo, ta), min(s_hi, tb)
        if ok and s_lo <= s_hi:
            lo, hi = min(lo, s_lo), max(hi, s_hi)
    return lo, hi


def capsule_interval(ax, ay, dx, dy, A, px, py, qx, qy, r, r2) -> Optional[Tuple[float, float]]:
    """capsule_interval_raw clipped to [0, 1]; None when empty or a single point."""
    lo, hi = capsule_interval_raw(ax, ay, dx, dy, A, px, py, qx, qy, r, r2)
    lo, hi = max(lo, 0.0), min(hi, 1.0)
    return (lo, hi) if lo < hi else None


def segment_measure(a, b, polys: Sequence[np.ndarray], r: float) -> float:
    """Metres of the segment a -> b inside O."""
    ax, ay, bx, by = float(a[0]), float(a[1]), float(b[0]), float(b[1])
    dx, dy = bx - ax, by - ay
    A = dx * dx + dy * dy
    if A == 0.0 or not polys:
        return 0.0
    r2 = r * r
    bps = {0.0, 1.0}
    for o in polys:
        n = len(o)
        for k in range(n):
            iv = capsule_interval(ax, ay, dx, dy, A, float(o[k, 0]), float(o[k, 1]), float(o[(k + 1) % n, 0]),
                                  float(o[(k + 1) % n, 1]), r, r2)
            if iv is not None:
                bps.update(iv)
    ts = sorted(bps)
    s = 0.0
    for t0, t1 in zip(ts[:-1], ts[1:]):
        tm = 0.5 * (t0 + t1)
        if in_region(ax + tm * dx, ay + tm * dy, polys, r2):
            s += t1 - t0
    return s * math.sqrt(A)


def segment_measures(path, obstacles, working_width: float) -> np.ndarray:
    """m of every segment i -> i + 1 of ``path`` [n, 2]."""
    p = np.asarray(path, dtype=np.float64).reshape(-1, 2)
    polys = _polys(obstacles)
    r = working_width / 2
    return np.array([segment_measure(p[i], p[i + 1], polys, r) for i in range(len(p) - 1)], dtype=np.float64)


def sweep(path, obstacles, working_width: float, n_main: Optional[int] = None) -> dict:
    """The per-path record of fcpp_sweep: segments of main_work.path (points [0, n_main)) and of headland.path
    (points [n_main, n)); the junction n_main - 1 -> n_main belongs to neither.  Sums left to right."""
    p = np.asarray(path, dtype=np.float64).reshape(-1, 2)
    n = len(p)
    nm = n if n_main is None else int(n_main)
    m = segment_measures(p, obstacles, working_width)
    out = {"n_seg_main": 0, "n_seg_head": 0, "len_main": 0.0, "len_head": 0.0}
    for i, v in enumerate(m):
        if i + 1 < nm:
            layer = "main"
        elif i >= nm:
            layer = "head"
        else:
            continue
        if v > 0.0:
            out["n_seg_" + layer] += 1
            out["len_" + layer] += float(v)
    return out


def knife_edges(path, obstacles, working_width: float) -> int:
    """Number of knife-edge segments of ``path`` (see knife_mask)."""
    return int(np.count_nonzero(knife_mask(path, obstacles, working_width)))


def knife_mask(path, obstacles, working_width: float) -> np.ndarray:
    """[n - 1] bool: the segments whose measure or hit flag hinges on the last bits: a line tangent to a vertex disc (discriminant
    within KNIFE_REL of zero, relative), a segment parallel to an edge at distance r (relative), or a capsule interval
    that touches the segment only at an end (within KNIFE_REL of t = 0 or t = 1)."""
    p = np.asarray(path, dtype=np.float64).reshape(-1, 2)
    polys = _polys(obstacles)
    r = working_width / 2
    r2 = r * r
    mask = np.zeros(max(len(p) - 1, 0), dtype=bool)
    for i in range(len(p) - 1):
        ax, ay, bx, by = map(float, (p[i, 0], p[i, 1], p[i + 1, 0], p[i + 1, 1]))
        dx, dy = bx - ax, by - ay
        A = dx * dx + dy * dy
        if A == 0.0:
            continue
        knife = False
        for o in polys:
            n = len(o)
            for k in range(n):
                px, py = float(o[k, 0]), float(o[k, 1])
                qx, qy = float(o[(k + 1) % n, 0]), float(o[(k + 1) % n, 1])
                for cx, cy in ((px, py), (qx, qy)):
                    wx, wy = ax - cx, ay - cy
                    B = dx * wx + dy * wy
                    Cc = (wx * wx + wy * wy) - r2
                    disc = B * B - A * Cc
                    if abs(disc) <= KNIFE_REL * max(B * B, abs(A * Cc)):
                        knife = True
                ex, ey = qx - px, qy - py
                ee = ex * ex + ey * ey
                if ee > 0.0:
                    h1 = ex * dy - ey * dx
                    h0 = ex * (ay - py) - ey * (ax - px)
                    rl = r * math.sqrt(ee)
                    if abs(h1) <= KNIFE_REL * (abs(ex * dy) + abs(ey * dx)) and abs(abs(h0) - rl) <= KNIFE_REL * rl:
                        knife = True
                lo, hi = capsule_interval_raw(ax, ay, dx, dy, A, px, py, qx, qy, r, r2)
                if lo <= hi and (abs(hi) <= KNIFE_REL or abs(lo - 1.0) <= KNIFE_REL):
                    knife = True
        mask[i] = knife
    return mask

