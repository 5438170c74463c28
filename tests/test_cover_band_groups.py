"""The coverage kernel evaluates the headland bands of all start corners of one (field, R) together when every
headland straight is axis-aligned (csrc/fcpp_cover.cu: band_grouped): one rectangle set, and at each physical
corner an ARC variant (turn arcs + reverse fill, shared by the three other start corners) and a START variant
(the loops' first points and the joins between loops).  Checked here:

  * on the CPU, a restatement of that decomposition (band_groups below) gives the brute-force counts of
    raster_oracle.c for every start corner;
  * on the GPU, the de-duplicated batches (grouped bands) give the same summaries, byte for byte, as the batches
    without de-duplication (cover mode bit 1: one band per candidate), across start-corner subsets, candidate
    orders, duplicates, dead candidates, shards, turn models and working widths.
"""
import math
from dataclasses import replace

import numpy as np
import pytest

from oracle import geom, raster, ref_planner as rp
from oracle.zoned_model import _in_quad_mask


def band_groups(fs, h=0.1):
    """[(band cells, covered cells) or None] for start corners 0..3 of the field and R of ``fs``, evaluated
    the way band_grouped does: the straights of every loop (the same for every start corner) are the
    rectangles; at physical corner c lies either its ARC material (per loop: corner, turn arc, loop-0 reverse
    fill, corner) when c is not the start corner, or its START material (the loops' first points and the
    joins between them).  Start corner sc uses arc(c) for c != sc and start(sc), and
        cov(sc) = |U ∩ W| + sum over its zones Z of (bits(Z) - |U ∩ W ∩ Z|).
    None for every start corner when a straight is not axis-aligned (the kernel keeps those bands apart), and
    for a start corner whose zones overlap or hold an entry outside their corner's quadrant (per-candidate
    fall-back)."""
    v = fs.vehicle
    W, R = v.working_width, v.min_turn_radius
    r = int(raster.q(W / 2))
    X0, Y0, H, nx, ny = raster.band_dims(fs.field_vertices, h)
    Xc0, Yc0 = X0 + H // 2, Y0 + H // 2
    org = np.array([Xc0, Yc0], dtype=np.int64)
    fq = raster.q(np.asarray(fs.field_vertices, dtype=np.float64)) - org
    mq = raster.q(np.asarray(geom.inset_convex(fs.field_vertices, fs.headland_width), dtype=np.float64)) - org
    xs, ys = np.arange(nx, dtype=np.int64) * H, np.arange(ny, dtype=np.int64) * H
    band = _in_quad_mask(fq, xs, ys) & ~_in_quad_mask(mq, xs, ys)
    K = math.ceil(fs.headland_width / W)
    rings = [np.asarray(geom.inset_convex(fs.field_vertices, W / 2 + k * W), dtype=np.float64) for k in range(K)]
    snapped = [raster.q(ring) - org for ring in rings]

    # the rectangles: straight c -> c + 1 of every loop
    rmask = np.zeros((ny, nx), dtype=bool)
    for p4 in snapped:
        for c in range(4):
            p, qq = p4[c], p4[(c + 1) % 4]
            if (p[0] == qq[0]) == (p[1] == qq[1]):
                return [None] * 4                     # slanted (or degenerate) straight: no grouping
            if p[0] == qq[0]:
                x, ylo, yhi = int(p[0]), int(min(p[1], qq[1])), int(max(p[1], qq[1]))
                ia, ib, ja, jb = (x - r) // H + 1, -((-(x + r)) // H) - 1, -((-ylo) // H), yhi // H
            else:
                y, xlo, xhi = int(p[1]), int(min(p[0], qq[0])), int(max(p[0], qq[0]))
                ia, ib, ja, jb = -((-xlo) // H), xhi // H, (y - r) // H + 1, -((-(y + r)) // H) - 1
            ia, ib, ja, jb = max(ia, 0), min(ib, nx - 1), max(ja, 0), min(jb, ny - 1)
            if ia <= ib and ja <= jb:
                rmask[ja:jb + 1, ia:ib + 1] = True

    # the materials, as polyline pieces (metres): m = c the arc material of corner c, m = 4 + c its start material
    pieces = {}
    for c in range(4):
        arc_pieces = []
        for k in range(K):
            corner = rings[k][c]
            arc = rp.corner_turn_arc(tuple(corner), c, R, rp.CORNER_ARC_POINTS, fs.turn_model, fs.clothoid_share)
            part = [corner[None, :], arc]
            if k == 0 and rp.should_apply_reverse_filling(fs, c) and rp.gap_gate(tuple(corner), c, R, W):
                part.append(rp.optimal_reverse_path(fs, arc[-1], arc[-2])[0])
            part.append(corner[None, :])
            arc_pieces.append(np.vstack(part))
        pieces[c] = arc_pieces
        pieces[4 + c] = [np.vstack([rings[0][c][None, :]] + [ring[c][None, :] for ring in rings])]

    def inside_main(x, y):
        return all((int(mq[(k + 1) % 4][0]) - int(mq[k][0])) * (y - int(mq[k][1])) -
                   (int(mq[(k + 1) % 4][1]) - int(mq[k][1])) * (x - int(mq[k][0])) >= 0 for k in range(4))

    L = raster.lib()
    midx2, midy2 = (nx - 1) * H, (ny - 1) * H
    zone, bad, gmask = {}, set(), {}
    for m, plist in pieces.items():
        c0 = snapped[0][m % 4]
        quad = (2 if 2 * int(c0[1]) >= midy2 else 0) | (1 if 2 * int(c0[0]) >= midx2 else 0)
        bits = np.zeros((nx * ny + 7) // 8, dtype=np.uint8)
        box = None
        for piece in plist:
            pts = raster.q(piece) - org
            for a, b in zip(pts[:-1], pts[1:]):
                x0, x1 = min(a[0], b[0]) - r, max(a[0], b[0]) + r
                y0, y1 = min(a[1], b[1]) - r, max(a[1], b[1]) + r
                if inside_main(x0, y0) and inside_main(x1, y0) and inside_main(x1, y1) and inside_main(x0, y1):
                    continue                          # C2
                jlo = max((min(a[1], b[1]) - r) // H + 1, 0)
                jhi = min(-((-(max(a[1], b[1]) + r)) // H) - 1, ny - 1)
                cl, ch = max((min(a[0], b[0]) - r) // H, 0), min(-((-(max(a[0], b[0]) + r)) // H), nx - 1)
                if jlo > jhi or cl > ch:
                    continue
                if ((2 if (a[1] + b[1]) >= midy2 else 0) | (1 if (a[0] + b[0]) >= midx2 else 0)) != quad:
                    bad.add(m)
                box = (cl, ch, jlo, jhi) if box is None else \
                    (min(box[0], cl), max(box[1], ch), min(box[2], jlo), max(box[3], jhi))
                seg = np.ascontiguousarray(np.array([a, b], dtype=np.int64) + org)
                L.fcpo_raster(raster._i64p(seg), 2, r, Xc0, Yc0, H, nx, ny, bits.ctypes.data)
        gmask[m] = np.unpackbits(bits, bitorder="little")[:nx * ny].reshape(ny, nx).astype(bool)
        zone[m] = box

    uw = rmask & band
    out = []
    for sc in range(4):
        used = [m for m in [c for c in range(4) if c != sc] + [4 + sc] if zone[m] is not None]
        boxes = [zone[m] for m in used]
        overlap = any(a[0] <= b[1] and b[0] <= a[1] and a[2] <= b[3] and b[2] <= a[3]
                      for i, a in enumerate(boxes) for b in boxes[i + 1:])
        if overlap or any(m in bad for m in used):
            out.append(None)
            continue
        cov = int(uw.sum())
        for m in used:
            cl, ch, jlo, jhi = zone[m]
            z = np.zeros((ny, nx), dtype=bool)
            z[jlo:jhi + 1, cl:ch + 1] = True
            assert not (gmask[m] & band & ~z).any(), "C3 violated: a general entry covers a band cell outside its zone"
            cov += int(((rmask | gmask[m]) & band & z).sum()) - int((uw & z).sum())
        out.append((int(band.sum()), cov))
    return out


FIELDS = {
    "rect120x80": ([(0, 0), (120, 0), (120, 80), (0, 80)], 3.2, (5.0, 8.0, 11.0), 0.1),
    "rect500x200": ([(0, 0), (500, 0), (500, 200), (0, 200)], 3.2, (7.2,), 0.1),
    "offset_rect": ([(1000.3, 2000.7), (1180.3, 2000.7), (1180.3, 2075.7), (1000.3, 2075.7)], 3.2, (6.4, 9.6), 0.25),
    "narrow_loops": ([(0, 0), (90, 0), (90, 70), (0, 70)], 0.8, (6.0,), 0.1),
    "sheared": ([(0, 0), (200, 0), (230, 90), (30, 90)], 3.2, (8.0,), 0.25),
    "tilted": ([(0, 0), (150, 20), (140, 95), (-10, 75)], 3.2, (8.0,), 0.25),
    # 16 loops (K = ceil(R / W) at its maximum)
    "k16": ([(0, 0), (140, 0), (140, 90), (0, 90)], 0.5, (8.0,), 0.1),
    # off the origin, so the reverse fills (rays to the lines x = 0, x = extent, ...) differ per corner
    "asym_fills": ([(30.0, 10.0), (150.0, 10.0), (150.0, 95.0), (30.0, 95.0)], 3.2, (4.0, 1.7), 0.1),
}


def _setup(verts, W, R):
    return rp.setup_field(replace(rp.VehicleParams(), working_width=W, min_turn_radius=R),
                          field_vertices=[tuple(map(float, v)) for v in verts], obstacles=[])


@pytest.mark.parametrize("case", sorted(FIELDS))
def test_grouped_band_model_equals_brute_force(case):
    """band_groups == raster.band_coverage of each start corner's own headland path, for every start corner that
    the grouped evaluation takes; rectangular fields take all four, fields with a slanted straight none."""
    verts, W, radii, h = FIELDS[case]
    grouped = 0
    for R in radii:
        fs = _setup(verts, W, R)
        model = band_groups(fs, h)
        for sc in range(4):
            if model[sc] is None:
                continue
            hp = rp.plan_complete_coverage(fs, start_corner=sc)["headland"]["path"]
            assert model[sc] == raster.band_coverage(fs, hp, h), (case, R, sc, model[sc])
            grouped += 1
    if case in ("sheared", "tilted"):
        assert grouped == 0, case
    else:
        assert grouped == 4 * len(radii), (case, grouped)


def test_grouped_band_model_covers_asymmetric_fills():
    """The asym_fills field really has reverse fills of different lengths at different corners."""
    verts, W, radii, _ = FIELDS["asym_fills"]
    lens = []
    for R in radii:
        fs = _setup(verts, W, R)
        ring = geom.inset_convex(fs.field_vertices, W / 2)
        n = []
        for c in range(4):
            if rp.should_apply_reverse_filling(fs, c) and rp.gap_gate(tuple(ring[c]), c, R, W):
                arc = rp.corner_turn_arc(tuple(ring[c]), c, R)
                n.append(len(rp.optimal_reverse_path(fs, arc[-1], arc[-2])[0]))
            else:
                n.append(0)
        lens.append(n)
    assert len(set(lens[0])) > 1 and min(lens[0]) > 0, lens


# ------------------------------------------------------------------------------------------------------------------
# GPU: grouped (default, de-duplicated) == one band per candidate (cover mode bit 1)
# ------------------------------------------------------------------------------------------------------------------
RECT = [(0, 0), (500, 0), (500, 200), (0, 200)]


@pytest.fixture(scope="module")
def fc():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import field_coverage_path_planning_b200 as fc
    return fc


def _per_candidate(fc, fields, veh, cand, **kw):
    from field_coverage_path_planning_b200 import _lib
    h = _lib.handle(0)
    try:
        h.check(h.lib.fcpp_set_cover_mode(h.h, 2))
        return fc.plan_batch(fields, veh, cand, **kw).summary
    finally:
        h.check(h.lib.fcpp_set_cover_mode(h.h, 0))


def _same(fc, fields, veh, cand, **kw):
    got = fc.plan_batch(fields, veh, cand, **kw).summary
    ref = _per_candidate(fc, fields, veh, cand, **kw)
    assert got.tobytes() == ref.tobytes()
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("corners", [[0, 1, 2, 3], [1], [0, 2], [3, 1]])
def test_gpu_grouped_band_equals_per_candidate(fc, corners):
    veh = fc.VehicleParams()
    cand = fc.make_candidates(1, radii=np.linspace(5.0, 12.0, 64), start_corners=corners)
    s = _same(fc, [RECT], veh, cand)
    assert (s["status"] == 0).all() and (s["cov_cells"] > 0).all()
    # shuffled explicit order, duplicates and dead candidates (a radius whose R-inset is empty)
    rng = np.random.default_rng(len(corners))
    n = len(cand["field_id"])
    idx = np.concatenate([rng.permutation(n), rng.integers(0, n, 17)])
    mixed = {k: v[idx] for k, v in cand.items()}
    mixed["R"] = mixed["R"].copy()
    mixed["R"][rng.integers(0, len(idx), 5)] = 150.0
    s = _same(fc, [RECT], veh, mixed)
    assert (s["status"] != 0).sum() >= 1
    # groups cut by shard ranges
    from field_coverage_path_planning_b200.dist import shard_candidates
    for rank in range(3):
        part, _ = shard_candidates(mixed, 3, rank)
        _same(fc, [RECT], veh, part)


@pytest.mark.gpu
@pytest.mark.parametrize("turn_model", ["clothoid", "omega"])
def test_gpu_grouped_band_turn_models(fc, turn_model):
    cand = fc.make_candidates(2, radii=[5.0, 8.0, 11.0], start_corners=[0, 1, 2, 3])
    _same(fc, [RECT, [(0, 0), (120, 0), (120, 80), (0, 80)]], fc.VehicleParams(), cand, turn_model=turn_model)


@pytest.mark.gpu
@pytest.mark.parametrize("width", [2.4, 0.5])
def test_gpu_grouped_band_working_widths(fc, width):
    veh = replace(fc.VehicleParams(), working_width=width)
    cand = fc.make_candidates(2, radii=[5.0, 7.9], start_corners=[0, 1, 2, 3])
    _same(fc, [RECT, [(30.0, 10.0), (150.0, 10.0), (150.0, 95.0), (30.0, 95.0)]], veh, cand)


@pytest.mark.gpu
def test_gpu_grouped_band_fallbacks(fc):
    """Narrow fields whose corner zones overlap (the start corners fall back to the per-candidate evaluation inside
    the group's CTA), a field with slanted straights (not grouped), and a coarse and a fine grid."""
    fields = [
        [(0, 0), (45, 0), (45, 300), (0, 300)],
        [(0, 0), (24, 0), (24, 60), (0, 60)],
        [(0, 0), (500, 0), (580, 200), (80, 200)],
        [(-250.05, -100.02), (249.95, -100.02), (249.95, 99.98), (-250.05, 99.98)],
    ]
    cand = fc.make_candidates(len(fields), radii=[5.0, 6.4, 8.0, 11.0], start_corners=[0, 1, 2, 3])
    for grid_h in (0.1, 0.25):
        _same(fc, fields, fc.VehicleParams(), cand, grid_h=grid_h)
