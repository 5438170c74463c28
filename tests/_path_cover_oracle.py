"""Brute-force statement of the whole-field and headland-band coverage of a path (TEST INFRASTRUCTURE ONLY).

Built on the integer rasterisation oracle (oracle/raster.py, oracle/raster_oracle.c): every cell of every segment's
bounding box is tested with the exact predicate, independently of the span rasteriser of csrc/fcpp_cover.cu.
"""
import numpy as np

from oracle import geom
from oracle.raster import _i64p, band_dims, lib, q

# ---- whole-field and headland-band coverage of a path (include/fcpp.h fcpp_path_cover, DESIGN.md §3.10) ----
# Lattice: A11's, cell centres q(bbox_min) + H/2 + (i H, j H).  A path is main work (its first n_main points) then
# headland; the segment joining the two layers belongs to neither.  Field cells = centre inside-or-on the field quad;
# covered by the segments of both layers.  Band cells = A11's band (field minus the closed mitred R-inset, D1; an
# empty inset or |area| < 1 m^2 leaves the whole field; R <= 0: no band), covered by the headland layer only.

def _cell_lattice(field_vertices, h):
    X0, Y0, H, nx, ny = band_dims(field_vertices, h)
    return X0 + H // 2, Y0 + H // 2, H, nx, ny


def _layer_bits(path, n_main, r, Xc0, Yc0, H, nx, ny, with_main):
    """Cover bits (fcpo_raster, row-major nx x ny) of the headland layer of ``path`` (its points from n_main on) and,
    with ``with_main``, of its main layer (the points before n_main)."""
    pts = np.ascontiguousarray(q(np.asarray(path, dtype=np.float64)).reshape(-1, 2))
    bits = np.zeros((nx * ny + 7) // 8, dtype=np.uint8)
    for part in ((pts[:n_main], pts[n_main:]) if with_main else (pts[n_main:],)):
        part = np.ascontiguousarray(part)
        if len(part) >= 2:
            lib().fcpo_raster(_i64p(part), len(part), int(q(r)), Xc0, Yc0, H, nx, ny, bits.ctypes.data)
    return bits


def _count_cells(field_q, inset_q, bits, Xc0, Yc0, H, nx, ny, rows=256):
    """(cells whose centre is in the closed field quad and not in the closed inset, those with their bit set):
    the exact integer test of raster_oracle.c in_convex, row block by row block."""
    total = cov = 0
    px = Xc0 + H * np.arange(nx, dtype=np.int64)[None, :]

    def inside(poly, py):
        ok = np.ones((py.shape[0], nx), dtype=bool)
        for k in range(4):
            ax, ay = int(poly[k][0]), int(poly[k][1])
            bx, by = int(poly[(k + 1) % 4][0]), int(poly[(k + 1) % 4][1])
            ok &= (bx - ax) * (py - ay) - (by - ay) * (px - ax) >= 0
        return ok

    for j0 in range(0, ny, rows):
        j1 = min(ny, j0 + rows)
        py = Yc0 + H * np.arange(j0, j1, dtype=np.int64)[:, None]
        m = inside(field_q, py)
        if inset_q is not None:
            m &= ~inside(inset_q, py)
        c0, c1 = j0 * nx, j1 * nx
        b = np.unpackbits(bits[c0 // 8:(c1 + 7) // 8], bitorder="little")[c0 % 8:c0 % 8 + (c1 - c0)]
        total += int(m.sum())
        cov += int((b.reshape(j1 - j0, nx).astype(bool) & m).sum())
    return total, cov


def field_coverage(field_vertices, path, W, h=0.1, n_main=0):
    """(field cells, field cells covered by the W/2 buffer of both layers of ``path``)."""
    Xc0, Yc0, H, nx, ny = _cell_lattice(field_vertices, h)
    assert H % 2 == 0
    bits = _layer_bits(path, int(n_main), W / 2, Xc0, Yc0, H, nx, ny, True)
    return _count_cells(q(np.asarray(field_vertices, dtype=np.float64)), None, bits, Xc0, Yc0, H, nx, ny)


def band_coverage_of(field_vertices, R, path, W, h=0.1, n_main=0):
    """A11 of (field, headland width R): (band cells, band cells covered by the W/2 buffer of the HEADLAND layer of
    ``path``, its points from n_main on).  oracle.raster.band_coverage for (field, R) instead of a FieldSetup; R <= 0:
    no band, (0, 0)."""
    if not R > 0:
        return 0, 0
    main = geom.inset_convex(field_vertices, R)
    if main is not None and abs(geom.signed_area(main)) < 1.0:
        main = None
    Xc0, Yc0, H, nx, ny = _cell_lattice(field_vertices, h)
    assert H % 2 == 0
    bits = _layer_bits(path, int(n_main), W / 2, Xc0, Yc0, H, nx, ny, False)
    inset_q = None if main is None else q(np.asarray(main, dtype=np.float64))
    return _count_cells(q(np.asarray(field_vertices, dtype=np.float64)), inset_q, bits, Xc0, Yc0, H, nx, ny)
