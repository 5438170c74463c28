"""Path coverage without a device: the host-side checks of verify_paths / plan_batch(field_coverage=True), the C layout
of fcpp_path_cover against its numpy mirror, and the oracle's field and band coverage on hand-countable cases."""
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _path_cover_oracle as pco  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SQ = [(0.0, 0.0), (10.0, 0.0), (10.0, 10.0), (0.0, 10.0)]


def test_path_cover_struct_matches_c_layout(tmp_path):
    from field_coverage_path_planning_b200 import _lib
    names = _lib.PATH_COVER_DTYPE.names
    src = tmp_path / "pc.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "fcpp.h"\nint main(){printf("%zu'
                   + ' %zu' * len(names) + '\\n",sizeof(fcpp_path_cover)'
                   + "".join(f",offsetof(fcpp_path_cover,{n})" for n in names) + ');return 0;}')
    exe = tmp_path / "pc"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = list(map(int, subprocess.check_output([str(exe)]).split()))
    assert got[0] == _lib.PATH_COVER_DTYPE.itemsize == 48
    assert got[1:] == [_lib.PATH_COVER_DTYPE.fields[n][1] for n in names]


BAD = [
    (dict(paths=[np.zeros((3, 3))]), "every path"),
    (dict(paths=[np.array([[0.0, np.nan]])]), "finite"),
    (dict(paths=[np.zeros((2, 2))], fields=[SQ, SQ]), "path_field is required"),
    (dict(paths=[np.zeros((2, 2))], fields=[SQ, SQ], path_field=[2]), "path_field must lie"),
    (dict(paths=[np.zeros((2, 2))], path_field=[-1]), "path_field must lie"),
    (dict(paths=[np.zeros((2, 2))], fields=[SQ[::-1]]), "counter-clockwise"),
    (dict(paths=[np.zeros((2, 2))], fields=[[(0, 0), (1, 0), (1, np.inf), (0, 1)]]), "finite"),
    (dict(paths=[np.zeros((2, 2))], grid_h=0.0), "grid_h"),
    (dict(paths=[np.zeros((2, 2))], grid_h=0.00015), "grid_h"),
    (dict(paths=[np.zeros((2, 2)), np.zeros((4, 2))], n_main=[1]), "one integer per path"),
    (dict(paths=[np.zeros((2, 2))], n_main=[3]), r"\[0, len\(path\)\]"),
    (dict(paths=[np.zeros((2, 2))], n_main=[-1]), r"\[0, len\(path\)\]"),
    (dict(paths=[np.zeros((2, 2))], headland_width=[1.0, 2.0]), "headland_width"),
    (dict(paths=[np.zeros((2, 2))], headland_width=np.nan), "finite"),
    (dict(paths=[np.zeros((2, 2))], obstacles=[[[(0, 0), (1, 0)]]]), "obstacle"),
    (dict(paths=[np.zeros((2, 2))], obstacles=[[], [[(0, 0), (1, 0), (1, 1)]]]), "one .* polygon list per field"),
]


@pytest.mark.parametrize("kw,msg", BAD)
def test_verify_paths_rejects_bad_input_on_the_host(kw, msg):
    """Every check runs before the device is looked for: without a GPU these raise ValueError, not FcppError."""
    import field_coverage_path_planning_b200 as fc
    kw = dict(kw)
    paths, fields = kw.pop("paths"), kw.pop("fields", [SQ])
    with pytest.raises(ValueError, match=msg):
        fc.verify_paths(paths, fields, **kw)


def test_plan_batch_field_coverage_needs_paths():
    import field_coverage_path_planning_b200 as fc
    with pytest.raises(ValueError, match="outputs='paths'"):
        fc.plan_batch([SQ], field_coverage=True)


def test_verify_paths_empty_batch_needs_no_device():
    import field_coverage_path_planning_b200 as fc
    from field_coverage_path_planning_b200 import _lib
    out = fc.verify_paths([], [SQ])
    assert out.dtype == _lib.PATH_COVER_DTYPE and len(out) == 0


# Hand-countable oracle cases: the 10 m square at h = 1 m has the cell centres 0.5, 1.5, ..., 9.5 on both axes.
def test_oracle_single_segment():
    seg = np.array([[0.0, 5.0], [10.0, 5.0]])
    # r = 1: the rows y = 4.5 and 5.5 (|y - 5| < 1), all ten columns
    assert pco.field_coverage(SQ, seg, 2.0, 1.0) == (100, 20)
    # the same segment as main work, a point as headland: the field counts both layers
    assert pco.field_coverage(SQ, np.vstack([seg, [[0.5, 0.5], [0.5, 0.5]]]), 2.0, 1.0, n_main=2) == (100, 21)
    # a one-point layer has no segment
    assert pco.field_coverage(SQ, np.vstack([seg, [[0.5, 0.5]]]), 2.0, 1.0, n_main=2) == (100, 20)
    # band of R = 2: the centres outside the closed inset [2, 8]^2, 100 - 36 = 64
    head = np.array([[0.0, 1.0], [10.0, 1.0]])
    assert pco.band_coverage_of(SQ, 2.0, head, 2.0, 1.0) == (64, 20)
    # ... counted from the headland layer only (n_main = 2: the segment is main work, nothing is headland)
    assert pco.band_coverage_of(SQ, 2.0, head, 2.0, 1.0, n_main=2) == (64, 0)
    assert pco.band_coverage_of(SQ, 2.0, np.vstack([head, head[::-1]]), 2.0, 1.0, n_main=2) == (64, 20)
    # an inset that collapses makes the band the whole field; a width <= 0 means no band
    assert pco.band_coverage_of(SQ, 6.0, head, 2.0, 1.0) == (100, 20)
    assert pco.band_coverage_of(SQ, 0.0, head, 2.0, 1.0) == (0, 0)


def test_oracle_cell_centre_tie():
    """A centre exactly r from the segment is not covered (strict predicate); a hair more radius covers it."""
    seg = np.array([[0.0, 5.0], [10.0, 5.0]])
    assert pco.field_coverage(SQ, seg, 1.0, 1.0) == (100, 0)
    assert pco.field_coverage(SQ, seg, 1.0002, 1.0) == (100, 20)
    # end discs: a degenerate segment on a cell corner reaches the four nearest centres (sqrt(0.5) m away) once r,
    # snapped to 1e-4 m, exceeds that distance
    pt = np.array([[5.0, 5.0], [5.0, 5.0]])
    assert pco.field_coverage(SQ, pt, 1.4144, 1.0)[1] == 4
    assert pco.field_coverage(SQ, pt, 1.4142, 1.0)[1] == 0
