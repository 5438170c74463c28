"""CPU-side tests (no GPU): the C-ABI library loads and exports every symbol include/fcpp.h
declares, the ctypes mirrors match the C structs, host set-up logic (A2) is right, and the product
fails LOUDLY without a CUDA device (no CPU fallback)."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    import field_coverage_path_planning_b200 as fc
    return fc


def test_library_exports_match_header_and_abi_version(built):
    from field_coverage_path_planning_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "fcpp.h")).read()
    declared = set(re.findall(r"\b(fcpp_[a-z_0-9]+)\s*\(", hdr))
    declared -= {"fcpp_handle"}
    L = _lib.load()
    for name in declared:
        assert hasattr(L, name), name
    assert declared == set(_lib.EXPORTS)
    assert L.fcpp_abi_version() == _lib.ABI_VERSION == 5


def test_struct_mirrors_match_c_layout(built, tmp_path):
    """sizeof/offsetof of the C structs (compiled with gcc from include/fcpp.h) == ctypes/numpy mirrors."""
    from field_coverage_path_planning_b200 import _lib
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "fcpp.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu\\n",'
                   'sizeof(fcpp_vehicle),sizeof(fcpp_batch),sizeof(fcpp_summary),sizeof(fcpp_outputs),'
                   'offsetof(fcpp_batch,n_cand),offsetof(fcpp_batch,grid_h),offsetof(fcpp_summary,cov_cells));return 0;}')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = list(map(int, subprocess.check_output([str(exe)]).split()))
    assert got[0] == ctypes.sizeof(_lib.Vehicle)
    assert got[1] == ctypes.sizeof(_lib.Batch)
    assert got[2] == _lib.SUMMARY_DTYPE.itemsize == 176
    assert got[3] == ctypes.sizeof(_lib.Outputs)
    assert got[4] == _lib.Batch.n_cand.offset
    assert got[5] == _lib.Batch.grid_h.offset
    assert got[6] == _lib.SUMMARY_DTYPE.fields["cov_cells"][1]


def test_no_cpu_fallback(built):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    fc = built
    from field_coverage_path_planning_b200 import _lib
    h = ctypes.c_void_p()
    assert _lib.load().fcpp_create(0, ctypes.byref(h)) == -3          # FCPP_ERR_NO_DEVICE
    with pytest.raises(fc.FcppError):
        fc.plan_batch([[(0, 0), (500, 0), (500, 200), (0, 200)]])
    with pytest.raises(fc.FcppError):
        fc.TwoLayerPathPlannerV37(fc.VehicleParams(), field_length=500, field_width=200).plan()
    with pytest.raises(fc.FcppError):
        fc.tour_lengths(np.zeros((3, 3)), np.array([[0, 1, 2]], dtype=np.int32))
    with pytest.raises(fc.FcppError):
        fc.plan_batch([[(0, 0), (500, 0), (500, 200), (0, 200)]], device="cpu")


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing under the package may import it."""
    pkg = os.path.join(ROOT, "field_coverage_path_planning_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f), encoding="utf-8").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, re.M), f
                assert "oracle/_build" not in txt and "libfcpo" not in txt, f


def test_constructor_contract(built):
    """mlp3:63-135 constructor behaviour and the aliases callers expect (SURVEY.md F2/F3)."""
    fc = built
    from oracle import ref_planner as rp
    with pytest.raises(ValueError):
        fc.TwoLayerPathPlannerV37(fc.VehicleParams())                      # mlp3:135
    p = fc.TwoLayerPlannerV35(vehicle=fc.VehicleParams(3.2, 8.0, 9.0, 15.0), field_length=500, field_width=200,
                              start_point=(10, 10), end_point=(600, 10))  # README.md:257-276 spelling
    assert p.start_point == (10, 10) and p.end_point is None               # out-of-bbox point ignored (mlp3:339-341)
    assert p.headland_width == 8.0 and p.field_shape == "rectangle" and p.main_work_pattern == "U型往复"
    assert p.field_polygon.area == 100000.0 and p.field_polygon.centroid.coords[0] == (250.0, 100.0)
    assert fc.TwoLayerPathPlannerV35 is fc.TwoLayerPathPlannerV36 is fc.TwoLayerPathPlannerV37
    assert p._select_best_start_corner((10, 10))[0] == 0
    for verts in ([(0, 0), (500, 0), (580, 200), (80, 200)], [(0, 0), (300, 0), (250, 150), (20, 120)],
                  [(0, 0), (100, 0), (100, 90), (0, 90)]):
        q = fc.TwoLayerPathPlannerV37(fc.VehicleParams(), field_vertices=verts)
        o = rp.setup_field(rp.VehicleParams(), field_vertices=verts)
        assert q.field_shape == o.field_shape and q.main_work_pattern == o.main_work_pattern
        np.testing.assert_allclose(q.corner_angles, o.corner_angles, rtol=0, atol=1e-12)
        assert (q.field_length, q.field_width) == (o.field_length, o.field_width)
    import multi_layer_planner_v3_optimized as alias                       # test/test_v37_complete.py:15
    assert alias.TwoLayerPathPlannerV35 is fc.TwoLayerPathPlannerV37 and alias.VehicleParams is fc.VehicleParams


def test_prepare_batch_host_setup(built):
    """A2 host set-up: flags, rotation tables, obstacle moments — against the oracle's scalars."""
    fc = built
    from field_coverage_path_planning_b200 import _lib, _geometry as G
    from oracle import geom, ref_planner as rp
    rect = [(0, 0), (500, 0), (500, 200), (0, 200)]
    sliver = [(0, 0), (400, 0), (700, 100), (300, 100)]                    # 18.4 deg corners: no reverse fill
    obst = [[(200, 80), (250, 80), (250, 120), (200, 120)]]
    cand = fc.make_candidates(2, headings=[0.0, 0.005, 0.3], radii=[5.0, 8.0], start_corners=[0, 1, 2, 3])
    assert len(cand["field_id"]) == 2 * 3 * 2 * 4
    assert list(cand["field_id"][:24]) == [0] * 24                         # field-major
    pb = fc.prepare_batch([rect, sliver], fc.VehicleParams(), cand, obstacles=[obst, []])
    a = pb.arrays
    assert a["field_flags"].tolist() == [15, 0b1010]
    np.testing.assert_array_equal(a["field_extent"], [[500, 200], [700, 100]])
    fl = a["cand_flags"]
    c = cand["start_corner"]
    assert ((fl & 3) == c).all()
    assert (((fl & _lib.FLAG_REVERSE_ORDER) != 0) == np.isin(c, (2, 3))).all()     # mlp3:650-653
    assert (((fl & _lib.FLAG_START_FROM_RIGHT) != 0) == np.isin(c, (1, 2))).all()  # mlp3:655-658
    assert (((fl & _lib.FLAG_ROTATED) != 0) == (np.abs(cand["heading"]) > 0.01)).all()  # mlp3:686
    assert ((fl & _lib.FLAG_GAP_GATE) != 0).all()
    np.testing.assert_array_equal(a["cand_rot"][:, 2], np.cos(cand["heading"]))
    np.testing.assert_array_equal(a["cand_rot"][:, 1], np.sin(-cand["heading"]))
    assert a["obs_poly_start"].tolist() == [0, 1, 1] and a["obs_vert_start"].tolist() == [0, 4]
    np.testing.assert_array_equal(a["obs_moments"][0], geom.round_buffer_moments(obst[0], 1.6))
    assert pb.max_obs_verts == 4 and pb.max_obs_polys == 1
    # gap gate: analytic lower bound vs numeric area for a degenerate (R, W)
    assert G.gap_gate(np.array([8.0]), 3.2)[0] == rp.gap_gate((0, 0), 0, 8.0, 3.2)
    assert bool(G.gap_gate(np.array([0.3]), 3.2)[0]) == rp.gap_gate((0, 0), 0, 0.3, 3.2)
    # D1 inset, product copy == oracle copy
    for verts in (rect, sliver, [(10, 5), (510, 40), (470, 260), (-20, 190)]):
        for dd in (1.6, 8.0, 30.0, 400.0):
            assert G.mitred_inset(verts, dd) == geom.inset_convex(verts, dd)
    with pytest.raises(ValueError):
        fc.prepare_batch([rect], fc.VehicleParams(), {"field_id": np.array([1], dtype=np.int32)})
    with pytest.raises(ValueError):
        fc.prepare_batch([rect], fc.VehicleParams(), {"field_id": np.array([0], dtype=np.int32),
                                                      "start_corner": np.array([4], dtype=np.int32)})
    # without a heading axis the heading is the field's (mlp3:244-263): trig per field, gathered per candidate
    tilted = [(10, 5), (510, 40), (470, 260), (-20, 190)]
    c2 = fc.make_candidates(3, radii=[6.0, 9.5], start_corners=[3, 0])
    p2 = fc.prepare_batch([rect, tilted, sliver], fc.VehicleParams(), c2)
    ang = np.array([0.0, np.arctan2(35.0, 500.0), 0.0])[c2["field_id"]]
    np.testing.assert_array_equal(p2.arrays["cand_rot"],
                                  np.stack([np.cos(-ang), np.sin(-ang), np.cos(ang), np.sin(ang)], axis=1))
    f2 = p2.arrays["cand_flags"]
    assert (((f2 & _lib.FLAG_ROTATED) != 0) == (c2["field_id"] == 1)).all()
    assert ((f2 & 3) == c2["start_corner"]).all() and f2.dtype == np.int32
    assert (((f2 & _lib.FLAG_REVERSE_ORDER) != 0) == (c2["start_corner"] == 3)).all()
    assert ((f2 & _lib.FLAG_START_FROM_RIGHT) == 0).all()
    # coverage de-duplication is requested when a candidate axis repeats coverage work (fcpp_batch.cover_dedupe)
    assert pb.dedupe == 2 and p2.dedupe == 1     # 2: a heading axis (few coverage representatives expected)
    assert not fc.prepare_batch([rect], fc.VehicleParams(), fc.make_candidates(1, radii=[5.0, 6.0])).dedupe
    assert not fc.prepare_batch([rect, tilted], fc.VehicleParams(), fc.make_candidates(2, start_corners=[1])).dedupe


def test_candidate_axes_host_setup(built):
    """Factored candidate sets (fcpp_batch: cand_field == NULL): the host computes per AXIS value exactly what the
    explicit form computes per candidate; enumeration order, ranges and shards agree with make_candidates."""
    fc = built
    from field_coverage_path_planning_b200 import _lib, batch as B, dist
    rect = [(0, 0), (500, 0), (500, 200), (0, 200)]
    tilted = [(10, 5), (510, 40), (470, 260), (-20, 190)]
    hs, rs, cs = [0.0, 0.005, 0.3], [5.0, 8.0], [3, 0, 1]
    ax = fc.candidate_axes(2, headings=hs, radii=rs, start_corners=cs)
    ex = fc.make_candidates(2, headings=hs, radii=rs, start_corners=cs)
    got = fc.expand_axes(ax)
    assert set(got) == set(ex) and all(np.array_equal(got[k], ex[k]) for k in ex)
    pick = np.array([35, 0, 17, 4])
    sub = fc.expand_axes(ax, pick)
    assert all(np.array_equal(sub[k], ex[k][pick]) for k in ex)
    pa = fc.prepare_batch([rect, tilted], fc.VehicleParams(), ax)
    pe = fc.prepare_batch([rect, tilted], fc.VehicleParams(), ex)
    assert pa.n_cand == pe.n_cand == 36 and pa.dedupe == pe.dedupe and pa.cand_first == 0
    assert "cand_field" not in pa.arrays and pa.h2d_bytes() < pe.h2d_bytes()
    g = np.arange(36)
    ih, ir, ic = g % 18 // 6, g // 3 % 2, g % 3
    np.testing.assert_array_equal(pa.arrays["ax_heading_rot"][ih], pe.arrays["cand_rot"])
    c = np.asarray(cs)[ic]
    want = (c | np.where(c >= 2, _lib.FLAG_REVERSE_ORDER, 0) | np.where(np.isin(c, (1, 2)), _lib.FLAG_START_FROM_RIGHT, 0)
            | pa.arrays["ax_heading_flags"][ih] | pa.arrays["ax_radius_flags"][ir])
    np.testing.assert_array_equal(want, pe.arrays["cand_flags"])          # the device decodes exactly this
    np.testing.assert_array_equal(pa.arrays["ax_radii"][ir], pe.arrays["cand_R"])
    # no heading axis: the field's own rotation per FIELD
    ax2 = fc.candidate_axes(2, radii=rs)
    p2 = fc.prepare_batch([rect, tilted], fc.VehicleParams(), ax2)
    e2 = fc.prepare_batch([rect, tilted], fc.VehicleParams(), fc.make_candidates(2, radii=rs))
    np.testing.assert_array_equal(p2.arrays["field_rot"][[0, 0, 1, 1]], e2.arrays["cand_rot"])
    assert p2.arrays["field_rot_flags"].tolist() == [0, _lib.FLAG_ROTATED]
    # contiguous shards: ranges of the product, nothing sliced
    parts = [dist.shard_candidates(ax, 3, r) for r in range(3)]
    assert [p[1] for p in parts] == [0, 12, 24] and [B.axes_count(p[0]) for p in parts] == [12, 12, 12]
    pr = fc.prepare_batch([rect, tilted], fc.VehicleParams(), parts[1][0])
    assert (pr.n_cand, pr.cand_first) == (12, 12)
    again, lo = dist.shard_candidates(parts[1][0], 2, 1)                   # a shard of a shard
    assert lo == 18 and again["range"] == (18, 24)
    with pytest.raises(ValueError):
        fc.prepare_batch([rect], fc.VehicleParams(), ax)                   # made for two fields
    with pytest.raises(ValueError):
        fc.prepare_batch([rect, tilted], fc.VehicleParams(), ax, start_points=np.zeros((36, 2)))
    with pytest.raises(ValueError):
        fc.prepare_batch([rect, tilted], fc.VehicleParams(), dict(ax, range=(30, 40)))
    with pytest.raises(ValueError):
        fc.candidate_axes(1, radii=[])
    # the bench workloads: the factored form enumerates the same candidates in the same order as the explicit arrays
    from benchmarks import workloads as wl
    for w in (wl.c2(1), wl.c2(2, 16), wl.c3(2, 8), wl.c5(1, 64), wl.c5(8, 64)):
        e = fc.expand_axes(w.axes)
        assert set(e) == set(w.cands) and all(np.array_equal(e[k], w.cands[k]) for k in e), w.name


def test_first_handle_call_in_a_fresh_process_returns():
    """_lib.handle() as the FIRST library call of a process (bench.py does that): the library load inside the
    Handle constructor must not dead-lock on the module lock.  Without a GPU it fails loudly instead."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from field_coverage_path_planning_b200 import _lib\n"
            "try:\n    _lib.handle(0); _lib.handle(0, 1); print('HANDLES')\n"
            "except _lib.FcppError as e:\n    print('RAISED', e)\n" % root)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert "RAISED" in out.stdout or "HANDLES" in out.stdout, out.stdout + out.stderr
