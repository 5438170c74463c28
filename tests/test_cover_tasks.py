"""Coverage task list of de-duplicated batches (csrc/fcpp_cover.cu: cover_rep_kernel / cover_list_kernel): every
(representative, part) — A10 corner windows or A11 headland band — is one task, the tasks are dispatched in
non-increasing estimated cost, and the two parts of one candidate may run in two CTAs at once.  Checked here:

  * the summaries are byte-identical to those of the same batch without de-duplication (cover mode bit 1: one
    CTA per candidate running both parts), with one CTA per task (mode bit 6) and the persistent grid (bit 7),
    across start-corner subsets, shuffled orders, duplicates, dead candidates, per-candidate band fall-backs, a band
    grid too large for the tile and a slanted heading search;
  * read back from a trace build (-DFCPP_COVER_TRACE), the list holds every required task exactly once, in
    non-increasing cost bucket, and A10 and A11 of a group are separate tasks.
"""
import json
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RECT = [(0.0, 0.0), (500.0, 0.0), (500.0, 200.0), (0.0, 200.0)]
SLANT = [(0.0, 0.0), (300.0, 0.0), (360.0, 120.0), (60.0, 120.0)]


@pytest.fixture(scope="module")
def fc():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import field_coverage_path_planning_b200 as fc
    return fc


def _same(fc, fields, cand, **kw):
    """the de-duplicated summaries (default launch form, one CTA per task, persistent grid) == without
    de-duplication"""
    from field_coverage_path_planning_b200 import _lib
    h = _lib.handle(0)
    veh = fc.VehicleParams()
    got = fc.plan_batch(fields, veh, cand, **kw).summary
    try:
        for mode in (2, 64, 128):
            h.check(h.lib.fcpp_set_cover_mode(h.h, mode))
            other = fc.plan_batch(fields, veh, cand, **kw).summary
            assert got.tobytes() == other.tobytes(), mode
    finally:
        h.check(h.lib.fcpp_set_cover_mode(h.h, 0))
    return got


def _shuffled(cand, seed, n_dup=9, n_dead=4):
    """shuffled order, duplicates and dead candidates (a radius whose R-inset is empty)"""
    rng = np.random.default_rng(seed)
    n = len(cand["field_id"])
    idx = np.concatenate([rng.permutation(n), rng.integers(0, n, n_dup)])
    out = {k: v[idx].copy() for k, v in cand.items()}
    if "R" in out:
        out["R"][rng.integers(0, len(idx), n_dead)] = 150.0
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("corners", [[0, 1, 2, 3], [2], [1, 3]])
def test_tasks_equal_per_candidate(fc, corners):
    cand = fc.make_candidates(1, radii=np.linspace(5.0, 12.0, 48), start_corners=corners)
    s = _same(fc, [RECT], cand)
    assert (s["status"] == 0).all() and (s["cov_cells"] > 0).all() and (s["corner_after"] > 0).all()
    s = _same(fc, [RECT], _shuffled(cand, len(corners)))
    assert (s["status"] != 0).any()


@pytest.mark.gpu
def test_tasks_fallbacks_and_slanted_straights(fc):
    """narrow fields whose corner zones overlap (per-candidate band fall-back inside the group's task) and a field with
    slanted straights (one band task per start corner), in a shuffled order"""
    fields = [[(0, 0), (45, 0), (45, 300), (0, 300)], [(0, 0), (24, 0), (24, 60), (0, 60)], SLANT, RECT]
    cand = fc.make_candidates(len(fields), radii=[5.0, 6.4, 8.0, 11.0], start_corners=[0, 1, 2, 3])
    _same(fc, fields, _shuffled(cand, 7))


@pytest.mark.gpu
def test_tasks_band_grid_too_large(fc):
    """a band row wider than the shared-memory tile (slanted field at 2 mm): the band tasks report the band detail bit,
    the corner-window tasks of the same candidates run and report nothing, exactly as without de-duplication"""
    cand = fc.make_candidates(1, radii=[5.0, 6.0], start_corners=[0, 1, 2, 3])
    s = _same(fc, [[(0.0, 0.0), (600.0, 0.0), (660.0, 200.0), (60.0, 200.0)]], cand, grid_h=0.002)
    assert (s["status"] == 16 | 64).all()
    assert (s["corner_after"] > 0).all()


@pytest.mark.gpu
def test_tasks_slanted_heading_search(fc):
    """a heading search over tilted fields (cover_dedupe = 2, the persistent grid by default): one A10 and one A11 task
    per field"""
    from benchmarks import workloads as wl
    fields = wl.c3_fields(6, seed=5)
    cand = fc.make_candidates(6, headings=np.deg2rad(np.arange(0.0, 180.0, 4.5)))
    _same(fc, fields, cand)
    _same(fc, fields, _shuffled(cand, 3, n_dead=0))


_LIST_CHECK = textwrap.dedent("""
    import ctypes as C, json, sys
    import numpy as np
    import field_coverage_path_planning_b200 as fc
    from field_coverage_path_planning_b200 import _lib
    h = _lib.handle(0)
    take = h.lib.fcpp_cover_trace_take
    take.restype, take.argtypes = C.c_int, [C.c_void_p, C.c_int]
    buf = np.zeros((1 << 16, 4), dtype=np.uint64)
    RECT = [(0.0, 0.0), (500.0, 0.0), (500.0, 200.0), (0.0, 200.0)]
    SLANT = [(0.0, 0.0), (300.0, 0.0), (360.0, 120.0), (60.0, 120.0)]
    cand = fc.make_candidates(2, radii=np.linspace(5.0, 12.0, 24), start_corners=[0, 1, 2, 3])
    perm = np.random.default_rng(11).permutation(len(cand["R"]))
    cand = {k: v[perm] for k, v in cand.items()}
    out = {}
    for mode in (64, 128):
        h.check(h.lib.fcpp_set_cover_mode(h.h, mode))
        take(buf.ctypes.data, len(buf))
        s = fc.plan_batch([RECT, SLANT], fc.VehicleParams(), cand).summary
        assert (s["status"] == 0).all()
        n = take(buf.ctypes.data, len(buf))
        t = buf[:n]
        out[mode] = {"pos": (t[:, 2] >> 32).astype(int).tolist(), "bucket": ((t[:, 2] >> 16) & 0xffff).astype(int).tolist(),
                     "cand": (t[:, 3] >> 2).astype(int).tolist(), "part": (t[:, 3] & 3).astype(int).tolist()}
    h.check(h.lib.fcpp_set_cover_mode(h.h, 0))
    out["field"] = cand["field_id"].tolist()
    out["R"] = cand["R"].tolist()
    json.dump(out, sys.stdout)
""")


@pytest.mark.gpu
def test_task_list_order_and_completeness(fc, tmp_path):
    """builds the trace variant of the library into a temporary directory and reads the task list back through it"""
    csrc = os.path.join(ROOT, "field_coverage_path_planning_b200", "csrc")
    lib = str(tmp_path / "libfcpp_trace.so")
    subprocess.check_call(["make", "-s", "-C", csrc, "-j8", f"BUILD={tmp_path / 'build'}", f"OUT={lib}",
                           "DEFS=-DFCPP_COVER_TRACE"], stdout=subprocess.DEVNULL)
    env = dict(os.environ, FCPP_LIB=lib, PYTHONPATH=ROOT)
    res = json.loads(subprocess.check_output([sys.executable, "-c", _LIST_CHECK], env=env, cwd=ROOT))
    field, R = np.asarray(res["field"]), np.asarray(res["R"])
    for mode in ("64", "128"):
        r = res[mode]
        pos, bucket, cnd, part = (np.asarray(r[k]) for k in ("pos", "bucket", "cand", "part"))
        assert (pos > 0).all(), "every task comes from the list"
        order = np.argsort(pos)
        assert np.array_equal(pos[order], np.arange(1, len(pos) + 1)), "each list position runs exactly once"
        assert (np.diff(bucket[order]) <= 0).all(), "non-increasing estimated cost"
        tasks = set(zip(cnd.tolist(), part.tolist()))
        assert len(tasks) == len(pos), "each (candidate, part) exactly once"
        # A10: one task per (field, R), run by its lowest-index candidate
        want10 = {min(np.flatnonzero((field == f) & (R == x))) for f, x in set(zip(field.tolist(), R.tolist()))}
        assert {c for c, p in tasks if p == 1} == want10
        # A11: the rectangle's bands are grouped per (field, R) (the same representative as A10, in a task of its
        # own); the slanted field keeps one band task per start corner
        want11 = {c for c in want10 if field[c] == 0} | set(np.flatnonzero(field == 1).tolist())
        assert {c for c, p in tasks if p == 2} == want11
